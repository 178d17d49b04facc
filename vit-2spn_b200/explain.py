"""Attention-based explanations of a ViTModel prediction, from the attentions and their retained gradients.

``attention_relevance`` is the relevance rule of Chefer, Gur and Wolf for self-attention encoders ("Generic
Attention-model Explainability for Interpreting Bi-Modal and Encoder-Decoder Transformers", ICCV 2021, eqs. 5-6; the
gradient-weighted attention of "Transformer Interpretability Beyond Attention Visualization", CVPR 2021)::

    out = model(x, output_attentions=True)
    for a in out.attentions:
        a.retain_grad()
    score.backward()                      # score: the logit to explain, summed over the batch
    maps = attention_relevance(out.attentions, [a.grad for a in out.attentions])    # [B,14,14]
"""
import torch


def attention_relevance(attentions, attention_grads, token="cls"):
    """Relevance of the 14 x 14 patches: ``R = I``; per block ``R += mean_h((dA * A).clamp(min=0)) @ R``; then the
    row of the CLS token (``token="cls"``) or the mean of all rows (``"mean"``, for the mean-pooled ViTBackbone /
    FineTunedModel), without the CLS column.  ``attentions`` / ``attention_grads``: the 12 [B,3,197,197] tensors of one
    backward; a None gradient (a block above the layers the score depends on) contributes nothing."""
    if token not in ("cls", "mean"):
        raise ValueError(f"token must be 'cls' or 'mean', got {token!r}")
    if len(attentions) != len(attention_grads):
        raise ValueError(f"{len(attentions)} attentions but {len(attention_grads)} gradients")
    a0 = attentions[0]
    B, n = a0.shape[0], a0.shape[-1]
    R = torch.eye(n, dtype=a0.dtype, device=a0.device).expand(B, n, n).clone()
    for a, g in zip(attentions, attention_grads):
        if g is not None:
            R = R + (g * a).clamp(min=0).mean(dim=1) @ R
    rel = R[:, 0] if token == "cls" else R.mean(dim=1)
    side = int(round((n - 1) ** 0.5))
    return rel[:, 1:].reshape(B, side, side)
