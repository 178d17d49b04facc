"""CPU reference of the classification head of transformers' ``ViTForImageClassification`` (test helper, not a test
module): the final LayerNorm of the CLS token, the linear classifier and transformers' ``ForSequenceClassificationLoss``
(MSE, cross-entropy with ignore_index -100, BCE with logits), on hidden_states[12].  With `lp` (torch.bfloat16 /
torch.float16) the normalised CLS rows and the classifier weight are rounded to that format as the 16-bit modes'
tensor-core GEMMs read them, and the logits' gradient is rounded to it on the way back (the GEMM operand G of the
library's backward); everything else stays in the input's precision.  ``model_loss`` adds the oracle's backbone, so its
``rounding`` model applies there.  Pinned to transformers by ``tests/test_cls_cpu.py``."""
import torch

import masked_tokens_oracle as mo
from oracle import vit2spn_oracle as orc


def _round(t, lp):
    return t if lp is None else t + (t.to(lp).to(t.dtype) - t).detach()


class _RoundGrad(torch.autograd.Function):
    @staticmethod
    def forward(ctx, t, lp):
        ctx.lp = lp
        return t.view_as(t)

    @staticmethod
    def backward(ctx, g):
        return g.to(ctx.lp).to(g.dtype), None


def loss_fn(labels, logits, problem_type):
    """transformers' ForSequenceClassificationLoss for a fixed problem_type."""
    n = logits.shape[-1]
    if problem_type == "regression":
        y = labels.to(logits.dtype)
        return torch.nn.functional.mse_loss(logits.squeeze(), y.squeeze()) if n == 1 else \
            torch.nn.functional.mse_loss(logits, y)
    if problem_type == "single_label_classification":
        return torch.nn.functional.cross_entropy(logits.view(-1, n), labels.view(-1).long(), ignore_index=-100)
    return torch.nn.functional.binary_cross_entropy_with_logits(logits, labels.to(logits.dtype))


def head(h12, ln_w, ln_b, w, b, labels=None, problem_type=None, lp=None):
    """(logits [B, N], loss or None) from hidden_states[12] [B,197,192]."""
    x = _round(torch.nn.functional.layer_norm(h12[:, 0], (192,), ln_w, ln_b, 1e-12), lp)
    z = x @ _round(w, lp).t() + b
    if lp is not None:
        z = _RoundGrad.apply(z, lp)
    return z, (loss_fn(labels, z, problem_type) if labels is not None else None)


def model_loss(p, w, b, x, labels=None, problem_type=None, lp=None, dlogits=None):
    """The whole model: (loss, logits, grads) for the objective loss + sum(logits * dlogits) (either term may be
    absent).  grads maps every name of `p` (HF ViTModel keys), "classifier.weight", "classifier.bias" and "pixels" to
    its gradient.  Call inside ``orc.rounding`` for the 16-bit modes' rounding model of the backbone."""
    with torch.enable_grad():
        q = {k: v.detach().clone().requires_grad_(True) for k, v in p.items()}
        ww = w.detach().clone().requires_grad_(True)
        bb = b.detach().clone().requires_grad_(True)
        xx = x.detach().clone().requires_grad_(True)
        h = mo.patch_embed(q, xx)
        for l in range(orc.LAYERS):
            h = orc.vit_layer(q, l, h)
        logits, loss = head(h, q["layernorm.weight"], q["layernorm.bias"], ww, bb, labels, problem_type, lp)
        obj = 0
        if loss is not None:
            obj = obj + loss
        if dlogits is not None:
            obj = obj + (logits * dlogits.to(logits.dtype)).sum()
        obj.backward()
    grads = {k: v.grad for k, v in q.items() if v.grad is not None}
    grads.update({"classifier.weight": ww.grad, "classifier.bias": bb.grad, "pixels": xx.grad})
    return (loss.detach() if loss is not None else None), logits.detach(), grads
