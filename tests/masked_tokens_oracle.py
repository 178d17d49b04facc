"""CPU reference of ViTModel with masked patch tokens (test helper, not a test module): transformers'
``ViTModel(config, use_mask_token=True)(x, bool_masked_pos=mask)`` with eager attention, stated with the oracle's own
functions (``oracle/vit2spn_oracle.py``), so the oracle's ``rounding`` model of the bf16 / fp16 modes applies as well.
Pinned to transformers by ``tests/test_masked_tokens_cpu.py``."""
import torch

import vit_outputs_oracle as vo
from oracle import vit2spn_oracle as orc


def patch_embed(p, x, mask=None, token=None):
    """``orc.patch_embed`` where each masked patch row is ``token + pos[1+p]`` (HF:ViTEmbeddings.forward, as a select:
    for finite values ``e (1 - m) + t m`` is ``e`` or ``t`` exactly).  mask [B,196] (nonzero = masked), token [192]."""
    h = orc.patch_embed(p, x)
    if mask is None:
        return h
    m = (mask != 0).unsqueeze(-1)
    tok = token.reshape(1, 1, orc.HIDDEN) + p["embeddings.position_embeddings"][:, 1:]
    return torch.cat([h[:, :1], torch.where(m, tok, h[:, 1:])], dim=1)


def backbone_outputs(p, x, mask=None, token=None):
    """(hidden_states, attentions) as ``vit_outputs_oracle.backbone_outputs``, with the patch mask applied."""
    hs, probs = [patch_embed(p, x, mask, token)], []
    for l in range(orc.LAYERS):
        probs.append(vo.attention_probs(p, l, hs[-1]))
        hs.append(orc.vit_layer(p, l, hs[-1]))
    return tuple(hs), tuple(probs)


def hidden_and_grads(p, x, mask, token, up, names=()):
    """hidden_states[-1] and the gradients of ``(hidden_states[-1] * up).sum()`` w.r.t. the pixels, the mask token and
    the parameters ``names`` of ``p``: (h, dx, dtoken [192], {name: grad})."""
    with torch.enable_grad():
        q = {k: (v.detach().clone().requires_grad_(k in names)) for k, v in p.items()}
        xx = x.detach().clone().requires_grad_(True)
        t = token.detach().clone().reshape(orc.HIDDEN).requires_grad_(True)
        h = patch_embed(q, xx, mask, t)
        for l in range(orc.LAYERS):
            h = orc.vit_layer(q, l, h)
        (h * up).sum().backward()
    return h.detach(), xx.grad, t.grad, {k: q[k].grad for k in names}
