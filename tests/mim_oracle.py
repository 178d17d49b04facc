"""CPU reference of the SimMIM head of transformers' ``ViTForMaskedImageModeling`` (test helper, not a test module): the
final LayerNorm, the 1x1-conv decoder with PixelShuffle(16) and the masked L1 loss, on hidden_states[12].  With `lp`
(torch.bfloat16 / torch.float16) the normalised patch rows and the decoder weight are rounded to that format as the
16-bit modes' tensor-core GEMMs read them (straight through: their gradients stay fp32, as the library computes them).
``model_loss`` adds the backbone (``masked_tokens_oracle``), so the oracle's ``rounding`` model applies to it.  Pinned to
transformers by ``tests/test_mim_cpu.py``."""
import torch

import masked_tokens_oracle as mo
from oracle import vit2spn_oracle as orc


def pixel_mask(mask):
    """[B,196] patch mask -> [B,1,224,224] pixel mask (as ViTForMaskedImageModeling builds it)."""
    return mask.reshape(-1, 14, 14).repeat_interleave(16, 1).repeat_interleave(16, 2).unsqueeze(1)


def _round(t, lp):
    return t if lp is None else t + (t.to(lp).to(t.dtype) - t).detach()


def head(h12, ln_w, ln_b, dec_w, dec_b, x, mask, lp=None):
    """(reconstruction [B,3,224,224], loss or None) from hidden_states[12] [B,197,192]."""
    B = h12.shape[0]
    last = torch.nn.functional.layer_norm(h12, (192,), ln_w, ln_b, 1e-12)
    seq = _round(last[:, 1:], lp)
    rows = seq @ _round(dec_w.reshape(768, 192), lp).t() + dec_b                        # [B,196,768]
    rec = torch.nn.functional.pixel_shuffle(rows.permute(0, 2, 1).reshape(B, 768, 14, 14), 16)
    if mask is None:
        return rec, None
    pm = pixel_mask(mask).to(x.dtype)
    l1 = torch.nn.functional.l1_loss(x, rec, reduction="none")
    return rec, (l1 * pm).sum() / (pm.sum() + 1e-5) / 3


def model_loss(p, token, dec_w, dec_b, x, mask, lp=None):
    """The whole model: (loss, reconstruction, grads) where grads maps every name of `p` (HF ViTModel keys),
    "mask_token", "decoder.0.weight", "decoder.0.bias" and "pixels" to d loss / d it.  Call inside ``orc.rounding`` for
    the 16-bit modes' rounding model of the backbone."""
    with torch.enable_grad():
        q = {k: v.detach().clone().requires_grad_(True) for k, v in p.items()}
        t = token.detach().clone().reshape(192).requires_grad_(True)
        w = dec_w.detach().clone().requires_grad_(True)
        b = dec_b.detach().clone().requires_grad_(True)
        xx = x.detach().clone().requires_grad_(True)
        h = mo.patch_embed(q, xx, mask, t)
        for l in range(orc.LAYERS):
            h = orc.vit_layer(q, l, h)
        rec, loss = head(h, q["layernorm.weight"], q["layernorm.bias"], w, b, xx, mask, lp)
        loss.backward()
    grads = {k: v.grad for k, v in q.items() if v.grad is not None}
    grads.update({"mask_token": t.grad, "decoder.0.weight": w.grad, "decoder.0.bias": b.grad, "pixels": xx.grad})
    return loss.detach(), rec.detach(), grads
