"""CPU reference of ``ViTModel(x, interpolate_pos_encoding=True)`` at any input of at most 197 tokens (test helper, not a
test module): transformers' ``ViTEmbeddings`` rule (the 14 x 14 position table resized bicubically, align_corners
False, to the patch grid; used unchanged for square 196-patch inputs) stated with the oracle's own functions
(``oracle/vit2spn_oracle.py``), so its ``rounding`` model of the bf16 / fp16 modes applies as well.  Pinned to stock
transformers by ``tests/test_interpolate_cpu.py``."""
import torch
import torch.nn.functional as F

import vit_outputs_oracle as vo
from oracle import vit2spn_oracle as orc


def position_table(pos, H, W):
    """[1,N,192] position table of an H x W input from the stored [1,197,192] one (HF:ViTEmbeddings.interpolate_pos_encoding)."""
    gh, gw = H // orc.PATCH, W // orc.PATCH
    if gh * gw == orc.GRID * orc.GRID and H == W:
        return pos
    grid = pos[:, 1:].reshape(1, orc.GRID, orc.GRID, orc.HIDDEN).permute(0, 3, 1, 2)
    grid = F.interpolate(grid, size=(gh, gw), mode="bicubic", align_corners=False)
    return torch.cat([pos[:, :1], grid.permute(0, 2, 3, 1).reshape(1, gh * gw, orc.HIDDEN)], dim=1)


def patch_embed(p, x, mask=None, token=None):
    """``orc.patch_embed`` at an H x W input: im2col over the gh x gw grid + GEMM, CLS, the interpolated table; a masked
    patch row (mask [B, gh*gw], nonzero = masked) takes ``token`` before the table is added."""
    B, _, H, W = x.shape
    gh, gw = H // orc.PATCH, W // orc.PATCH
    cols = x.reshape(B, 3, gh, orc.PATCH, gw, orc.PATCH).permute(0, 2, 4, 1, 3, 5).reshape(B, gh * gw, -1)
    w = orc._rnd(p["embeddings.patch_embeddings.projection.weight"].reshape(orc.HIDDEN, -1), "w")
    tok = orc._rnd(cols, "patches") @ w.t() + p["embeddings.patch_embeddings.projection.bias"]
    if mask is not None:
        tok = torch.where((mask != 0).unsqueeze(-1), token.reshape(1, 1, orc.HIDDEN).to(tok.dtype), tok)
    cls = p["embeddings.cls_token"].expand(B, -1, -1)
    return torch.cat([cls, tok], dim=1) + position_table(p["embeddings.position_embeddings"], H, W)


def backbone_outputs(p, x, mask=None, token=None):
    """(hidden_states, attentions): 13 x [B,N,192] (before the final LayerNorm) and 12 x [B,3,N,N]."""
    hs, probs = [patch_embed(p, x, mask, token)], []
    for l in range(orc.LAYERS):
        probs.append(vo.attention_probs(p, l, hs[-1]))
        hs.append(orc.vit_layer(p, l, hs[-1]))
    return tuple(hs), tuple(probs)


def grads(p, x, up, mask=None, token=None, retain=(), names=None):
    """Gradients of ``(hidden_states[-1] * up).sum()``: (hidden_states, attentions, dx, dtoken or None,
    {name: grad} over ``names`` (default: every tensor of ``p``), {l: d loss / d attentions[l]} for l in ``retain``).
    The attentions of ``retain`` are the ones the blocks use, so their gradients are transformers' retain_grad()."""
    names = list(p) if names is None else list(names)
    with torch.enable_grad():
        q = {k: v.detach().clone().requires_grad_(k in names) for k, v in p.items()}
        xx = x.detach().clone().requires_grad_(True)
        t = token.detach().clone().reshape(orc.HIDDEN).requires_grad_(True) if token is not None else None
        hs, probs = [patch_embed(q, xx, mask, t)], []
        for l in range(orc.LAYERS):
            h = hs[-1]
            pre = f"encoder.layer.{l}."
            xn = orc._rnd(orc.layer_norm(h, q[pre + "layernorm_before.weight"], q[pre + "layernorm_before.bias"]), "xn")
            a = pre + "attention.attention."
            qkv = [orc._rnd(xn @ orc._rnd(q[a + n + ".weight"], "w").t() + q[a + n + ".bias"], "qkv")
                   for n in ("query", "key", "value")]
            B, N, _ = qkv[0].shape
            qh, kh, vh = (z.view(B, N, orc.HEADS, orc.HEAD_DIM).transpose(1, 2) for z in qkv)
            pr = torch.softmax((qh @ kh.transpose(-1, -2)) * (orc.HEAD_DIM ** -0.5), dim=-1)
            if l in retain:
                pr.retain_grad()
            probs.append(pr)
            ctx = orc._rnd((pr @ vh).transpose(1, 2).reshape(B, N, orc.HIDDEN), "ctx")
            h = h + ctx @ orc._rnd(q[pre + "attention.output.dense.weight"], "w").t() + q[pre + "attention.output.dense.bias"]
            xn = orc._rnd(orc.layer_norm(h, q[pre + "layernorm_after.weight"], q[pre + "layernorm_after.bias"]), "xn")
            u = xn @ orc._rnd(q[pre + "intermediate.dense.weight"], "w").t() + q[pre + "intermediate.dense.bias"]
            h = h + orc._rnd(orc.gelu_erf(u), "h") @ orc._rnd(q[pre + "output.dense.weight"], "w").t() + q[pre + "output.dense.bias"]
            hs.append(h)
        (hs[-1] * up).sum().backward()
    return (tuple(h.detach() for h in hs), tuple(a.detach() for a in probs), xx.grad, t.grad if t is not None else None,
            {k: q[k].grad for k in names if q[k].grad is not None}, {l: probs[l].grad for l in retain})
