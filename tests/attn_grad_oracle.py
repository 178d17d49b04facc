"""CPU reference of the gradients w.r.t. ViTModel's attention probabilities (test helper, not a test module).

The oracle's block (``orc.vit_layer``) is restated with the probabilities as an explicit tensor ``A``, so that autograd
gives ``d loss / d A_l``: the total derivative that ``retain_grad()`` on transformers' ``attentions[l]`` reports.  Under
``orc.rounding(...)`` the block rounds where the oracle does (with the "p" stage, ``A V`` takes the value of the oracle's
rounded numerators over the fp32 row sum, and the gradient of ``A V``).  Pinned to
transformers by ``tests/test_attn_grad_cpu.py``."""
import torch

from oracle import vit2spn_oracle as orc


def block(p, l, h):
    """``orc.vit_layer(p, l, h)`` with the attention probabilities explicit: (block output, A [B,3,197,197])."""
    pre = f"encoder.layer.{l}."
    x = orc._rnd(orc.layer_norm(h, p[pre + "layernorm_before.weight"], p[pre + "layernorm_before.bias"]), "xn")
    a = pre + "attention.attention."
    q, k, v = (orc._rnd(x @ orc._rnd(p[a + n + ".weight"], "w").t() + p[a + n + ".bias"], "qkv")
               for n in ("query", "key", "value"))
    B, N, _ = q.shape
    q, k, v = (t.view(B, N, orc.HEADS, orc.HEAD_DIM).transpose(1, 2) for t in (q, k, v))
    s = (q @ k.transpose(-1, -2)) * (orc.HEAD_DIM ** -0.5)
    if "p" in orc._ROUND["stages"]:
        e = torch.exp(s - s.max(dim=-1, keepdim=True).values)
        r = e.sum(dim=-1, keepdim=True)
        A = e / r
        av = A @ v
        o = av + ((orc._rnd(e, "p") @ v) / r - av).detach()      # the oracle's value, the gradient of A V
    else:
        A = torch.softmax(s, dim=-1)
        o = A @ v
    ctx = orc._rnd(o.transpose(1, 2).reshape(B, N, orc.HIDDEN), "ctx")
    h = h + ctx @ orc._rnd(p[pre + "attention.output.dense.weight"], "w").t() + p[pre + "attention.output.dense.bias"]
    x = orc._rnd(orc.layer_norm(h, p[pre + "layernorm_after.weight"], p[pre + "layernorm_after.bias"]), "xn")
    u = x @ orc._rnd(p[pre + "intermediate.dense.weight"], "w").t() + p[pre + "intermediate.dense.bias"]
    h = h + orc._rnd(orc.gelu_erf(u), "h") @ orc._rnd(p[pre + "output.dense.weight"], "w").t() + p[pre + "output.dense.bias"]
    return h, A


def attention_grads(p, x, loss_fn):
    """(hidden_states, attentions, d loss / d attentions) for ``loss_fn(hidden_states)``; a block the loss does not reach
    gets None, as transformers' retained ``.grad`` does."""
    with torch.enable_grad():
        hs, probs = [orc.patch_embed(p, x.detach().requires_grad_(True))], []    # so that every A_l requires grad
        for l in range(orc.LAYERS):
            h, A = block(p, l, hs[-1])
            hs.append(h)
            probs.append(A)
        grads = torch.autograd.grad(loss_fn(tuple(hs)), probs, allow_unused=True)
    return tuple(t.detach() for t in hs), tuple(a.detach() for a in probs), grads


def relevance_loop(attentions, grads, token="cls"):
    """Chefer et al.'s relevance, one image at a time, as the equations are published: R = I; R += Ebar_h[(grad A * A)^+] R
    per block; the CLS row (or the mean over rows) without the CLS column, as [B,14,14]."""
    out = []
    for b in range(attentions[0].shape[0]):
        R = torch.eye(attentions[0].shape[-1], dtype=torch.float64)
        for a, g in zip(attentions, grads):
            if g is None:
                continue
            cam = (g[b].double() * a[b].double()).clamp(min=0).mean(dim=0)
            R = R + cam @ R
        row = R[0] if token == "cls" else R.mean(dim=0)
        out.append(row[1:].reshape(14, 14))
    return torch.stack(out)
