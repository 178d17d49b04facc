"""GPU: ``ViTModel(interpolate_pos_encoding=True)`` at inputs other than 224 x 224 (v2s_set_image_size).

* the attention operators (``v2s_test_attention``: forward, backward, probabilities and their gradient; tensor-core and
  SIMT kernels, bf16 and fp16) at N tokens against a torch fp32 reference on the same 16-bit inputs, with the tolerances
  of ``tests/test_gpu_attention.py``; 128 / 129 sit on the query-tile boundary;
* ``ViTModel`` end to end against ``interp_oracle`` (fp32 check mode at 1e-5; bf16 / fp16 at the 224 x 224 gates);
* 224 x 224 with the flag is bit-identical to a run without it, with the same launches; 128 x 128 launches one more
  kernel in the forward and one more in a full backward with weight gradients; the deterministic flag; a combined case.
"""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import interp_oracle as io  # noqa: E402  (helper module, not a test)

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
TOKENS = [2, 17, 65, 101, 128, 129, 145, 170, 197]
SIZES = [(64, 64), (128, 128), (96, 160), (112, 448)]


def _get_lib():
    import vit2spn  # noqa: F401
    from vit2spn import _lib
    _lib.init_device(0)
    return _lib


def _set_tokens(_lib, n):
    """an image size with n tokens: one row of n - 1 patches"""
    _lib.check(_lib.lib.v2s_set_image_size(16, 16 * (n - 1)), "set_image_size")


def _ref(qkv, dctx, n):
    B = qkv.shape[0]
    x = qkv.float().requires_grad_(True)
    q, k, v = [t.view(B, n, 3, 64).transpose(1, 2) for t in x.split(192, dim=-1)]
    s = (q @ k.transpose(-1, -2)) * 0.125
    lse = torch.logsumexp(s, dim=-1)
    p = torch.softmax(s, dim=-1)
    o = (p @ v).transpose(1, 2).reshape(B, n, 192)
    o.backward(dctx.float())
    dvt = dctx.float().view(B, n, 3, 64).transpose(1, 2) @ v.detach().transpose(-1, -2)
    return o.detach(), lse.detach(), x.grad, p.detach(), dvt


@pytest.mark.parametrize("n", TOKENS)
@pytest.mark.parametrize("variant", [0, 1, 2, 3])    # bit 0: SIMT kernels; bit 1: fp16
def test_attention_operators_at_n_tokens(n, variant):
    _lib = _get_lib()
    batch = 3
    g = torch.Generator(device=DEV).manual_seed(n * 10 + variant)
    lp = torch.float16 if variant & 2 else torch.bfloat16
    qkv = torch.randn(batch, n, 576, device=DEV, generator=g).to(lp)
    dctx = torch.randn(batch, n, 192, device=DEV, generator=g).to(lp)
    o_ref, lse_ref, dqkv_ref, p_ref, dp_ref = _ref(qkv, dctx, n)
    _set_tokens(_lib, n)
    try:
        ctx = torch.full((batch, n, 192), float("nan"), device=DEV, dtype=lp)
        lse = torch.full((batch, 3, n), float("nan"), device=DEV)
        _lib.check(_lib.lib.v2s_test_attention(0, _lib.ptr(qkv), _lib.ptr(ctx), _lib.ptr(lse), None, None, batch, variant,
                                               _lib.stream_ptr()), "attention fwd")
        torch.cuda.synchronize()
        assert _lib.lib.v2s_debug_flag() == 0
        assert torch.isfinite(ctx.float()).all()
        assert (ctx.float() - o_ref).abs().max().item() <= 0.02 * max(1.0, o_ref.abs().max().item())
        assert (lse - lse_ref).abs().max().item() <= 2e-3 * max(1.0, lse_ref.abs().max().item())
        dqkv = torch.full((batch, n, 576), float("nan"), device=DEV, dtype=lp)
        _lib.check(_lib.lib.v2s_test_attention(1, _lib.ptr(qkv), _lib.ptr(ctx), _lib.ptr(lse), _lib.ptr(dctx),
                                               _lib.ptr(dqkv), batch, variant, _lib.stream_ptr()), "attention bwd")
        torch.cuda.synchronize()
        assert _lib.lib.v2s_debug_flag() == 0
        assert torch.isfinite(dqkv.float()).all()
        for i, name in enumerate(("dq", "dk", "dv")):
            got, ref = dqkv[..., i * 192:(i + 1) * 192].float(), dqkv_ref[..., i * 192:(i + 1) * 192]
            rel = (got - ref).norm().item() / max(ref.norm().item(), 1e-12)
            assert rel <= 2e-2, (name, rel)
            assert (got - ref).abs().max().item() <= 0.03 * max(1.0, ref.abs().max().item()), name
        for which, ref in ((2, p_ref), (3, dp_ref)):
            out = torch.full((batch, 3, n, n), float("nan"), device=DEV)
            _lib.check(_lib.lib.v2s_test_attention(which, _lib.ptr(qkv), _lib.ptr(out), _lib.ptr(lse), _lib.ptr(dctx), None,
                                                   batch, variant, _lib.stream_ptr()), f"attention which {which}")
            torch.cuda.synchronize()
            assert _lib.lib.v2s_debug_flag() == 0
            assert torch.isfinite(out).all(), which
            rel = (out - ref).norm().item() / max(ref.norm().item(), 1e-12)
            assert rel <= 2e-2, (which, rel)
    finally:
        _lib.check(_lib.lib.v2s_set_image_size(224, 224), "set_image_size")


def _state(seed=11):
    from oracle import vit2spn_oracle as orc
    return orc.sub_state(orc.init_state(seed, 0.01), "online_network_1")


def _token(seed=12):
    return 0.02 * torch.randn(192, generator=torch.Generator().manual_seed(seed))


def _model(p, mode, token=None, frozen=False):
    import vit2spn
    m = vit2spn.ViTModel(use_mask_token=token is not None)
    sd = dict(p)
    if token is not None:
        sd["embeddings.mask_token"] = token.view(1, 1, 192)
    m.load_state_dict(sd, strict=True)
    m.to(DEV)
    m.compute_mode = mode
    if frozen:
        m.requires_grad_(False)
    return m


def _rel(a, b):
    return ((a.double().cpu() - b.double().cpu()).norm() / b.double().cpu().norm().clamp_min(1e-30)).item()


_ORACLE = {}


def _oracle(p, x, up, key, **kw):
    """io.grads, computed once per input set"""
    if key not in _ORACLE:
        _ORACLE[key] = io.grads(p, x, up, **kw)
    return _ORACLE[key]


def _inputs(B, H, W, seed=0):
    g = torch.Generator().manual_seed(seed + H * 7 + W)
    n = (H // 16) * (W // 16)
    return torch.randn(B, 3, H, W, generator=g), torch.randn(B, n + 1, 192, generator=g)


def _active(p):
    return [k for k in p if not k.startswith(("pooler.", "layernorm."))]


def _run(m, x, up, mask=None, attn=False, retain=(), interp=True):
    xd = x.to(DEV).requires_grad_(True)
    out = m(xd, output_hidden_states=True, output_attentions=attn, interpolate_pos_encoding=interp,
            bool_masked_pos=None if mask is None else mask.to(DEV))
    for l in retain:
        out.attentions[l].retain_grad()
    (out.hidden_states[-1] * up.to(DEV)).sum().backward()
    return out, xd.grad


def _wrel(m, ref, names):
    got = dict(m.named_parameters())
    num = sum(float(((got[k].grad.double().cpu() - ref[k].double()) ** 2).sum()) for k in names if not k.endswith("key.bias"))
    den = sum(float((ref[k].double() ** 2).sum()) for k in names if not k.endswith("key.bias"))
    return (num / den) ** 0.5


@pytest.mark.parametrize("H,W", SIZES)
@pytest.mark.parametrize("B", [3, 128])
def test_fp32_matches_oracle(H, W, B):
    p = _state()
    x, up = _inputs(B, H, W)
    names = _active(p)
    hs, probs, dx, _, dp, da = _oracle(p, x, up, (H, W, B), retain=(0, 11), names=names)
    m = _model(p, "fp32")
    out, gx = _run(m, x, up, attn=True, retain=(0, 11))
    torch.cuda.synchronize()
    from vit2spn import _lib
    assert _lib.lib.v2s_debug_flag() == 0
    for k in range(13):
        assert _rel(out.hidden_states[k].detach(), hs[k]) <= 1e-5, k
    for k in range(12):
        assert _rel(out.attentions[k].detach(), probs[k]) <= 1e-5, k
    assert _rel(gx, dx) <= 1e-5
    assert _wrel(m, dp, names) <= 1e-5
    assert _rel(m.embeddings.position_embeddings.grad, dp["embeddings.position_embeddings"]) <= 1e-5
    for l in (0, 11):
        assert _rel(out.attentions[l].grad, da[l]) <= 1e-5, l


@pytest.mark.parametrize("H,W", SIZES)
@pytest.mark.parametrize("B", [3, 128])
@pytest.mark.parametrize("mode,dtype", [("bf16", torch.bfloat16), ("fp16", torch.float16)])
def test_16bit_matches_oracle(H, W, B, mode, dtype):
    p = _state()
    x, up = _inputs(B, H, W)
    names = _active(p)
    hs, _, dx, _, dp, _ = _oracle(p, x, up, (H, W, B), retain=(0, 11), names=names)
    m = _model(p, mode)
    out, gx = _run(m, x, up)
    torch.cuda.synchronize()
    from vit2spn import _lib
    assert _lib.lib.v2s_debug_flag() == 0
    assert _rel(gx, dx) <= 2e-2
    assert _wrel(m, dp, names) <= 2e-2
    # features (the mean over the tokens of hidden_states[-1]): no further from fp32 than torch.autocast of the oracle on
    # the same inputs, with the tolerance of the 224 x 224 gate (tests/test_gpu_parity.py)
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        hs_ac, _ = io.backbone_outputs({k: v.to(DEV) for k, v in p.items()}, x.to(DEV))
    ref = hs[-1].mean(dim=1)
    e_torch = _rel(hs_ac[-1].float().mean(dim=1), ref)
    e_ours = _rel(out.hidden_states[-1].detach().mean(dim=1), ref)
    assert e_ours <= 1e-2 and e_ours <= 1.5 * e_torch + 1e-4, (e_ours, e_torch)


def _launches(fn):
    from vit2spn import _lib
    torch.cuda.synchronize()
    a = _lib.lib.v2s_launch_count()
    fn()
    torch.cuda.synchronize()
    return _lib.lib.v2s_launch_count() - a


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_224_with_flag_is_bit_identical(mode, monkeypatch):
    # fixed-order weight-gradient sums, so that two runs can be compared bit for bit
    monkeypatch.setattr(torch, "are_deterministic_algorithms_enabled", lambda: True)
    p = _state()
    x, up = _inputs(3, 224, 224)
    res = []
    for interp in (False, True):
        m = _model(p, mode)
        box = {}

        def go():
            box["r"] = _run(m, x, up, attn=True, retain=(3,), interp=interp)
        n = _launches(go)
        out, gx = box["r"]
        res.append((n, out, gx, {k: v.grad.clone() for k, v in m.named_parameters() if v.grad is not None}))
    (n0, o0, g0, w0), (n1, o1, g1, w1) = res
    assert n0 == n1
    for a, b in zip(o0.hidden_states + o0.attentions, o1.hidden_states + o1.attentions):
        assert torch.equal(a, b)
    assert torch.equal(o0.attentions[3].grad, o1.attentions[3].grad)
    assert torch.equal(g0, g1)
    assert w0.keys() == w1.keys() and all(torch.equal(w0[k], w1[k]) for k in w0)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_launch_counts_at_128(mode):
    p = _state()
    x, up = _inputs(4, 128, 128)
    x224, up224 = _inputs(4, 224, 224)
    counts = {}
    for name, xx, uu in (("224", x224, up224), ("128", x, up)):
        m = _model(p, mode)
        xd = xx.to(DEV)
        with torch.no_grad():
            fwd = _launches(lambda: m(xd, interpolate_pos_encoding=True, output_hidden_states=True))
        box = {}
        full = _launches(lambda: box.setdefault("o", m(xd, interpolate_pos_encoding=True, output_hidden_states=True)))
        bwd = _launches(lambda: (box["o"].hidden_states[-1] * uu.to(DEV)).sum().backward())
        counts[name] = (fwd, full, bwd)
    assert counts["128"][0] == counts["224"][0] + 1
    assert counts["128"][1] == counts["224"][1] + 1
    assert counts["128"][2] == counts["224"][2] + 1


@pytest.mark.parametrize("mode", ["fp32", "bf16", "fp16"])
def test_deterministic_at_128(mode):
    p = _state()
    x, up = _inputs(6, 128, 128)
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        runs = []
        for _ in range(2):
            m = _model(p, mode, token=_token())
            mask = torch.rand(6, 64, generator=torch.Generator().manual_seed(5)) < 0.3
            out, gx = _run(m, x, up, mask=mask)
            runs.append((gx, {k: v.grad.clone() for k, v in m.named_parameters() if v.grad is not None}))
        (g0, w0), (g1, w1) = runs
        assert torch.equal(g0, g1)
        assert w0.keys() == w1.keys() and all(torch.equal(w0[k], w1[k]) for k in w0)
    finally:
        torch.use_deterministic_algorithms(prev)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_combined_mask_frozen_pixels_retained_attention_at_128(mode):
    p, token = _state(), _token()
    B = 3
    x, up = _inputs(B, 128, 128)
    mask = torch.rand(B, 64, generator=torch.Generator().manual_seed(9)) < 0.4
    hs, _, dx, dtok, _, da = io.grads(p, x, up, mask=mask, token=token, retain=(2, 7), names=())
    m = _model(p, mode, token=token, frozen=True)
    m.embeddings.mask_token.requires_grad_(True)
    out, gx = _run(m, x, up, mask=mask, attn=True, retain=(2, 7))
    torch.cuda.synchronize()
    from vit2spn import _lib
    assert _lib.lib.v2s_debug_flag() == 0
    tol = 1e-5 if mode == "fp32" else 2e-2
    assert out.attentions[2].grad.shape == (B, 3, 65, 65)
    assert _rel(gx, dx) <= tol
    assert _rel(m.embeddings.mask_token.grad.view(192), dtok) <= tol
    for l in (2, 7):
        assert _rel(out.attentions[l].grad, da[l]) <= (tol if mode == "fp32" else 5e-2), l
    assert all(v.grad is None for k, v in m.named_parameters() if k != "embeddings.mask_token")


def test_host_passes_the_forward_size_to_the_backward():
    _lib = _get_lib()
    p = _state()
    m = _model(p, "bf16")
    x, up = _inputs(2, 128, 128)
    out = m(x.to(DEV), interpolate_pos_encoding=True, output_hidden_states=True)
    m2 = _model(p, "bf16")
    with torch.no_grad():
        m2(torch.zeros(2, 3, 64, 64, device=DEV), interpolate_pos_encoding=True)   # another size in between
    (out.hidden_states[-1] * up.to(DEV)).sum().backward()                          # the host passes the forward's size
    assert m.embeddings.position_embeddings.grad is not None
    torch.cuda.synchronize()
    assert _lib.lib.v2s_debug_flag() == 0


@pytest.mark.parametrize("fwd_size,bwd_size", [((128, 128), (64, 64)), ((128, 128), (224, 224)), ((224, 224), (112, 448))])
def test_c_backward_at_another_size_is_refused(fwd_size, bwd_size):
    """v2s_backbone_backward refuses a stash filled at another image size (the library's own check, below the host)"""
    _lib = _get_lib()
    from vit2spn import modules
    p = _state()
    m = _model(p, "bf16")
    B, mode = 2, _lib.MODE_BF16
    store = m._store
    store.ensure()
    x = torch.randn(B, 3, *fwd_size, device=DEV)
    n = 1 + (bwd_size[0] // 16) * (bwd_size[1] // 16)
    dh = torch.randn(B, max(n, 1 + (fwd_size[0] // 16) * (fwd_size[1] // 16)), 192, device=DEV)
    grads = torch.zeros(store.numel, dtype=torch.float32, device=DEV)
    ws = modules._new_workspace(DEV, B, mode, 1, 1, fwd_size)
    modules._run_forward([modules._group(store, mode, x, 0)], B, mode, ws, size=fwd_size)
    g = modules._group(store, mode, x, 0, grads=grads, dhidden=dh)
    with pytest.raises(RuntimeError, match="image size"):
        modules._run_backward([g], B, mode, ws, size=bwd_size)
    # at the forward's size the same call runs
    modules._run_backward([g], B, mode, ws, size=fwd_size)
    torch.cuda.synchronize()
    assert _lib.lib.v2s_debug_flag() == 0
    assert grads.abs().sum().item() > 0
