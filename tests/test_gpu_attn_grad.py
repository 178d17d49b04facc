"""GPU: gradients w.r.t. the attention probabilities (retain_grad() on ViTModel's attentions,
v2s_backbone_backward_attn_grads).  The dP = d ctx V^T operator against float64; the retained .grad of all 12 blocks
against the oracle (fp32 check mode; bf16 / fp16 against the fp32 oracle and its rounding model); transformers' None
pattern; weight gradients and reproducibility; the frozen backbone with pixel gradients; launch counts; the relevance map.

Measured errors go to $V2S_ATTN_GRAD_REPORT (JSON) when set."""
import json
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import attn_grad_oracle as ag  # noqa: E402  (helper module, not a test)

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
_REPORT = {}


def _report(key, value):
    _REPORT[key] = value
    path = os.environ.get("V2S_ATTN_GRAD_REPORT")
    if path:
        with open(path, "w") as f:
            json.dump(_REPORT, f, indent=1, sort_keys=True)


def _state(seed=11):
    from oracle import vit2spn_oracle as orc
    return orc.sub_state(orc.init_state(seed, 0.01), "online_network_1")


def _model(p, mode, frozen=False):
    import vit2spn
    m = vit2spn.ViTModel()
    m.load_state_dict(p, strict=True)
    m.to(DEV)
    m.compute_mode = mode
    if frozen:
        m.requires_grad_(False)
    return m


def _images(B, seed=0):
    from oracle import vit2spn_oracle as orc
    return orc.preprocess_u8(orc.synthetic_octmnist_u8(B, seed))


def _rel(a, b):
    return ((a.double().cpu() - b.double().cpu()).norm() / b.double().cpu().norm().clamp_min(1e-30)).item()


def _flag_clear():
    from vit2spn import _lib
    torch.cuda.synchronize()
    assert _lib.lib.v2s_debug_flag() == 0


def _weights(B, seed=5):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, 197, 192, generator=g), torch.randn(B, 192, generator=g)


def _loss_fn(w7, wf):
    """hidden_states[7] and the mean-pooled last state: every block is reached, blocks 0-6 along two paths"""
    return lambda hs: (hs[7] * w7.to(hs[7].device)).sum() + (hs[12].mean(1) * wf.to(hs[12].device)).sum()


def _run(m, x, loss_fn, retain=range(12), **kw):
    """forward with all outputs, retain_grad() on the attentions of the blocks in `retain`, backward of the loss"""
    out = m(x, output_hidden_states=True, output_attentions=True, **kw)
    for l in retain:
        out.attentions[l].retain_grad()
    loss_fn(out.hidden_states).backward()
    return out


# ---- the operator ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("batch", [1, 3, 5, 64])
@pytest.mark.parametrize("variant", [0, 1, 2, 3])    # bit 0: SIMT kernel instead of tensor-core; bit 1: fp16 tensors
def test_attention_probability_gradient_operator(batch, variant):
    from vit2spn import _lib
    _lib.init_device(0)
    g = torch.Generator(device=DEV).manual_seed(batch + 7)
    lp = torch.float16 if variant & 2 else torch.bfloat16
    qkv = torch.randn(batch, 197, 576, device=DEV, generator=g).to(lp)
    dctx = (torch.randn(batch, 197, 192, device=DEV, generator=g) * 1e-2).to(lp)
    outs = []
    for _ in range(2):
        out = torch.full((batch, 3, 197, 197), float("nan"), device=DEV)
        _lib.check(_lib.lib.v2s_test_attention(3, _lib.ptr(qkv), _lib.ptr(out), None, _lib.ptr(dctx), None, batch, variant,
                                               _lib.stream_ptr()), "attention probability gradient")
        outs.append(out)
    _flag_clear()
    do = dctx.double().view(batch, 197, 3, 64).transpose(1, 2)
    v = qkv.double()[..., 384:].reshape(batch, 197, 3, 64).transpose(1, 2)
    ref = do @ v.transpose(-1, -2)
    scale = (do.abs() @ v.abs().transpose(-1, -2)).max().item()
    err = (outs[0].double() - ref).abs().max().item()
    _report(f"op_b{batch}_v{variant}", {"maxabs": err, "maxabs_over_scale": err / scale, "rel_l2": _rel(outs[0], ref)})
    assert torch.isfinite(outs[0]).all()
    assert err <= 1e-6 * scale, (err, scale)
    assert torch.equal(outs[0], outs[1])


# ---- end to end against the oracle --------------------------------------------------------------------------------
def test_fp32_attention_gradients_match_oracle():
    p = _state()
    B = 3
    x = _images(B, seed=2)
    loss_fn = _loss_fn(*_weights(B))
    _, _, ref = ag.attention_grads(p, x, loss_fn)
    out = _run(_model(p, "fp32"), x.to(DEV), loss_fn)
    _flag_clear()
    rels = [_rel(a.grad, r) for a, r in zip(out.attentions, ref)]
    _report("fp32_B3", rels)
    assert max(rels) <= 1e-4, rels


@pytest.mark.parametrize("mode,dtype", [("bf16", torch.bfloat16), ("fp16", torch.float16)])
def test_16bit_attention_gradients_match_oracle(mode, dtype):
    from oracle import vit2spn_oracle as orc
    p = _state()
    B = 3
    x = _images(B, seed=3)
    loss_fn = _loss_fn(*_weights(B, 6))
    _, _, exact = ag.attention_grads(p, x, loss_fn)
    with orc.rounding("all", dtype):
        _, _, rounded = ag.attention_grads(p, x, loss_fn)
    out = _run(_model(p, mode), x.to(DEV), loss_fn)
    _flag_clear()
    rel = [_rel(a.grad, r) for a, r in zip(out.attentions, exact)]
    rel_r = [_rel(a.grad, r) for a, r in zip(out.attentions, rounded)]
    _report(f"{mode}_B3", {"vs_fp32_oracle": rel, "vs_rounding_model": rel_r})
    assert max(rel) <= 2e-2 and max(rel_r) <= 2e-2, (rel, rel_r)


def test_blocks_the_loss_does_not_reach_keep_grad_none():
    p = _state()
    B = 2
    x = _images(B, seed=4)
    w, _ = _weights(B, 7)

    def loss_fn(hs):
        return (hs[4] * w.to(hs[4].device)).sum()

    _, _, ref = ag.attention_grads(p, x, loss_fn)
    m = _model(p, "fp32")
    out = _run(m, x.to(DEV), loss_fn)
    _flag_clear()
    assert [a.grad is not None for a in out.attentions] == [l < 4 for l in range(12)]
    assert [r is not None for r in ref] == [l < 4 for l in range(12)]
    rels = [_rel(out.attentions[l].grad, ref[l]) for l in range(4)]
    _report("reach4_fp32", rels)
    assert max(rels) <= 1e-4, rels


def test_retained_gradient_accumulates_like_retain_grad():
    m = _model(_state(), "fp32")
    x = _images(2, seed=8).to(DEV)
    out = m(x, output_attentions=True)
    out.attentions[2].retain_grad()
    out.attentions[2].grad = torch.ones_like(out.attentions[2])
    out.hidden_states[-1].sum().backward()
    got = out.attentions[2].grad
    out = m(x, output_attentions=True)
    out.attentions[2].retain_grad()
    out.hidden_states[-1].sum().backward()
    _flag_clear()
    assert torch.allclose(got, out.attentions[2].grad + 1, rtol=1e-6, atol=1e-7)


# ---- weight gradients, reproducibility --------------------------------------------------------------------------
def test_weight_gradients_bit_identical_and_attention_gradients_reproducible():
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        p = _state()
        B = 16
        x = _images(B, 7).to(DEV)
        loss_fn = _loss_fn(*_weights(B, 9))
        m = _model(p, "bf16")
        runs = []
        for retain in ((), range(12), range(12)):
            m.zero_grad(set_to_none=True)
            out = _run(m, x, loss_fn, retain)
            runs.append(({n: q.grad.clone() for n, q in m.named_parameters() if q.grad is not None},
                         [a.grad if a.retains_grad else None for a in out.attentions]))
        _flag_clear()
        assert all(g is None for g in runs[0][1])
        for wg, _ in runs[1:]:
            assert wg.keys() == runs[0][0].keys()
            bad = [n for n in wg if not torch.equal(wg[n], runs[0][0][n])]
            assert not bad, bad[:8]
        assert all(torch.equal(a, b) for a, b in zip(runs[1][1], runs[2][1]))
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


# ---- frozen backbone with pixel gradients; launch counts ----------------------------------------------------------
def _launches(fn):
    from vit2spn import _lib
    fn()                                  # warm-up: kernel attributes, workspace
    torch.cuda.synchronize()
    n0 = _lib.lib.v2s_launch_count()
    fn()
    torch.cuda.synchronize()
    return _lib.lib.v2s_launch_count() - n0


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_frozen_backbone_pixel_and_attention_gradients(mode):
    p = _state()
    B = 3
    x = _images(B, seed=5)
    loss_fn = _loss_fn(*_weights(B, 10))
    m = _model(p, mode, frozen=True)
    xd = x.to(DEV).requires_grad_(True)
    out = _run(m, xd, loss_fn)
    _flag_clear()
    from oracle import vit2spn_oracle as orc
    ctx = orc.rounding("all", torch.bfloat16) if mode == "bf16" else torch.enable_grad()
    xo = x.clone().requires_grad_(True)
    with ctx:
        _, _, ref = ag.attention_grads(p, x, loss_fn)
        hs = [orc.patch_embed(p, xo)]
        for l in range(orc.LAYERS):
            hs.append(orc.vit_layer(p, l, hs[-1]))
        loss_fn(hs).backward()
    gate = 2e-2 if mode == "bf16" else 1e-4
    rels = [_rel(a.grad, r) for a, r in zip(out.attentions, ref)]
    rel_x = _rel(xd.grad, xo.grad)
    _report(f"frozen_{mode}", {"attn": rels, "pixels": rel_x})
    assert max(rels) <= gate and rel_x <= gate, (rels, rel_x)
    assert all(prm.grad is None for prm in m.parameters())
    if os.environ.get("V2S_GEMM_DEBUG"):
        return

    def step(retain):
        def fn():
            xx = x.to(DEV).requires_grad_(True)
            _run(m, xx, loss_fn, retain)
        return fn

    base, three, all12 = (_launches(step(r)) for r in ((), (0, 6, 11), range(12)))
    _report(f"frozen_{mode}_launches", [base, three, all12])
    assert (three - base, all12 - base) == (3, 12), (base, three, all12)


def test_launch_count_grows_by_the_retained_blocks():
    if os.environ.get("V2S_GEMM_DEBUG"):
        pytest.skip("launch counts are pinned for the uninstrumented kernels")
    m = _model(_state(), "bf16")
    x = _images(4).to(DEV)
    loss_fn = _loss_fn(*_weights(4, 11))
    counts = [_launches(lambda r=r: _run(m, x, loss_fn, r)) for r in ((), (3,), (1, 2, 9, 10), range(12))]
    _report("launches_bf16", counts)
    assert [c - counts[0] for c in counts] == [0, 1, 4, 12], counts


# ---- relevance map, realistic size --------------------------------------------------------------------------------
@pytest.mark.parametrize("token", ["cls", "mean"])
def test_relevance_map_matches_oracle(token):
    """The FineTunedModel pattern: attentions of the backbone's ViTModel, the head on the mean-pooled last state."""
    import vit2spn
    from vit2spn import explain
    torch.manual_seed(0)
    ft = vit2spn.FineTunedModel(4)
    p = _state(12)
    ft.backbone.vit.load_state_dict(p, strict=True)
    ft.to(DEV).eval()
    ft.backbone.vit.compute_mode = "fp32"
    x = _images(2, seed=6)
    out = ft.backbone.vit(x.to(DEV), output_attentions=True)
    for a in out.attentions:
        a.retain_grad()
    ft.fc(out.hidden_states[-1].mean(1))[:, 1].sum().backward()
    _flag_clear()
    got = explain.attention_relevance(out.attentions, [a.grad for a in out.attentions], token=token)
    fc = ft.fc.cpu()
    _, attn, grads = ag.attention_grads(p, x, lambda hs: fc(hs[12].mean(1))[:, 1].sum())
    want = ag.relevance_loop(attn, grads, token=token)
    rel = _rel(got, want)
    _report(f"relevance_{token}_fp32", rel)
    assert got.shape == (2, 14, 14) and rel <= 1e-4, rel


def test_realistic_batch_bf16():
    p = _state()
    B = 128
    x = _images(B, seed=13)
    loss_fn = _loss_fn(*_weights(B, 14))
    out = _run(_model(p, "bf16"), x.to(DEV), loss_fn)
    _flag_clear()
    assert all(torch.isfinite(a.grad).all() for a in out.attentions)
    rows = [0, B // 2, B - 1]      # the images of a batch are independent: the oracle checks three
    w7, wf = _weights(B, 14)
    _, _, ref = ag.attention_grads(p, x[rows], _loss_fn(w7[rows], wf[rows]))
    rels = [_rel(a.grad[rows], r) for a, r in zip(out.attentions, ref)]
    _report("bf16_B128_vs_fp32_oracle", rels)
    assert max(rels) <= 2e-2, rels
