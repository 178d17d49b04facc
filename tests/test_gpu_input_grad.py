"""GPU: gradients w.r.t. pixel_values (v2s_backbone_input_backward).  fp32 check mode and bf16 / fp16 against the oracle's
autograd (16-bit modes against its rounding model), a frozen model computing no parameter gradient, the joint backward
leaving the weight gradients bit-identical, the launch counts, the other entry points (FineTunedModel, DualStreamNetwork,
an intermediate hidden state, an integrated-gradients chain) and the image-gradient GEMM operator.

Measured errors go to $V2S_INPUT_GRAD_REPORT (JSON) when set."""
import json
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
_REPORT = {}


def _report(key, value):
    _REPORT[key] = value
    path = os.environ.get("V2S_INPUT_GRAD_REPORT")
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


def _upstream(B, seed=1):
    return torch.randn(B, 197, 192, generator=torch.Generator().manual_seed(seed))


def _rel(a, b):
    return ((a.double().cpu() - b.double().cpu()).norm() / b.double().cpu().norm().clamp_min(1e-30)).item()


def _oracle_dx(p, x, up, dtype=None):
    from oracle import vit2spn_oracle as orc
    xx = x.clone().requires_grad_(True)
    ctx = orc.rounding("all", dtype) if dtype is not None else torch.enable_grad()
    with ctx:
        (orc.backbone_hidden(p, xx) * up).sum().backward()
    return xx.grad


def _flag_clear():
    from vit2spn import _lib
    torch.cuda.synchronize()
    assert _lib.lib.v2s_debug_flag() == 0


def test_fp32_pixel_gradient_matches_oracle():
    p = _state()
    x, up = _images(3), _upstream(3)
    m = _model(p, "fp32")
    xd = x.to(DEV).requires_grad_(True)
    (m(xd).hidden_states[-1] * up.to(DEV)).sum().backward()
    _flag_clear()
    rel = _rel(xd.grad, _oracle_dx(p, x, up))
    _report("fp32_B3", rel)
    assert rel <= 1e-5, rel


@pytest.mark.parametrize("B", [1, 3, 128])
@pytest.mark.parametrize("mode,dtype", [("bf16", torch.bfloat16), ("fp16", torch.float16)])
def test_16bit_pixel_gradient_matches_rounding_model(mode, dtype, B):
    p = _state()
    x, up = _images(B, seed=B), _upstream(B, seed=B)
    m = _model(p, mode)
    xd = x.to(DEV).requires_grad_(True)
    (m(xd).hidden_states[-1] * up.to(DEV)).sum().backward()
    _flag_clear()
    rel = _rel(xd.grad, _oracle_dx(p, x, up, dtype))
    exact = _oracle_dx(p, x, up)
    entry = {"vs_rounding_model": rel, "vs_fp32_oracle": _rel(xd.grad, exact)}
    if B <= 3:     # torch.autocast's own error on the same inputs (oracle under autocast on the GPU)
        from oracle import vit2spn_oracle as orc
        pd = {k: v.to(DEV) for k, v in p.items()}
        xa = x.to(DEV).requires_grad_(True)
        with torch.autocast("cuda", dtype=dtype):
            h = orc.backbone_hidden(pd, xa)
        (h.float() * up.to(DEV)).sum().backward()
        entry["autocast_vs_fp32_oracle"] = _rel(xa.grad, exact)
    _report(f"{mode}_B{B}", entry)
    assert rel <= 2e-2, rel


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_frozen_model_gives_pixel_gradient_and_no_parameter_gradient(mode):
    from vit2spn import _lib
    p = _state()
    B = 3
    x, up = _images(B, 5), _upstream(B, 5)
    m = _model(p, mode, frozen=True)
    xd = x.to(DEV).requires_grad_(True)
    _lib.prof_enable(True)
    (m(xd).hidden_states[-1] * up.to(DEV)).sum().backward()
    rep = _lib.prof_report()
    _lib.prof_enable(False)
    _flag_clear()
    ref = _oracle_dx(p, x, up, torch.bfloat16 if mode == "bf16" else None)
    rel = _rel(xd.grad, ref)
    _report(f"frozen_{mode}", {"rel": rel, "classes": {k: v[0] for k, v in rep.items()}})
    assert rel <= (2e-2 if mode == "bf16" else 1e-5), rel
    assert all(prm.grad is None for prm in m.parameters())
    assert "gemm_wgrad" not in rep and "colsum" not in rep, rep
    assert rep["gemm_pixels"][0] == 1


def test_joint_backward_keeps_weight_gradients_bit_identical():
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        p = _state()
        B = 16
        x, up = _images(B, 7).to(DEV), _upstream(B, 7).to(DEV)
        m = _model(p, "bf16")
        runs = []
        for want_x in (False, True, True):
            m.zero_grad(set_to_none=True)
            xd = x.clone().requires_grad_(want_x)
            (m(xd).hidden_states[-1] * up).sum().backward()
            runs.append(({n: q.grad.clone() for n, q in m.named_parameters() if q.grad is not None},
                         xd.grad.clone() if want_x else None))
        _flag_clear()
        for ga in runs[1:]:
            assert ga[0].keys() == runs[0][0].keys()
            bad = [n for n in ga[0] if not torch.equal(ga[0][n], runs[0][0][n])]
            assert not bad, bad[:8]
        assert torch.equal(runs[1][1], runs[2][1])           # the pixel gradient is reproducible too
        assert _rel(runs[1][1], _oracle_dx(p, x.cpu(), up.cpu(), torch.bfloat16)) <= 2e-2
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


def test_launch_counts():
    """No request, no change (155 / 363, as tests/test_gpu_deterministic.py pins); the frozen input-only backward."""
    import vit2spn
    from vit2spn import _lib
    from oracle import vit2spn_oracle as orc
    if os.environ.get("V2S_GEMM_DEBUG"):
        pytest.skip("launch counts are pinned for the uninstrumented kernels")
    x = _images(4).to(DEV)
    m = _model(_state(), "bf16")
    m(x).hidden_states[-1].mean().backward()
    n0 = _lib.lib.v2s_launch_count()
    m(x).hidden_states[-1].mean().backward()
    vit = _lib.lib.v2s_launch_count() - n0
    d = vit2spn.DualStreamNetwork()
    d.load_state_dict(orc.init_state(3), strict=True)
    d.to(DEV).train()
    d.compute_mode = "bf16"
    d.ssp_step(x, x)
    n0 = _lib.lib.v2s_launch_count()
    d.ssp_step(x, x)
    pred, tgt = d(x, x)
    (pred * tgt).sum().backward()
    dual = _lib.lib.v2s_launch_count() - n0
    assert (vit, dual) == (155, 363)
    f = _model(_state(), "bf16", frozen=True)
    xd = x.clone().requires_grad_(True)
    f(xd).hidden_states[-1].mean().backward()
    n0 = _lib.lib.v2s_launch_count()
    f(xd).hidden_states[-1].mean().backward()
    frozen = _lib.lib.v2s_launch_count() - n0
    _report("launches", {"vit": vit, "dual": dual, "frozen_input_only": frozen})
    # 155 - 24 merged wgrads - the fc2 bias column sum of block 11 - embed_bwd - the patch wgrad + the image-gradient GEMM
    assert frozen == 129, frozen


def test_finetuned_saliency_matches_oracle_backbone_plus_head():
    import vit2spn
    from oracle import vit2spn_oracle as orc
    torch.manual_seed(0)
    ft = vit2spn.FineTunedModel(4)
    ft.backbone.vit.load_state_dict(orc.sub_state(orc.init_state(11, 0.01), "online_network_1"), strict=True)
    ft.to(DEV).eval()
    ft.backbone.vit.compute_mode = "fp32"
    x = _images(3, 9)
    xd = x.to(DEV).requires_grad_(True)
    ft(xd)[:, 2].sum().backward()
    _flag_clear()
    p = {k: v.detach().cpu() for k, v in ft.backbone.vit.state_dict().items()}
    xo = x.clone().requires_grad_(True)
    fc = ft.fc.cpu()
    fc(orc.backbone_features(p, xo))[:, 2].sum().backward()
    rel = _rel(xd.grad, xo.grad)
    _report("finetuned_saliency_fp32", rel)
    assert rel <= 1e-5, rel


def test_dual_stream_pixel_gradients_match_oracle():
    import vit2spn
    from oracle import vit2spn_oracle as orc
    state = orc.init_state(3, 0.01)
    d = vit2spn.DualStreamNetwork()
    d.load_state_dict(state, strict=True)
    d.to(DEV).train()
    d.projection_head[2].p = 0.0
    d.compute_mode = "fp32"
    x1, x2 = orc.synthetic_views(2, seed=4)
    a, b = x1.to(DEV).requires_grad_(True), x2.to(DEV).requires_grad_(True)
    pred, tgt = d(a, b)
    orc.ssp_loss(pred, tgt).backward()
    _flag_clear()
    o1, o2 = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)
    op, ot = orc.dual_stream_forward(state, o1, o2)
    orc.ssp_loss(op, ot.detach()).backward()
    r1, r2 = _rel(a.grad, o1.grad), _rel(b.grad, o2.grad)
    _report("dual_stream_fp32", [r1, r2])
    assert r1 <= 1e-4 and r2 <= 1e-4, (r1, r2)


def test_intermediate_hidden_state_and_integrated_gradients_chain():
    p = _state()
    m = _model(p, "fp32", frozen=True)
    img = _images(2, 3).to(DEV)
    base = torch.zeros_like(img)
    x = img.clone().requires_grad_(True)
    out = m(x, output_hidden_states=True)
    out.hidden_states[4].square().mean().backward()
    assert x.grad is not None and x.grad.abs().sum().item() > 0
    alpha = torch.tensor(0.5, device=DEV, requires_grad=True)
    xi = base + alpha * (img - base)
    xi.retain_grad()
    m(xi).hidden_states[-1].sum().backward()
    _flag_clear()
    want = (xi.grad * (img - base)).sum()
    assert torch.allclose(alpha.grad, want, rtol=1e-5, atol=1e-6), (alpha.grad.item(), want.item())


@pytest.mark.parametrize("B,variant", [(1, 0), (3, 2), (5, 0)])
def test_image_gradient_gemm_operator(B, variant):
    from vit2spn import _lib
    _lib.init_device(0)
    dt = torch.float16 if variant & 2 else torch.bfloat16
    g = torch.Generator(device=DEV).manual_seed(B)
    a = torch.randn(B * 196, 192, device=DEV, generator=g).to(dt)
    w = torch.randn(192, 768, device=DEV, generator=g).to(dt)
    c = torch.full((B, 3, 224, 224), float("nan"), device=DEV)
    _lib.check(_lib.lib.v2s_test_gemm(5, _lib.ptr(a), _lib.ptr(w), _lib.ptr(c), B * 196, 768, 192, variant,
                                      _lib.stream_ptr()), "test_gemm 5")
    _flag_clear()
    rows = a.float() @ w.float()
    ref = rows.view(B, 14, 14, 3, 16, 16).permute(0, 3, 1, 4, 2, 5).reshape(B, 3, 224, 224)
    assert _rel(c, ref) <= 1e-5
