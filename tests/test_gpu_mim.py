"""GPU: ``vit2spn.ViTForMaskedImageModeling`` (SimMIM head on the CUDA path).  The fp32 check mode against
``mim_oracle`` (loss, reconstruction, decoder / LayerNorm / mask-token / backbone / pixel gradients); bf16 and fp16
against its rounding model, the whole model at B=3 and the head at B=128; agreement with the torch-head recipe on the
same backbone; bit-reproducibility; fp16 with a GradScaler; frozen backbone and frozen decoder; launch counts of the head;
a FusedAdam loop; the non-differentiable reconstruction.

Measured errors go to $V2S_MIM_REPORT (JSON) when set."""
import json
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import mim_oracle as mim  # noqa: E402  (helper module, not a test)

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
_REPORT = {}
_LP = {"bf16": torch.bfloat16, "fp16": torch.float16}


def _report(key, value):
    _REPORT[key] = value
    path = os.environ.get("V2S_MIM_REPORT")
    if path:
        with open(path, "w") as f:
            json.dump(_REPORT, f, indent=1, sort_keys=True)


def _weights(seed=11):
    from oracle import vit2spn_oracle as orc
    p = orc.sub_state(orc.init_state(seed, 0.01), "online_network_1")
    g = torch.Generator().manual_seed(seed + 100)
    token = 0.02 * torch.randn(192, generator=g)
    dec_w, dec_b = 0.02 * torch.randn(768, 192, 1, 1, generator=g), 0.01 * torch.randn(768, generator=g)
    return p, token, dec_w, dec_b


def _model(w, mode):
    import vit2spn
    p, token, dec_w, dec_b = w
    m = vit2spn.ViTForMaskedImageModeling()
    sd = {"vit." + k: v for k, v in p.items() if not k.startswith("pooler.")}
    sd.update({"vit.embeddings.mask_token": token.view(1, 1, 192), "decoder.0.weight": dec_w, "decoder.0.bias": dec_b})
    m.load_state_dict(sd, strict=True)
    m.to(DEV)
    m.compute_mode = mode
    return m


def _images(B, seed=0):
    from oracle import vit2spn_oracle as orc
    return orc.preprocess_u8(orc.synthetic_octmnist_u8(B, seed))


def _mask(B, seed, edge=True, frac=0.6):
    m = torch.rand(B, 196, generator=torch.Generator().manual_seed(seed)) < frac
    if edge:                                        # one unmasked image, one fully masked, the rest mixed
        m[0] = False
        m[1] = True
    return m


def _rel(a, b):
    return ((a.double().cpu() - b.double().cpu()).norm() / b.double().cpu().norm().clamp_min(1e-30)).item()


def _flag_clear():
    from vit2spn import _lib
    torch.cuda.synchronize()
    assert _lib.lib.v2s_debug_flag() == 0


def _step(m, x, mask, want_x=True, scale=1.0):
    """forward + backward; `scale` multiplies the loss as a GradScaler does (fp16: the backbone's 16-bit gradients would
    underflow at SimMIM's ~1e-7 per-pixel scale) and the returned pixel gradient is divided by it again"""
    xd = x.detach().to(DEV).clone().requires_grad_(want_x)
    out = m(xd, bool_masked_pos=mask.to(DEV) if mask is not None else None)
    if out.loss is not None:
        (out.loss * scale).backward()
    return out, (xd.grad / scale if xd.grad is not None else None)


_SCALE = {"fp32": 1.0, "bf16": 1.0, "fp16": 2.0 ** 14}


def _pixels(got, ref, mask):
    """The pixel gradient in two parts.  Unmasked pixels carry the backbone's term only: relative L2 error.  Masked
    pixels carry only the loss's own term -c sign(r - x) (a masked patch gives the backbone no pixel gradient), which is
    discontinuous: where the reconstruction is within rounding of the input the sign can differ from the reference's, so
    the fraction of masked pixels whose sign differs is reported instead."""
    pm = mim.pixel_mask(mask).expand_as(ref).cpu()
    got, ref = got.detach().cpu().double(), ref.double()
    c = ref[pm].abs().max().clamp_min(1e-30)
    flips = ((got[pm] - ref[pm]).abs() > 0.5 * c).double().mean().item() if pm.any() else 0.0
    return _rel(got[~pm], ref[~pm]), flips


def _scaled_grads(m, dx, scale):
    return {k: (v / scale if v is not None else None) for k, v in _grads(m, dx).items()} if scale != 1.0 else _grads(m, dx)


_CHECKED = ("decoder.0.weight", "decoder.0.bias", "layernorm.weight", "layernorm.bias", "mask_token",
            "embeddings.patch_embeddings.projection.weight", "encoder.layer.5.intermediate.dense.weight", "pixels")


def _grads(m, dx):
    named = dict(m.named_parameters())
    g = {k: named["vit." + k].grad for k in _CHECKED if "vit." + k in named}
    g.update({"decoder.0.weight": m.decoder[0].weight.grad, "decoder.0.bias": m.decoder[0].bias.grad,
              "mask_token": m.vit.embeddings.mask_token.grad.view(192), "pixels": dx})
    return g


# ---- fp32 check mode against the oracle ----------------------------------------------------------------------------
def test_fp32_matches_oracle_b3():
    w = _weights()
    B = 3
    x, mask = _images(B, seed=1), _mask(B, seed=2)
    m = _model(w, "fp32")
    out, dx = _step(m, x, mask)
    _flag_clear()
    loss, rec, ref = mim.model_loss(*w, x, mask)
    got = _grads(m, dx)
    rel = {"loss": abs(out.loss.item() - loss.item()) / abs(loss.item()), "reconstruction": _rel(out.reconstruction, rec)}
    rel.update({k: _rel(got[k], ref[k]) for k in _CHECKED})
    _report("fp32_B3", rel)
    assert max(rel.values()) <= 1e-5, rel


def test_fp32_all_false_mask_and_no_mask():
    w = _weights()
    B = 2
    x = _images(B, seed=3)
    m = _model(w, "fp32")
    out, dx = _step(m, x, torch.zeros(B, 196, dtype=torch.bool))
    _flag_clear()
    assert out.loss.item() == 0.0
    for k, g in _grads(m, dx).items():
        assert g is not None and torch.count_nonzero(g) == 0, k
    out2, _ = _step(m, x, None)
    assert out2.loss is None and torch.equal(out2.reconstruction, out.reconstruction)
    _, rec, _ = mim.model_loss(*w, x, torch.zeros(B, 196, dtype=torch.bool))
    assert _rel(out2.reconstruction, rec) <= 1e-5


# ---- 16-bit modes ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["bf16", "fp16"])
def test_16bit_matches_rounding_model_b3(mode):
    from oracle import vit2spn_oracle as orc
    w = _weights()
    B = 3
    x, mask = _images(B, seed=4), _mask(B, seed=5)
    m = _model(w, mode)
    out, dx = _step(m, x, mask, scale=_SCALE[mode])
    _flag_clear()
    with orc.rounding("all", _LP[mode]):
        loss, rec, ref = mim.model_loss(*w, x, mask, lp=_LP[mode])
    got = _scaled_grads(m, dx, _SCALE[mode])
    rel = {"loss": abs(out.loss.item() - loss.item()) / abs(loss.item()), "reconstruction": _rel(out.reconstruction, rec)}
    rel.update({k: _rel(got[k], ref[k]) for k in _CHECKED if k != "pixels"})
    rel["pixels_unmasked"], rel["pixels_masked_sign_flips"] = _pixels(dx, ref["pixels"], mask)
    _report(f"{mode}_B3", rel)
    assert rel["loss"] <= 1e-3, rel
    assert rel["pixels_masked_sign_flips"] <= 1e-3, rel
    assert max(v for k, v in rel.items() if k not in ("loss", "pixels_masked_sign_flips")) <= 2e-2, rel


@pytest.mark.parametrize("mode", ["bf16", "fp16"])
def test_16bit_head_matches_rounding_model_b128(mode):
    """The head at B=128 on the backbone's own hidden_states[12]: loss, reconstruction and every head gradient."""
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)       # both backbone backwards below give the same pixel gradient
    try:
        _head_b128(mode)
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


def _head_b128(mode):
    w = _weights()
    B = 128
    x, mask = _images(B, seed=6), _mask(B, seed=7)
    m = _model(w, mode)
    xd = x.to(DEV).requires_grad_(True)
    out = m(xd, bool_masked_pos=mask.to(DEV), output_hidden_states=True)
    h12 = out.hidden_states[-1]
    h12.retain_grad()
    out.loss.backward()
    _flag_clear()
    # the pixel term of the head alone: x.grad minus the backbone's share (the backbone run again, head-free)
    with torch.enable_grad():
        xb = x.to(DEV).requires_grad_(True)
        hb = m.vit(xb, bool_masked_pos=mask.to(DEV)).hidden_states[-1]
        hb.backward(h12.grad)
    direct = xd.grad - xb.grad
    _flag_clear()
    with torch.enable_grad():
        hh = h12.detach().cpu().requires_grad_(True)
        lw, lb = (m.vit.layernorm.weight.detach().cpu().requires_grad_(True),
                  m.vit.layernorm.bias.detach().cpu().requires_grad_(True))
        dw, db = w[2].clone().requires_grad_(True), w[3].clone().requires_grad_(True)
        xx = x.clone().requires_grad_(True)
        rec, loss = mim.head(hh, lw, lb, dw, db, xx, mask, _LP[mode])
        loss.backward()
    rel = {"loss": abs(out.loss.item() - loss.item()) / abs(loss.item()),
           "reconstruction": _rel(out.reconstruction, rec.detach()),
           "hidden12": _rel(h12.grad, hh.grad), "layernorm.weight": _rel(m.vit.layernorm.weight.grad, lw.grad),
           "layernorm.bias": _rel(m.vit.layernorm.bias.grad, lb.grad),
           "decoder.0.weight": _rel(m.decoder[0].weight.grad, dw.grad), "decoder.0.bias": _rel(m.decoder[0].bias.grad, db.grad),
           "pixels_direct": _rel(direct, xx.grad)}
    _report(f"{mode}_head_B128", rel)
    assert rel["loss"] <= 1e-3, rel
    assert max(v for k, v in rel.items() if k != "loss") <= 2e-2, rel
    assert torch.count_nonzero(h12.grad[:, 0]) == 0


def test_agrees_with_the_torch_head_recipe():
    """The same CUDA backbone with the eager-torch SimMIM head (final LayerNorm, fp32 Conv2d, PixelShuffle, masked L1)."""
    from test_masked_tokens_cpu import simmim_loss
    w = _weights()
    B = 16
    x, mask = _images(B, seed=8).to(DEV), _mask(B, seed=9).to(DEV)
    m = _model(w, "bf16")
    out, dx = _step(m, x, mask)
    ours = {k: v.clone() for k, v in _grads(m, dx).items()}
    m.zero_grad(set_to_none=True)
    xd = x.clone().requires_grad_(True)
    ref = simmim_loss(m.vit(xd, bool_masked_pos=mask).last_hidden_state, m.decoder[0], xd, mask)
    ref.backward()
    _flag_clear()
    theirs = _grads(m, xd.grad)
    rel = {"loss": abs(out.loss.item() - ref.item()) / abs(ref.item())}
    rel.update({k: _rel(ours[k], theirs[k]) for k in _CHECKED if k != "pixels"})
    rel["pixels_unmasked"], rel["pixels_masked_sign_flips"] = _pixels(ours["pixels"], theirs["pixels"].cpu(), mask)
    _report("torch_head_bf16_B16", rel)
    assert rel["loss"] <= 1e-3, rel
    assert rel["pixels_masked_sign_flips"] <= 1e-3, rel
    assert max(v for k, v in rel.items() if k != "pixels_masked_sign_flips") <= 2e-2, rel


# ---- determinism -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_deterministic_steps_are_bit_identical(mode):
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        w = _weights()
        B = 8
        x, mask = _images(B, seed=10), _mask(B, seed=11)
        m = _model(w, mode)
        runs = []
        for _ in range(2):
            m.zero_grad(set_to_none=True)
            out, dx = _step(m, x, mask)
            runs.append((out.loss.detach().clone(), out.reconstruction.clone(), dx,
                         {n: q.grad.clone() for n, q in m.named_parameters() if q.grad is not None}))
        _flag_clear()
        (l0, r0, x0, g0), (l1, r1, x1, g1) = runs
        assert torch.equal(l0, l1) and torch.equal(r0, r1) and torch.equal(x0, x1)
        assert g0.keys() == g1.keys() and "decoder.0.weight" in g0 and "vit.layernorm.weight" in g0
        bad = [n for n in g0 if not torch.equal(g0[n], g1[n])]
        assert not bad, bad[:8]
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


def test_loss_is_bit_identical_without_the_flag():
    from vit2spn import _lib
    w = _weights()
    B = 64
    x, mask = _images(B, seed=12).to(DEV), _mask(B, seed=13).to(DEV)
    m = _model(w, "bf16")
    losses = []
    with torch.no_grad():
        for sms in (0, 37, 0):                      # the tile partials do not depend on the grid
            _lib.check(_lib.lib.v2s_set_sm_limit(sms), "set_sm_limit")
            losses.append(m(x, bool_masked_pos=mask).loss.clone())
    _lib.check(_lib.lib.v2s_set_sm_limit(0), "set_sm_limit")
    _flag_clear()
    assert all(torch.equal(losses[0], t) for t in losses[1:]), losses


# ---- fp16 with a GradScaler, frozen parts ----------------------------------------------------------------------------
def test_fp16_gradscaler_step():
    import vit2spn
    w = _weights()
    B = 8
    x, mask = _images(B, seed=14).to(DEV), _mask(B, seed=15).to(DEV)
    m = _model(w, "fp16")
    out, _ = _step(m, x, mask, want_x=False, scale=2.0 ** 14)          # the same scale applied by hand
    plain = {k: v.clone() for k, v in _scaled_grads(m, None, 2.0 ** 14).items() if k != "pixels"}
    m.zero_grad(set_to_none=True)
    opt = vit2spn.FusedAdam(m.parameters(), lr=1e-4)
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 14)
    loss = m(x, bool_masked_pos=mask).loss
    scaler.scale(loss).backward()
    scaled = {k: v.clone() / scaler.get_scale() for k, v in _grads(m, None).items() if k != "pixels"}
    w0 = m.decoder[0].weight.detach().clone()
    scaler.step(opt)
    scaler.update()
    _flag_clear()
    rel = {k: _rel(scaled[k], plain[k]) for k in plain}
    _report("fp16_gradscaler", rel)
    assert max(rel.values()) <= 1e-3, rel
    assert not torch.equal(w0, m.decoder[0].weight.detach())
    assert all(torch.isfinite(q).all().item() for q in m.parameters())


@pytest.mark.parametrize("mode", ["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("deterministic", [False, True])
def test_frozen_backbone_or_decoder(mode, deterministic):
    from vit2spn import _lib
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(deterministic)
    try:
        w = _weights()
        B = 3
        x, mask = _images(B, seed=16), _mask(B, seed=17)
        m = _model(w, mode)
        sc = _SCALE[mode]
        _, _ = _step(m, x, mask, want_x=False, scale=sc)
        full = {k: v.clone() for k, v in _grads(m, None).items() if k != "pixels"}
        tol = 1e-5 if mode == "fp32" else 1e-3
        # frozen backbone (its final LayerNorm and mask token too), trainable decoder: no backbone weight gradient at all
        m.zero_grad(set_to_none=True)
        m.vit.requires_grad_(False)
        _lib.prof_enable(True)
        _step(m, x, mask, want_x=False, scale=sc)
        rep = _lib.prof_report()
        _lib.prof_enable(False)
        assert rep.get("gemm_wgrad", (0,))[0] == 0 and rep["mim_bwd"][0] == 1, rep
        assert [n for n, q in m.named_parameters() if q.grad is not None] == ["decoder.0.weight", "decoder.0.bias"]
        assert _rel(m.decoder[0].weight.grad, full["decoder.0.weight"]) <= tol
        assert _rel(m.decoder[0].bias.grad, full["decoder.0.bias"]) <= tol
        # frozen decoder, trainable backbone
        m.zero_grad(set_to_none=True)
        m.vit.requires_grad_(True)
        m.decoder.requires_grad_(False)
        _step(m, x, mask, want_x=False, scale=sc)
        assert m.decoder[0].weight.grad is None and m.decoder[0].bias.grad is None
        got = _grads(m, None)
        for k in ("layernorm.weight", "mask_token", "encoder.layer.5.intermediate.dense.weight"):
            assert _rel(got[k], full[k]) <= tol, k
        _flag_clear()
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


# ---- launch counts, training loop, reconstruction --------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["bf16", "fp16"])
def test_head_launch_counts(mode):
    """The head adds 4 kernels to a masked forward (W_dec cast, final LayerNorm, decoder GEMM, loss), 3 without a mask,
    and 5 to the backward (decoder wgrad, its scaling, dgrad, LayerNorm backward, pixel term; 4 without the pixels)."""
    from vit2spn import _lib
    from vit2spn import modules
    w = _weights()
    B = 4
    m = _model(w, mode)
    x, mask = _images(B, seed=18).to(DEV), _mask(B, seed=19).to(DEV).to(torch.uint8)
    hidden = torch.randn(B, 197, 192, device=DEV, requires_grad=True)
    ln, conv = m.vit.layernorm, m.decoder[0]

    def count(fn):
        fn()
        torch.cuda.synchronize()
        n0 = _lib.lib.v2s_launch_count()
        r = fn()
        torch.cuda.synchronize()
        return _lib.lib.v2s_launch_count() - n0, r

    def fwd(msk, xx=x):
        return modules._MIMHeadFn.apply(hidden, xx, ln.weight, ln.bias, conv.weight, conv.bias, m, msk, True)
    n_fwd, _ = count(lambda: fwd(mask))
    n_fwd_plain, _ = count(lambda: fwd(None))
    xg = x.clone().requires_grad_(True)
    n_all, _ = count(lambda: fwd(mask)[1].backward())
    n_all_x, _ = count(lambda: fwd(mask, xg)[1].backward())
    _flag_clear()
    _report(f"launches_{mode}", {"forward": n_fwd, "forward_no_mask": n_fwd_plain, "fwd_bwd": n_all, "fwd_bwd_pixels": n_all_x})
    assert (n_fwd, n_fwd_plain) == (4, 3)
    assert n_all - n_fwd == 4 and n_all_x - n_fwd == 5


def test_fused_adam_loop_does_not_accumulate_the_layernorm_grad():
    import vit2spn
    w = _weights()
    B = 4
    x, mask = _images(B, seed=20).to(DEV), _mask(B, seed=21).to(DEV)
    m = _model(w, "bf16")
    opt = vit2spn.FusedAdam(m.parameters(), lr=1e-4)
    for _ in range(3):
        opt.zero_grad()
        assert m.vit.layernorm.weight.grad is None and m.decoder[0].weight.grad is None
        m(x, bool_masked_pos=mask).loss.backward()
        g = m.vit.layernorm.weight.grad
        assert g is not None and torch.isfinite(g).all().item()
        opt.step()
    m.zero_grad(set_to_none=True)
    m(x, bool_masked_pos=mask).loss.backward()
    g_fresh = m.vit.layernorm.weight.grad.clone()
    m(x, bool_masked_pos=mask).loss.backward()
    _flag_clear()
    assert _rel(m.vit.layernorm.weight.grad, 2 * g_fresh) <= 1e-3     # accumulation without zero_grad is torch's


def test_reconstruction_is_not_differentiable():
    w = _weights()
    m = _model(w, "bf16")
    x, mask = _images(2, seed=22).to(DEV), _mask(2, seed=23).to(DEV)
    out = m(x, bool_masked_pos=mask)
    with pytest.raises(RuntimeError, match="not differentiable"):
        (out.loss + out.reconstruction.sum()).backward()
    with torch.no_grad():
        out = m(x, bool_masked_pos=mask)
    assert out.loss is not None and out.reconstruction.shape == (2, 3, 224, 224)
    _flag_clear()
