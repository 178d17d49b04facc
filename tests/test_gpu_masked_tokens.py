"""GPU: masked patch tokens (``ViTModel(use_mask_token=True)``, ``forward(..., bool_masked_pos=...)``).  The fp32 check
mode through the whole backbone against ``masked_tokens_oracle`` (hidden states, final-LayerNorm features, attentions,
every weight gradient, d mask_token, the pixel gradient); bf16 / fp16 against the oracle's rounding model and the fp32
oracle; an all-False mask against no mask; bit-reproducibility under the deterministic flag; a frozen backbone; retained
attention gradients; a SimMIM step at B=128; launch counts; the checks on the mask and its forward / backward pairing.

Measured errors go to $V2S_MASKED_TOKENS_REPORT (JSON) when set."""
import json
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import masked_tokens_oracle as mo  # noqa: E402  (helper module, not a test)

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
_REPORT = {}


def _report(key, value):
    _REPORT[key] = value
    path = os.environ.get("V2S_MASKED_TOKENS_REPORT")
    if path:
        with open(path, "w") as f:
            json.dump(_REPORT, f, indent=1, sort_keys=True)


def _state(seed=11):
    from oracle import vit2spn_oracle as orc
    return orc.sub_state(orc.init_state(seed, 0.01), "online_network_1")


def _token(seed=12):
    return 0.02 * torch.randn(192, generator=torch.Generator().manual_seed(seed))


def _model(p, mode, token, frozen=False):
    import vit2spn
    m = vit2spn.ViTModel(use_mask_token=True)
    m.load_state_dict({**p, "embeddings.mask_token": token.view(1, 1, 192)}, strict=True)
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


def _masks(B, kind, seed=2):
    """per-image masks of different density; 'edge': image 0 fully masked, image 1 not at all"""
    if kind == "all":
        return torch.ones(B, 196, dtype=torch.bool)
    if kind == "none":
        return torch.zeros(B, 196, dtype=torch.bool)
    g = torch.Generator().manual_seed(seed)
    frac = torch.linspace(0.15, 0.75, B).unsqueeze(1)
    m = torch.rand(B, 196, generator=g) < frac
    if kind == "edge":
        m[0] = True
        m[1] = False
    return m


def _rel(a, b):
    return ((a.double().cpu() - b.double().cpu()).norm() / b.double().cpu().norm().clamp_min(1e-30)).item()


def _flag_clear():
    from vit2spn import _lib
    torch.cuda.synchronize()
    assert _lib.lib.v2s_debug_flag() == 0


def _active_names(p):
    return [k for k in p if not k.startswith(("pooler.", "layernorm."))]


def _run(m, x, mask, up, attn=False, retain=()):
    xd = x.to(DEV).requires_grad_(True)
    out = m(xd, output_hidden_states=True, output_attentions=attn, bool_masked_pos=mask.to(DEV))
    for l in retain:
        out.attentions[l].retain_grad()
    (out.hidden_states[-1] * up.to(DEV)).sum().backward()
    return out, xd.grad


def _weight_grad_rel(m, ref):
    got = dict(m.named_parameters())
    num = sum(float(((got[k].grad.double().cpu() - g.double()) ** 2).sum()) for k, g in ref.items())
    den = sum(float((g.double() ** 2).sum()) for g in ref.values())
    return (num / den) ** 0.5


# ---- fp32 check mode against the oracle ----------------------------------------------------------------------------
@pytest.mark.parametrize("B,kind", [(1, "rand"), (3, "rand"), (5, "edge"), (2, "all"), (2, "none")])
def test_fp32_masked_backbone_matches_oracle(B, kind):
    p, token = _state(), _token()
    x, up, mask = _images(B, seed=B), _upstream(B, seed=B + 1), _masks(B, kind, seed=B + 2)
    m = _model(p, "fp32", token)
    out, dx = _run(m, x, mask, up, attn=True)
    _flag_clear()
    hs, probs = mo.backbone_outputs(p, x, mask, token)
    names = _active_names(p)
    _, rdx, rtok, rgrads = mo.hidden_and_grads(p, x, mask, token, up, names)
    feat = torch.nn.functional.layer_norm(hs[-1], (192,), p["layernorm.weight"], p["layernorm.bias"], 1e-12)
    rel = {
        "hidden": max(_rel(a, b) for a, b in zip(out.hidden_states, hs)),
        "features": _rel(out.last_hidden_state.detach(), feat),
        "attentions": max(_rel(a, b) for a, b in zip(out.attentions, probs)),
        "weight_grads": _weight_grad_rel(m, rgrads),
        "patch_weight": _rel(m.embeddings.patch_embeddings.projection.weight.grad, rgrads[names[2]]),
        "patch_bias": _rel(m.embeddings.patch_embeddings.projection.bias.grad, rgrads[names[3]]),
        "pos": _rel(m.embeddings.position_embeddings.grad, rgrads["embeddings.position_embeddings"]),
        "pixels": _rel(dx, rdx),
    }
    if kind != "none":
        rel["mask_token"] = _rel(m.embeddings.mask_token.grad.view(192), rtok)
    else:
        assert torch.count_nonzero(m.embeddings.mask_token.grad) == 0
    _report(f"fp32_B{B}_{kind}", rel)
    assert max(rel.values()) <= 1e-5, rel
    pm = mask.reshape(B, 14, 14).repeat_interleave(16, 1).repeat_interleave(16, 2).unsqueeze(1).expand(B, 3, 224, 224)
    assert torch.count_nonzero(dx.cpu()[pm]) == 0
    if kind == "all":
        assert torch.count_nonzero(m.embeddings.patch_embeddings.projection.weight.grad) == 0
        assert torch.count_nonzero(m.embeddings.patch_embeddings.projection.bias.grad) == 0


# ---- 16-bit modes ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode,dtype", [("bf16", torch.bfloat16), ("fp16", torch.float16)])
def test_16bit_masked_backbone_matches_oracle(mode, dtype):
    from oracle import vit2spn_oracle as orc
    p, token = _state(), _token()
    B = 4
    x, up, mask = _images(B, seed=20), _upstream(B, seed=21), _masks(B, "edge", seed=22)
    m = _model(p, mode, token)
    out, dx = _run(m, x, mask, up)
    _flag_clear()
    names = _active_names(p)
    h, rdx, rtok, rgrads = mo.hidden_and_grads(p, x, mask, token, up, names)
    with orc.rounding("all", dtype):
        hr, rdx_r, rtok_r, rgrads_r = mo.hidden_and_grads(p, x, mask, token, up, names)
    loss, loss_r = out.hidden_states[-1].detach().cpu().abs().mean(), hr.abs().mean()      # a forward-only "loss"
    rel = {"loss_vs_rounding_model": abs(loss.item() - loss_r.item()) / abs(loss_r.item()),
           "hidden_vs_rounding_model": _rel(out.hidden_states[-1], hr),
           "weight_grads_vs_rounding_model": _weight_grad_rel(m, rgrads_r),
           "mask_token_vs_rounding_model": _rel(m.embeddings.mask_token.grad.view(192), rtok_r),
           "pixels_vs_rounding_model": _rel(dx, rdx_r),
           "weight_grads_vs_fp32_oracle": _weight_grad_rel(m, rgrads),
           "mask_token_vs_fp32_oracle": _rel(m.embeddings.mask_token.grad.view(192), rtok),
           "pixels_vs_fp32_oracle": _rel(dx, rdx)}
    _report(f"{mode}_B4", rel)
    assert rel["loss_vs_rounding_model"] <= 1e-3, rel
    assert max(v for k, v in rel.items() if k.startswith(("weight", "mask", "pixels"))) <= 2e-2, rel
    pm = mask.reshape(B, 14, 14).repeat_interleave(16, 1).repeat_interleave(16, 2).unsqueeze(1).expand(B, 3, 224, 224)
    assert torch.count_nonzero(dx.cpu()[pm]) == 0


# ---- all-False mask, determinism ------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "bf16", "fp16"])
def test_all_false_mask_is_bit_identical_to_no_mask(mode):
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        p, token = _state(), _token()
        B = 8
        x, up = _images(B, seed=30).to(DEV), _upstream(B, seed=31).to(DEV)
        m = _model(p, mode, token)
        runs = []
        for mask in (None, torch.zeros(B, 196, dtype=torch.bool, device=DEV)):
            m.zero_grad(set_to_none=True)
            xd = x.clone().requires_grad_(True)
            out = m(xd, output_hidden_states=True, output_attentions=True, bool_masked_pos=mask)
            (out.hidden_states[-1] * up).sum().backward()
            runs.append(([h.detach() for h in out.hidden_states], [a for a in out.attentions], xd.grad,
                         {n: q.grad.clone() for n, q in m.named_parameters()
                          if q.grad is not None and n != "embeddings.mask_token"}))
        _flag_clear()
        (h0, a0, x0, g0), (h1, a1, x1, g1) = runs
        assert all(torch.equal(a, b) for a, b in zip(h0, h1))
        assert all(torch.equal(a, b) for a, b in zip(a0, a1))
        assert torch.equal(x0, x1)
        assert g0.keys() == g1.keys()
        bad = [n for n in g0 if not torch.equal(g0[n], g1[n])]
        assert not bad, bad[:8]
        assert torch.count_nonzero(m.embeddings.mask_token.grad) == 0
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_masked_runs_are_bit_identical_under_deterministic_flag(mode):
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        p, token = _state(), _token()
        B = 16
        x, up, mask = _images(B, seed=40), _upstream(B, seed=41), _masks(B, "edge", seed=42)
        m = _model(p, mode, token)
        runs = []
        for _ in range(2):
            m.zero_grad(set_to_none=True)
            _, dx = _run(m, x, mask, up)
            runs.append((dx, {n: q.grad.clone() for n, q in m.named_parameters() if q.grad is not None}))
        _flag_clear()
        assert "embeddings.mask_token" in runs[0][1]
        assert torch.equal(runs[0][0], runs[1][0])
        bad = [n for n in runs[0][1] if not torch.equal(runs[0][1][n], runs[1][1][n])]
        assert not bad, bad[:8]
        # the fixed-order sums also split the masked rows correctly: d b_pe, d mask_token and the rest against the oracle
        from oracle import vit2spn_oracle as orc
        names = _active_names(p)
        ctx = orc.rounding("all", torch.bfloat16) if mode == "bf16" else torch.enable_grad()
        with ctx:
            _, rdx, rtok, rgrads = mo.hidden_and_grads(p, x, mask, token, up, names)
        g = runs[0][1]
        rel = {"patch_bias": _rel(g["embeddings.patch_embeddings.projection.bias"],
                                  rgrads["embeddings.patch_embeddings.projection.bias"]),
               "patch_weight": _rel(g["embeddings.patch_embeddings.projection.weight"],
                                    rgrads["embeddings.patch_embeddings.projection.weight"]),
               "pos": _rel(g["embeddings.position_embeddings"], rgrads["embeddings.position_embeddings"]),
               "mask_token": _rel(g["embeddings.mask_token"].view(192), rtok),
               "weight_grads": _weight_grad_rel(m, rgrads),
               "pixels": _rel(runs[0][0], rdx)}
        _report(f"deterministic_{mode}_B16", rel)
        assert max(rel.values()) <= (2e-2 if mode == "bf16" else 1e-5), rel
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


# ---- frozen backbone, retained attentions ----------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("token_trainable", [False, True])
def test_frozen_backbone_pixel_gradient(mode, token_trainable):
    from oracle import vit2spn_oracle as orc
    p, token = _state(), _token()
    B = 3
    x, up, mask = _images(B, seed=50), _upstream(B, seed=51), _masks(B, "rand", seed=52)
    m = _model(p, mode, token, frozen=True)
    m.embeddings.mask_token.requires_grad_(token_trainable)
    _, dx = _run(m, x, mask, up)
    _flag_clear()
    ctx = orc.rounding("all", torch.bfloat16) if mode == "bf16" else torch.enable_grad()
    with ctx:
        _, rdx, rtok, _ = mo.hidden_and_grads(p, x, mask, token, up)
    tol = 2e-2 if mode == "bf16" else 1e-5
    rel = {"pixels": _rel(dx, rdx)}
    with_grad = [n for n, q in m.named_parameters() if q.grad is not None]
    if token_trainable:
        assert with_grad == ["embeddings.mask_token"]
        rel["mask_token"] = _rel(m.embeddings.mask_token.grad.view(192), rtok)
    else:
        assert with_grad == []
    _report(f"frozen_{mode}_token{int(token_trainable)}", rel)
    assert max(rel.values()) <= tol, rel


def test_masked_forward_with_retained_attention_gradients():
    import attn_grad_oracle as ag
    from oracle import vit2spn_oracle as orc
    p, token = _state(), _token()
    B = 2
    x, up, mask = _images(B, seed=60), _upstream(B, seed=61), _masks(B, "rand", seed=62)
    m = _model(p, "fp32", token)
    out, _ = _run(m, x, mask, up, attn=True, retain=(0, 5, 11))
    _flag_clear()
    # the oracle's blocks with explicit probabilities, from the masked embedding output
    with torch.enable_grad():
        hs, probs = [mo.patch_embed(p, x, mask, token).requires_grad_(True)], []
        for l in range(orc.LAYERS):
            h, A = ag.block(p, l, hs[-1])
            hs.append(h)
            probs.append(A)
        grads = torch.autograd.grad((hs[-1] * up).sum(), probs)
    assert [a.grad is not None for a in out.attentions] == [l in (0, 5, 11) for l in range(12)]
    rels = [_rel(out.attentions[l].grad, grads[l]) for l in (0, 5, 11)]
    _report("retained_attn_fp32", rels)
    assert max(rels) <= 1e-4, rels


# ---- SimMIM step at B=128 ------------------------------------------------------------------------------------------
def test_simmim_step_bf16_b128():
    import vit2spn
    from oracle import vit2spn_oracle as orc
    from test_masked_tokens_cpu import simmim_loss
    p, token = _state(), _token()
    B = 128
    x = _images(B, seed=70)
    mask = torch.rand(B, 196, generator=torch.Generator().manual_seed(71)) < 0.4
    torch.manual_seed(72)
    conv0 = torch.nn.Conv2d(192, 768, kernel_size=1)
    xd, md = x.to(DEV), mask.to(DEV)
    # one SimMIM step: torch decoder, FusedAdam over the backbone, its mask token and the decoder
    m = _model(p, "bf16", token)
    conv = torch.nn.Conv2d(192, 768, kernel_size=1).to(DEV)
    conv.load_state_dict(conv0.state_dict())
    opt = vit2spn.FusedAdam(list(m.parameters()) + list(conv.parameters()), lr=1e-3)
    opt.zero_grad()
    loss = simmim_loss(m(xd, bool_masked_pos=md).last_hidden_state, conv, xd, md)
    loss.backward()
    t0 = m.embeddings.mask_token.detach().clone()
    opt.step()
    _flag_clear()
    assert torch.isfinite(loss).item()
    assert all(torch.isfinite(q).all().item() for q in m.parameters())
    assert not torch.equal(t0, m.embeddings.mask_token.detach())        # updated, outside the flat store
    # the same step's loss and d mask_token on 3 rows against the oracle's rounding model of the bf16 mode
    rows = [0, 57, 127]
    m3 = _model(p, "bf16", token)
    conv3 = torch.nn.Conv2d(192, 768, kernel_size=1).to(DEV)
    conv3.load_state_dict(conv0.state_dict())
    loss3 = simmim_loss(m3(xd[rows], bool_masked_pos=md[rows]).last_hidden_state, conv3, xd[rows], md[rows])
    loss3.backward()
    _flag_clear()
    t = token.clone().requires_grad_(True)
    with orc.rounding("all", torch.bfloat16):
        h = mo.patch_embed(p, x[rows], mask[rows], t)
        for l in range(orc.LAYERS):
            h = orc.vit_layer(p, l, h)
    last = torch.nn.functional.layer_norm(h, (192,), p["layernorm.weight"], p["layernorm.bias"], 1e-12)
    ref = simmim_loss(last, conv0, x[rows], mask[rows])
    ref.backward()
    rel = {"loss_3rows": abs(loss3.item() - ref.item()) / abs(ref.item()),
           "mask_token_3rows": _rel(m3.embeddings.mask_token.grad.view(192), t.grad)}
    _report("simmim_bf16_B128", {**rel, "loss_B128": loss.item()})
    assert rel["loss_3rows"] <= 1e-3 and rel["mask_token_3rows"] <= 2e-2, rel


# ---- launch counts ---------------------------------------------------------------------------------------------------
def _launches(fn):
    from vit2spn import _lib
    fn()                                  # warm-up: kernel attributes, workspace
    torch.cuda.synchronize()
    n0 = _lib.lib.v2s_launch_count()
    fn()
    torch.cuda.synchronize()
    return _lib.lib.v2s_launch_count() - n0


@pytest.mark.parametrize("mode", ["bf16", "fp16"])
def test_masked_launch_count_equals_unmasked(mode):
    p, token = _state(), _token()
    B = 4
    x, up = _images(B, seed=80).to(DEV), _upstream(B, seed=81).to(DEV)
    mask = _masks(B, "rand", seed=82).to(DEV)
    m = _model(p, mode, token)

    def step(mk, want_x):
        m.zero_grad(set_to_none=True)
        xd = x.clone().requires_grad_(want_x)
        (m(xd, bool_masked_pos=mk).hidden_states[-1] * up).sum().backward()

    for want_x in (False, True):
        n_plain, n_masked = _launches(lambda: step(None, want_x)), _launches(lambda: step(mask, want_x))
        _report(f"launches_{mode}_x{int(want_x)}", {"unmasked": n_plain, "masked": n_masked})
        assert n_masked == n_plain, (want_x, n_plain, n_masked)
    _flag_clear()


# ---- argument checks on the GPU --------------------------------------------------------------------------------------
def test_mask_on_cpu_is_refused():
    m = _model(_state(), "bf16", _token())
    x = _images(2, seed=90).to(DEV)
    with pytest.raises(ValueError, match="device"):
        m(x, bool_masked_pos=torch.zeros(2, 196, dtype=torch.bool))


def test_backward_outputs_with_another_mask_or_a_partial_range_are_refused():
    from vit2spn import _lib, modules as M
    p, token = _state(), _token()
    B = 2
    m = _model(p, "bf16", token)
    x = _images(B, seed=91).to(DEV)
    mask = _masks(B, "rand", seed=92).to(DEV).to(torch.uint8)
    other = mask.clone()
    mode = m._mode()
    store = m._store
    ws = M._new_workspace(DEV, B, mode, 1, 1)
    hid = torch.empty(B, 197, 192, device=DEV)
    tok = m.embeddings.mask_token.detach().reshape(192)
    g = M._group(store, mode, x, 0, hidden=hid)

    def outputs(patch_mask, dtok=None):
        o = _lib.GroupOutputs()
        o.mask, o.mask_token = patch_mask.data_ptr(), tok.data_ptr()
        o.dmask_token = dtok.data_ptr() if dtok is not None else None
        return [o]
    M._run_forward([g], B, mode, ws, outputs(mask))
    dh = torch.ones(B, 197, 192, device=DEV)
    gb = M._group(store, mode, x, 0, grads=store.grads(), dhidden=dh)
    with pytest.raises(RuntimeError, match="patch mask"):
        M._run_backward([gb], B, mode, ws, outputs(other))
    with pytest.raises(RuntimeError, match="patch mask"):
        M._run_backward([gb], B, mode, ws, None, 12, 6)          # a partial range after a masked forward
    with pytest.raises(RuntimeError, match="patch mask"):
        M._run_backward([gb], B, mode, ws)                       # no mask
    with pytest.raises(RuntimeError, match="whole range"):
        M._run_backward([gb], B, mode, ws, outputs(mask), 12, 6)  # the forward's own mask over a partial range
    dtok = torch.zeros(192, device=DEV)
    M._run_backward([gb], B, mode, ws, outputs(mask, dtok))      # the forward's own mask: accepted
    _flag_clear()
    assert torch.count_nonzero(dtok) > 0
