"""GPU: ViTModel(x, output_hidden_states=True, output_attentions=True) — the 13 hidden states and 12 attention
probabilities against the oracle (fp32 check mode; bf16 / fp16 against the oracle's rounding model), gradients into
intermediate hidden states, the probabilities operator, and the no-request path launching what it launched before.

Measured errors go to $V2S_OUTPUTS_REPORT (JSON) when set."""
import json
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import vit_outputs_oracle as vo  # noqa: E402  (helper module, not a test)

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
_REPORT = {}


def _report(key, value):
    _REPORT[key] = value
    path = os.environ.get("V2S_OUTPUTS_REPORT")
    if path:
        with open(path, "w") as f:
            json.dump(_REPORT, f, indent=1, sort_keys=True)


def _state(seed=11):
    from oracle import vit2spn_oracle as orc
    return orc.sub_state(orc.init_state(seed, 0.01), "online_network_1")


def _model(p, mode):
    import vit2spn
    m = vit2spn.ViTModel()
    m.load_state_dict(p, strict=True)
    m.to(DEV)
    m.compute_mode = mode
    return m


def _images(B, seed=0):
    from oracle import vit2spn_oracle as orc
    return orc.preprocess_u8(orc.synthetic_octmnist_u8(B, seed))


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def _debug_flag_clear():
    from vit2spn import _lib
    torch.cuda.synchronize()
    assert _lib.lib.v2s_debug_flag() == 0


# ---- 3: fp32 check mode, odd batch --------------------------------------------------------------------------------
def test_fp32_outputs_match_oracle():
    from oracle import vit2spn_oracle as orc
    p = _state()
    x = _images(3)
    m = _model(p, "fp32")
    with torch.no_grad():
        out = m(x.to(DEV), output_hidden_states=True, output_attentions=True)
        plain = m(x.to(DEV))
        hs, attn = vo.backbone_outputs(p, x)
    _debug_flag_clear()
    assert len(out.hidden_states) == 13 and len(out.attentions) == 12
    err_h = max((a.cpu() - b).abs().max().item() for a, b in zip(out.hidden_states, hs))
    err_a = max((a.cpu() - b).abs().max().item() for a, b in zip(out.attentions, attn))
    err_sum = max((a.sum(-1) - 1).abs().max().item() for a in out.attentions)
    _report("fp32_B3", {"hidden_maxabs": err_h, "attn_maxabs": err_a, "row_sum_maxabs": err_sum})
    assert err_h <= 5e-4 and err_a <= 1e-5 and err_sum <= 1e-5, (err_h, err_a, err_sum)
    assert all(a.dtype == torch.float32 and a.shape == (3, 3, 197, 197) for a in out.attentions)
    assert torch.equal(out.hidden_states[-1], plain.hidden_states[-1])
    assert out.hidden_states[-1] is out.hidden_states[12]
    assert torch.equal(out.last_hidden_state, plain.last_hidden_state)


# ---- 4: bf16 / fp16 against the rounding model ------------------------------------------------------------------
# Gates: about 3x the largest error measured on a B200 (B = 1 and 128): hidden-state rel-L2 1.34e-3 (bf16) / 1.74e-4
# (fp16), attention max-abs 1.39e-5 / 2.20e-6, row sums 1.2e-6 off 1.  The images of a batch are independent, so the
# oracle checks three of the 128.
GATE_16 = {"bf16": {"hidden_rel": 4e-3, "attn_maxabs": 5e-5}, "fp16": {"hidden_rel": 6e-4, "attn_maxabs": 1e-5}}


@pytest.mark.parametrize("mode,dtype", [("bf16", torch.bfloat16), ("fp16", torch.float16)])
@pytest.mark.parametrize("B", [1, 128])
def test_16bit_outputs_match_rounding_model(mode, dtype, B):
    from oracle import vit2spn_oracle as orc
    p = _state()
    x = _images(B, seed=1)
    m = _model(p, mode)
    with torch.no_grad():
        out = m(x.to(DEV), output_hidden_states=True, output_attentions=True)
        plain = m(x.to(DEV))
    _debug_flag_clear()
    rows = sorted({0, B // 2, B - 1})
    with torch.no_grad(), orc.rounding("all", dtype):
        hs, attn = vo.backbone_outputs(p, x[rows])
    err_h = max(_rel(a[rows].cpu(), b) for a, b in zip(out.hidden_states, hs))
    err_a = max((a[rows].cpu() - b).abs().max().item() for a, b in zip(out.attentions, attn))
    err_sum = max((a.sum(-1) - 1).abs().max().item() for a in out.attentions)
    _report(f"{mode}_B{B}", {"hidden_rel_l2": err_h, "attn_maxabs": err_a, "row_sum_maxabs": err_sum})
    assert err_h <= GATE_16[mode]["hidden_rel"] and err_a <= GATE_16[mode]["attn_maxabs"], (err_h, err_a)
    assert err_sum <= 1e-5, err_sum
    assert torch.equal(out.hidden_states[-1], plain.hidden_states[-1])


# ---- 5: gradients into intermediate hidden states ---------------------------------------------------------------
def _weights(B, seed=5):
    g = torch.Generator().manual_seed(seed)
    return {k: torch.randn(B, 197, 192, generator=g) for k in (2, 7, 12)}, torch.randn(B, 192, generator=g)


def _oracle_grads(p, x, loss_fn, rounding=None):
    from oracle import vit2spn_oracle as orc
    leaves = {k: v.detach().clone().requires_grad_(k not in ("layernorm.weight", "layernorm.bias")
                                                     and not k.startswith("pooler.")) for k, v in p.items()}
    ctx = orc.rounding("all", rounding) if rounding is not None else torch.enable_grad()
    with ctx:
        hs, _ = vo.backbone_outputs(leaves, x)
        loss = loss_fn(hs)
    names = [k for k, v in leaves.items() if v.requires_grad]
    grads = torch.autograd.grad(loss, [leaves[k] for k in names], allow_unused=True)
    return {k: g if g is not None else torch.zeros_like(leaves[k]) for k, g in zip(names, grads)}


def _grad_rel(model, ref):
    num = den = 0.0
    for n, prm in model.named_parameters():
        if n in ref:
            g = prm.grad.detach().cpu().double() if prm.grad is not None else torch.zeros_like(ref[n]).double()
            num += float(((g - ref[n].double()) ** 2).sum())
            den += float((ref[n].double() ** 2).sum())
    return (num / den) ** 0.5


@pytest.mark.parametrize("mode,gate", [("fp32", 1e-4), ("bf16", 2e-2)])
def test_gradients_through_intermediate_hidden_states(mode, gate):
    p = _state()
    B = 3
    x = _images(B, seed=2)
    w, wf = _weights(B)

    def loss_fn(hs):
        return sum((hs[k] * w[k].to(hs[k].device)).sum() for k in (2, 7)) + (hs[12].mean(1) * wf.to(hs[12].device)).sum()

    ref = _oracle_grads(p, x, loss_fn, torch.bfloat16 if mode == "bf16" else None)
    m = _model(p, mode)
    out = m(x.to(DEV), output_hidden_states=True, output_attentions=True)
    loss_fn(out.hidden_states).backward()
    _debug_flag_clear()
    rel = _grad_rel(m, ref)
    _report(f"grad_{mode}", rel)
    assert rel <= gate, rel


def test_gradient_from_one_intermediate_state_skips_the_blocks_above():
    p = _state()
    B = 2
    x = _images(B, seed=4)
    w, _ = _weights(B)

    def loss_fn(hs):
        return (hs[4] * w[2].to(hs[4].device)).sum()

    ref = _oracle_grads(p, x, loss_fn)
    m = _model(p, "fp32")
    loss_fn(m(x.to(DEV), output_hidden_states=True).hidden_states).backward()
    _debug_flag_clear()
    assert _grad_rel(m, ref) <= 1e-4
    for n, prm in m.named_parameters():
        if n.startswith("encoder.layer."):
            l = int(n.split(".")[2])
            if l >= 4:
                assert prm.grad is None or not prm.grad.any(), n
            else:
                assert prm.grad.abs().sum() > 0, n


def test_backward_with_other_hidden_tensors_than_the_forward_is_refused():
    import ctypes as C
    from vit2spn import _lib, modules
    m = _model(_state(), "bf16")
    B = 2
    x = _images(B).to(DEV)
    hidden = [torch.empty(B, 197, 192, device=DEV) for _ in range(13)]
    o = _lib.GroupOutputs()
    for i, t in enumerate(hidden):
        o.hidden[i] = t.data_ptr()
    ws = modules._new_workspace(DEV, B, _lib.MODE_BF16, 1, 1)
    g = modules._group(m._store, _lib.MODE_BF16, x, 0)
    with torch.cuda.device(DEV):
        modules._run_forward([g], B, _lib.MODE_BF16, ws, [o])
        dh = torch.ones(B, 197, 192, device=DEV)
        gb = modules._group(m._store, _lib.MODE_BF16, x, 0, grads=m._store.grads(), dhidden=dh)
        with pytest.raises(RuntimeError, match="differs from the forward"):
            modules._run_backward([gb], B, _lib.MODE_BF16, ws)          # no hidden[] this time
        o2 = _lib.GroupOutputs()
        for i, t in enumerate(hidden):
            o2.hidden[i] = t.data_ptr()
        modules._run_backward([gb], B, _lib.MODE_BF16, ws, [o2])     # the same tensors: accepted
    _debug_flag_clear()


# ---- 6: the probabilities operator ------------------------------------------------------------------------------
@pytest.mark.parametrize("batch,scale", [(1, 1.0), (3, 1.0), (5, 4.0), (64, 0.5)])
@pytest.mark.parametrize("variant", [0, 1, 2, 3])    # bit 0: SIMT kernels instead of tensor-core; bit 1: fp16 tensors
def test_attention_probabilities_operator(batch, scale, variant):
    from vit2spn import _lib
    _lib.init_device(0)
    g = torch.Generator(device=DEV).manual_seed(batch)
    lp = torch.float16 if variant & 2 else torch.bfloat16
    qkv = (torch.randn(batch, 197, 576, device=DEV, generator=g) * scale).to(lp)
    ctx = torch.empty(batch, 197, 192, device=DEV, dtype=lp)
    lse = torch.full((batch, 3, 197), float("nan"), device=DEV)
    _lib.check(_lib.lib.v2s_test_attention(0, _lib.ptr(qkv), _lib.ptr(ctx), _lib.ptr(lse), None, None, batch, variant,
                                           _lib.stream_ptr()), "attention fwd")
    probs = torch.full((batch, 3, 197, 197), float("nan"), device=DEV)
    _lib.check(_lib.lib.v2s_test_attention(2, _lib.ptr(qkv), _lib.ptr(probs), _lib.ptr(lse), None, None, batch, variant,
                                           _lib.stream_ptr()), "attention probabilities")
    torch.cuda.synchronize()
    assert _lib.lib.v2s_debug_flag() == 0
    q, k, _ = [t.view(batch, 197, 3, 64).transpose(1, 2) for t in qkv.double().split(192, dim=-1)]
    ref = torch.softmax((q @ k.transpose(-1, -2)) * 0.125, dim=-1)
    err = (probs.double() - ref).abs().max().item()
    err_sum = (probs.double().sum(-1) - 1).abs().max().item()
    _report(f"op_b{batch}_s{scale}_v{variant}", {"maxabs": err, "row_sum": err_sum})
    assert torch.isfinite(probs).all()
    assert err <= 1e-5 and err_sum <= 2e-5, (err, err_sum)


# ---- 7: training with output_attentions=True ----------------------------------------------------------------------
def test_attentions_are_not_differentiable():
    m = _model(_state(), "bf16")
    x = _images(2).to(DEV)
    out = m(x, output_hidden_states=True, output_attentions=True)
    (out.hidden_states[5].square().mean() + out.hidden_states[-1].mean()).backward()
    assert m.encoder.layer[0].attention.attention.query.weight.grad.abs().sum() > 0
    out = m(x, output_attentions=True)
    with pytest.raises(RuntimeError, match="not differentiable"):
        (out.attentions[3].sum() + out.hidden_states[-1].sum()).backward()
    out = m(x, output_attentions=True)
    out.hidden_states[-1].sum().backward()                 # attentions requested but unused: trains as before
    _debug_flag_clear()


# ---- 8: nothing requested -> the kernels of the previous release --------------------------------------------------
# v2s_launch_count() of one forward + backward with no per-layer output requested, as the release before the per-layer
# outputs launched it (bf16).
PARENT_LAUNCHES = {"vit": 155, "dual": 363}


def _count_launches():
    import vit2spn
    from vit2spn import _lib
    from oracle import vit2spn_oracle as orc
    x = _images(4).to(DEV)
    m = _model(_state(), "bf16")
    m(x).hidden_states[-1].mean().backward()                # warm-up (the first call sets up kernel attributes)
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
    torch.cuda.synchronize()
    return vit, dual


def test_launch_count_unchanged_without_outputs():
    if os.environ.get("V2S_GEMM_DEBUG"):
        pytest.skip("launch counts are pinned for the uninstrumented kernels")
    vit, dual = _count_launches()
    _report("launches", {"vit": vit, "dual": dual})
    assert vit == PARENT_LAUNCHES["vit"], vit
    assert dual == PARENT_LAUNCHES["dual"], dual
