"""GPU: ``vit2spn.ViTForImageClassification`` (classification head on the CUDA path).  The fp32 check mode against
``cls_oracle`` for the three problem types and num_labels 4 and 1000 (logits, loss, classifier / LayerNorm / backbone /
pixel gradients); bf16 and fp16 against its rounding model, the whole model at B=3 and the head at B=128; agreement
with the eager-head recipe on the same backbone; a loss of the user's own on the logits; the linear probe (frozen vit)
and the head's launch counts; saliency on a frozen model; bit-reproducibility; fp16 with a GradScaler; a FusedAdam
fine-tune loop; an out-of-range label.

Measured errors go to $V2S_CLS_REPORT (JSON) when set."""
import json
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import cls_oracle as co  # noqa: E402  (helper module, not a test)

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
_REPORT = {}
_LP = {"bf16": torch.bfloat16, "fp16": torch.float16}
_KINDS = ("single_label_classification", "regression", "multi_label_classification")


def _report(key, value):
    _REPORT[key] = value
    path = os.environ.get("V2S_CLS_REPORT")
    if path:
        with open(path, "w") as f:
            json.dump(_REPORT, f, indent=1, sort_keys=True)


def _weights(n, seed=11):
    from oracle import vit2spn_oracle as orc
    p = orc.sub_state(orc.init_state(seed, 0.01), "online_network_1")
    g = torch.Generator().manual_seed(seed + 100)
    return p, 0.05 * torch.randn(n, 192, generator=g), 0.02 * torch.randn(n, generator=g)


def _model(w, mode, problem_type=None):
    import vit2spn
    p, cw, cb = w
    m = vit2spn.ViTForImageClassification(vit2spn.ViTConfig(num_labels=cw.shape[0], problem_type=problem_type))
    sd = {"vit." + k: v for k, v in p.items() if not k.startswith("pooler.")}
    sd.update({"classifier.weight": cw, "classifier.bias": cb})
    m.load_state_dict(sd, strict=True)
    m.to(DEV)
    m.compute_mode = mode
    return m


def _images(B, seed=0):
    from oracle import vit2spn_oracle as orc
    return orc.preprocess_u8(orc.synthetic_octmnist_u8(B, seed))


def _labels(kind, B, n, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "single_label_classification":
        y = torch.randint(0, n, (B,), generator=g)
        if B > 2:
            y[1] = -100                              # one ignored row
        return y
    if kind == "regression":
        return torch.randn(B, n, generator=g)
    return (torch.rand(B, n, generator=g) < 0.3).float()


def _rel(a, b):
    return ((a.double().cpu() - b.double().cpu()).norm() / b.double().cpu().norm().clamp_min(1e-30)).item()


def _flag_clear():
    from vit2spn import _lib
    torch.cuda.synchronize()
    assert _lib.lib.v2s_debug_flag() == 0


_CHECKED = ("classifier.weight", "classifier.bias", "layernorm.weight", "layernorm.bias",
            "embeddings.patch_embeddings.projection.weight", "encoder.layer.5.intermediate.dense.weight", "pixels")


def _grads(m, dx):
    named = dict(m.named_parameters())
    g = {k: named["vit." + k].grad for k in _CHECKED if "vit." + k in named}
    g.update({"classifier.weight": m.classifier.weight.grad, "classifier.bias": m.classifier.bias.grad, "pixels": dx})
    return g


def _step(m, x, y, want_x=True, scale=1.0, dlogits=None):
    xd = x.detach().to(DEV).clone().requires_grad_(want_x)
    out = m(xd, labels=y.to(DEV) if y is not None else None)
    obj = 0
    if out.loss is not None:
        obj = obj + out.loss * scale
    if dlogits is not None:
        obj = obj + (out.logits * dlogits.to(DEV)).sum() * scale
    obj.backward()
    return out, (xd.grad / scale if xd.grad is not None else None)


def _double(w):
    p, cw, cb = w
    return {k: v.double() for k, v in p.items()}, cw.double(), cb.double()


# ---- fp32 check mode against the float64 oracle ----------------------------------------------------------------------
@pytest.mark.parametrize("n", [4, 1000])
@pytest.mark.parametrize("kind", _KINDS)
def test_fp32_matches_oracle(kind, n):
    w = _weights(n)
    B = 3
    x, y = _images(B, seed=1), _labels(kind, B, n, seed=2)
    m = _model(w, "fp32", problem_type=kind if kind == "regression" else None)   # else inferred from the labels
    out, dx = _step(m, x, y)
    _flag_clear()
    assert m.config.problem_type == kind
    loss, logits, ref = co.model_loss(*_double(w), x.double(), y, m.config.problem_type)
    got = _grads(m, dx)
    rel = {"loss": abs(out.loss.item() - loss.item()) / abs(loss.item()), "logits": _rel(out.logits, logits)}
    rel.update({k: _rel(got[k], ref[k]) for k in _CHECKED})
    _report(f"fp32_{kind}_{n}", rel)
    assert max(rel.values()) <= 1e-5, rel


def test_fp32_custom_loss_on_logits():
    """A user's own loss on the logits (here a fixed cotangent), alone and together with the model's loss."""
    n = 4
    w = _weights(n)
    B = 3
    x, y = _images(B, seed=3), _labels("single_label_classification", B, n, seed=4)
    dl = torch.randn(B, n, generator=torch.Generator().manual_seed(5))
    m = _model(w, "fp32")
    for labels in (None, y):
        m.zero_grad(set_to_none=True)
        out, dx = _step(m, x, labels, dlogits=dl)
        _flag_clear()
        _, _, ref = co.model_loss(*_double(w), x.double(), labels, "single_label_classification", dlogits=dl.double())
        got = _grads(m, dx)
        rel = {k: _rel(got[k], ref[k]) for k in _CHECKED}
        _report(f"fp32_custom_loss_labels_{labels is not None}", rel)
        assert max(rel.values()) <= 1e-5, rel


def test_fp32_all_ignored_batch():
    n = 4
    w = _weights(n)
    x = _images(2, seed=6)
    y = torch.full((2,), -100, dtype=torch.int64)
    m = _model(w, "fp32")
    out, dx = _step(m, x, y)
    _flag_clear()
    ref = torch.nn.functional.cross_entropy(torch.zeros(2, n, requires_grad=True), y, ignore_index=-100)
    assert torch.isnan(out.loss).item() and torch.isnan(ref).item()
    for k, g in _grads(m, dx).items():
        assert g is not None and torch.count_nonzero(g) == 0, k


# ---- 16-bit modes ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["bf16", "fp16"])
def test_16bit_matches_rounding_model_b3(mode):
    from oracle import vit2spn_oracle as orc
    n = 4
    w = _weights(n)
    B = 3
    x, y = _images(B, seed=7), _labels("single_label_classification", B, n, seed=8)
    m = _model(w, mode)
    out, dx = _step(m, x, y)
    _flag_clear()
    with orc.rounding("all", _LP[mode]):
        loss, logits, ref = co.model_loss(*w, x, y, "single_label_classification", lp=_LP[mode])
    got = _grads(m, dx)
    rel = {"loss": abs(out.loss.item() - loss.item()) / abs(loss.item()), "logits": _rel(out.logits, logits)}
    rel.update({k: _rel(got[k], ref[k]) for k in _CHECKED})
    _report(f"{mode}_B3", rel)
    assert rel["loss"] <= 1e-3, rel
    assert max(rel.values()) <= 2e-2, rel


@pytest.mark.parametrize("n", [4, 1000])
@pytest.mark.parametrize("mode", ["bf16", "fp16"])
def test_16bit_head_matches_rounding_model_b128(mode, n):
    """The head at B=128 on the backbone's own hidden_states[12]: loss, logits and every head gradient."""
    w = _weights(n)
    B = 128
    x, y = _images(B, seed=9), _labels("single_label_classification", B, n, seed=10)
    m = _model(w, mode)
    out = m(x.to(DEV), labels=y.to(DEV), output_hidden_states=True)
    h12 = out.hidden_states[-1]
    h12.retain_grad()
    out.loss.backward()
    _flag_clear()
    with torch.enable_grad():
        hh = h12.detach().cpu().requires_grad_(True)
        lw = m.vit.layernorm.weight.detach().cpu().requires_grad_(True)
        lb = m.vit.layernorm.bias.detach().cpu().requires_grad_(True)
        cw, cb = w[1].clone().requires_grad_(True), w[2].clone().requires_grad_(True)
        logits, loss = co.head(hh, lw, lb, cw, cb, y, "single_label_classification", _LP[mode])
        loss.backward()
    rel = {"loss": abs(out.loss.item() - loss.item()) / abs(loss.item()), "logits": _rel(out.logits, logits.detach()),
           "hidden12": _rel(h12.grad, hh.grad), "layernorm.weight": _rel(m.vit.layernorm.weight.grad, lw.grad),
           "layernorm.bias": _rel(m.vit.layernorm.bias.grad, lb.grad),
           "classifier.weight": _rel(m.classifier.weight.grad, cw.grad),
           "classifier.bias": _rel(m.classifier.bias.grad, cb.grad)}
    _report(f"{mode}_head_B128_{n}", rel)
    assert rel["loss"] <= 1e-3, rel
    assert max(rel.values()) <= 2e-2, rel
    assert torch.count_nonzero(h12.grad[:, 1:]) == 0


def test_agrees_with_the_eager_head_recipe():
    """The same CUDA backbone with the eager head users wrote before: last_hidden_state[:, 0] -> Linear -> CE."""
    n = 4
    w = _weights(n)
    B = 16
    x, y = _images(B, seed=11).to(DEV), _labels("single_label_classification", B, n, seed=12).to(DEV)
    m = _model(w, "bf16")
    out, dx = _step(m, x, y)
    ours = {k: v.clone() for k, v in _grads(m, dx).items()}
    logits = out.logits.detach().clone()
    m.zero_grad(set_to_none=True)
    xd = x.clone().requires_grad_(True)
    z = m.classifier(m.vit(xd).last_hidden_state[:, 0])
    ref = torch.nn.functional.cross_entropy(z, y)
    ref.backward()
    _flag_clear()
    theirs = _grads(m, xd.grad)
    rel = {"loss": abs(out.loss.item() - ref.item()) / abs(ref.item()), "logits": _rel(logits, z.detach())}
    rel.update({k: _rel(ours[k], theirs[k]) for k in _CHECKED})
    _report("eager_head_bf16_B16", rel)
    assert rel["loss"] <= 1e-2, rel
    assert max(rel.values()) <= 3e-2, rel


# ---- linear probe, launch counts, saliency ---------------------------------------------------------------------------
def _count(fn):
    from vit2spn import _lib
    fn()
    torch.cuda.synchronize()
    n0 = _lib.lib.v2s_launch_count()
    r = fn()
    torch.cuda.synchronize()
    return _lib.lib.v2s_launch_count() - n0, r


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_head_launch_counts(mode):
    """The head adds 5 kernels to a forward with labels in the 16-bit modes (W_cls cast, final LayerNorm, logit GEMM,
    loss rows, loss finish; 4 in fp32, which has no cast), one fewer without labels.  A trained backward is 4 (logit
    gradient, wgrad with the bias row sums, dgrad, LayerNorm backward; fp32 adds the bias column sums), a linear probe's
    is 2 (logit gradient, wgrad; fp32: 3)."""
    from vit2spn import modules
    n = 4
    m = _model(_weights(n), mode)
    B = 4
    y = _labels("single_label_classification", B, n, seed=13).to(DEV)
    hidden = torch.randn(B, 197, 192, device=DEV, requires_grad=True)
    ln, fc = m.vit.layernorm, m.classifier
    ce = 1

    def fwd(labels, h=hidden):
        return modules._ClsHeadFn.apply(h, ln.weight, ln.bias, fc.weight, fc.bias, m, ce if labels is not None else 0,
                                        labels, True)
    n_fwd, _ = _count(lambda: fwd(y))
    n_fwd_plain, _ = _count(lambda: fwd(None))
    n_all, _ = _count(lambda: fwd(y)[1].backward())
    ln.requires_grad_(False)
    n_probe, _ = _count(lambda: fwd(y, hidden.detach())[1].backward())
    ln.requires_grad_(True)
    _flag_clear()
    counts = {"forward": n_fwd, "forward_no_labels": n_fwd_plain, "fwd_bwd": n_all, "fwd_bwd_probe": n_probe}
    _report(f"launches_{mode}", counts)
    lp = mode != "fp32"
    assert (n_fwd, n_fwd_plain) == ((5, 4) if lp else (4, 3)), counts
    assert n_all - n_fwd == (4 if lp else 5) and n_probe - n_fwd == (2 if lp else 3), counts


@pytest.mark.parametrize("mode", ["fp32", "bf16", "fp16"])
def test_linear_probe_runs_no_backbone_backward(mode):
    from vit2spn import _lib
    n = 4
    w = _weights(n)
    B = 3
    x, y = _images(B, seed=14).to(DEV), _labels("single_label_classification", B, n, seed=15).to(DEV)
    m = _model(w, mode)
    _step(m, x, y, want_x=False)
    full = {k: m.classifier.get_parameter(k).grad.clone() for k in ("weight", "bias")}
    m.zero_grad(set_to_none=True)
    m.vit.requires_grad_(False)
    n_fwd, _ = _count(lambda: m(x, labels=y))
    _lib.prof_enable(True)
    n_step, _ = _count(lambda: m(x, labels=y).loss.backward())      # twice: the gradients accumulate
    rep = _lib.prof_report()
    _lib.prof_enable(False)
    _flag_clear()
    _report(f"probe_{mode}", {"forward": n_fwd, "step": n_step})
    assert n_step - n_fwd == (3 if mode == "fp32" else 2), (n_fwd, n_step)
    assert rep.get("gemm_wgrad", (0,))[0] == 0 and rep.get("attn_bwd", (0,))[0] == 0 and rep["cls_bwd"][0] == 2, rep
    assert [k for k, q in m.named_parameters() if q.grad is not None] == ["classifier.weight", "classifier.bias"]
    tol = 1e-5 if mode == "fp32" else 1e-3
    for k in ("weight", "bias"):        # the second step accumulated onto the first: twice one step's gradient
        assert _rel(m.classifier.get_parameter(k).grad, 2 * full[k]) <= tol, k
    # a frozen classifier still propagates to the backbone
    m.vit.requires_grad_(True)
    m.classifier.requires_grad_(False)
    m.zero_grad(set_to_none=True)
    _step(m, x, y, want_x=False)
    _flag_clear()
    assert m.classifier.weight.grad is None and m.vit.layernorm.weight.grad is not None
    assert m.vit.encoder.layer[3].output.dense.weight.grad.abs().sum().item() > 0


def test_saliency_on_a_frozen_model():
    n = 4
    w = _weights(n)
    B = 3
    x = _images(B, seed=16)
    m = _model(w, "fp32")
    m.requires_grad_(False)
    xd = x.to(DEV).requires_grad_(True)
    m(xd).logits[:, 2].sum().backward()
    _flag_clear()
    dl = torch.zeros(B, n, dtype=torch.float64)
    dl[:, 2] = 1
    _, _, ref = co.model_loss(*_double(w), x.double(), None, None, dlogits=dl)
    assert _rel(xd.grad, ref["pixels"]) <= 1e-5
    assert all(q.grad is None for q in m.parameters())


# ---- determinism, GradScaler, training loop, bad labels --------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_deterministic_steps_are_bit_identical(mode):
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        n = 1000
        m = _model(_weights(n), mode)
        B = 8
        x, y = _images(B, seed=17), _labels("single_label_classification", B, n, seed=18)
        runs = []
        for _ in range(2):
            m.zero_grad(set_to_none=True)
            out, dx = _step(m, x, y)
            runs.append((out.loss.detach().clone(), out.logits.detach().clone(), dx,
                         {k: q.grad.clone() for k, q in m.named_parameters() if q.grad is not None}))
        _flag_clear()
        (l0, z0, x0, g0), (l1, z1, x1, g1) = runs
        assert torch.equal(l0, l1) and torch.equal(z0, z1) and torch.equal(x0, x1)
        assert "classifier.weight" in g0 and "vit.layernorm.weight" in g0 and g0.keys() == g1.keys()
        bad = [k for k in g0 if not torch.equal(g0[k], g1[k])]
        assert not bad, bad[:8]
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


def test_loss_is_bit_identical_across_runs_and_grids():
    from vit2spn import _lib
    n = 1000
    m = _model(_weights(n), "bf16")
    B = 128
    x, y = _images(B, seed=19).to(DEV), _labels("single_label_classification", B, n, seed=20).to(DEV)
    losses = []
    with torch.no_grad():
        for sms in (0, 37, 0):
            _lib.check(_lib.lib.v2s_set_sm_limit(sms), "set_sm_limit")
            losses.append(m(x, labels=y).loss.clone())
    _lib.check(_lib.lib.v2s_set_sm_limit(0), "set_sm_limit")
    _flag_clear()
    assert all(torch.equal(losses[0], t) for t in losses[1:]), losses


def test_fp16_gradscaler_step():
    import vit2spn
    n = 4
    m = _model(_weights(n), "fp16")
    B = 8
    x, y = _images(B, seed=21).to(DEV), _labels("single_label_classification", B, n, seed=22).to(DEV)
    sc = 2.0 ** 14
    _step(m, x, y, want_x=False, scale=sc)
    plain = {k: v.clone() / sc for k, v in _grads(m, None).items() if k != "pixels"}
    m.zero_grad(set_to_none=True)
    opt = vit2spn.FusedAdam(m.parameters(), lr=1e-4)
    scaler = torch.amp.GradScaler("cuda", init_scale=sc)
    scaler.scale(m(x, labels=y).loss).backward()
    scaled = {k: v.clone() / scaler.get_scale() for k, v in _grads(m, None).items() if k != "pixels"}
    w0 = m.classifier.weight.detach().clone()
    scaler.step(opt)
    scaler.update()
    _flag_clear()
    rel = {k: _rel(scaled[k], plain[k]) for k in plain}
    _report("fp16_gradscaler", rel)
    assert max(rel.values()) <= 1e-3, rel
    assert not torch.equal(w0, m.classifier.weight.detach())
    assert all(torch.isfinite(q).all().item() for q in m.parameters())


def test_fused_adam_finetune_reduces_the_loss():
    import vit2spn
    n = 4
    m = _model(_weights(n), "bf16")
    B = 32
    x = _images(B, seed=23).to(DEV)
    y = torch.arange(B, device=DEV) % n
    opt = vit2spn.FusedAdam(m.parameters(), lr=1e-4)
    losses = []
    for _ in range(40):
        opt.zero_grad()
        loss = m(x, labels=y).loss
        loss.backward()
        opt.step()
        losses.append(loss.item())
    _flag_clear()
    _report("finetune_losses", losses)
    assert losses[-1] < 0.9 * losses[0] and losses[-1] < losses[-10], losses


def test_out_of_range_label_gives_nan_loss():
    n = 4
    m = _model(_weights(n), "bf16")
    x = _images(3, seed=24).to(DEV)
    for bad in (4, -1, 1 << 40):
        y = torch.tensor([0, bad, 2], device=DEV)
        out = m(x, labels=y)
        assert torch.isnan(out.loss).item(), bad
        assert torch.isfinite(out.logits).all().item()
    _flag_clear()
