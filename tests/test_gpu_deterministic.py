"""GPU: the deterministic mode.  With ``torch.use_deterministic_algorithms(True)`` every cross-CTA reduction of the
backward pass sums in a fixed order (v2s_set_deterministic): the split-K weight gradients, the bias / LayerNorm /
embedding column sums.  Results are then bit-identical from run to run, including under an SM
limit and across the range-wise backward of the data-parallel overlap, and the launch sequence is the default one."""
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
LP = {0: torch.bfloat16, 2: torch.float16}      # v2s_test_gemm variant bit 1: fp16 instead of bf16 tensors


@pytest.fixture
def deterministic():
    """torch's flag on for the test; restored (with the library switch and the SM limit) afterwards."""
    from vit2spn import _lib
    _lib.init_device(0)
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    _lib.lib.v2s_set_deterministic(1)       # the operator test calls the library directly; the modules set it themselves
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)
        _lib.lib.v2s_set_deterministic(int(prev))
        _lib.lib.v2s_set_sm_limit(0)
        torch.cuda.synchronize()
        assert _lib.lib.v2s_debug_flag() == 0, "tcgen05 pipeline protocol timeout"


def _set_flag(on):
    torch.use_deterministic_algorithms(on)


def _views(B, seed):
    from oracle import vit2spn_oracle as orc
    x1, x2 = orc.synthetic_views(B, seed=seed)
    return x1.to(DEV), x2.to(DEV)


def _dual(mode, seed=3):
    import vit2spn
    from oracle import vit2spn_oracle as orc
    model = vit2spn.DualStreamNetwork()
    model.load_state_dict(orc.init_state(seed, 0.02), strict=True)
    model.to(DEV).train()
    model.projection_head[2].p = 0.0
    model.compute_mode = mode
    return model


def _grads(model):
    return {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}


def _assert_equal(ga, gb):
    assert ga.keys() == gb.keys()
    bad = [n for n in ga if not torch.equal(ga[n], gb[n])]
    assert not bad, bad[:8]


# ---- 1: the tcgen05 split-K weight gradient ---------------------------------------------------------------------
@pytest.mark.parametrize("m,n,k", [(192, 192, 25216), (192, 768, 9456), (576, 192, 4000), (768, 192, 25216)])
@pytest.mark.parametrize("fmt", [0, 2])
def test_wgrad_split_k_is_bit_identical(deterministic, m, n, k, fmt):
    """v2s_test_gemm which 4 (TN, fp32 += into a nonzero C, with the bias row sums of A += into a nonzero vector):
    bit-identical over repeats and under an SM limit, and within fp32 summation tolerance of an fp64 reference.
    M = 192 / 576 leave partial 128-row tiles.  The scratch follows the outputs in the caller's buffer."""
    from vit2spn import _lib
    g = torch.Generator(device=DEV).manual_seed(m + n + k + fmt)
    a = torch.randn(k, m, device=DEV, generator=g).to(LP[fmt])
    b = torch.randn(k, n, device=DEV, generator=g).to(LP[fmt])
    base = torch.randn(m * n + m, device=DEV, generator=g)
    scratch = 1024 + torch.cuda.get_device_properties(DEV).multi_processor_count * (128 * 192 + 128)

    def run():
        buf = torch.empty(m * n + m + scratch, device=DEV)
        buf[:m * n + m] = base
        _lib.check(_lib.lib.v2s_test_gemm(4, _lib.ptr(a), _lib.ptr(b), _lib.ptr(buf), m, n, k, fmt, _lib.stream_ptr()))
        torch.cuda.synchronize()
        return buf[:m * n + m].clone()

    first = run()
    for _ in range(3):
        assert torch.equal(run(), first)
    try:
        _lib.lib.v2s_set_sm_limit(100)
        assert torch.equal(run(), first)
    finally:
        _lib.lib.v2s_set_sm_limit(0)
    ad, bd, bs = a.cpu().double(), b.cpu().double(), base.cpu().double()
    ref = ad.t() @ bd + bs[:m * n].view(m, n)
    err = (first[:m * n].cpu().double().view(m, n) - ref).abs().max().item()
    assert err <= 2e-5 * ref.abs().max().item() + 1e-3, err
    ref_b = ad.sum(0) + bs[m * n:]
    err_b = (first[m * n:].cpu().double() - ref_b).abs().max().item()
    assert err_b <= 2e-5 * ref_b.abs().max().item() + 1e-3, err_b


# ---- 2: the fused step, all three compute modes ------------------------------------------------------------------
def _steps(mode, n_steps=10, B=32):
    model = _dual(mode)
    scaler = torch.amp.GradScaler("cuda") if mode == "fp16" else None
    losses = []
    for i in range(n_steps):
        x1, x2 = _views(B, 100 + i)
        losses.append(model.ssp_step(x1, x2, accumulation_steps=4, grad_scale=scaler if scaler else 1.0).clone())
    return torch.stack(losses), _grads(model)


@pytest.mark.parametrize("mode", ["bf16", "fp16", "fp32"])
def test_ssp_steps_are_bit_identical(deterministic, mode):
    """Two freshly built models from one seed, 10 accumulated ssp_steps each (fp16 through a GradScaler): equal losses
    and gradients.  The default path's gradients agree with them within its own run-to-run spread (5e-4 rel-L2)."""
    la, ga = _steps(mode)
    lb, gb = _steps(mode)
    assert torch.equal(la, lb)
    _assert_equal(ga, gb)
    _set_flag(False)
    lc, gc = _steps(mode)
    num = sum(float((gc[k].double() - ga[k].double()).square().sum()) for k in ga)
    den = sum(float(ga[k].double().square().sum()) for k in ga)
    assert (num / den) ** 0.5 <= 5e-4, (num / den) ** 0.5
    # per tensor too, so that a wrong fix-up of a small tensor (a bias, a LayerNorm parameter) cannot hide in the total.
    # Each tensor is measured against its own norm, or that of a tensor of its size at the average gradient magnitude
    # when larger: the key biases' gradient is zero in exact arithmetic (softmax ignores a per-query constant), so their
    # computed value is pure rounding noise in either mode.
    rms = (den / sum(ga[k].numel() for k in ga)) ** 0.5
    worst = max(((gc[k].double() - ga[k].double()).norm().item() / max(ga[k].double().norm().item(), rms * ga[k].numel() ** 0.5), k)
                for k in ga)
    assert worst[0] <= 1e-2, worst
    assert torch.allclose(lc, la, rtol=1e-4, atol=0)


# ---- 3: the training loop --------------------------------------------------------------------------------------
def test_training_loop_state_is_bit_identical(deterministic, tmp_path):
    """train_self_supervised with accumulation over the boundary and the epoch's tail step, FusedAdam and the EMA
    update, run twice from one seed: bit-identical state_dicts."""
    import vit2spn
    from oracle import vit2spn_oracle as orc
    batches = [orc.synthetic_views(4, seed=300 + 2 * i) for i in range(9)]
    loader = [((a, b), torch.zeros(a.shape[0], 1)) for a, b in batches]
    states = []
    for run in range(2):
        model = _dual("bf16", seed=21)
        opt = vit2spn.FusedAdam(model.parameters(), lr=1e-4)
        vit2spn.train_self_supervised(model, loader, 2, opt, torch.nn.CosineSimilarity(dim=1),
                                      checkpoint_path=str(tmp_path / f"ckpt{run}.pth"), accumulation_steps=8, device=DEV,
                                      log=lambda s: None)
        states.append({k: v.detach().clone() for k, v in model.state_dict().items()})
    _assert_equal(*states)


# ---- 4: the range-wise backward of the data-parallel overlap -------------------------------------------------------
class _RangeSync:
    """The calls ssp_step makes on an OverlappedGradSync, without NCCL: ranges 12 -> 8 -> 4 -> 0, and the SM limit
    set after the first range as the overlapped all-reduce does."""
    ranges = [(12, 8), (8, 4), (4, 0)]

    def begin(self):
        pass

    def heads_ready(self):
        pass

    def range_ready(self, hi, lo):
        from vit2spn import _lib
        if hi == 12:
            _lib.lib.v2s_set_sm_limit(100)


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_range_wise_backward_under_sm_limit_equals_plain(deterministic, mode):
    from vit2spn import _lib
    x1, x2 = _views(32, 7)
    plain = _dual(mode)
    lp = plain.ssp_step(x1, x2)
    ranged = _dual(mode)
    try:
        lr = ranged.ssp_step(x1, x2, grad_sync=_RangeSync())
    finally:
        _lib.lib.v2s_set_sm_limit(0)
    assert torch.equal(lp, lr)
    _assert_equal(_grads(plain), _grads(ranged))


# ---- 5: autograd paths -----------------------------------------------------------------------------------------
def _vit(mode="bf16"):
    import vit2spn
    from oracle import vit2spn_oracle as orc
    m = vit2spn.ViTModel()
    m.load_state_dict(orc.sub_state(orc.init_state(11, 0.01), "online_network_1"), strict=True)
    m.to(DEV).train()
    m.compute_mode = mode
    return m


def _images(B, seed=0):
    from oracle import vit2spn_oracle as orc
    return orc.preprocess_u8(orc.synthetic_octmnist_u8(B, seed)).to(DEV)


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_vit_hidden_state_gradients_are_bit_identical(deterministic, mode):
    """A loss on an intermediate hidden state (its gradient joins the residual stream and the fc2 bias gradient of the
    block that produced it) and on the last one."""
    m = _vit(mode)
    x = _images(16)
    runs = []
    for _ in range(2):
        m.zero_grad(set_to_none=True)
        out = m(x, output_hidden_states=True)
        (out.hidden_states[6].square().mean() + out.hidden_states[-1].mean()).backward()
        runs.append(_grads(m))
    _assert_equal(*runs)


def test_vit_features_backward_is_bit_identical(deterministic):
    """ViTModel.features: the backbone half of FineTunedModel."""
    m = _vit()
    x = _images(16, seed=1)
    w = torch.randn(192, device=DEV, generator=torch.Generator(device=DEV).manual_seed(0))
    runs = []
    for _ in range(2):
        m.zero_grad(set_to_none=True)
        (m.features(x) @ w).square().sum().backward()
        runs.append(_grads(m))
    _assert_equal(*runs)


# ---- 6: CUDA graph -----------------------------------------------------------------------------------------------
def test_graphed_step_matches_eager_and_recaptures_on_toggle(deterministic):
    x1, x2 = _views(32, 9)
    eager = _dual("bf16")
    le = [eager.ssp_step(x1, x2).clone() for _ in range(3)]
    graphed = _dual("bf16")
    lg = [graphed.ssp_step_graphed(x1, x2).clone() for _ in range(3)]       # capture on the first call, then replays
    assert torch.equal(torch.stack(le), torch.stack(lg))
    _assert_equal(_grads(eager), _grads(graphed))
    assert len(graphed._graphs) == 1
    _set_flag(False)
    graphed.ssp_step_graphed(x1, x2)
    assert len(graphed._graphs) == 2


# ---- 7: launch counts --------------------------------------------------------------------------------------------
def test_launch_counts_match_default_mode(deterministic):
    """The fixed-order reductions add no launch: 155 per ViTModel forward + backward and 363 per DualStreamNetwork step
    (fused step + autograd step), as in the default mode (tests/test_gpu_vit_outputs.py)."""
    import os
    import vit2spn
    from vit2spn import _lib
    from oracle import vit2spn_oracle as orc
    if os.environ.get("V2S_GEMM_DEBUG"):
        pytest.skip("launch counts are pinned for the uninstrumented kernels")
    x = _images(4)
    m = _vit()
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
