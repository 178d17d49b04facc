#!/usr/bin/env python
"""bench.py — dual-view SSP pairs/sec, ViT-Tiny, batch 128 per GPU (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on host cores
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's outputs (dump_outputs)

A "step" (default workload `ssp`) is one full SSP step of the reference recipe with accumulation_steps=1
(BASELINE.md §3): zero_grad → 4 backbones forward (2 online with grad, 2 EMA targets) → heads → -mean(cos)/1 →
backward → [gradient all-reduce, overlapped with backward, if N>1] → Adam(lr 1e-4) → EMA(0.999), on one batch of 128
synthetic OCTMNIST-shaped pairs per GPU (uint8 28x28 → bilinear 224 → 3ch → ImageNet-normalised fp32).
Other workloads (`--workload`): `accum8` = the reference recipe proper (8 micro-steps per optimizer step, ref:39,
215), `finetune` = FineTunedModel step (BASELINE config 4), `eval1024` = forward-only feature extraction at batch
1024 (config 5).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
# random-init ViT-Tiny weights by specification (north_star: no ImageNet checkpoint offline)
os.environ.setdefault("V2S_ALLOW_RANDOM_INIT", "1")
COMM_SMS = int(os.environ.get("V2S_COMM_SMS", "8"))
# the gradient all-reduce overlaps the backward pass on the SMs the compute grids leave free (parallel.py)
os.environ.setdefault("NCCL_MAX_CTAS", str(COMM_SMS))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLOP_PER_PAIR = 19.945e9          # SURVEY.md §8(d): algorithmic FLOPs of one pair per micro-step
FLOP_PER_IMAGE_FT = 7.463e9       # fine-tune step per image, FLOP_PER_IMAGE_FWD forward only (SURVEY §8d)
FLOP_PER_IMAGE_FWD = 2.507e9
METRIC = "dual-view SSP pairs/sec, ViT-Tiny b128/GPU"
SYNC_SPLITS = tuple(int(x) for x in os.environ.get("V2S_SYNC_SPLITS", "8,4").split(","))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ssp", choices=["ssp", "accum8", "finetune", "eval1024"])
    ap.add_argument("--loss", default="cosine", choices=["cosine", "infonce"],
                    help="cosine = the reference's loss (ref:174,211; default); infonce = opt-in global-negative InfoNCE "
                         "(BASELINE config 3: all-gather of the target projections over the ranks)")
    ap.add_argument("--graph", action="store_true", help="replay the micro-step from a CUDA graph (ssp_step_graphed; 1 GPU)")
    ap.add_argument("--batch", type=int, default=None, help="samples per GPU (default 128; eval1024: 1024)")
    ap.add_argument("--mode", default="bf16", choices=["bf16", "fp16", "fp32"])
    ap.add_argument("--cpu-batch", type=int, default=32, help="bounded CPU sample (pairs per CPU step)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-input", default="auto", choices=["auto", "u8p", "u8", "fp32"],
                    help="host format of the e2e leg: raw uint8 28x28 source images (0.2 MB/step) turned on the GPU into the "
                         "16-bit patch matrix (u8p, one kernel; default where the step accepts it) or into fp32 views (u8), "
                         "or the reference DataLoader's fp32 views (fp32, 154 MB/step)")
    ap.add_argument("--no-overlap", action="store_true", help="N>1: plain all-reduce after backward instead of the overlapped one")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned, and the model state it left, to DIR/<name>.npy "
                         "(float32 / float64, at most 64 MB) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.t0 = self.t1 = None

    def start(self):
        """Started well before the timed region (nvidia-smi takes a while to come up); samples are time-stamped on
        arrival and only those inside [mark_begin, mark_end] are used."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()

        def parse(rows):
            sm, mx, reasons = [], None, set()
            for _, ln in rows:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx = float(f[2])
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, reasons

        inside = [r for r in self.lines if self.t0 is not None and self.t0 <= r[0] <= (self.t1 or r[0]) + 0.03]
        scope = "timed region"
        if not inside:                       # region shorter than the sampling period: nearest samples under load
            inside, scope = self.lines[-3:], "nearest samples (timed region shorter than the sampling period)"
        sm, mx, reasons = parse(inside)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm), "scope": scope}


def cpu_reference_step_fn(batch):
    """The reference algorithm on host cores: oracle port of ref:ssp_vit2spn_tiny.py:205-219
    (fp32, accumulation_steps=1: fwd → loss → bwd → Adam → EMA).  /root/reference itself does not
    exist on the GPU box, so kind = "port"."""
    import torch
    from oracle import vit2spn_oracle as orc
    torch.set_num_threads(os.cpu_count() or 1)
    state = orc.init_state(42, 0.0)
    x1, x2 = orc.synthetic_views(batch, seed=0)
    opt = {}

    def step():
        nonlocal state, opt
        loss, _, state, opt = orc.ssp_step(state, opt, x1, x2, lr=1e-4, momentum=0.999)
        return float(loss)
    return step, torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    step, cores = cpu_reference_step_fn(args.cpu_batch)
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = args.cpu_batch * args.steps / dt
    sample = (f"{args.steps} full SSP steps (fwd+bwd+Adam+EMA, fp32) of {args.cpu_batch} pairs each on "
              f"{cores} host threads; oracle port of the reference algorithm (bounded sample of the 128-pair batch: "
              "a 128-pair fp32 step is ~13 GB of autograd state and tens of seconds on these cores)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "ViT-Tiny dual-stream SSP full step, accumulation 1 (BASELINE config 2 recipe), "
                               f"bounded CPU sample of {args.cpu_batch} pairs/step"},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


_STDOUT_FD = None


def claim_stdout():
    """stdout carries exactly ONE JSON line: anything a library prints there (NCCL's version banner at
    communicator creation, for one) is sent to stderr instead."""
    global _STDOUT_FD
    sys.stdout.flush()
    _STDOUT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_STDOUT_FD if _STDOUT_FD is not None else 1, (json.dumps(line) + "\n").encode())


def eager_gpu_baseline(dev, B):
    """The practical bar of SURVEY §8(d): the reference's own PyTorch path (the oracle's restatement of its classes)
    under bf16 autocast on THIS GPU — stock eager kernels (cuBLAS / SDPA), full step incl. Adam + EMA."""
    import torch
    from oracle import vit2spn_oracle as orc
    state = {k: v.to(dev) for k, v in orc.init_state(42, 0.0).items()}
    x1, x2 = (t.to(dev) for t in orc.synthetic_views(B, seed=0))
    names = orc.trainable_names()
    params = [state[k].clone().requires_grad_(True) for k in names]
    opt = torch.optim.Adam(params, lr=1e-4)

    def step():
        st = dict(state)
        st.update(dict(zip(names, params)))
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            p, t = orc.dual_stream_forward(st, x1, x2)
        loss = orc.ssp_loss(p.float(), t.float())
        loss.backward()
        opt.step()
        with torch.no_grad():                       # EMA as one foreach pass (kinder than the reference's Python loop)
            for o, t_ in (("online_network_1", "target_network_1"), ("online_network_2", "target_network_2")):
                ks = list(orc.backbone_param_shapes())
                tg = [state[f"{t_}.vit.{k}"] for k in ks]
                on = [st[f"{o}.vit.{k}"].detach() for k in ks]
                torch._foreach_mul_(tg, 0.999)
                torch._foreach_add_(tg, on, alpha=0.001)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 5
    e0.record()
    for _ in range(n):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    return {"value": B / (ms * 1e-3), "unit": "pairs/s", "ms_per_step": ms, "steps": n,
            "what": "oracle restatement of the reference classes, torch.autocast(bf16), torch.optim.Adam, foreach EMA, "
                    f"batch {B}, same GPU (stock PyTorch kernels)"}


DUMP_SAMPLE = 1 << 23     # float32 elements of the parameter sample: 32 MB, within the 64 MB budget of a dump


def dump_outputs(dirname, result, model, probs=None):
    """What the last timed step hands its caller: its return value (`result.npy`), the class probabilities of the
    forward-only workload (`probs.npy`), and for training workloads the parameters and buffers the step updated, as
    the L2 norm of every state_dict tensor (`state_norms.npy`, float64, state_dict order) and the values of the
    concatenated state_dict at DUMP_SAMPLE positions drawn without replacement by numpy's default_rng(0), in
    ascending order (`state_sample.npy`; every value when the state is smaller than that)."""
    import numpy as np
    import torch
    os.makedirs(dirname, exist_ok=True)
    out = {"result": result.detach().float().reshape(-1).cpu().numpy()}
    if probs is not None:
        out["probs"] = probs.detach().float().cpu().numpy()
    else:
        sd = list(model.state_dict().values())
        out["state_norms"] = np.array([float(v.detach().double().norm()) for v in sd])
        flat = torch.cat([v.detach().reshape(-1).float() for v in sd])
        if flat.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(flat.numel(), DUMP_SAMPLE, replace=False))
        else:
            idx = np.arange(flat.numel())
        out["state_sample"] = flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy()
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    for name, a in out.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def main():
    args = parse()
    claim_stdout()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import vit2spn
    from vit2spn import _lib
    import numpy as np

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch or (1024 if args.workload == "eval1024" else 128)
    vit2spn.set_compute_mode(args.mode)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    _lib.init_device(local)

    # ---- synthetic data: seeded raw OCTMNIST-shaped source images, uint8 [2B,1,28,28] (SURVEY §8d); rank-dependent --
    u8_host = torch.from_numpy(np.random.default_rng(1000 + rank).integers(0, 256, size=(2 * B, 1, 28, 28), dtype=np.uint8))
    u8 = u8_host.to(dev)
    views = torch.empty(2, B, 3, 224, 224, device=dev)

    def preprocess(src_u8, dst):
        _lib.check(_lib.lib.v2s_preprocess_u8(_lib.ptr(src_u8), _lib.ptr(dst), 2 * B, _lib.stream_ptr()))
    preprocess(u8, views)
    x1, x2 = views[0], views[1]

    # ---- model / optimizer / step of the chosen workload --------------------------------------------------------
    torch.manual_seed(42)
    sync = None
    step_out = {}           # what the most recent step returned (and, forward-only, its class probabilities)
    if args.workload in ("ssp", "accum8"):
        model = vit2spn.DualStreamNetwork().to(dev).train()
        model.loss_mode = args.loss
        vit2spn.parallel.broadcast_parameters(model)     # identical replicas
        opt = vit2spn.FusedAdam(model.parameters(), lr=1e-4)
        if world > 1 and not args.no_overlap:
            sync = vit2spn.parallel.OverlappedGradSync(model, splits=SYNC_SPLITS, comm_sms=COMM_SMS)
        micro = 8 if args.workload == "accum8" else 1

        def step(a, b):
            loss = None
            for i in range(micro):
                last = i == micro - 1
                if args.graph and world == 1:
                    loss = model.ssp_step_graphed(a, b, accumulation_steps=micro)
                else:
                    loss = model.ssp_step(a, b, accumulation_steps=micro, grad_sync=sync if (last and world > 1) else None)
            if world > 1:
                if sync is not None:
                    sync.finish(opt)
                else:       # one collective per optimizer step over 3 flat fp32 buckets; 1/world folded into Adam
                    vit2spn.parallel.allreduce_gradients(model, optimizer=opt)
            opt.step()
            opt.zero_grad()
            model.update_target_network()
            return loss
        units_per_step, unit, flop_per_unit = B * micro, "pairs/s", FLOP_PER_PAIR
        metric = METRIC
        loss_name = "cosine loss" if args.loss == "cosine" else ("InfoNCE loss (temperature 0.2) over the target projections "
                                                                  "all-gathered from every rank (NCCL)")
        workload = (f"ViT-Tiny dual-stream SSP full step (4 backbones fwd, 2 bwd, heads, {loss_name}, Adam lr 1e-4, EMA 0.999), "
                    + ("accumulation 1, batch 128/GPU (BASELINE config 2)" if micro == 1 else
                       "reference recipe: 8 accumulated micro-steps of 128 pairs per optimizer step (ref:39,215)")
                    + ("; micro-step replayed from a CUDA graph" if args.graph and world == 1 else ""))
    elif args.workload == "finetune":
        model = vit2spn.FineTunedModel(num_classes=4).to(dev).train()
        opt = vit2spn.FusedAdam(model.parameters(), lr=1e-4, weight_decay=1e-4)          # ref:octmnist_ft_vit2spn.py:192
        y = (torch.arange(B, device=dev) % 4)
        crit = torch.nn.CrossEntropyLoss(weight=torch.tensor([1.0, 2.0, 0.5, 1.5], device=dev))

        def step(a, b):
            opt.zero_grad()
            loss = crit(model(a), y)
            loss.backward()
            if world > 1:       # BatchNorm1d statistics stay per-rank (the reference is single-GPU); gradients are averaged
                for p in model.parameters():
                    if p.grad is not None:
                        dist.all_reduce(p.grad)
                opt.grad_multiplier = 1.0 / world
            opt.step()
            return loss.detach()
        units_per_step, unit, flop_per_unit = B, "images/s", FLOP_PER_IMAGE_FT
        metric = "ViT-2SPN fine-tune images/sec, ViT-Tiny b128/GPU (BASELINE config 4)"
        workload = "FineTunedModel step: backbone fwd+bwd, BatchNorm/Dropout head (torch), weighted CE, Adam lr 1e-4 + L2 1e-4"
    else:
        model = vit2spn.FineTunedModel(num_classes=4).to(dev).eval()

        def step(a, b):
            with torch.no_grad():
                step_out["probs"] = torch.softmax(model(a), dim=1)
                return step_out["probs"][:, 0].sum()
        units_per_step, unit, flop_per_unit = B, "images/s", FLOP_PER_IMAGE_FWD
        metric = "forward-only feature extraction images/sec, ViT-Tiny b1024 (BASELINE config 5)"
        workload = "FineTunedModel eval forward (backbone + head + softmax), batch 1024, no_grad (ref:octmnist_ft_vit2spn.py:129-137)"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, finish=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if finish is not None:
            finish()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    if hasattr(model, "ssp_step"):
        opt.zero_grad()
    warm = max(args.warmup, 3)
    for _ in range(warm):
        step(x1, x2)

    def timed_step():
        step_out["result"] = step(x1, x2)

    l0 = _lib.lib.v2s_launch_count() + getattr(model, "graph_replayed_kernels", 0)
    sampler.mark_begin()
    ms_total = timed(timed_step, args.steps)
    sampler.mark_end()
    # kernels of this library launched in the timed region (those replayed from a CUDA graph included)
    launches = int(_lib.lib.v2s_launch_count() + getattr(model, "graph_replayed_kernels", 0) - l0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step_out["result"], model, step_out.get("probs"))
    # host-side cost of enqueueing one step (no device wait inside): tells CPU-bound from GPU-bound
    torch.cuda.synchronize()
    h0 = time.perf_counter()
    for _ in range(5):
        step(x1, x2)
    host_ms = (time.perf_counter() - h0) / 5 * 1e3
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    flag = _lib.lib.v2s_debug_flag()
    ms_per_step = ms_total / args.steps
    value = world * units_per_step * args.steps / (ms_total * 1e-3)

    # ---- end to end through the public API with HOST buffers: every step copies its inputs from pinned host memory
    #      (double-buffered on a copy stream) and reads its result back on the host ------------------------------
    e2e = None
    e2e_in = args.e2e_input
    if e2e_in == "auto":      # the fused uint8 -> patch-matrix kernel where the step takes it (SSP step, 16-bit modes)
        e2e_in = "u8p" if (args.workload in ("ssp", "accum8") and args.mode in ("bf16", "fp16")) else "u8"
    if not args.no_e2e:
        if e2e_in == "u8p":
            host = u8_host.pin_memory()
            raw = [torch.empty_like(u8) for _ in range(2)]
            lp_dtype = torch.bfloat16 if args.mode == "bf16" else torch.float16
            bufs = [torch.empty(2, B, 196, 768, dtype=lp_dtype, device=dev) for _ in range(2)]
            h2d = int(host.numel())
            what = ("raw uint8 source images [2B,1,28,28] in pinned host memory → H2D → bilinear 224 / 3 channels / normalise / "
                    "im2col in one kernel (v2s_preprocess_u8_patches: the 16-bit patch matrix the patch-embed GEMM reads) → step")
        elif e2e_in == "u8":
            # the dataset's native format (28x28 uint8, ref:ssp_vit2spn_tiny.py:100-104): 2*B*784 bytes per step; the
            # resize / normalise of the reference's transform runs on the GPU inside the timed region
            host = u8_host.pin_memory()
            raw = [torch.empty_like(u8) for _ in range(2)]
            bufs = [torch.empty_like(views) for _ in range(2)]
            h2d = int(host.numel())
            what = ("raw uint8 source images [2B,1,28,28] in pinned host memory → H2D → bilinear 224 / 3 channels / "
                    "normalise on the GPU (v2s_preprocess_u8) → step")
        else:
            host = [views[i].cpu().pin_memory() for i in range(2)]
            bufs = [torch.empty_like(views) for _ in range(2)]
            h2d = int(2 * B * 3 * 224 * 224 * 4)
            what = "fp32 views [2,B,3,224,224] in pinned host memory (the reference DataLoader's format), double-buffered H2D"
        copy_stream = torch.cuda.Stream()
        ready = [torch.cuda.Event() for _ in range(2)]
        done = [torch.cuda.Event() for _ in range(2)]

        def upload(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done[i])
                if e2e_in == "u8p":
                    raw[i].copy_(host, non_blocking=True)
                    vit2spn.preprocess_u8_patches(raw[i], out=bufs[i].view(2 * B, 196, 768))
                elif e2e_in == "u8":
                    raw[i].copy_(host, non_blocking=True)
                    preprocess(raw[i], bufs[i])
                else:
                    bufs[i][0].copy_(host[0], non_blocking=True)
                    bufs[i][1].copy_(host[1], non_blocking=True)
                ready[i].record(copy_stream)

        # the result of every step is read on the host (ref:220 `loss.item()`), through a pinned buffer and an event,
        # one step behind: step k's value is fetched after step k+1 has been enqueued, so the host-side enqueue
        # cost of a step never leaves the GPU idle; the last value is fetched before the timed region closes
        loss_host = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
        loss_ev = [torch.cuda.Event() for _ in range(2)]
        state = {"i": 0, "pending": None, "last": None}
        for d in done:
            d.record()

        def fetch():
            j = state["pending"]
            if j is not None:
                loss_ev[j].synchronize()
                state["last"] = float(loss_host[j])
                state["pending"] = None

        def e2e_step():
            i = state["i"]
            torch.cuda.current_stream().wait_event(ready[i])
            loss = step(bufs[i][0], bufs[i][1])
            loss_host[i].copy_(loss.detach().reshape(()).float(), non_blocking=True)   # D2H of the step's result
            loss_ev[i].record()
            done[i].record()
            upload(i)                      # refill this buffer for step i+2 while step i+1 computes
            fetch()                        # previous step's result
            state["pending"] = i
            state["i"] = i ^ 1

        upload(0); upload(1)
        for _ in range(3):
            e2e_step()
        fetch()
        ms_e2e = timed(e2e_step, args.steps, finish=fetch)
        if state["last"] is None or state["last"] != state["last"]:
            raise RuntimeError("e2e: result readback failed")
        e2e = {"value": world * units_per_step * args.steps / (ms_e2e * 1e-3), "unit": unit,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps, "input": what,
               "result": "the step's loss / output checksum copied to pinned host memory and read there, one step behind the enqueue"}

    # ---- per-kernel-class device timing (CUDA events on the launching stream) → roofline ---------
    pk, pk_src = peaks()
    _lib.prof_enable(True)
    nprof = 3
    for _ in range(nprof):
        step(x1, x2)
    rep = _lib.prof_report()
    _lib.prof_enable(False)
    classes = {}
    for k, (n, ms, w, nb) in rep.items():
        c = {"launches": n // nprof, "ms_per_step": ms / nprof, "work_per_step": w / nprof, "bytes_per_step": nb / nprof}
        sec = c["ms_per_step"] * 1e-3
        is_tc = k.startswith("gemm") or k.startswith("attn")
        c["achieved_GBps"] = c["bytes_per_step"] / sec / 1e9 if sec > 0 else None
        c["frac_of_hbm_peak"] = c["achieved_GBps"] / pk["hbm_gbs"] if sec > 0 else None
        if is_tc and sec > 0:
            c["achieved_TFLOPs"] = c["work_per_step"] / sec / 1e12
            c["frac_of_bf16_burst_peak"] = c["achieved_TFLOPs"] / pk["bf16_tflops"]
            c["bound"] = "hbm" if c["bytes_per_step"] / (pk["hbm_gbs"] * 1e9) >= c["work_per_step"] / (pk["bf16_tflops_sustained"] * 1e12) else "tensor"
        else:
            c["bound"] = "hbm"
        classes[k] = c
    tensor_classes = [k for k in classes if k.startswith("gemm") or k.startswith("attn")]
    step_tflops = value / world * flop_per_unit / 1e12
    roofline = None
    traffic_file = "ncu_r02_traffic.json" if os.path.exists(os.path.join(ROOT, "profiles", "ncu_r02_traffic.json")) else "ncu_r01_traffic.json"
    try:
        ncu_traffic = json.load(open(os.path.join(ROOT, "profiles", traffic_file)))
    except Exception:
        ncu_traffic = {}
    if tensor_classes:
        # dominant kernel class by device time; its bound is whichever roofline time is larger for its
        # ALGORITHMIC flops / bytes (operands and outputs once, SURVEY §8d)
        dom = max(tensor_classes, key=lambda k: classes[k]["ms_per_step"])
        c = classes[dom]
        tr = ncu_traffic.get(dom, {}).get("dram_bytes_per_launch")
        if c["bound"] == "hbm":
            roofline = {"kernel": dom, "bound": "hbm", "achieved": c["achieved_GBps"], "peak": pk["hbm_gbs"], "unit": "GB/s",
                        "frac": c["frac_of_hbm_peak"], "traffic": tr, "peak_source": f"hbm_gbs ({pk_src})"}
        else:
            roofline = {"kernel": dom, "bound": "tensor", "achieved": c["achieved_TFLOPs"], "peak": pk["bf16_tflops_sustained"],
                        "unit": "TFLOP/s", "frac": c["achieved_TFLOPs"] / pk["bf16_tflops_sustained"], "traffic": tr,
                        "peak_source": f"bf16_tflops_sustained ({pk_src}; the kernel runs inside a long step)"}
        roofline.update({"launches_per_step": c["launches"], "ms_per_step": c["ms_per_step"],
                         "share_of_step": c["ms_per_step"] / ms_per_step,
                         "algorithmic_bytes_per_launch": c["bytes_per_step"] / max(c["launches"], 1),
                         "algorithmic_flops_per_launch": c["work_per_step"] / max(c["launches"], 1),
                         "traffic_source": "ncu dram__bytes_read.sum + dram__bytes_write.sum per launch, "
                                           f"profiles/{traffic_file} (cold-cache capture)",
                         # SURVEY §8(d): the step as a whole against the bf16 tensor roofline, both denominators
                         "step": {"algorithmic_tflops_per_gpu": step_tflops,
                                  "frac_of_bf16_burst_peak": step_tflops / pk["bf16_tflops"],
                                  "frac_of_bf16_sustained_peak": step_tflops / pk["bf16_tflops_sustained"],
                                  "algorithmic_hbm_bytes_per_step": sum(v["bytes_per_step"] for v in classes.values()),
                                  "hbm_floor_ms": sum(v["bytes_per_step"] for v in classes.values()) / (pk["hbm_gbs"] * 1e9) * 1e3,
                                  "tensor_floor_ms": units_per_step * flop_per_unit / (pk["bf16_tflops"] * 1e12) * 1e3},
                         "classes": {k: {kk: v[kk] for kk in ("launches", "ms_per_step", "bound", "achieved_GBps", "frac_of_hbm_peak",
                                                               "achieved_TFLOPs", "frac_of_bf16_burst_peak") if kk in v}
                                     for k, v in sorted(classes.items(), key=lambda kv: -kv[1]["ms_per_step"])}})

    cpu_baseline = gpu_eager = None
    if rank == 0 and world == 1 and args.workload == "ssp":
        if not args.no_eager_baseline:
            torch.cuda.empty_cache()
            try:
                gpu_eager = eager_gpu_baseline(dev, B)
            except Exception as e:  # noqa: BLE001  (a baseline must never take the line down)
                gpu_eager = {"error": str(e)[:200]}
        if not args.no_cpu_baseline:
            cstep, cores = cpu_reference_step_fn(args.cpu_batch)
            cstep()
            n = 0
            t0 = time.perf_counter()
            while n < 3 or (time.perf_counter() - t0 < 15 and n < 30):
                cstep(); n += 1
            dt = time.perf_counter() - t0
            cpu_baseline = {"value": args.cpu_batch * n / dt, "unit": "pairs/s", "cores": cores, "kind": "port",
                            "sample": f"{n} full SSP steps (fwd+bwd+Adam+EMA, fp32) of {args.cpu_batch} pairs each; "
                                      "oracle port of the reference algorithm (the reference's CPU path is torch fp32)"}

    if rank == 0:
        par = f"dp{world}"
        if world > 1:
            par += (f" (gradient all-reduce in {len(SYNC_SPLITS) + 1} block ranges + heads overlapped with backward, {COMM_SMS} SMs left to NCCL, 1/world folded into Adam)" if sync is not None
                    else " (3 flat all-reduces after backward)")
        line = {
            "metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.mode, "data": "synthetic",
            "config": {"workload": workload, "batch_per_gpu": B, "parallelism": par,
                       "l2": "inputs (154 MB/step) and activations (>2 GB/step) exceed the 126 MB L2; no explicit flush"},
            "step_tflops_per_gpu": step_tflops,
            "step_frac_of_bf16_peak": step_tflops / pk["bf16_tflops"],
            "roofline": roofline, "cpu_baseline": cpu_baseline, "gpu_eager_baseline": gpu_eager, "e2e": e2e,
            "gpu_launches": launches, "clocks": clocks, "kernel_classes": classes, "debug_flag": flag,
            "host_enqueue_ms_per_step": host_ms,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
