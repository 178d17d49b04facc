"""Cost of ViTModel's per-layer outputs on the GPU: a bf16 eval forward at B = 128 with and without
output_hidden_states / output_attentions (CUDA events, the four variants alternated round by round), the
attention-probabilities kernel's time per launch and its achieved write bandwidth against the 6.5 TB/s copy rate
measured on the B200 (DESIGN §4), and a launcher-shaped training step (``vit(x).hidden_states[-1].mean(1)``, the
reference's own call, which asks for output_hidden_states=True) with the flag off and on: step time and peak memory.

    python tools/vit_outputs_cost.py [--batch 128] [--rounds 10] [--out profiles/vit_outputs_cost.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("V2S_ALLOW_RANDOM_INIT", "1")

import torch  # noqa: E402

COPY_PEAK_TBS = 6.5


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # noqa: BLE001  (the numbers stand without it, but say why it is missing)
        info["power_limit"] = f"unavailable: {e}"
    return info


def timed(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "vit_outputs_cost.json"))
    a = ap.parse_args()
    import vit2spn
    from vit2spn import _lib
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: there is nothing to measure on the CPU")
    dev = torch.device("cuda", 0)
    B = a.batch
    m = vit2spn.ViTModel().to(dev).eval()
    m.compute_mode = "bf16"
    x = torch.randn(B, 3, 224, 224, device=dev)
    variants = {"none": (False, False), "hidden": (True, False), "attn": (False, True), "both": (True, True)}
    res = {"card": card(), "batch": B, "mode": "bf16", "forward_ms": {}}
    times = {k: [] for k in variants}
    with torch.no_grad():
        for k, (h, at) in variants.items():                       # warm-up of every shape
            m(x, output_hidden_states=h, output_attentions=at)
        for _ in range(a.rounds):
            for k, (h, at) in variants.items():
                times[k].append(timed(lambda: m(x, output_hidden_states=h, output_attentions=at), a.iters))
        for k, ts in times.items():
            ts = sorted(ts)
            res["forward_ms"][k] = {"median": ts[len(ts) // 2], "min": ts[0], "max": ts[-1]}
        _lib.prof_enable(True)
        for _ in range(a.iters):
            m(x, output_attentions=True)
        rep = _lib.prof_report()
        _lib.prof_enable(False)
    n, ms, work, nbytes = rep["attn_probs"]
    us = ms * 1e3 / n
    gbs = nbytes / (ms * 1e-3) / 1e9
    res["attn_probs_kernel"] = {"launches": n, "us_per_launch": us, "algorithmic_bytes_per_launch": nbytes / n,
                                "GB_per_s": gbs, "fraction_of_copy_peak": gbs / (COPY_PEAK_TBS * 1e3)}
    # launcher-shaped training step: the reference reads hidden_states[-1] of a model built with output_hidden_states=True
    step = {}
    for flag in (False, True):
        t = vit2spn.ViTModel.from_pretrained("WinKawaks/vit-tiny-patch16-224", output_hidden_states=flag).to(dev).train()
        t.compute_mode = "bf16"

        def one():
            t.zero_grad(set_to_none=False)
            t(x).hidden_states[-1].mean(dim=1).square().mean().backward()
        one()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        ms_step = sorted(timed(one, a.iters) for _ in range(a.rounds))
        step[f"output_hidden_states={flag}"] = {"step_ms_median": ms_step[len(ms_step) // 2],
                                                "peak_allocated_above_start_MB": (torch.cuda.max_memory_allocated(dev) - base) / 2 ** 20}
        del t
    res["launcher_step"] = step
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
