"""Cost of the deterministic mode (torch.use_deterministic_algorithms(True)) on the default SSP step: DualStreamNetwork,
B = 128, bf16, one fused micro-step (ssp_step), with the flag off and on alternated round by round in one process (CUDA
events).  Also the per-kernel-class device times of both (v2s_prof_report, a separate pass), the launches per step, and
the card's name and power limit.

    python tools/deterministic_cost.py [--batch 128] [--rounds 8] [--out profiles/deterministic_cost_r01.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
os.environ.setdefault("V2S_ALLOW_RANDOM_INIT", "1")

import torch  # noqa: E402

from vit_outputs_cost import card, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "deterministic_cost_r01.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: there is nothing to measure on the CPU")
    import vit2spn
    from vit2spn import _lib
    from oracle import vit2spn_oracle as orc
    dev = torch.device("cuda", 0)
    B = a.batch
    model = vit2spn.DualStreamNetwork()
    model.load_state_dict(orc.init_state(3, 0.02), strict=True)
    model.to(dev).train()
    model.compute_mode = "bf16"
    g = torch.Generator(device=dev).manual_seed(0)
    x1 = torch.randn(B, 3, 224, 224, device=dev, generator=g)
    x2 = torch.randn(B, 3, 224, 224, device=dev, generator=g)
    prev = torch.are_deterministic_algorithms_enabled()
    res = {"card": card(), "batch": B, "mode": "bf16", "workload": "DualStreamNetwork.ssp_step (fused micro-step)",
           "step_ms": {}, "launches_per_step": {}, "classes_ms_per_step": {}}
    flags = {"default": False, "deterministic": True}
    times = {k: [] for k in flags}
    try:
        for k, on in flags.items():                 # warm-up of both paths (workspaces, kernel attributes)
            torch.use_deterministic_algorithms(on)
            for _ in range(3):
                model.ssp_step(x1, x2)
            torch.cuda.synchronize()
            n0 = _lib.lib.v2s_launch_count()
            model.ssp_step(x1, x2)
            res["launches_per_step"][k] = int(_lib.lib.v2s_launch_count() - n0)
        for _ in range(a.rounds):
            for k, on in flags.items():
                torch.use_deterministic_algorithms(on)
                times[k].append(timed(lambda: model.ssp_step(x1, x2), a.iters))
        for k, ts in times.items():
            ts = sorted(ts)
            res["step_ms"][k] = {"median": ts[len(ts) // 2], "min": ts[0], "max": ts[-1], "rounds": ts}
        res["step_cost_relative"] = res["step_ms"]["deterministic"]["median"] / res["step_ms"]["default"]["median"] - 1.0
        for k, on in flags.items():
            torch.use_deterministic_algorithms(on)
            _lib.prof_enable(True)
            for _ in range(a.iters):
                model.ssp_step(x1, x2)
            rep = _lib.prof_report()
            _lib.prof_enable(False)
            res["classes_ms_per_step"][k] = {c: v[1] / a.iters for c, v in sorted(rep.items())}
    finally:
        torch.use_deterministic_algorithms(prev)
    d, o = res["classes_ms_per_step"]["deterministic"], res["classes_ms_per_step"]["default"]
    res["class_delta_ms_per_step"] = {c: d.get(c, 0.0) - o.get(c, 0.0) for c in sorted(set(d) | set(o))}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
