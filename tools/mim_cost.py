"""What the SimMIM head costs next to the backbone, on one GPU: a training step (forward, backward, FusedAdam) of
``vit2spn.ViTForMaskedImageModeling`` against the same CUDA backbone with the eager-torch head of the earlier recipe
(``tests/test_masked_tokens_cpu.simmim_loss``: final LayerNorm, fp32 Conv2d(192, 768, 1), PixelShuffle(16), masked L1).
B = 128, bf16, a fixed 60 % random mask; the two arms alternate in one process, device-event timed, several rounds.
A separate profiled pass gives the head's own kernel classes (mim_fwd / mim_bwd) with their algorithmic bytes and FLOPs.

    python tools/mim_cost.py [--batch 128] [--steps 20] [--rounds 5] [--out profiles/mim_cost_r01.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
os.environ.setdefault("V2S_ALLOW_RANDOM_INIT", "1")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mim_cost_r01.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("mim_cost: no CUDA device (this measurement runs on the GPU only)")
    import vit2spn
    from oracle import vit2spn_oracle as orc
    from test_masked_tokens_cpu import simmim_loss
    dev = torch.device("cuda", 0)
    B = a.batch
    x = orc.preprocess_u8(orc.synthetic_octmnist_u8(B, 0)).to(dev)
    mask = (torch.rand(B, 196, generator=torch.Generator().manual_seed(1)) < 0.6).to(dev)
    torch.manual_seed(0)
    fused = vit2spn.ViTForMaskedImageModeling().to(dev)
    fused.compute_mode = "bf16"
    opt_f = vit2spn.FusedAdam(fused.parameters(), lr=1e-4)
    vit = vit2spn.ViTModel(use_mask_token=True).to(dev)
    vit.compute_mode = "bf16"
    conv = torch.nn.Conv2d(192, 768, kernel_size=1).to(dev)
    vit.load_state_dict({k[4:]: v for k, v in fused.state_dict().items() if k.startswith("vit.")}, strict=False)
    conv.load_state_dict({"weight": fused.decoder[0].weight.detach(), "bias": fused.decoder[0].bias.detach()})
    opt_t = vit2spn.FusedAdam(list(vit.parameters()) + list(conv.parameters()), lr=1e-4)

    def step_fused():
        opt_f.zero_grad()
        loss = fused(x, bool_masked_pos=mask).loss
        loss.backward()
        opt_f.step()
        return loss

    def step_torch():
        opt_t.zero_grad()
        loss = simmim_loss(vit(x, bool_masked_pos=mask).last_hidden_state, conv, x, mask)
        loss.backward()
        opt_t.step()
        return loss

    arms = {"cuda_head": step_fused, "torch_head": step_torch}
    for fn in arms.values():                     # warm-up: every shape, workspaces, kernel attributes
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(a.rounds):
        for k, fn in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / a.steps)
    loss_f, loss_t = step_fused().item(), step_torch().item()

    from vit2spn import _lib
    _lib.prof_enable(True)
    nprof = 5
    for _ in range(nprof):
        step_fused()
    rep = _lib.prof_report()
    _lib.prof_enable(False)
    prof = {k: {"launches": n // nprof, "ms_per_step": ms / nprof, "work_per_step": w / nprof, "bytes_per_step": nb / nprof}
            for k, (n, ms, w, nb) in rep.items() if n}
    for k in ("mim_fwd", "mim_bwd"):
        c = prof.get(k)
        if c and c["ms_per_step"] > 0:
            c["achieved_GBps"] = c["bytes_per_step"] / (c["ms_per_step"] * 1e-3) / 1e9
            c["achieved_TFLOPs"] = c["work_per_step"] / (c["ms_per_step"] * 1e-3) / 1e12
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    res = {"card": card(), "batch": B, "mode": "bf16", "mask_fraction": 0.6, "steps_per_round": a.steps,
           "rounds": a.rounds, "step_ms": {k: {"median": med[k], "min": min(v), "max": max(v), "all": v}
                                            for k, v in times.items()},
           "head_saving_ms_per_step": med["torch_head"] - med["cuda_head"],
           "loss_after_timing": {"cuda_head": loss_f, "torch_head": loss_t},
           "prof_classes_cuda_head": prof,
           "note": "step = forward + backward + FusedAdam; prof classes from a separate profiled pass (CUDA events per "
                   "launch), bytes and FLOPs algorithmic"}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "head_saving_ms_per_step")} | {"median_ms": med}))


if __name__ == "__main__":
    main()
