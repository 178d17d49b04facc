"""Device cost of masked patch tokens at B=128, bf16.  Two arms alternated in one process, both forward + backward of a
trainable vit2spn.ViTModel(use_mask_token=True) with the loss on hidden_states[-1]:
  unmasked  forward(x)
  masked    forward(x, bool_masked_pos=m), m a fixed 40 % random mask (every GEMM still runs on all rows)
then per-class device times (v2s_prof) of one call of each arm in a separate pass.  Writes --out (JSON)."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("V2S_ALLOW_RANDOM_INIT", "1")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "masked_tokens_cost_r01.json"))
    a = ap.parse_args()
    import vit2spn
    from vit2spn import _lib
    from oracle import vit2spn_oracle as orc
    dev = torch.device("cuda", 0)
    B = a.batch
    m = vit2spn.ViTModel(use_mask_token=True)
    m.load_state_dict({**orc.sub_state(orc.init_state(11, 0.01), "online_network_1"),
                       "embeddings.mask_token": 0.02 * torch.randn(1, 1, 192)}, strict=True)
    m.to(dev).compute_mode = "bf16"
    x = orc.preprocess_u8(orc.synthetic_octmnist_u8(B, 0)).to(dev)
    up = torch.randn(B, 197, 192, device=dev)
    mask = torch.rand(B, 196, device=dev, generator=torch.Generator(device=dev).manual_seed(1)) < 0.4

    def run(mk):
        m.zero_grad(set_to_none=False)
        (m(x, bool_masked_pos=mk).hidden_states[-1] * up).sum().backward()
    arms = {"unmasked": lambda: run(None), "masked": lambda: run(mask)}
    for f in arms.values():
        for _ in range(3):
            f()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(a.rounds):
        for k, f in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.iters):
                f()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / a.iters)
    classes = {}
    for k, f in arms.items():
        f()
        torch.cuda.synchronize()
        _lib.prof_enable(True)
        f()
        classes[k] = _lib.prof_report()
        _lib.prof_enable(False)
    assert _lib.lib.v2s_debug_flag() == 0

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0), "batch": B, "mode": "bf16",
           "masked_fraction": round(mask.float().mean().item(), 4),
           "ms_per_fwd_bwd": {k: {"median": sorted(v)[len(v) // 2], "min": min(v), "max": max(v), "all": v}
                              for k, v in times.items()},
           "classes_ms": {k: {c: [cnt, round(t, 4)] for c, (cnt, t, _, _) in v.items()} for k, v in classes.items()},
           "note": "CUDA events around iters forward+backward calls, arms alternated per round; classes: one call with "
                   "v2s_prof enabled (launches, device ms); the mask is applied inside assemble_tokens (forward), "
                   "gather_patch_rows and embed_bwd (backward), counted under misc"}
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v["median"] for k, v in res["ms_per_fwd_bwd"].items()}), res["gpu"])


if __name__ == "__main__":
    main()
