"""Device time of a gradient w.r.t. pixel_values at B=128, bf16, four arms alternated in one process:
  frozen      vit2spn.ViTModel, parameters frozen: forward + pixel backward (no weight gradient at all)
  trainable   forward + backward without x grad (the training path)
  joint       trainable + x grad (weight and pixel gradients)
  hf_eager    transformers.ViTModel (eager attention) under torch.autocast(bf16), frozen, forward + pixel backward
then per-class device times (v2s_prof) of the three vit2spn arms in a separate pass.  Writes --out (JSON)."""
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
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="input_grad_cost.json")
    a = ap.parse_args()
    import vit2spn
    import transformers
    from vit2spn import _lib
    from oracle import vit2spn_oracle as orc
    dev = torch.device("cuda", 0)
    p = orc.sub_state(orc.init_state(11, 0.01), "online_network_1")

    def vit(frozen):
        m = vit2spn.ViTModel()
        m.load_state_dict(p, strict=True)
        m.to(dev).compute_mode = "bf16"
        m.requires_grad_(not frozen)
        return m
    frozen, train = vit(True), vit(False)
    cfg = transformers.ViTConfig(hidden_size=192, num_hidden_layers=12, num_attention_heads=3, intermediate_size=768,
                                 layer_norm_eps=1e-12, attn_implementation="eager")
    hf = transformers.ViTModel(cfg, add_pooling_layer=False)
    hf.load_state_dict({k: v for k, v in p.items() if not k.startswith("pooler.")}, strict=True)
    hf.to(dev).eval().requires_grad_(False)
    x = orc.preprocess_u8(orc.synthetic_octmnist_u8(a.batch, 0)).to(dev)
    up = torch.randn(a.batch, 197, 192, device=dev)

    def run_vit(m, want_x):
        xd = x.clone().requires_grad_(want_x)
        m.zero_grad(set_to_none=False)
        (m(xd).hidden_states[-1] * up).sum().backward()

    def run_hf():
        xd = x.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            h = hf(pixel_values=xd, output_hidden_states=True).hidden_states[-1]
        (h.float() * up).sum().backward()
    arms = {"frozen": lambda: run_vit(frozen, True), "trainable": lambda: run_vit(train, False),
            "joint": lambda: run_vit(train, True), "hf_eager": run_hf}
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
    for k in ("frozen", "trainable", "joint"):
        arms[k]()
        torch.cuda.synchronize()
        _lib.prof_enable(True)
        arms[k]()
        classes[k] = _lib.prof_report()
        _lib.prof_enable(False)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0), "batch": a.batch, "mode": "bf16",
           "ms_per_fwd_bwd": {k: {"median": sorted(v)[len(v) // 2], "min": min(v), "max": max(v)} for k, v in times.items()},
           "classes_ms": {k: {c: [n, round(ms, 4)] for c, (n, ms, _, _) in v.items()} for k, v in classes.items()},
           "note": "host clock-free: CUDA events around iters forward+backward calls, arms alternated per round; "
                   "classes: one call with v2s_prof enabled (launches, device ms)"}
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["ms_per_fwd_bwd"]), res["gpu"])


if __name__ == "__main__":
    main()
