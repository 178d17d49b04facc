"""Time per image of ViTModel(interpolate_pos_encoding=True) against the input size, bf16, B200.

For 224, 160, 128 and 64 px square inputs (197, 101, 65 and 17 tokens) at batches with about the same number of tokens
per batch (B = 128, 250, 388, 1483), two arms on the same weights, alternated per round:
  vit2spn       vit2spn.ViTModel, compute_mode bf16
  transformers  stock transformers.ViTModel (eager attention) under torch.autocast(bfloat16)
each timed for the forward (no grad) and the forward + backward (loss on hidden_states[-1]).  Then, with --bench, the
default bench.py line of this tree and of --parent-tree (the parent commit's tree, built), in ABBA order.  The card's name
and power limit are read in the same call.  Writes --out (JSON)."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("V2S_ALLOW_RANDOM_INIT", "1")

POINTS = [(224, 128), (160, 250), (128, 388), (64, 1483)]


def _time(f, iters, rounds_out):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        f()
    e1.record()
    torch.cuda.synchronize()
    rounds_out.append(e0.elapsed_time(e1) / iters)


def _stats(v):
    s = sorted(v)
    return {"median": s[len(s) // 2], "min": s[0], "max": s[-1], "all": v}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--bench", action="store_true")
    ap.add_argument("--parent-tree", default="")
    ap.add_argument("--bench-rounds", type=int, default=6)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "interp_cost_r01.json"))
    a = ap.parse_args()
    import transformers
    import vit2spn
    from vit2spn import _lib
    from oracle import vit2spn_oracle as orc
    dev = torch.device("cuda", 0)
    p = orc.sub_state(orc.init_state(11, 0.01), "online_network_1")
    m = vit2spn.ViTModel()
    m.load_state_dict(p, strict=True)
    m.to(dev).compute_mode = "bf16"
    cfg = transformers.ViTConfig(hidden_size=192, num_hidden_layers=12, num_attention_heads=3, intermediate_size=768,
                                 patch_size=16, image_size=224, layer_norm_eps=1e-12, hidden_act="gelu", qkv_bias=True,
                                 attn_implementation="eager")
    hf = transformers.ViTModel(cfg, add_pooling_layer=False)
    hf.load_state_dict({k: v for k, v in p.items() if not k.startswith("pooler.")}, strict=True)
    hf.to(dev)

    res = {"points": {}}
    for side, B in POINTS:
        n = 1 + (side // 16) ** 2
        x = torch.randn(B, 3, side, side, device=dev)
        up = torch.randn(B, n, 192, device=dev)

        def ours_fwd():
            with torch.no_grad():
                m(x, interpolate_pos_encoding=True)

        def ours_fb():
            m.zero_grad(set_to_none=False)
            (m(x, interpolate_pos_encoding=True, output_hidden_states=True).hidden_states[-1] * up).sum().backward()

        def hf_fwd():
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                hf(pixel_values=x, interpolate_pos_encoding=True)

        def hf_fb():
            hf.zero_grad(set_to_none=False)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                out = hf(pixel_values=x, interpolate_pos_encoding=True, output_hidden_states=True)
            (out.hidden_states[-1].float() * up).sum().backward()
        arms = {"vit2spn_fwd": ours_fwd, "transformers_fwd": hf_fwd, "vit2spn_fwd_bwd": ours_fb, "transformers_fwd_bwd": hf_fb}
        for f in arms.values():
            for _ in range(2):
                f()
        torch.cuda.synchronize()
        times = {k: [] for k in arms}
        for _ in range(a.rounds):
            for k, f in arms.items():
                _time(f, a.iters, times[k])
        assert _lib.lib.v2s_debug_flag() == 0
        res["points"][f"{side}px"] = {"tokens": n, "batch": B, "tokens_per_batch": n * B,
                                      "ms_per_call": {k: _stats(v) for k, v in times.items()},
                                      "us_per_image": {k: 1000.0 * _stats(v)["median"] / B for k, v in times.items()}}
        print(side, B, {k: round(1000.0 * _stats(v)["median"] / B, 2) for k, v in times.items()}, flush=True)

    if a.bench:
        lines = {"this": [], "parent": []}
        order = (("parent", a.parent_tree), ("this", ROOT))
        for r in range(a.bench_rounds):        # ABBA: neither tree always runs first
            for name, tree in (order if r % 2 == 0 else order[::-1]):
                if not tree:
                    continue
                proc = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "30", "--warmup", "10"],
                                      cwd=tree, capture_output=True, text=True)
                line = [L for L in proc.stdout.splitlines() if L.startswith("{")]
                lines[name].append(json.loads(line[-1]) if line else {"error": proc.stderr[-400:]})
        res["bench"] = lines

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res["gpu"] = smi[0] if smi else torch.cuda.get_device_name(0)
    res["note"] = ("CUDA events around --iters calls, the four arms alternated over --rounds rounds (median, min, max); "
                   "transformers: stock eager ViTModel under torch.autocast(bfloat16), same weights; bench: the default "
                   "bench.py line (30 steps, 10 warm-up) of this tree and of the parent commit, in ABBA order")
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(res["gpu"])


if __name__ == "__main__":
    main()
