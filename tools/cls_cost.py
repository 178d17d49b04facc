"""What the classification head costs next to the backbone, on one GPU: ``vit2spn.ViTForImageClassification`` against
the same CUDA backbone with the eager recipe users wrote before it (``ViTModel(...).last_hidden_state[:, 0]`` ->
``nn.Linear`` -> ``F.cross_entropy``), in three arms each: a fine-tune step (forward, backward, FusedAdam), a
linear-probe step (frozen ``vit``: forward, backward, FusedAdam on the classifier) and an inference forward.  B = 128,
bf16, num_labels 4 (OCTMNIST) and 1000 (ImageNet-1k); all arms alternate in one process, device-event timed, several
rounds.  The card's name and power limit are read in the same run.

    python tools/cls_cost.py [--batch 128] [--steps 20] [--rounds 5] [--out profiles/cls_cost_r01.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("V2S_ALLOW_RANDOM_INIT", "1")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def arms_for(n_labels, x, y, dev):
    import torch
    import vit2spn
    torch.manual_seed(0)
    fused = vit2spn.ViTForImageClassification(vit2spn.ViTConfig(num_labels=n_labels)).to(dev)
    fused.compute_mode = "bf16"
    vit = vit2spn.ViTModel(add_pooling_layer=False).to(dev)
    vit.compute_mode = "bf16"
    fc = torch.nn.Linear(192, n_labels).to(dev)
    vit.load_state_dict({k[4:]: v for k, v in fused.state_dict().items() if k.startswith("vit.")}, strict=True)
    fc.load_state_dict({"weight": fused.classifier.weight.detach(), "bias": fused.classifier.bias.detach()})
    opt_f = vit2spn.FusedAdam(fused.parameters(), lr=1e-5)
    opt_t = vit2spn.FusedAdam(list(vit.parameters()) + list(fc.parameters()), lr=1e-5)
    opt_fp = vit2spn.FusedAdam(fused.classifier.parameters(), lr=1e-5)
    opt_tp = vit2spn.FusedAdam(fc.parameters(), lr=1e-5)

    def eager(v):
        return fc(v(x).last_hidden_state[:, 0])

    def finetune_cuda():
        fused.vit.requires_grad_(True)
        opt_f.zero_grad()
        fused(x, labels=y).loss.backward()
        opt_f.step()

    def finetune_eager():
        vit.requires_grad_(True)
        opt_t.zero_grad()
        torch.nn.functional.cross_entropy(eager(vit), y).backward()
        opt_t.step()

    def probe_cuda():
        fused.vit.requires_grad_(False)
        opt_fp.zero_grad()
        fused(x, labels=y).loss.backward()
        opt_fp.step()

    def probe_eager():
        vit.requires_grad_(False)
        opt_tp.zero_grad()
        torch.nn.functional.cross_entropy(eager(vit), y).backward()
        opt_tp.step()

    def infer_cuda():
        with torch.no_grad():
            return fused(x).logits

    def infer_eager():
        with torch.no_grad():
            return eager(vit)

    return {"finetune": (finetune_cuda, finetune_eager), "probe": (probe_cuda, probe_eager),
            "inference": (infer_cuda, infer_eager)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "cls_cost_r01.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("cls_cost: no CUDA device (this measurement runs on the GPU only)")
    from oracle import vit2spn_oracle as orc
    dev = torch.device("cuda", 0)
    B = a.batch
    x = orc.preprocess_u8(orc.synthetic_octmnist_u8(B, 0)).to(dev)
    res = {"card": card(), "batch": B, "mode": "bf16", "steps_per_round": a.steps, "rounds": a.rounds, "labels": {},
           "note": "finetune / probe step = forward + backward + FusedAdam (probe: frozen vit, classifier only); "
                   "inference = no-grad forward; cuda = ViTForImageClassification, eager = the same CUDA backbone's "
                   "last_hidden_state[:, 0] -> nn.Linear -> F.cross_entropy; ms per step, device events"}
    for n in (4, 1000):
        y = torch.randint(0, n, (B,), generator=torch.Generator().manual_seed(n)).to(dev)
        arms = arms_for(n, x, y, dev)
        fns = {f"{arm}_{side}": fn for arm, pair in arms.items() for side, fn in zip(("cuda", "eager"), pair)}
        for fn in fns.values():                   # warm-up: every shape, workspaces, kernel attributes
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        times = {k: [] for k in fns}
        for _ in range(a.rounds):
            for k, fn in fns.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.steps):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1) / a.steps)
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        res["labels"][str(n)] = {
            "step_ms": {k: {"median": med[k], "min": min(v), "max": max(v), "all": v} for k, v in times.items()},
            "eager_minus_cuda_ms": {arm: med[f"{arm}_eager"] - med[f"{arm}_cuda"] for arm in arms}}
        print(json.dumps({"num_labels": n, "median_ms": med}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))


if __name__ == "__main__":
    main()
