"""Device cost of the gradients w.r.t. the attention probabilities at B=128, bf16.  Two arms alternated in one process,
both forward + backward of a trainable vit2spn.ViTModel(x, output_attentions=True) with the loss on hidden_states[-1]:
  plain       no attention retains its gradient (the kernels of a backward without the feature)
  retain_all  retain_grad() on all 12 attentions (12 more launches of the dP = d ctx V^T kernel)
then per-class device times (v2s_prof) of one call of each arm in a separate pass, and the kernel on its own
(v2s_test_attention which = 3, back to back, CUDA events) next to the probabilities kernel it mirrors (which = 2).
Writes --out (JSON)."""
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
    ap.add_argument("--kernel-iters", type=int, default=200)
    ap.add_argument("--out", default="attn_grad_cost.json")
    a = ap.parse_args()
    import vit2spn
    from vit2spn import _lib
    from oracle import vit2spn_oracle as orc
    dev = torch.device("cuda", 0)
    B = a.batch
    m = vit2spn.ViTModel()
    m.load_state_dict(orc.sub_state(orc.init_state(11, 0.01), "online_network_1"), strict=True)
    m.to(dev).compute_mode = "bf16"
    x = orc.preprocess_u8(orc.synthetic_octmnist_u8(B, 0)).to(dev)
    up = torch.randn(B, 197, 192, device=dev)

    def run(retain):
        m.zero_grad(set_to_none=False)
        out = m(x, output_attentions=True)
        if retain:
            for t in out.attentions:
                t.retain_grad()
        (out.hidden_states[-1] * up).sum().backward()
    arms = {"plain": lambda: run(False), "retain_all": lambda: run(True)}
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
    n, ms, _, nbytes = classes["retain_all"]["attn_dprobs"]

    # the kernel alone: dP of one block (which 3) and the probabilities (which 2), bf16, back to back
    g = torch.Generator(device=dev).manual_seed(0)
    qkv = torch.randn(B, 197, 576, device=dev, generator=g).to(torch.bfloat16)
    dctx = (torch.randn(B, 197, 192, device=dev, generator=g) * 1e-2).to(torch.bfloat16)
    lse = torch.empty(B, 3, 197, device=dev)
    ctx = torch.empty(B, 197, 192, device=dev, dtype=torch.bfloat16)
    outp = torch.empty(B, 3, 197, 197, device=dev)
    _lib.check(_lib.lib.v2s_test_attention(0, _lib.ptr(qkv), _lib.ptr(ctx), _lib.ptr(lse), None, None, B, 0,
                                           _lib.stream_ptr()), "attention fwd")
    alone = {}
    for which, name in ((3, "attn_dprobs"), (2, "attn_probs")):
        def launch():
            _lib.check(_lib.lib.v2s_test_attention(which, _lib.ptr(qkv), _lib.ptr(outp), _lib.ptr(lse), _lib.ptr(dctx),
                                                   None, B, 0, _lib.stream_ptr()), name)
        for _ in range(10):
            launch()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.kernel_iters):
            launch()
        e1.record()
        torch.cuda.synchronize()
        alone[name] = round(e0.elapsed_time(e1) * 1e3 / a.kernel_iters, 2)
    assert _lib.lib.v2s_debug_flag() == 0

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    written = B * 3 * 197 * 197 * 4
    res = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0), "batch": B, "mode": "bf16",
           "ms_per_fwd_bwd": {k: {"median": sorted(v)[len(v) // 2], "min": min(v), "max": max(v)} for k, v in times.items()},
           "attn_dprobs_per_launch": {"launches": n, "us_in_backward": round(ms * 1e3 / n, 2),
                                      "us_alone": alone["attn_dprobs"], "attn_probs_us_alone": alone["attn_probs"],
                                      "algorithmic_bytes": nbytes / n, "bytes_written": written,
                                      "bytes_read": nbytes / n - written,
                                      "GB_per_s_in_backward": round(nbytes / n / (ms / n * 1e-3) / 1e9, 1)},
           "classes_ms": {k: {c: [cnt, round(t, 4)] for c, (cnt, t, _, _) in v.items()} for k, v in classes.items()},
           "note": "CUDA events around iters forward+backward calls, arms alternated per round; classes: one call with "
                   "v2s_prof enabled (launches, device ms); us_alone: CUDA events around kernel_iters back-to-back "
                   "launches of the test hook on the same inputs (the 79 MB working set is partly L2-resident)"}
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["ms_per_fwd_bwd"]), json.dumps(res["attn_dprobs_per_launch"]), res["gpu"])


if __name__ == "__main__":
    main()
