"""Golden layout of the checkpoint the reference's training script writes (ref:ssp_vit2spn_tiny.py:53-61:
``save_checkpoint`` = ``torch.save`` of {epoch, model_state_dict, optimizer_state_dict, loss} for its
``DualStreamNetwork`` and ``torch.optim.Adam(model.parameters(), lr=1e-4)``, ref:173), stored in
tests/golden/reference_checkpoint_layout.json:   python tests/golden/make_checkpoint_golden.py

The reference side is built from what the repository already pins to the reference: the 808 state_dict keys in
registration order (``oracle.model_param_names()``, asserted equal to the reference's ``named_parameters()`` by
make_golden.py), frozen target networks (ref:128-131), and stock ``torch.optim.Adam`` after one step.  With
V2S_REFERENCE_DIR naming a checkout of the original ViT-2SPN, the reference's own ``DualStreamNetwork`` and
``save_checkpoint`` (AST-extracted, executed unmodified) also write a file, and its layout must be the same."""
import json
import os
import sys
import tempfile
from collections import OrderedDict

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from oracle import vit2spn_oracle as orc  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_checkpoint_layout.json")
FROZEN = ("target_network_1.", "target_network_2.")


def _seeded_adam_step(params):
    """torch.optim.Adam (lr 1e-4) over `params` after one step on seeded gradients for every trainable tensor."""
    opt = torch.optim.Adam(params, lr=1e-4)
    g = torch.Generator().manual_seed(0)
    for p in params:
        if p.requires_grad:
            p.grad = torch.randn(p.shape, generator=g) * 1e-3
    opt.step()
    return opt


def reference_checkpoint(epoch, loss):
    """A checkpoint dict as the reference writes it: oracle state (seed 31, perturbation 0.01) and Adam state."""
    state = orc.init_state(31, 0.01)
    names = orc.model_param_names()
    params = [nn.Parameter(state[k].clone(), requires_grad=not k.startswith(FROZEN)) for k in names]
    opt = _seeded_adam_step(params)
    sd = OrderedDict((k, p.detach()) for k, p in zip(names, params))
    return {"epoch": epoch, "model_state_dict": sd, "optimizer_state_dict": opt.state_dict(), "loss": loss}


def _describe(v, param_shape):
    if not torch.is_tensor(v):
        return [type(v).__name__]
    return ["Tensor", str(v.dtype), "param" if list(v.shape) == param_shape else list(v.shape)]


def layout(ck):
    """Everything about a checkpoint dict that another reader depends on, except the values: top-level keys, state_dict
    keys in order with shapes and dtypes, optimizer param_groups, which parameters have Adam state and the type, dtype
    and shape of each state field."""
    sd, opt = ck["model_state_dict"], ck["optimizer_state_dict"]
    shapes = [list(v.shape) for v in sd.values()]
    groups = [dict({k: (list(v) if isinstance(v, tuple) else v) for k, v in g.items() if k != "params"},
                   params=list(g["params"])) for g in opt["param_groups"]]
    fields = {json.dumps({f: _describe(v, shapes[i]) for f, v in sorted(st.items())}) for i, st in opt["state"].items()}
    return {"keys": sorted(ck),
            "model_state_dict": [[k, list(v.shape), str(v.dtype)] for k, v in sd.items()],
            "param_groups": groups,
            "state_indices": sorted(opt["state"]),
            "state_fields": [json.loads(f) for f in sorted(fields)]}


def main():
    out = layout(reference_checkpoint(10, 0.25))
    ref = os.environ.get("V2S_REFERENCE_DIR", "")
    if ref:
        import make_golden as mg
        script = os.path.join(ref, "ssp_vit2spn_tiny.py")
        ns = mg.reference_namespace("ssp_vit2spn_tiny.py")
        ns["os"] = os
        mg.extract_classes(script, {"save_checkpoint"}, ns)
        model = ns["DualStreamNetwork"]()
        model.load_state_dict(orc.init_state(31, 0.01), strict=True)
        opt = _seeded_adam_step(list(model.parameters()))
        with tempfile.TemporaryDirectory() as d:
            path = os.path.join(d, "ref_ckpt.pth")
            ns["save_checkpoint"](model, opt, 10, 0.25, path)
            assert layout(torch.load(path)) == out, "the original ViT-2SPN writes another checkpoint layout"
        print("the original's save_checkpoint writes the same layout")
    with open(GOLDEN, "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print("wrote", GOLDEN, os.path.getsize(GOLDEN), "bytes")


if __name__ == "__main__":
    main()
