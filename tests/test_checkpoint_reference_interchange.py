"""Checkpoint interchange with the reference (SURVEY §8f N4): a file in the layout the reference's ``save_checkpoint``
writes (ref:ssp_vit2spn_tiny.py:53-61, stored in tests/golden/reference_checkpoint_layout.json by
tests/golden/make_checkpoint_golden.py) loads here bit for bit, and the file this library writes has that same layout
and loads the way the reference's ``load_checkpoint`` reads it (ref:63-72: ``torch.load``, then ``load_state_dict``
into the model and into ``torch.optim.Adam``)."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_checkpoint_golden as mk  # noqa: E402  (helpers only)

with open(mk.GOLDEN) as _f:
    G = json.load(_f)


def _same_adam_state(a, b):
    assert set(a) == set(b) and len(a) == 408                   # Adam state of the 400 + 8 trainable tensors
    for k in a:
        for f in ("exp_avg", "exp_avg_sq"):
            assert torch.equal(a[k][f].cpu(), b[k][f].cpu()), (k, f)
        assert float(a[k]["step"]) == float(b[k]["step"])


def test_reference_checkpoint_loads_here_and_ours_loads_there(tmp_path):
    import vit2spn
    ref = mk.reference_checkpoint(10, 0.25)
    assert mk.layout(ref) == G                                  # torch.optim.Adam still writes the stored layout
    path = os.path.join(tmp_path, "ref_ckpt.pth")
    torch.save(ref, path)
    ours = vit2spn.DualStreamNetwork()
    ours_opt = vit2spn.FusedAdam(ours.parameters(), lr=1e-4)
    _, _, epoch, loss = vit2spn.load_checkpoint(ours, ours_opt, path)           # a reference file, read here
    assert epoch == 10 and loss == 0.25
    ref_sd, our_sd = ref["model_state_dict"], ours.state_dict()
    assert list(ref_sd) == list(our_sd)
    assert all(torch.equal(ref_sd[k], our_sd[k]) for k in ref_sd)
    _same_adam_state(ref["optimizer_state_dict"]["state"], ours_opt.state_dict()["state"])

    # and back: this library writes the reference's layout, and the reference's way of reading it restores the state
    back = os.path.join(tmp_path, "our_ckpt.pth")
    vit2spn.save_checkpoint(ours, ours_opt, 11, 0.5, back)
    ck = torch.load(back)
    assert mk.layout(ck) == G
    assert ck["epoch"] == 11 and ck["loss"] == 0.5
    assert all(torch.equal(ck["model_state_dict"][k], ref_sd[k]) for k in ref_sd)
    params = [torch.nn.Parameter(torch.zeros(shape), requires_grad=not name.startswith(mk.FROZEN))
              for name, shape, _ in G["model_state_dict"]]
    torch_opt = torch.optim.Adam(params, lr=1e-4)
    torch_opt.load_state_dict(ck["optimizer_state_dict"])
    _same_adam_state(ref["optimizer_state_dict"]["state"], torch_opt.state_dict()["state"])
