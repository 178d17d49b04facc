"""Golden vectors that pin the fine-tune / evaluation path (SURVEY §8f N2) to the REFERENCE.

Needs the original ViT-2SPN:   V2S_REFERENCE_DIR=/path/to/ViT-2SPN python tests/golden/make_finetune_golden.py

`ViTBackbone` and `FineTunedModel` are AST-extracted from $V2S_REFERENCE_DIR/octmnist_ft_vit2spn.py:63-87 and executed
unmodified (``from_pretrained`` redirected to the random-init tiny config: no checkpoint offline).  One training step
as the script does it (ref:95-104,187-192: train mode, weighted CrossEntropyLoss, Adam lr 1e-4 with L2 1e-4) and one
evaluation forward (ref:129-137: eval mode, softmax) are recorded in tests/golden/finetune_golden.npz.  Dropout(0.5)
is neutralised (p = 0) on the reference side, as every parity test does on the build side.  No reference source is
copied: the class bodies are read and exec'd from where they lie."""
import os
import sys

import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from oracle import vit2spn_oracle as orc  # noqa: E402
from make_golden import REF, extract_classes  # noqa: E402

NUM_CLASSES, BATCH, SLICE = 4, 6, 64
CLASS_WEIGHTS = [1.0, 2.0, 0.5, 1.5]
LABELS = [0, 1, 2, 3, 1, 2]


def head_state(seed=5):
    """deterministic fc head: Linear(192,128) - BatchNorm1d(128) - ReLU - Dropout - Linear(128,C)"""
    rng = np.random.Generator(np.random.PCG64(seed))
    t = lambda *s, scale=0.05: torch.from_numpy((rng.standard_normal(s) * scale).astype(np.float32))  # noqa: E731
    return {"fc.0.weight": t(128, 192), "fc.0.bias": t(128), "fc.1.weight": 1.0 + t(128), "fc.1.bias": t(128),
            "fc.1.running_mean": t(128), "fc.1.running_var": 1.0 + t(128).abs(),
            "fc.1.num_batches_tracked": torch.tensor(3), "fc.4.weight": t(NUM_CLASSES, 128), "fc.4.bias": t(NUM_CLASSES)}


def full_state():
    sub = orc.sub_state(orc.init_state(9, 0.02), "online_network_1")
    st = {"backbone.vit." + k: v for k, v in sub.items()}
    st.update(head_state())
    return st


def inputs():
    return orc.synthetic_views(BATCH, seed=2)[0], torch.tensor(LABELS)


def main():
    from transformers import ViTConfig, ViTModel

    class _OfflineViTModel(ViTModel):
        @classmethod
        def from_pretrained(cls, name, **kw):
            return ViTModel(ViTConfig(hidden_size=192, num_hidden_layers=12, num_attention_heads=3,
                                      intermediate_size=768, patch_size=16, image_size=224, **kw))

    ns = {"torch": torch, "nn": nn, "ViTModel": _OfflineViTModel}
    extract_classes(os.path.join(REF, "octmnist_ft_vit2spn.py"), {"ViTBackbone", "FineTunedModel"}, ns)
    model = ns["FineTunedModel"](NUM_CLASSES)
    state = full_state()
    res = model.load_state_dict(state, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    x, y = inputs()
    out = {"keys": np.array(list(model.state_dict().keys()))}
    # evaluation forward (ref:129-137)
    model.eval()
    with torch.no_grad():
        out["eval_probs"] = torch.softmax(model(x), dim=1).numpy()
    # one training step (ref:95-104, 187-192)
    model.train()
    model.fc[3].p = 0.0
    crit = nn.CrossEntropyLoss(weight=torch.tensor(CLASS_WEIGHTS))
    opt = torch.optim.Adam(model.parameters(), lr=1e-4, weight_decay=1e-4)
    opt.zero_grad()
    logits = model(x)
    loss = crit(logits, y)
    loss.backward()
    names = [n for n, p in model.named_parameters() if p.grad is not None]
    out["logits"] = logits.detach().numpy()
    out["loss"] = np.array(loss.item(), np.float64)
    out["grad_names"] = np.array(names)
    grads = dict(model.named_parameters())
    out["grad_norms"] = np.array([grads[n].grad.double().norm().item() for n in names])
    out["grad_slices"] = np.stack([np.pad(grads[n].grad.flatten()[:SLICE].numpy(), (0, max(0, SLICE - grads[n].numel())))
                                   for n in names])
    opt.step()
    post = model.state_dict()
    out["post_norms"] = np.array([post[k].double().norm().item() for k in post])
    out["post_fc0_weight_slice"] = post["fc.0.weight"].flatten()[:SLICE].numpy()
    out["post_bn_running_mean"] = post["fc.1.running_mean"].numpy()
    out["post_bn_running_var"] = post["fc.1.running_var"].numpy()
    # the oracle backbone under the same head, reported at generation time
    leaves = {k: v.clone().requires_grad_(True) for k, v in orc.sub_state(orc.init_state(9, 0.02), "online_network_1").items()}
    head = nn.Sequential(nn.Linear(192, 128), nn.BatchNorm1d(128), nn.ReLU(), nn.Dropout(0.0), nn.Linear(128, NUM_CLASSES))
    head.load_state_dict({k[3:]: v for k, v in head_state().items()})
    head.train()
    o_loss = crit(head(orc.backbone_features(leaves, x)), y)
    print(f"reference loss {loss.item():.8f}  oracle backbone + same head {o_loss.item():.8f}  "
          f"rel {abs(o_loss.item() - loss.item()) / abs(loss.item()):.2e}; {len(names)} tensors with gradients")
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "finetune_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
