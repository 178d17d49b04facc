"""Golden vectors that pin the single-stream variant (SURVEY §8f N3) to the REFERENCE.

Needs the original ViT-2SPN:   V2S_REFERENCE_DIR=/path/to/ViT-2SPN python tests/golden/make_single_golden.py

`ViTBackbone` and `SingleStreamNetwork` are AST-extracted from $V2S_REFERENCE_DIR/dsn_ssn/ssp_single.py:93-138 and
executed unmodified (``from_pretrained`` redirected to the random-init tiny config).  One micro-step as the script does
it (ref:195-206: loss = -mean(cos)/accumulation_steps with accumulation_steps = 8, backward, Adam lr 1e-4,
`update_target_network()` with its default momentum 0.99) is recorded in tests/golden/single_golden.npz; Dropout(0.3)
neutralised (p = 0).  No reference source is copied."""
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

BATCH, SLICE, ACCUM = 3, 64, 8


def heads_state(seed=6):
    rng = np.random.Generator(np.random.PCG64(seed))
    t = lambda *s, scale=0.03: torch.from_numpy((rng.standard_normal(s) * scale).astype(np.float32))  # noqa: E731
    return {"projection_head.0.weight": t(1024, 192), "projection_head.0.bias": t(1024),
            "projection_head.3.weight": t(128, 1024), "projection_head.3.bias": t(128),
            "prediction_head.0.weight": t(128, 128, scale=0.08), "prediction_head.0.bias": t(128),
            "prediction_head.2.weight": t(128, 128, scale=0.08), "prediction_head.2.bias": t(128)}


def full_state():
    base = orc.init_state(13, 0.01)
    st = {"online_network.vit." + k: v for k, v in orc.sub_state(base, "online_network_1").items()}
    st.update({"target_network.vit." + k: v for k, v in orc.sub_state(base, "target_network_1").items()})
    st.update(heads_state())
    return st


def inputs():
    return orc.synthetic_views(BATCH, seed=4)


def main():
    from transformers import ViTConfig, ViTModel

    class _OfflineViTModel(ViTModel):
        @classmethod
        def from_pretrained(cls, name, **kw):
            return ViTModel(ViTConfig(hidden_size=192, num_hidden_layers=12, num_attention_heads=3,
                                      intermediate_size=768, patch_size=16, image_size=224, **kw))

    ns = {"torch": torch, "nn": nn, "ViTModel": _OfflineViTModel}
    extract_classes(os.path.join(REF, "dsn_ssn", "ssp_single.py"), {"ViTBackbone", "SingleStreamNetwork"}, ns)
    model = ns["SingleStreamNetwork"]()
    res = model.load_state_dict(full_state(), strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    model.train()
    model.projection_head[2].p = 0.0
    v1, v2 = inputs()
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    opt.zero_grad()
    pred, tgt = model(v1, v2)
    loss = -torch.mean(nn.CosineSimilarity(dim=1)(pred, tgt)) / ACCUM
    loss.backward()
    named = dict(model.named_parameters())
    names = [n for n, p in named.items() if p.grad is not None]
    out = {"keys": np.array(list(model.state_dict().keys())), "pred": pred.detach().numpy(), "tgt": tgt.detach().numpy(),
           "loss": np.array(loss.item(), np.float64), "grad_names": np.array(names),
           "grad_norms": np.array([named[n].grad.double().norm().item() for n in names]),
           "grad_slices": np.stack([np.pad(named[n].grad.flatten()[:SLICE].numpy(), (0, max(0, SLICE - named[n].numel())))
                                    for n in names])}
    opt.step()
    model.update_target_network()
    post = model.state_dict()
    out["post_norms"] = np.array([post[k].double().norm().item() for k in post])
    out["post_target_pos_slice"] = post["target_network.vit.embeddings.position_embeddings"].flatten()[:SLICE].numpy()
    print(f"reference single-stream loss {loss.item():.8f}; {len(names)} tensors with gradients, {len(post)} state tensors")
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "single_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
