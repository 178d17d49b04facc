"""Generate the golden vectors that pin ``oracle/vit2spn_oracle.py`` to the REFERENCE.

Needs a checkout of the original mrsaraei/ViT-2SPN, which the repository does not contain:

    V2S_REFERENCE_DIR=/path/to/ViT-2SPN python tests/golden/make_golden.py

The reference scripts train at import time, so their class definitions (``ViTBackbone``,
``DualStreamNetwork``) are AST-extracted from
  * $V2S_REFERENCE_DIR/ssp_ssl/ssl_vit2spn_scratch.py  (random-init ``ViTModel(ViTConfig(...))``)
  * $V2S_REFERENCE_DIR/ssp_vit2spn_tiny.py             (``from_pretrained`` redirected to the same
    random-init tiny config: no checkpoint / network offline)
and executed, unmodified, against the installed ``transformers`` / ``torch``.  The oracle's
deterministic state (numpy PCG64) is loaded into them with ``load_state_dict(strict=True)``;
the outputs of the reference modules (loss, pred/target projections, features, per-tensor
gradient norms and slices, post-Adam and post-EMA weights) are stored in
``tests/golden/ssp_golden.npz``.  Dropout(0.3) of the projection head is neutralised (p=0) on
the reference side (SURVEY D11), exactly as every parity test does on the build side.
No reference source is copied into the repo: the class bodies are read and exec'd from where
they lie.
"""
import ast
import os
import sys

import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import vit2spn_oracle as orc  # noqa: E402

REF = os.environ.get("V2S_REFERENCE_DIR", "")        # empty: the original is not available


def extract_classes(path, names, namespace):
    src = open(path).read()
    tree = ast.parse(src)
    for node in tree.body:
        if isinstance(node, (ast.ClassDef, ast.FunctionDef)) and node.name in names:
            code = compile(ast.Module(body=[node], type_ignores=[]), path, "exec")
            exec(code, namespace)
    return namespace


def reference_namespace(script):
    from transformers import ViTConfig, ViTModel

    class _OfflineViTModel(ViTModel):
        @classmethod
        def from_pretrained(cls, name, **kw):   # no HF checkpoint offline → same tiny config
            return ViTModel(ViTConfig(hidden_size=192, num_hidden_layers=12, num_attention_heads=3,
                                      intermediate_size=768, patch_size=16, image_size=224, **kw))

    ns = {"torch": torch, "nn": nn, "ViTModel": _OfflineViTModel, "ViTConfig": ViTConfig,
          "momentum": 0.999}
    return extract_classes(os.path.join(REF, script), {"ViTBackbone", "DualStreamNetwork"}, ns)


def run_reference(script, state, x1, x2, accumulation_steps):
    ns = reference_namespace(script)
    torch.manual_seed(0)
    model = ns["DualStreamNetwork"]()
    missing = model.load_state_dict(state, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    model.train()
    model.projection_head[2].p = 0.0          # neutralise Dropout(0.3) (D11)
    names = [n for n, _ in model.named_parameters()]
    assert names == orc.model_param_names(), "state_dict order differs from oracle.model_param_names()"
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    crit = nn.CosineSimilarity(dim=1)
    opt.zero_grad()
    pred, tgt = model(x1, x2)
    loss = -torch.mean(crit(pred, tgt)) / accumulation_steps
    loss.backward()
    with torch.no_grad():
        f1 = model.online_network_1(x1)
        hid = model.online_network_1.vit(x1).hidden_states[-1]
    grads = {n: (p.grad.detach().clone() if p.grad is not None else None) for n, p in model.named_parameters()}
    opt.step()
    model.update_target_network()
    post = {k: v.detach().clone() for k, v in model.state_dict().items()}
    return dict(loss=loss.detach(), pred=pred.detach(), tgt=tgt.detach(), feat1=f1, hidden1=hid,
                grads=grads, post=post)


SLICE = 64   # elements of each flattened tensor kept in the fixture


def main():
    out = {}
    cases = [("init", 42, 0.0, 4, 1), ("perturbed", 8, 0.02, 3, 8)]
    for tag, seed, perturb, B, accum in cases:
        state = orc.init_state(seed, perturb)
        x1, x2 = orc.synthetic_views(B, seed=seed)
        ref = run_reference("ssp_ssl/ssl_vit2spn_scratch.py", state, x1, x2, accum)
        ref2 = run_reference("ssp_vit2spn_tiny.py", state, x1, x2, accum)
        # the two reference variants must agree bit-for-bit (same classes modulo constructor)
        assert torch.equal(ref["loss"], ref2["loss"]) and torch.equal(ref["pred"], ref2["pred"])
        for k in ref["grads"]:
            a, b = ref["grads"][k], ref2["grads"][k]
            assert (a is None) == (b is None) and (a is None or torch.equal(a, b)), k

        # oracle vs reference, reported at generation time
        loss, pred, tgt, g = orc.loss_and_grads(dict(state), x1, x2, accum)
        rel = abs(loss.item() - ref["loss"].item()) / abs(ref["loss"].item())
        num = sum(((g[k] - ref["grads"][k]) ** 2).sum().item() for k in g)
        den = sum((ref["grads"][k] ** 2).sum().item() for k in g)
        none_names = sorted(k for k, v in ref["grads"].items() if v is None)
        print(f"[{tag}] ref loss {ref['loss'].item():.8f} oracle {loss.item():.8f} rel {rel:.2e}; "
              f"grad rel-L2 {np.sqrt(num / den):.2e}; grad-None tensors {len(none_names)}")
        assert sorted(set(orc.model_param_names()) - set(orc.trainable_names())) == none_names

        out[f"{tag}/meta"] = np.array([seed, perturb, B, accum], dtype=np.float64)
        out[f"{tag}/loss"] = ref["loss"].numpy().astype(np.float64)
        out[f"{tag}/pred"] = ref["pred"].numpy()
        out[f"{tag}/tgt"] = ref["tgt"].numpy()
        out[f"{tag}/feat1"] = ref["feat1"].numpy()
        out[f"{tag}/hidden1_slice"] = ref["hidden1"][:, ::49, :].numpy()   # tokens 0,49,98,147,196
        gn, gs, pn, ps = [], [], [], []
        for k in orc.model_param_names():
            gr = ref["grads"][k]
            if gr is not None:
                gn.append(gr.double().norm().item())
                gs.append(gr.flatten()[:SLICE].numpy())
            pn.append(ref["post"][k].double().norm().item())
            ps.append(ref["post"][k].flatten()[:SLICE].numpy())
        out[f"{tag}/grad_norms"] = np.array(gn)
        out[f"{tag}/grad_slices"] = np.stack([np.pad(s, (0, SLICE - len(s))) for s in gs])
        out[f"{tag}/post_norms"] = np.array(pn)
        out[f"{tag}/post_slices"] = np.stack([np.pad(s, (0, SLICE - len(s))) for s in ps])
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ssp_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
