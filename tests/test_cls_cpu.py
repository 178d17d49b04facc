"""CPU: ``vit2spn.ViTForImageClassification`` and what it needs from the rest of the package.

* ``state_dict`` keys and order equal ``transformers.ViTForImageClassification``'s 200 keys, and load strictly both ways;
* ``cls_oracle`` (the head in float64 on the oracle's backbone) equals transformers' logits, loss and gradients for the
  three problem types, ignored labels, an all-ignored batch and num_labels 1, 4 and 1000;
* ``problem_type`` inference and its config mutation match transformers';
* the errors raised before anything runs on the device, and the C entry points' argument checks;
* ``from_pretrained`` with classification, ViTModel and SimMIM checkpoints, a classifier-size mismatch and a bad one.
"""
import ctypes as C
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import cls_oracle as co  # noqa: E402  (helper module, not a test)


def _cfg(transformers, **kw):
    return transformers.ViTConfig(hidden_size=192, num_hidden_layers=12, num_attention_heads=3, intermediate_size=768,
                                  patch_size=16, image_size=224, layer_norm_eps=1e-12, hidden_act="gelu", qkv_bias=True,
                                  attn_implementation="eager", **kw)


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def _weights(seed, n):
    from oracle import vit2spn_oracle as orc
    p = orc.sub_state(orc.init_state(seed, 0.01), "online_network_1")
    g = torch.Generator().manual_seed(seed + 100)
    return p, 0.05 * torch.randn(n, 192, generator=g), 0.02 * torch.randn(n, generator=g)


def _labels(kind, B, n, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "single_label_classification":
        y = torch.randint(0, n, (B,), generator=g)
        y[1] = -100
        return y
    if kind == "regression":
        return torch.randn(B, n, generator=g)
    return (torch.rand(B, n, generator=g) < 0.3).float()


def test_state_dict_keys_order_and_strict_loads_match_transformers():
    transformers = pytest.importorskip("transformers")
    import vit2spn
    hf = transformers.ViTForImageClassification(_cfg(transformers, num_labels=4))
    ours = vit2spn.ViTForImageClassification(vit2spn.ViTConfig(num_labels=4))
    assert list(ours.state_dict()) == list(hf.state_dict()) and len(hf.state_dict()) == 200
    assert sum(k.startswith("vit.") for k in ours.state_dict()) == 198
    w = ours.classifier.weight.detach()
    assert tuple(w.shape) == (4, 192) and abs(w.std().item() - 0.02) < 4e-3
    assert torch.count_nonzero(ours.classifier.bias) == 0
    for t in hf.state_dict().values():
        if t.is_floating_point():
            t.normal_()
    ours.load_state_dict(hf.state_dict(), strict=True)
    for k, v in hf.state_dict().items():
        assert torch.equal(ours.state_dict()[k], v), k
    hf2 = transformers.ViTForImageClassification(_cfg(transformers, num_labels=4))
    hf2.load_state_dict(ours.state_dict(), strict=True)
    assert vit2spn.ViTForImageClassification().classifier.out_features == 2      # transformers' default num_labels


@pytest.mark.parametrize("n,kind", [(4, "single_label_classification"), (1000, "single_label_classification"),
                                    (4, "regression"), (1, "regression"), (4, "multi_label_classification"),
                                    (1000, "multi_label_classification")])
def test_oracle_matches_transformers(n, kind):
    transformers = pytest.importorskip("transformers")
    p, cw, cb = _weights(7, n)
    B = 3
    hf = transformers.ViTForImageClassification(_cfg(transformers, num_labels=n, problem_type=kind)).double().eval()
    sd = {"vit." + k: v for k, v in p.items() if not k.startswith("pooler.")}
    sd.update({"classifier.weight": cw, "classifier.bias": cb})
    hf.load_state_dict(sd, strict=True)
    x = torch.randn(B, 3, 224, 224, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    y = _labels(kind, B, n, 5)
    y = y.double() if y.is_floating_point() else y
    xh = x.clone().requires_grad_(True)
    out = hf(pixel_values=xh, labels=y)
    out.loss.backward()
    loss, logits, grads = co.model_loss({k: v.double() for k, v in p.items()}, cw.double(), cb.double(), x, y, kind)
    assert abs(loss.item() - out.loss.item()) <= 1e-10 * abs(out.loss.item())
    assert _rel(logits, out.logits.detach()) <= 1e-10
    named = dict(hf.named_parameters())
    for k in ("classifier.weight", "classifier.bias"):
        assert _rel(grads[k], named[k].grad) <= 1e-10, k
    for k in ("layernorm.weight", "layernorm.bias", "embeddings.patch_embeddings.projection.weight",
              "encoder.layer.0.attention.attention.query.weight", "encoder.layer.11.output.dense.weight"):
        assert _rel(grads[k], named["vit." + k].grad) <= 1e-10, k
    assert _rel(grads["pixels"], xh.grad) <= 1e-10
    # the 16-bit rounding model stays within the formats' resolution of the exact head
    h12 = hf.vit(pixel_values=x, output_hidden_states=True).hidden_states[-1].detach().float()
    y = y.float() if y.is_floating_point() else y
    z, l32 = co.head(h12, p["layernorm.weight"], p["layernorm.bias"], cw, cb, y, kind)
    for lp, tol in ((torch.bfloat16, 3e-2), (torch.float16, 4e-3)):
        z2, l2 = co.head(h12, p["layernorm.weight"], p["layernorm.bias"], cw, cb, y, kind, lp)
        assert 0 < _rel(z2, z) <= tol and abs(l2.item() - l32.item()) <= tol * abs(l32.item())


def test_oracle_ignored_labels_match_torch():
    n = 4
    p, cw, cb = _weights(8, n)
    h = torch.randn(3, 197, 192, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    lw, lb = p["layernorm.weight"].double(), p["layernorm.bias"].double()
    all_ignored = torch.full((3,), -100)
    _, loss = co.head(h, lw, lb, cw.double(), cb.double(), all_ignored, "single_label_classification")
    assert torch.isnan(loss).item()
    y = torch.tensor([1, -100, 3])
    z, loss = co.head(h, lw, lb, cw.double(), cb.double(), y, "single_label_classification")
    assert torch.allclose(loss, torch.nn.functional.cross_entropy(z[[0, 2]], y[[0, 2]]))


@pytest.mark.parametrize("n,dtype,want", [(1, torch.int64, "regression"), (1, torch.float32, "regression"),
                                          (4, torch.int64, "single_label_classification"),
                                          (4, torch.int32, "single_label_classification"),
                                          (4, torch.float32, "multi_label_classification"),
                                          (4, torch.int16, "multi_label_classification")])
def test_problem_type_inference_matches_transformers(n, dtype, want):
    transformers = pytest.importorskip("transformers")
    from transformers.loss.loss_utils import ForSequenceClassificationLoss
    import vit2spn
    hf_cfg = _cfg(transformers, num_labels=n)
    y = torch.zeros(2, dtype=dtype) if "single" in want or n == 1 else torch.zeros(2, n, dtype=dtype)
    try:
        ForSequenceClassificationLoss(y, torch.zeros(2, n), hf_cfg)
    except RuntimeError:
        pass                             # int16 multi-label: BCE refuses the dtype; the config is set before
    m = vit2spn.ViTForImageClassification(vit2spn.ViTConfig(num_labels=n))
    try:
        m._labels(y, torch.zeros(2, 3, 224, 224))
    except RuntimeError:
        pass
    assert m.config.problem_type == hf_cfg.problem_type == want


def test_label_errors_are_torchs():
    import vit2spn
    m = vit2spn.ViTForImageClassification(vit2spn.ViTConfig(num_labels=4))
    x = torch.zeros(3, 3, 224, 224)
    with pytest.raises((ValueError, RuntimeError), match="batch_size|match"):
        m._labels(torch.zeros(5, dtype=torch.int64), x)
    m.config.problem_type = "multi_label_classification"
    with pytest.raises(ValueError, match="Target size"):
        m._labels(torch.zeros(3, 5), x)
    m.config.problem_type = "regression"
    kind, lab = m._labels(torch.zeros(3, 4, dtype=torch.float64), x)
    assert lab.dtype == torch.float32 and tuple(lab.shape) == (3, 4)
    m1 = vit2spn.ViTForImageClassification(vit2spn.ViTConfig(num_labels=1))
    kind, lab = m1._labels(torch.zeros(3, 1), x)             # a single label: both sides squeezed, as transformers
    assert tuple(lab.shape) == (3, 1)
    m.config.problem_type = "single_label_classification"
    with pytest.raises(RuntimeError, match="dtype"):
        m._labels(torch.zeros(3), x)                         # torch's own refusal of float class indices


def test_errors_before_the_device():
    import vit2spn
    with pytest.raises(ValueError, match="num_labels"):
        vit2spn.ViTForImageClassification(vit2spn.ViTConfig(num_labels=0))
    m = vit2spn.ViTForImageClassification()
    x = torch.zeros(2, 3, 224, 224)
    for kw in ({"head_mask": torch.ones(12, 3)}, {"interpolate_pos_encoding": True},
               {"bool_masked_pos": torch.zeros(2, 196, dtype=torch.bool)}, {"num_items_in_batch": 2}):
        with pytest.raises(ValueError, match=next(iter(kw))):
            m(x, **kw)
    with pytest.raises(ValueError, match="patch-row"):
        m(torch.zeros(2, 196, 768, dtype=torch.bfloat16))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(x, labels=torch.zeros(2, dtype=torch.int64))


def test_cls_entry_points_check_their_arguments():
    from vit2spn import _lib
    lib = _lib.lib
    M = _lib.MODE_BF16
    assert lib.v2s_cls_workspace_bytes(0, 4, 1) == -1 and lib.v2s_cls_workspace_bytes(2, 0, 1) == -1
    assert lib.v2s_cls_workspace_bytes(2, 65537, 1) == -1 and lib.v2s_cls_workspace_bytes(2, 4, 7) == -1
    n = lib.v2s_cls_workspace_bytes(2, 4, M)
    assert n >= 2 * 192 * 2 + 8 * 192 * 2
    ws = C.c_void_p(1 << 20)
    a = [C.c_void_p(0x10000 * (i + 1)) for i in range(10)]
    CE = _lib.CLS_LOSS_CE

    def fwd(*args, kind=CE, labels=a[5], loss=a[7], nbytes=n, wsp=ws, batch=2, nl=4):
        h, g, b, w, bias, logits = args if args else (a[0], a[1], a[2], a[3], a[4], a[6])
        return lib.v2s_cls_forward(h, g, b, w, bias, nl, kind, labels, logits, loss, 1, batch, M, wsp, nbytes, None)

    def err():
        return lib.v2s_last_error().decode()
    assert fwd(None, a[1], a[2], a[3], a[4], a[6]) != 0 and "null argument" in err()
    assert fwd(kind=CE, loss=None) != 0 and "null argument" in err()
    assert fwd(kind=_lib.CLS_LOSS_NONE) != 0 and "null argument" in err()            # a loss without a loss kind
    assert fwd(a[0], a[1], a[2], a[3], a[4], C.c_void_p(0x10004)) != 0 and "aligned" in err()
    assert fwd(kind=CE, labels=None) != 0 and "labels" in err()
    assert fwd(kind=9) != 0 and "loss_kind" in err()
    assert fwd(nbytes=n - 1024) != 0 and "workspace too small" in err()
    assert fwd(wsp=C.c_void_p((1 << 20) + 16)) != 0 and "1024-byte aligned" in err()
    assert fwd(batch=0) != 0 and "bad batch" in err()
    assert fwd(nl=70000) != 0 and "bad batch" in err()

    def bwd(dlogits=a[6], dloss=a[7], dg=a[9], dbeta=a[8], kind=CE, labels=a[5]):
        return lib.v2s_cls_backward(a[0], a[1], a[3], 4, kind, labels, dlogits, dloss, a[2], dg, dbeta, a[4], None, 2, M,
                                    ws, n, None)
    assert bwd(dlogits=None, dloss=None) != 0 and "null argument" in err()
    assert bwd(kind=_lib.CLS_LOSS_NONE, labels=None) != 0 and "null argument" in err()     # dloss without a loss
    assert bwd(dg=None) != 0 and "go together" in err()


def _save(sd, d, fmt="bin"):
    os.makedirs(d, exist_ok=True)
    if fmt == "safetensors":
        from safetensors.torch import save_file
        save_file({k: v.contiguous() for k, v in sd.items()}, os.path.join(d, "model.safetensors"))
    else:
        torch.save(sd, os.path.join(d, "pytorch_model.bin"))
    return d


def test_from_pretrained_classification_checkpoints(tmp_path, capfd):
    transformers = pytest.importorskip("transformers")
    import vit2spn
    hf = transformers.ViTForImageClassification(_cfg(transformers, num_labels=1000))
    for t in hf.parameters():
        t.data.normal_()
    d = _save(hf.state_dict(), str(tmp_path / "in1k"), "safetensors")
    m = vit2spn.ViTForImageClassification.from_pretrained(d)            # num_labels from the checkpoint
    assert m.config.num_labels == 1000
    for k, v in hf.state_dict().items():
        assert torch.equal(m.state_dict()[k], v), k
    # without the vit. prefix
    d2 = _save({k[4:] if k.startswith("vit.") else k: v for k, v in hf.state_dict().items()}, str(tmp_path / "bare"))
    assert torch.equal(vit2spn.ViTForImageClassification.from_pretrained(d2).classifier.weight, hf.classifier.weight)
    # another classifier size: an error naming ignore_mismatched_sizes, or a fresh classifier and a note on stderr
    with pytest.raises(RuntimeError, match="ignore_mismatched_sizes"):
        vit2spn.ViTForImageClassification.from_pretrained(d, num_labels=4)
    capfd.readouterr()
    m4 = vit2spn.ViTForImageClassification.from_pretrained(d, num_labels=4, ignore_mismatched_sizes=True)
    assert "newly initialized" in capfd.readouterr().err
    assert tuple(m4.classifier.weight.shape) == (4, 192) and torch.count_nonzero(m4.classifier.bias) == 0
    assert torch.equal(m4.vit.embeddings.cls_token, hf.vit.embeddings.cls_token)


def test_from_pretrained_backbone_and_simmim_checkpoints(tmp_path):
    transformers = pytest.importorskip("transformers")
    import vit2spn
    vm = transformers.ViTModel(_cfg(transformers))                     # pooler included
    for t in vm.parameters():
        t.data.normal_()
    m = vit2spn.ViTForImageClassification.from_pretrained(_save(vm.state_dict(), str(tmp_path / "vit")), num_labels=4)
    assert torch.equal(m.vit.embeddings.cls_token, vm.embeddings.cls_token) and m.config.num_labels == 4
    m2 = vit2spn.ViTForImageClassification.from_pretrained(_save(vm.state_dict(), str(tmp_path / "vit2")))
    assert m2.config.num_labels == 2
    # a ViT-2SPN backbone checkpoint (online_network_1.state_dict())
    net = vit2spn.DualStreamNetwork()
    ssp = str(tmp_path / "ssp.pth")
    torch.save(net.online_network_1.state_dict(), ssp)
    m3 = vit2spn.ViTForImageClassification.from_pretrained(ssp, num_labels=4)
    assert torch.equal(m3.vit.encoder.layer[2].output.dense.weight, net.online_network_1.vit.encoder.layer[2].output.dense.weight)
    mim = transformers.ViTForMaskedImageModeling(_cfg(transformers, encoder_stride=16))
    m4 = vit2spn.ViTForImageClassification.from_pretrained(_save(mim.state_dict(), str(tmp_path / "mim")), num_labels=4)
    assert torch.equal(m4.vit.layernorm.weight, mim.vit.layernorm.weight)
    bad = {k: v for k, v in vm.state_dict().items() if "encoder.layer.3." not in k}
    with pytest.raises(RuntimeError, match="missing"):
        vit2spn.ViTForImageClassification.from_pretrained(_save(bad, str(tmp_path / "bad")), num_labels=4)
    geo = transformers.ViTForImageClassification(transformers.ViTConfig(hidden_size=192, num_hidden_layers=2,
                                                                        num_attention_heads=3, intermediate_size=768,
                                                                        num_labels=4))
    with pytest.raises(RuntimeError, match="missing|size mismatch"):
        vit2spn.ViTForImageClassification.from_pretrained(_save(geo.state_dict(), str(tmp_path / "geo")))
