"""CPU: ``vit2spn.ViTForMaskedImageModeling`` (SimMIM) and what it needs from the rest of the package.

* ``state_dict`` keys and order equal ``transformers.ViTForMaskedImageModeling``'s 201 keys, and load strictly both
  ways; ``ViTModel(add_pooling_layer=False)`` equals transformers' keys, the default's keys are unchanged;
* ``mim_oracle`` (the head on hidden_states[12], and the whole model on the oracle's backbone) equals transformers' loss,
  reconstruction and gradients; its 16-bit rounding model stays close to the fp32 head;
* the errors raised before anything runs on the device, and the C entry points' argument checks;
* ``from_pretrained`` with a SimMIM checkpoint and with a ViTModel checkpoint;
* ``FusedAdam.zero_grad`` clears the final LayerNorm's own ``.grad`` (autograd's, not a flat-buffer view).
"""
import ctypes as C
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import mim_oracle as mim  # noqa: E402  (helper module, not a test)


def _cfg(transformers, **kw):
    return transformers.ViTConfig(hidden_size=192, num_hidden_layers=12, num_attention_heads=3, intermediate_size=768,
                                  patch_size=16, image_size=224, layer_norm_eps=1e-12, hidden_act="gelu", qkv_bias=True,
                                  attn_implementation="eager", **kw)


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def _weights(seed):
    from oracle import vit2spn_oracle as orc
    p = orc.sub_state(orc.init_state(seed, 0.01), "online_network_1")
    g = torch.Generator().manual_seed(seed + 100)
    token = 0.02 * torch.randn(192, generator=g)
    dec_w, dec_b = 0.02 * torch.randn(768, 192, 1, 1, generator=g), 0.01 * torch.randn(768, generator=g)
    return p, token, dec_w, dec_b


def _hf_model(transformers, p, token, dec_w, dec_b):
    hf = transformers.ViTForMaskedImageModeling(_cfg(transformers, encoder_stride=16)).eval()
    sd = {"vit." + k: v for k, v in p.items() if not k.startswith("pooler.")}
    sd.update({"vit.embeddings.mask_token": token.view(1, 1, 192), "decoder.0.weight": dec_w, "decoder.0.bias": dec_b})
    hf.load_state_dict(sd, strict=True)
    return hf


def test_state_dict_keys_order_and_strict_loads_match_transformers():
    transformers = pytest.importorskip("transformers")
    import vit2spn
    hf = transformers.ViTForMaskedImageModeling(_cfg(transformers, encoder_stride=16))
    ours = vit2spn.ViTForMaskedImageModeling()
    assert list(ours.state_dict()) == list(hf.state_dict()) and len(hf.state_dict()) == 201
    w = ours.decoder[0].weight.detach()
    assert abs(w.std().item() - 0.02) < 2e-3                  # transformers' trunc_normal_(std=0.02)
    assert torch.count_nonzero(ours.decoder[0].bias) == 0
    for t in hf.state_dict().values():
        if t.is_floating_point():
            t.normal_()
    ours.load_state_dict(hf.state_dict(), strict=True)
    for k, v in hf.state_dict().items():
        assert torch.equal(ours.state_dict()[k], v), k
    hf2 = transformers.ViTForMaskedImageModeling(_cfg(transformers, encoder_stride=16))
    hf2.load_state_dict(ours.state_dict(), strict=True)
    # the backbone's 200 tensors (pooler included) still live in its flat store
    store = ours.vit._store
    assert len(store.params) == 200
    for prm, o in zip(store.params, store.offsets):
        assert prm.data_ptr() == store.flat.data_ptr() + 4 * o


@pytest.mark.parametrize("add_pooling_layer", [True, False])
def test_vitmodel_add_pooling_layer_keys_match_transformers(add_pooling_layer):
    transformers = pytest.importorskip("transformers")
    import vit2spn
    from vit2spn import modules
    hf = transformers.ViTModel(_cfg(transformers), add_pooling_layer=add_pooling_layer)
    ours = vit2spn.ViTModel(vit2spn.ViTConfig(), add_pooling_layer=add_pooling_layer)
    assert list(ours.state_dict()) == list(hf.state_dict())
    assert len(list(ours.parameters())) == (200 if add_pooling_layer else 198) and len(ours._store.params) == 200
    if add_pooling_layer:
        assert list(ours.state_dict()) == list(vit2spn.ViTModel().state_dict())
        assert ours.pooler is not None
    else:
        assert ours.pooler is None
        assert modules.ViTModelOutput(ours, torch.zeros(1, 197, 192)).pooler_output is None
    ours.load_state_dict(hf.state_dict(), strict=True)
    hf.load_state_dict(ours.state_dict(), strict=True)


def test_head_oracle_matches_transformers():
    transformers = pytest.importorskip("transformers")
    from oracle import vit2spn_oracle as orc
    p, token, dec_w, dec_b = _weights(7)
    hf = _hf_model(transformers, p, token, dec_w, dec_b)
    g = torch.Generator().manual_seed(4)
    x = torch.randn(3, 3, 224, 224, generator=g)
    mask = torch.rand(3, 196, generator=g) < 0.5
    mask[0] = False                                  # an unmasked image, a fully masked one, a mixed one
    mask[1] = True
    xh = x.clone().requires_grad_(True)
    out = hf(pixel_values=xh, bool_masked_pos=mask)
    out.loss.backward()
    loss, rec, grads = mim.model_loss(p, token, dec_w, dec_b, x, mask)
    assert abs(loss.item() - out.loss.item()) <= 1e-5 * abs(out.loss.item())
    assert _rel(rec, out.reconstruction.detach()) <= 1e-5
    named = dict(hf.named_parameters())
    pairs = {"decoder.0.weight": named["decoder.0.weight"].grad, "decoder.0.bias": named["decoder.0.bias"].grad,
             "mask_token": named["vit.embeddings.mask_token"].grad.view(192), "pixels": xh.grad}
    for k in ("layernorm.weight", "layernorm.bias", "embeddings.patch_embeddings.projection.weight",
              "encoder.layer.0.attention.attention.query.weight", "encoder.layer.11.output.dense.weight"):
        pairs[k] = named["vit." + k].grad
    for k, ref in pairs.items():
        assert _rel(grads[k], ref) <= 1e-5, k
    # the head alone on transformers' own hidden_states[12]; without a mask there is no loss
    h12 = hf.vit(pixel_values=x, bool_masked_pos=mask, output_hidden_states=True).hidden_states[-1].detach()
    rec2, loss2 = mim.head(h12, p["layernorm.weight"], p["layernorm.bias"], dec_w, dec_b, x, mask)
    assert abs(loss2.item() - out.loss.item()) <= 1e-5 * abs(out.loss.item())
    assert mim.head(h12, p["layernorm.weight"], p["layernorm.bias"], dec_w, dec_b, x, None)[1] is None
    # the 16-bit rounding model differs from the fp32 head by about the formats' resolution, no more
    for lp, tol in ((torch.bfloat16, 2e-2), (torch.float16, 3e-3)):
        rec3, loss3 = mim.head(h12, p["layernorm.weight"], p["layernorm.bias"], dec_w, dec_b, x, mask, lp)
        assert 0 < _rel(rec3, rec2) <= tol and abs(loss3.item() - loss2.item()) <= tol * abs(loss2.item())
    assert orc.LAYERS == 12


def test_errors_before_the_device():
    import vit2spn
    with pytest.raises(ValueError, match="encoder_stride"):
        vit2spn.ViTForMaskedImageModeling(vit2spn.ViTConfig(encoder_stride=8))
    m = vit2spn.ViTForMaskedImageModeling()
    with pytest.raises(ValueError, match="fp32 pixels"):
        m(torch.zeros(2, 196, 768, dtype=torch.bfloat16), bool_masked_pos=torch.zeros(2, 196, dtype=torch.bool))
    with pytest.raises(ValueError, match="interpolate_pos_encoding"):
        m(torch.zeros(2, 3, 224, 224), interpolate_pos_encoding=True)
    with pytest.raises(ValueError, match=r"\[B,196\]"):
        m(torch.zeros(2, 3, 224, 224), bool_masked_pos=torch.zeros(2, 197, dtype=torch.bool))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(2, 3, 224, 224), bool_masked_pos=torch.zeros(2, 196, dtype=torch.bool))


def test_mim_entry_points_check_their_arguments():
    from vit2spn import _lib
    lib = _lib.lib
    assert lib.v2s_mim_workspace_bytes(0, 1) == -1 and lib.v2s_mim_workspace_bytes(2, 7) == -1
    n = lib.v2s_mim_workspace_bytes(2, _lib.MODE_BF16)
    assert n > 2 * 196 * 768 * 2
    ws = C.c_void_p(1 << 20)
    a = [C.c_void_p(0x10000 * (i + 1)) for i in range(9)]
    rc = lib.v2s_mim_forward(None, *a[1:5], a[5], a[6], a[7], a[8], 1, 2, _lib.MODE_BF16, ws, n, None)
    assert rc != 0 and "null argument" in lib.v2s_last_error().decode()
    rc = lib.v2s_mim_forward(*a[:5], None, a[6], a[7], a[8], 1, 2, _lib.MODE_BF16, ws, n, None)   # mask without pixels
    assert rc != 0 and "null argument" in lib.v2s_last_error().decode()
    rc = lib.v2s_mim_forward(*a[:5], a[5], a[6], C.c_void_p(0x10004), a[8], 1, 2, _lib.MODE_BF16, ws, n, None)
    assert rc != 0 and "aligned" in lib.v2s_last_error().decode()
    rc = lib.v2s_mim_forward(*a[:9], 1, 2, _lib.MODE_BF16, ws, n - 1024, None)
    assert rc != 0 and "workspace too small" in lib.v2s_last_error().decode()
    rc = lib.v2s_mim_backward(*a[:3], None, a[4], *a[5:9], None, None, 2, _lib.MODE_BF16, ws, n, None)
    assert rc != 0 and "null argument" in lib.v2s_last_error().decode()
    rc = lib.v2s_mim_backward(*a[:5], a[5], None, a[7], None, None, None, 2, _lib.MODE_BF16, ws, n, None)
    assert rc != 0 and "go together" in lib.v2s_last_error().decode()


def test_from_pretrained_simmim_and_vitmodel_checkpoints(tmp_path, monkeypatch):
    transformers = pytest.importorskip("transformers")
    import vit2spn
    monkeypatch.setenv("V2S_ALLOW_RANDOM_INIT", "1")
    hf = transformers.ViTForMaskedImageModeling(_cfg(transformers, encoder_stride=16))
    for t in hf.parameters():
        t.data.normal_()
    path = os.path.join(tmp_path, "mim.bin")
    torch.save(hf.state_dict(), path)
    m = vit2spn.ViTForMaskedImageModeling.from_pretrained(path)
    for k, v in hf.state_dict().items():
        assert torch.equal(m.state_dict()[k], v), k
    # a ViTModel checkpoint (pooler included, no decoder, no mask token): the backbone loads, the rest keeps its init
    vm = transformers.ViTModel(_cfg(transformers))
    path2 = os.path.join(tmp_path, "vit.bin")
    torch.save(vm.state_dict(), path2)
    m2 = vit2spn.ViTForMaskedImageModeling.from_pretrained(path2)
    assert torch.equal(m2.vit.embeddings.cls_token.detach(), vm.embeddings.cls_token.detach())
    assert torch.equal(m2.vit.embeddings.mask_token.detach(), torch.zeros(1, 1, 192))
    bad = os.path.join(tmp_path, "bad.bin")
    torch.save({k: v for k, v in hf.state_dict().items() if "encoder.layer.3." not in k}, bad)
    with pytest.raises(RuntimeError, match="missing"):
        vit2spn.ViTForMaskedImageModeling.from_pretrained(bad)


def test_fused_adam_zero_grad_clears_the_final_layernorm_grad():
    import vit2spn
    m = vit2spn.ViTModel(use_mask_token=True)
    m._store.grads()
    m.layernorm.weight.grad = torch.ones(192)           # what autograd leaves after a loss on last_hidden_state
    m.layernorm.bias.grad = torch.ones(192)
    m.embeddings.mask_token.grad = torch.ones(1, 1, 192)
    opt = vit2spn.FusedAdam(m.parameters(), lr=1e-3)
    opt.zero_grad()
    assert m.layernorm.weight.grad is None and m.layernorm.bias.grad is None and m.embeddings.mask_token.grad is None
    # the flat-buffer views stay attached and read as zeros
    q = m.encoder.layer[0].attention.attention.query.weight
    assert q.grad is not None and torch.count_nonzero(q.grad) == 0
    m.layernorm.weight.grad = torch.ones(192)
    opt.zero_grad(set_to_none=False)
    assert m.layernorm.weight.grad is not None and torch.count_nonzero(m.layernorm.weight.grad) == 0
