"""CPU: masked patch tokens (``ViTModel(use_mask_token=True)``, ``forward(..., bool_masked_pos=...)``).

* ``masked_tokens_oracle`` (the oracle's patch embedding with the mask-token select) equals stock
  ``transformers.ViTModel(config, use_mask_token=True)`` (eager, fp32, same weights, a non-zero mask token): hidden
  states and the gradients w.r.t. the mask token, the patch weight and bias, the position embeddings and the pixels, which
  are exactly zero on masked patches;
* a SimMIM loss built in torch on the oracle (final LayerNorm, 1x1 conv to 768 channels, PixelShuffle(16), masked L1)
  equals ``transformers.ViTForMaskedImageModeling``'s loss and gradients;
* ``state_dict`` keys equal transformers' with and without the mask token, and load strictly both ways;
* the new C entry points and ``ViTModel.forward`` check their arguments before touching the device.
"""
import ctypes as C
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import masked_tokens_oracle as mo  # noqa: E402  (helper module, not a test)


def _cfg(transformers, **kw):
    return transformers.ViTConfig(hidden_size=192, num_hidden_layers=12, num_attention_heads=3, intermediate_size=768,
                                  patch_size=16, image_size=224, layer_norm_eps=1e-12, hidden_act="gelu", qkv_bias=True,
                                  attn_implementation="eager", **kw)


def _weights(seed):
    from oracle import vit2spn_oracle as orc
    p = orc.sub_state(orc.init_state(seed, 0.01), "online_network_1")
    token = 0.02 * torch.randn(192, generator=torch.Generator().manual_seed(seed + 100))
    return p, token


def _mask(B, seed, frac=0.4):
    return torch.rand(B, 196, generator=torch.Generator().manual_seed(seed)) < frac


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def _patch_mask_pixels(mask):
    """[B,196] patch mask -> [B,1,224,224] pixel mask (as ViTForMaskedImageModeling builds it)."""
    return mask.reshape(-1, 14, 14).repeat_interleave(16, 1).repeat_interleave(16, 2).unsqueeze(1)


def test_oracle_masked_embedding_matches_transformers():
    transformers = pytest.importorskip("transformers")
    p, token = _weights(5)
    hf = transformers.ViTModel(_cfg(transformers), add_pooling_layer=False, use_mask_token=True).eval()
    hf.load_state_dict({**{k: v for k, v in p.items() if not k.startswith("pooler.")},
                        "embeddings.mask_token": token.view(1, 1, 192)}, strict=True)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(3, 3, 224, 224, generator=g)
    up = torch.randn(3, 197, 192, generator=g)
    mask = _mask(3, 1)
    mask[1] = False                                 # an unmasked image and a fully masked one
    mask[2] = True
    names = ("embeddings.patch_embeddings.projection.weight", "embeddings.patch_embeddings.projection.bias",
             "embeddings.position_embeddings", "embeddings.cls_token")
    h, dx, dtok, dp = mo.hidden_and_grads(p, x, mask, token, up, names)

    xh = x.clone().requires_grad_(True)
    out = hf(pixel_values=xh, bool_masked_pos=mask, output_hidden_states=True)
    (out.hidden_states[-1] * up).sum().backward()
    assert _rel(h, out.hidden_states[-1].detach()) <= 1e-5
    hs, _ = mo.backbone_outputs(p, x, mask, token)
    for k in range(13):
        assert _rel(hs[k], out.hidden_states[k].detach()) <= 1e-5, k
    emb = hf.embeddings
    assert _rel(dtok, emb.mask_token.grad.view(192)) <= 1e-5
    assert _rel(dp[names[0]], emb.patch_embeddings.projection.weight.grad) <= 1e-5
    assert _rel(dp[names[1]], emb.patch_embeddings.projection.bias.grad) <= 1e-5
    assert _rel(dp[names[2]], emb.position_embeddings.grad) <= 1e-5
    assert _rel(dp[names[3]], emb.cls_token.grad) <= 1e-5
    assert _rel(dx, xh.grad) <= 1e-5
    pm = _patch_mask_pixels(mask).expand_as(dx)
    assert torch.count_nonzero(dx[pm]) == 0 and torch.count_nonzero(xh.grad[pm]) == 0
    assert torch.count_nonzero(dx[~pm]) > 0
    # the patch bias sees the unmasked patches only: image 2 (all masked) contributes nothing
    _, _, _, dp_only2 = mo.hidden_and_grads(p, x[2:], mask[2:], token, up[2:], names[1:2])
    assert torch.count_nonzero(dp_only2[names[1]]) == 0


def simmim_loss(last_hidden, conv, x, mask):
    """ViTForMaskedImageModeling's loss (HF modeling_vit.py:559-581) on a final-LayerNorm output [B,197,192]."""
    B = last_hidden.shape[0]
    seq = last_hidden[:, 1:].permute(0, 2, 1).reshape(B, 192, 14, 14)
    rec = torch.nn.functional.pixel_shuffle(conv(seq), 16)
    pm = _patch_mask_pixels(mask).to(x.dtype)
    l1 = torch.nn.functional.l1_loss(x, rec, reduction="none")
    return (l1 * pm).sum() / (pm.sum() + 1e-5) / 3


def test_simmim_loss_on_the_oracle_matches_transformers():
    transformers = pytest.importorskip("transformers")
    from oracle import vit2spn_oracle as orc
    p, token = _weights(7)
    hf = transformers.ViTForMaskedImageModeling(_cfg(transformers, encoder_stride=16)).eval()
    torch.manual_seed(3)
    conv = torch.nn.Conv2d(192, 768, kernel_size=1)
    sd = {"vit." + k: v for k, v in p.items() if not k.startswith("pooler.")}
    sd.update({"vit.embeddings.mask_token": token.view(1, 1, 192), "decoder.0.weight": conv.weight.detach(),
               "decoder.0.bias": conv.bias.detach()})
    hf.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(4)
    x = torch.randn(2, 3, 224, 224, generator=g)
    mask = _mask(2, 5)
    out = hf(pixel_values=x, bool_masked_pos=mask)
    out.loss.backward()

    q = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    t = token.clone().requires_grad_(True)
    h = mo.patch_embed(q, x, mask, t)
    for l in range(orc.LAYERS):
        h = orc.vit_layer(q, l, h)
    last = torch.nn.functional.layer_norm(h, (192,), q["layernorm.weight"], q["layernorm.bias"], 1e-12)
    loss = simmim_loss(last, conv, x, mask)
    loss.backward()
    assert abs(loss.item() - out.loss.item()) <= 1e-5 * abs(out.loss.item())
    assert _rel(t.grad, hf.vit.embeddings.mask_token.grad.view(192)) <= 1e-5
    assert _rel(conv.weight.grad, hf.decoder[0].weight.grad) <= 1e-5
    for k in ("embeddings.patch_embeddings.projection.weight", "encoder.layer.0.attention.attention.query.weight",
              "encoder.layer.11.output.dense.weight", "layernorm.weight"):
        assert _rel(q[k].grad, dict(hf.vit.named_parameters())[k].grad) <= 1e-5, k


@pytest.mark.parametrize("use_mask_token", [False, True])
def test_state_dict_keys_and_strict_loads_match_transformers(use_mask_token):
    transformers = pytest.importorskip("transformers")
    import vit2spn
    hf = transformers.ViTModel(_cfg(transformers), use_mask_token=use_mask_token)
    ours = vit2spn.ViTModel(vit2spn.ViTConfig(), use_mask_token=use_mask_token)
    assert list(ours.state_dict()) == list(hf.state_dict())
    assert ("embeddings.mask_token" in ours.state_dict()) == use_mask_token
    assert len(ours._store.params) == 200 and len(list(ours.parameters())) == 200 + use_mask_token
    if use_mask_token:
        assert torch.equal(ours.embeddings.mask_token.detach(), torch.zeros(1, 1, 192))
        hf.embeddings.mask_token.data.normal_()
    ours.load_state_dict(hf.state_dict(), strict=True)
    for k, v in hf.state_dict().items():
        assert torch.equal(ours.state_dict()[k], v), k
    hf2 = transformers.ViTModel(_cfg(transformers), use_mask_token=use_mask_token)
    hf2.load_state_dict(ours.state_dict(), strict=True)
    # the flat store still backs the 200 tensors; the mask token is a parameter of its own
    for prm, o in zip(ours._store.params, ours._store.offsets):
        assert prm.data_ptr() == ours._store.flat.data_ptr() + 4 * o


def test_from_pretrained_loads_or_keeps_the_mask_token(tmp_path, monkeypatch):
    transformers = pytest.importorskip("transformers")
    import vit2spn
    monkeypatch.setenv("V2S_ALLOW_RANDOM_INIT", "1")
    hf = transformers.ViTModel(_cfg(transformers), use_mask_token=True)
    hf.embeddings.mask_token.data.normal_()
    sd = hf.state_dict()
    with_tok, without = os.path.join(tmp_path, "a.bin"), os.path.join(tmp_path, "b.bin")
    torch.save(sd, with_tok)
    torch.save({k: v for k, v in sd.items() if k != "embeddings.mask_token"}, without)
    m = vit2spn.ViTModel.from_pretrained(with_tok, use_mask_token=True)
    assert torch.equal(m.embeddings.mask_token.detach(), sd["embeddings.mask_token"])
    m = vit2spn.ViTModel.from_pretrained(without, use_mask_token=True)
    assert torch.equal(m.embeddings.mask_token.detach(), torch.zeros(1, 1, 192))
    assert torch.equal(m.embeddings.cls_token.detach(), sd["embeddings.cls_token"])
    assert getattr(vit2spn.ViTModel.from_pretrained(without).embeddings, "mask_token", None) is None


def test_forward_rejects_bad_masks():
    import vit2spn
    x = torch.zeros(2, 3, 224, 224)
    m = torch.zeros(2, 196, dtype=torch.bool)
    with pytest.raises(ValueError, match="use_mask_token"):
        vit2spn.ViTModel()(x, bool_masked_pos=m)
    model = vit2spn.ViTModel(use_mask_token=True)
    for bad in (torch.zeros(2, 14, 14, dtype=torch.bool), torch.zeros(3, 196, dtype=torch.bool),
                torch.zeros(2, 197, dtype=torch.bool), torch.zeros(392, dtype=torch.bool)):
        with pytest.raises(ValueError, match=r"\[B,196\]"):
            model(x, bool_masked_pos=bad)
    with pytest.raises(ValueError, match="integer"):
        model(x, bool_masked_pos=torch.zeros(2, 196))


def test_masked_entry_points_reject_bad_arguments():
    from vit2spn import _lib
    B, mode = 2, _lib.MODE_FP32
    nbytes = _lib.lib.v2s_workspace_bytes(B, mode, 1, 1)
    g = _lib.Group()
    g.params, g.x, g.grads, g.slot, g.dfeat = 0x10000, 0x20000, 0x30000, 0, 0x40000
    arr = (_lib.Group * 1)(g)
    ws = C.c_void_p(1 << 20)
    masks = (C.c_void_p * 1)(0x50000)
    rc = _lib.lib.v2s_backbone_forward_masked(arr, None, masks, None, 1, B, mode, ws, nbytes, None)
    err = _lib.lib.v2s_last_error().decode()
    assert rc != 0 and "no mask token" in err, err
    toks = (C.c_void_p * 1)(None)
    rc = _lib.lib.v2s_backbone_forward_masked(arr, None, masks, toks, 1, B, mode, ws, nbytes, None)
    assert rc != 0 and "no mask token" in _lib.lib.v2s_last_error().decode()
    toks[0] = 0x60008                                 # fp32 [192] read as float4: 16-byte rule
    rc = _lib.lib.v2s_backbone_forward_masked(arr, None, masks, toks, 1, B, mode, ws, nbytes, None)
    err = _lib.lib.v2s_last_error().decode()
    assert rc != 0 and "mask_tokens[0]" in err and "aligned" in err, err
    rc = _lib.lib.v2s_backbone_forward_masked(None, None, masks, toks, 1, B, mode, ws, nbytes, None)
    assert rc != 0 and "null" in _lib.lib.v2s_last_error().decode()

    dt = (C.c_void_p * 1)(0x70002)
    rc = _lib.lib.v2s_backbone_backward_masked(arr, None, masks, dt, None, None, 1, 1, B, mode, ws, nbytes, None)
    err = _lib.lib.v2s_last_error().decode()
    assert rc != 0 and "dmask_tokens[0]" in err and "aligned" in err, err
    dt[0] = 0x70004
    dp = (C.c_void_p * 1)(0x200004)
    rc = _lib.lib.v2s_backbone_backward_masked(arr, None, masks, dt, None, dp, 1, 1, B, mode, ws, nbytes, None)
    assert rc != 0 and "dpixels[0]" in _lib.lib.v2s_last_error().decode()
    da = (C.c_void_p * 12)()
    da[5] = 0x100002
    rc = _lib.lib.v2s_backbone_backward_masked(arr, None, masks, dt, da, None, 1, 1, B, mode, ws, nbytes, None)
    err = _lib.lib.v2s_last_error().decode()
    assert rc != 0 and "dattn[5]" in err and "aligned" in err, err
    rc = _lib.lib.v2s_backbone_backward_masked(None, None, masks, dt, None, None, 1, 1, B, mode, ws, nbytes, None)
    assert rc != 0 and "null" in _lib.lib.v2s_last_error().decode()
