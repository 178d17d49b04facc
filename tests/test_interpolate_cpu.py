"""CPU: ``ViTModel(interpolate_pos_encoding=True)`` for inputs other than 224 x 224 (up to 197 tokens).

* ``interp_oracle`` (the oracle at N tokens with transformers' bicubic position-table rule) equals stock
  ``transformers.ViTModel`` (eager, fp32, same weights): hidden states, attentions and the gradients w.r.t. the pixels,
  every parameter (the position table's border cells included), the mask token and the retained attentions;
* ``v2s_set_image_size`` accepts and refuses the sizes it should, and ``v2s_workspace_bytes`` follows it;
* ``ViTModel.forward`` refuses bad sizes and masks before touching the device;
* ``attention_relevance(..., grid=(gh, gw))`` gives non-square maps.
"""
import ctypes as C
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import interp_oracle as io  # noqa: E402  (helper module, not a test)

SIZES = [(16, 16), (64, 64), (128, 128), (96, 160), (112, 448), (224, 224)]


def _cfg(transformers, **kw):
    return transformers.ViTConfig(hidden_size=192, num_hidden_layers=12, num_attention_heads=3, intermediate_size=768,
                                  patch_size=16, image_size=224, layer_norm_eps=1e-12, hidden_act="gelu", qkv_bias=True,
                                  attn_implementation="eager", **kw)


def _weights(seed):
    from oracle import vit2spn_oracle as orc
    p = orc.sub_state(orc.init_state(seed, 0.01), "online_network_1")
    token = 0.02 * torch.randn(192, generator=torch.Generator().manual_seed(seed + 100))
    return p, token


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


@pytest.mark.parametrize("H,W", SIZES)
def test_oracle_matches_transformers(H, W):
    transformers = pytest.importorskip("transformers")
    p, token = _weights(7)
    hf = transformers.ViTModel(_cfg(transformers), add_pooling_layer=False, use_mask_token=True).eval()
    hf.load_state_dict({**{k: v for k, v in p.items() if not k.startswith("pooler.")},
                        "embeddings.mask_token": token.view(1, 1, 192)}, strict=True)
    B, n = 3, (H // 16) * (W // 16)
    g = torch.Generator().manual_seed(H * 1000 + W)
    x = torch.randn(B, 3, H, W, generator=g)
    up = torch.randn(B, n + 1, 192, generator=g)
    mask = torch.rand(B, n, generator=g) < 0.3
    retain = (0, 5, 11)

    hs, probs, dx, dtok, dp, da = io.grads(p, x, up, mask, token, retain)
    xh = x.clone().requires_grad_(True)
    out = hf(pixel_values=xh, bool_masked_pos=mask, interpolate_pos_encoding=True, output_hidden_states=True,
             output_attentions=True)
    for l in retain:
        out.attentions[l].retain_grad()
    (out.hidden_states[-1] * up).sum().backward()
    for k in range(13):
        assert _rel(hs[k], out.hidden_states[k].detach()) <= 1e-5, k
    for k in range(12):
        assert _rel(probs[k], out.attentions[k].detach()) <= 1e-5, k
    assert _rel(dx, xh.grad) <= 1e-5
    assert _rel(dtok, hf.embeddings.mask_token.grad.view(192)) <= 1e-5
    hp = dict(hf.named_parameters())
    for k, v in dp.items():
        if k.endswith("key.bias"):         # softmax ignores it: both gradients are rounding noise around 0
            assert v.norm() < 1e-5 and hp[k].grad.norm() < 1e-5, k
        elif k in hp:
            assert hp[k].grad is not None and _rel(v, hp[k].grad) <= 1e-5, k
    for l in retain:
        assert _rel(da[l], out.attentions[l].grad) <= 1e-5, l
    # the clamped bicubic taps fold onto the border cells of the stored 14 x 14 grid: check them on their own
    dpos, ref = dp["embeddings.position_embeddings"][0, 1:].reshape(14, 14, 192), \
        hp["embeddings.position_embeddings"].grad[0, 1:].reshape(14, 14, 192)
    border = torch.ones(14, 14, dtype=torch.bool)
    border[1:-1, 1:-1] = False
    assert _rel(dpos[border], ref[border]) <= 1e-5
    # the same hidden states without a mask (the unmasked embedding path)
    hs2, _ = io.backbone_outputs(p, x)
    out2 = hf(pixel_values=x, interpolate_pos_encoding=True, output_hidden_states=True)
    assert _rel(hs2[-1], out2.hidden_states[-1].detach()) <= 1e-5


def test_224_table_unchanged_and_112x448_interpolated():
    p, _ = _weights(3)
    pos = p["embeddings.position_embeddings"]
    assert io.position_table(pos, 224, 224) is pos
    t = io.position_table(pos, 112, 448)           # 7 x 28 = 196 patches, but H != W: interpolated
    assert t.shape == (1, 197, 192) and not torch.equal(t, pos)


def _lib():
    import vit2spn
    lib = C.CDLL(vit2spn.LIB_PATH)
    lib.v2s_set_image_size.argtypes = [C.c_int, C.c_int]
    lib.v2s_set_image_size.restype = C.c_int
    lib.v2s_workspace_bytes.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
    lib.v2s_workspace_bytes.restype = C.c_int64
    lib.v2s_last_error.restype = C.c_char_p
    return lib


def test_set_image_size_and_workspace_bytes():
    lib = _lib()
    before = lib.v2s_workspace_bytes(64, 1, 1, 1)
    try:
        for h, w in [(16, 16), (112, 448), (224, 224)]:
            assert lib.v2s_set_image_size(h, w) == 0, (h, w)
        assert lib.v2s_workspace_bytes(64, 1, 1, 1) == before
        for h, w in [(0, 0), (100, 100), (240, 240), (16, 3152)]:
            assert lib.v2s_set_image_size(h, w) != 0, (h, w)
        assert b"197" in lib.v2s_last_error() or b"196" in lib.v2s_last_error()
        assert lib.v2s_set_image_size(128, 128) == 0
        small = lib.v2s_workspace_bytes(64, 1, 1, 1)
        assert 0 < small < before
    finally:
        assert lib.v2s_set_image_size(224, 224) == 0
    assert lib.v2s_workspace_bytes(64, 1, 1, 1) == before


def _model(use_mask_token=False):
    import vit2spn
    return vit2spn.ViTModel(use_mask_token=use_mask_token)


def test_python_refusals_before_the_device():
    m = _model(use_mask_token=True)
    x = torch.zeros(2, 3, 128, 128)                # CPU tensors: every refusal below comes before the device check
    with pytest.raises(ValueError, match=r"Input image size \(128\*128\) doesn't match model \(224\*224\)"):
        m(x)
    with pytest.raises(ValueError, match=r"x\[\.\.\., :96, :128\]"):
        m(torch.zeros(2, 3, 100, 140), interpolate_pos_encoding=True)
    with pytest.raises(ValueError, match="197 tokens"):
        m(torch.zeros(2, 3, 240, 240), interpolate_pos_encoding=True)
    with pytest.raises(ValueError, match=r"\[B,64\]"):
        m(x, interpolate_pos_encoding=True, bool_masked_pos=torch.zeros(2, 196, dtype=torch.bool))
    with pytest.raises(ValueError, match=r"\[B,196\]"):
        m(torch.zeros(2, 3, 224, 224), interpolate_pos_encoding=True, bool_masked_pos=torch.zeros(2, 64, dtype=torch.bool))


def test_attention_relevance_grid():
    from vit2spn.explain import attention_relevance
    B, gh, gw = 2, 4, 8
    n = 1 + gh * gw
    g = torch.Generator().manual_seed(0)
    att = [torch.softmax(torch.randn(B, 3, n, n, generator=g), -1) for _ in range(12)]
    grads = [torch.randn(B, 3, n, n, generator=g) for _ in range(12)]
    r = attention_relevance(att, grads, grid=(gh, gw))
    assert r.shape == (B, gh, gw)
    assert torch.equal(r.reshape(B, -1), attention_relevance(att, grads, grid=(1, gh * gw)).reshape(B, -1))
    with pytest.raises(ValueError):
        attention_relevance(att, grads, grid=(5, 8))
    with pytest.raises(ValueError):
        attention_relevance(att, grads)            # 32 patches are no square grid
