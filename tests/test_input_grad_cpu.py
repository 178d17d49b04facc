"""CPU: the oracle's gradient w.r.t. pixel_values (autograd through orc.backbone_hidden, fp32) equals stock
transformers.ViTModel's (eager attention, same weights).  This pins the col2im index order k = c*256 + ky*16 + kx that
the library's image-gradient epilogue writes."""
import pytest
import torch


def test_oracle_pixel_gradient_matches_transformers():
    transformers = pytest.importorskip("transformers")
    from oracle import vit2spn_oracle as orc
    p = orc.sub_state(orc.init_state(5, 0.01), "online_network_1")
    cfg = transformers.ViTConfig(hidden_size=192, num_hidden_layers=12, num_attention_heads=3, intermediate_size=768,
                                 patch_size=16, image_size=224, layer_norm_eps=1e-12, hidden_act="gelu", qkv_bias=True,
                                 attn_implementation="eager")
    hf = transformers.ViTModel(cfg, add_pooling_layer=False).eval()
    hf.load_state_dict({k: v for k, v in p.items() if not k.startswith("pooler.")}, strict=True)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 3, 224, 224, generator=g)
    up = torch.randn(2, 197, 192, generator=g)
    xo = x.clone().requires_grad_(True)
    (orc.backbone_hidden(p, xo) * up).sum().backward()
    xh = x.clone().requires_grad_(True)
    (hf(pixel_values=xh, output_hidden_states=True).hidden_states[-1] * up).sum().backward()
    rel = ((xo.grad.double() - xh.grad.double()).norm() / xh.grad.double().norm()).item()
    assert rel <= 1e-5, rel
