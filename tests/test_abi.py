"""CPU: the C-ABI library loads and exports every symbol include/vit2spn.h declares; the flat layout
matches the HF parameter order; the host mirror keeps the reference's API surface."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "vit2spn.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(v2s_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol_and_abi_versions_agree():
    import vit2spn
    lib = ctypes.CDLL(vit2spn.LIB_PATH)
    syms = _declared_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/vit2spn.h but not exported"
    assert set(vit2spn.EXPORTED) == set(syms), set(vit2spn.EXPORTED) ^ set(syms)
    # 4: one entry point per operation; 3: InfoNCE, uint8 -> patch-matrix input format; 2: fp16 mode, amp entry points
    assert lib.v2s_abi_version() == 4
    header = open(os.path.join(ROOT, "include", "vit2spn.h")).read()
    assert int(re.search(r"#define V2S_ABI_VERSION (\d+)", header).group(1)) == vit2spn._lib.ABI_VERSION == 4


def test_layout_matches_hf_parameter_order():
    import vit2spn
    from vit2spn import _lib
    from oracle import vit2spn_oracle as orc
    offs = _lib.backbone_layout()
    shapes = list(orc.backbone_param_shapes().values())
    assert len(offs) == 200
    spans = sorted((o, o + int(torch.tensor(s).prod())) for o, s in zip(offs, shapes))
    assert spans[0][0] == 0 and spans[-1][1] == _lib.BACKBONE_NUMEL == 5_561_472
    for (a0, a1), (b0, b1) in zip(spans, spans[1:]):
        assert a1 == b0, "flat layout must tile the buffer without gaps or overlap"
    # q/k/v of a block are adjacent → one fused [576,192] matrix
    assert offs[6] - offs[4] == 192 * 192 and offs[8] - offs[6] == 192 * 192
    # never-used tensors (final LN, pooler) sit after the active prefix
    assert min(offs[196:]) == _lib.BACKBONE_ACTIVE_NUMEL == 5_524_032
    assert sum(1 for o in offs if o < _lib.BACKBONE_ACTIVE_NUMEL) == 196
    hoffs = _lib.heads_layout()
    assert hoffs[0] == 0 and _lib.HEADS_NUMEL == 558_464


def test_model_api_surface_and_state_dict_roundtrip():
    import vit2spn
    from oracle import vit2spn_oracle as orc
    model = vit2spn.DualStreamNetwork()
    names = [n for n, _ in model.named_parameters()]
    assert names == orc.model_param_names()                      # 808 tensors, reference order
    assert sum(p.numel() for p in model.parameters() if p.requires_grad) == 11_681_408
    assert all(not p.requires_grad for p in model.target_network_1.parameters())
    state = orc.init_state(3)
    model.load_state_dict(state, strict=True)
    sd = model.state_dict()
    assert list(sd.keys()) == orc.model_param_names()
    assert all(torch.equal(sd[k], state[k]) for k in state)
    # parameters are views of one flat buffer per backbone, in the library's layout
    store = model.online_network_1.vit._store
    from vit2spn import _lib
    for p, o in zip(store.params, _lib.backbone_layout()):
        assert p.data_ptr() == store.flat.data_ptr() + 4 * o
    # rebinding .data (the reference's EMA loop, SURVEY D7) is detected and re-flattened
    p0 = store.params[5]
    p0.data = p0.data * 2.0
    store.ensure()
    assert p0.data_ptr() == store.flat.data_ptr() + 4 * store.offsets[5]
    assert torch.equal(store.flat[store.offsets[5]:store.offsets[5] + p0.numel()].view(p0.shape), p0.data)
    # online_network_1.state_dict() loads strict into a fine-tune backbone (ref:octmnist_ft_vit2spn.py:190)
    ft = vit2spn.FineTunedModel(4)
    ft.backbone.load_state_dict(model.online_network_1.state_dict(), strict=True)


def test_no_cpu_fallback():
    import vit2spn
    m = vit2spn.ViTBackbone()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 3, 224, 224))
    with pytest.raises(NotImplementedError):
        vit2spn.ViTModel(vit2spn.ViTConfig(hidden_size=384, num_attention_heads=6))


def test_fused_adam_state_dict_layout_matches_torch_adam():
    import vit2spn
    lin = torch.nn.Linear(4, 3)
    a = vit2spn.FusedAdam(lin.parameters(), lr=1e-4)
    b = torch.optim.Adam(lin.parameters(), lr=1e-4)
    ka, kb = a.state_dict()["param_groups"][0], b.state_dict()["param_groups"][0]
    for k in ("lr", "betas", "eps", "weight_decay", "amsgrad", "params"):
        assert ka[k] == kb[k]
