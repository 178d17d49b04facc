"""CPU: ViTModel's per-layer outputs (output_hidden_states / output_attentions).

* ``vit_outputs_oracle.backbone_outputs`` (stated with the oracle's functions) is pinned to ``transformers.ViTModel``
  with eager attention on the same weights;
* the host API resolves the two flags as transformers does and keeps the old hidden-state accessor's contract;
* the C entry points reject malformed ``v2s_group_outputs`` and layer ranges before touching the device.
"""
import ctypes as C
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import vit_outputs_oracle as vo  # noqa: E402  (helper module, not a test)


def test_reference_outputs_match_transformers_eager():
    transformers = pytest.importorskip("transformers")
    from oracle import vit2spn_oracle as orc
    cfg = transformers.ViTConfig(hidden_size=192, num_hidden_layers=12, num_attention_heads=3, intermediate_size=768,
                                 patch_size=16, image_size=224, layer_norm_eps=1e-12, hidden_act="gelu", qkv_bias=True)
    cfg._attn_implementation = "eager"
    ref = transformers.ViTModel(cfg).eval()
    p = orc.sub_state(orc.init_state(7, 0.01), "online_network_1")
    missing, unexpected = ref.load_state_dict(p, strict=False)
    assert not unexpected and all(k.startswith("pooler.") for k in missing), (missing, unexpected)
    x, _ = orc.synthetic_views(2, seed=3)
    with torch.no_grad():
        out = ref(x, output_hidden_states=True, output_attentions=True)
        hs, attn = vo.backbone_outputs(p, x)
    assert len(out.hidden_states) == len(hs) == 13 and len(out.attentions) == len(attn) == 12
    for a, b in zip(hs, out.hidden_states):
        assert (a - b).abs().max().item() <= 1e-5
    for a, b in zip(attn, out.attentions):
        assert a.shape == (2, 3, 197, 197)
        assert (a - b).abs().max().item() <= 1e-5
    assert (hs[-1] - orc.backbone_hidden(p, x)).abs().max().item() == 0.0


def test_output_flags_and_accessors():
    import vit2spn
    from vit2spn import modules
    assert vit2spn.ViTConfig().output_attentions is False
    assert vit2spn.ViTConfig(output_attentions=True).output_attentions is True
    m = vit2spn.ViTModel.from_pretrained("no/such-checkpoint", output_hidden_states=True, output_attentions=True)
    assert m.config.output_hidden_states and m.config.output_attentions
    hs = modules.ViTModelOutput(m, torch.zeros(1, 197, 192)).hidden_states
    assert hs[-1].shape == (1, 197, 192) and len(hs) == 13
    with pytest.raises(NotImplementedError, match="output_hidden_states=True"):
        hs[3]
    assert modules.ViTModelOutput(m, torch.zeros(1, 197, 192)).attentions is None


def _call(fn, outputs, *, slot=0, dhidden=None, dfeat=None, layer_hi=12, layer_lo=0):
    """Calls a backbone entry point with fake (never dereferenced) device pointers: the argument checks run first.
    ``outputs=None`` passes NULL for the per-group outputs."""
    from vit2spn import _lib
    B, mode = 2, _lib.MODE_FP32
    nbytes = _lib.lib.v2s_workspace_bytes(B, mode, 1, 1)
    g = _lib.Group()
    g.params, g.x, g.grads, g.slot = 0x10000, 0x20000, 0x30000, slot
    g.dhidden, g.dfeat = dhidden, dfeat
    arr = (_lib.Group * 1)(g)
    outs = (_lib.GroupOutputs * 1)(outputs) if outputs is not None else None
    if fn == "forward":
        rc = _lib.lib.v2s_backbone_forward(arr, outs, 1, B, mode, C.c_void_p(1 << 20), nbytes, None)
    else:
        rc = _lib.lib.v2s_backbone_backward(arr, outs, 1, B, mode, C.c_void_p(1 << 20), nbytes, layer_hi, layer_lo, 1, None)
    return rc, _lib.lib.v2s_last_error().decode()


def test_backbone_calls_reject_malformed_outputs_and_ranges():
    from vit2spn import _lib
    assert C.sizeof(_lib.GroupOutputs) == (13 + 12 + 13 + 12 + 4) * 8
    o = _lib.GroupOutputs()
    for i in range(12):                       # 12 of 13 hidden states
        o.hidden[i] = 0x100000 * (i + 1)
    for fn in ("forward", "backward"):
        rc, err = _call(fn, o, dfeat=0x40000)
        assert rc != 0 and "hidden[]" in err and "all or none" in err, err
    o = _lib.GroupOutputs()
    o.attn[0] = 0x100000                     # 1 of 12 attention outputs
    rc, err = _call("forward", o)
    assert rc != 0 and "attn[]" in err, err
    o = _lib.GroupOutputs()
    o.hidden[0] = 0x100004                   # misaligned
    rc, err = _call("forward", o)
    assert rc != 0 and "aligned" in err, err
    o = _lib.GroupOutputs()
    o.dhidden[12] = 0x50000                  # both dhidden[12] and v2s_group.dhidden
    rc, err = _call("backward", o, dhidden=0x60000)
    assert rc != 0 and "both" in err, err
    rc, err = _call("backward", _lib.GroupOutputs())      # no gradient at all
    assert rc != 0 and "needs dfeat or dhidden" in err, err
    rc, err = _call("backward", None, dfeat=0x40000, layer_hi=4, layer_lo=8)    # empty layer range, no outputs
    assert rc != 0 and "bad layer range" in err, err
