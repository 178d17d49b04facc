"""CPU: gradients w.r.t. the attention probabilities.

* ``attn_grad_oracle.attention_grads`` (the oracle's block with the probabilities explicit) equals what ``retain_grad()``
  gives on stock ``transformers.ViTModel``'s attentions (eager attention, same weights), blocks the loss does not reach
  included (None on both sides), and keeps the oracle's values and a consistent gradient under its rounding model;
* ``vit2spn.explain.attention_relevance`` equals a per-image loop over the published equations;
* the new C entry point checks its arguments before touching the device.
"""
import ctypes as C
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import attn_grad_oracle as ag  # noqa: E402  (helper module, not a test)
import vit_outputs_oracle as vo  # noqa: E402


def _hf_and_weights(seed):
    transformers = pytest.importorskip("transformers")
    from oracle import vit2spn_oracle as orc
    p = orc.sub_state(orc.init_state(seed, 0.01), "online_network_1")
    cfg = transformers.ViTConfig(hidden_size=192, num_hidden_layers=12, num_attention_heads=3, intermediate_size=768,
                                 patch_size=16, image_size=224, layer_norm_eps=1e-12, hidden_act="gelu", qkv_bias=True,
                                 attn_implementation="eager")
    hf = transformers.ViTModel(cfg, add_pooling_layer=False).eval()
    hf.load_state_dict({k: v for k, v in p.items() if not k.startswith("pooler.")}, strict=True)
    return hf, p


def _hf_attention_grads(hf, x, loss_fn):
    out = hf(pixel_values=x, output_hidden_states=True, output_attentions=True)
    for a in out.attentions:
        a.retain_grad()
    loss_fn(out.hidden_states).backward()
    return out.attentions, [a.grad for a in out.attentions]


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm()).item()


@pytest.mark.parametrize("reach", [12, 4])
def test_oracle_attention_gradients_match_transformers_retain_grad(reach):
    hf, p = _hf_and_weights(5)
    g = torch.Generator().manual_seed(reach)
    x = torch.randn(2, 3, 224, 224, generator=g)
    up = torch.randn(2, 197, 192, generator=g)
    wf = torch.randn(2, 192, generator=g)

    def loss_fn(hs):
        if reach == 12:
            return (hs[7] * up).sum() + (hs[12].mean(1) * wf).sum()
        return (hs[4] * up).sum()

    _, hf_grads = _hf_attention_grads(hf, x, loss_fn)
    _, _, ref = ag.attention_grads(p, x, loss_fn)
    for l, (a, b) in enumerate(zip(hf_grads, ref)):
        if l >= reach:
            assert a is None and b is None, l
        else:
            assert a is not None and b is not None, l
            assert _rel(b, a) <= 1e-5, (l, _rel(b, a))


def test_oracle_rounding_branch_keeps_values_and_gradients():
    """With the "p" stage on, the block takes the oracle's values (its rounded-numerator form of A V); rounding to fp32
    itself makes that form exact, and the gradients w.r.t. A must then equal the softmax form's."""
    from oracle import vit2spn_oracle as orc
    p = orc.sub_state(orc.init_state(4, 0.01), "online_network_1")
    x = torch.randn(1, 3, 224, 224, generator=torch.Generator().manual_seed(0))
    w = torch.randn(1, 197, 192, generator=torch.Generator().manual_seed(1))

    def loss_fn(hs):
        return (hs[6] * w).sum() + hs[12].square().mean()

    with orc.rounding("all", torch.bfloat16):
        hs, attn, _ = ag.attention_grads(p, x, loss_fn)
        with torch.no_grad():
            hs_ref, attn_ref = vo.backbone_outputs(p, x)
    assert all(torch.equal(a, b) for a, b in zip(hs, hs_ref))
    assert max((a - b).abs().max().item() for a, b in zip(attn, attn_ref)) <= 1e-7
    _, _, exact = ag.attention_grads(p, x, loss_fn)
    with orc.rounding(("p",), torch.float32):
        _, _, same = ag.attention_grads(p, x, loss_fn)
    assert max(_rel(a, b) for a, b in zip(same, exact)) <= 1e-5


@pytest.mark.parametrize("token", ["cls", "mean"])
def test_relevance_matches_published_equations(token):
    from vit2spn import explain
    hf, _ = _hf_and_weights(6)
    x = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(1))
    w = torch.randn(2, 197, 192, generator=torch.Generator().manual_seed(2))
    attn, grads = _hf_attention_grads(hf, x, lambda hs: (hs[9] * w).sum())    # blocks 9-11: no gradient
    assert grads[9] is None and grads[8] is not None
    attn = [a.detach() for a in attn]
    got = explain.attention_relevance(attn, grads, token=token)
    want = ag.relevance_loop(attn, grads, token=token)
    assert got.shape == (2, 14, 14) and got.dtype == torch.float32
    assert (got.double() - want).abs().max().item() <= 1e-5 * want.abs().max().item()
    with pytest.raises(ValueError, match="token"):
        explain.attention_relevance(attn, grads, token="first")


def test_attn_grad_outputs_reject_bad_arguments():
    from vit2spn import _lib
    B, mode = 2, _lib.MODE_FP32
    nbytes = _lib.lib.v2s_workspace_bytes(B, mode, 1, 1)
    g = _lib.Group()
    g.params, g.x, g.grads, g.slot, g.dfeat = 0x10000, 0x20000, 0x30000, 0, 0x40000
    arr = (_lib.Group * 1)(g)
    o = _lib.GroupOutputs()
    o.dattn[3] = 0x100002                             # not 4-byte aligned
    outs = (_lib.GroupOutputs * 1)(o)
    rc = _lib.lib.v2s_backbone_backward(arr, outs, 1, B, mode, C.c_void_p(1 << 20), nbytes, 12, 0, 1, None)
    err = _lib.lib.v2s_last_error().decode()
    assert rc != 0 and "group 0: dattn[3]" in err and "aligned" in err, err
    outs[0].dattn[3] = 0x100004
    outs[0].dpixels = 0x200004                        # the image gradient keeps its 16-byte rule
    rc = _lib.lib.v2s_backbone_backward(arr, outs, 1, B, mode, C.c_void_p(1 << 20), nbytes, 12, 0, 1, None)
    err = _lib.lib.v2s_last_error().decode()
    assert rc != 0 and "group 0: dpixels" in err and "aligned" in err, err
