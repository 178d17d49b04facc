"""CPU reference of ViTModel's per-layer outputs (test helper, not a test module): the hidden states and attention
probabilities of ``transformers.ViTModel(x, output_hidden_states=True, output_attentions=True)`` with eager attention,
stated with the oracle's own functions (``oracle/vit2spn_oracle.py``), so the oracle's ``rounding`` model of the bf16 /
fp16 modes applies to them as well.  Pinned to transformers by ``tests/test_vit_outputs_cpu.py``."""
import torch

from oracle import vit2spn_oracle as orc


def attention_probs(p, l, h):
    """softmax(q k^T / sqrt(64)) of block ``l`` for its input ``h``: fp32 [B,3,197,197], what HF's eager attention returns
    (HF:eager_attention_forward).  q and k follow ``orc.vit_layer`` (and its rounding model); the probabilities
    themselves are not rounded - the library outputs them in fp32."""
    pre = f"encoder.layer.{l}."
    x = orc._rnd(orc.layer_norm(h, p[pre + "layernorm_before.weight"], p[pre + "layernorm_before.bias"]), "xn")
    a = pre + "attention.attention."
    q = orc._rnd(x @ orc._rnd(p[a + "query.weight"], "w").t() + p[a + "query.bias"], "qkv")
    k = orc._rnd(x @ orc._rnd(p[a + "key.weight"], "w").t() + p[a + "key.bias"], "qkv")
    B, N, _ = q.shape
    q = q.view(B, N, orc.HEADS, orc.HEAD_DIM).transpose(1, 2)
    k = k.view(B, N, orc.HEADS, orc.HEAD_DIM).transpose(1, 2)
    return torch.softmax((q @ k.transpose(-1, -2)) * (orc.HEAD_DIM ** -0.5), dim=-1)


def backbone_outputs(p, x):
    """``ViTModel(x, output_hidden_states=True, output_attentions=True)`` with eager attention: (hidden_states, attentions)
    = the embedding output and the 12 block outputs (13 x [B,197,192], before the final LayerNorm) and the 12 attention
    probabilities [B,3,197,197] (HF:ViTEncoder)."""
    hs, probs = [orc.patch_embed(p, x)], []
    for l in range(orc.LAYERS):
        probs.append(attention_probs(p, l, hs[-1]))
        hs.append(orc.vit_layer(p, l, hs[-1]))
    return tuple(hs), tuple(probs)
