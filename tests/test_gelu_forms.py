"""CPU: the one-MUFU GELU forms of the chained MLP kernel (vit-2spn_b200/csrc/tc_math.cuh, used by mlp_tc.cu) restated
in numpy fp32 with the coefficients PARSED from the header, against the exact erf GELU of the reference (HF
hidden_act="gelu", HF:modeling_vit.py:296-299) and its derivative: the approximation error must disappear inside the
16-bit rounding of the activations (bf16 2^-9, fp16 2^-11 relative).  tools/fit_gelu.py regenerates the coefficients."""
import os
import re

import numpy as np
from scipy.special import erf

HDR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "vit-2spn_b200", "csrc", "tc_math.cuh")


def _body(name):
    src = open(HDR).read()
    i = src.index(f"float {name}(float x)")
    return src[i:src.index("\n}\n", i)]


def _floats(text):
    return [np.float32(v) for v in re.findall(r"(-?\d\.\d+e[+-]\d+)f", text)]


def _exponent(ax, c):
    r = np.full_like(ax, c[0])
    for cc in c[1:]:
        r = (r * ax + cc).astype(np.float32)
    return (r * ax).astype(np.float32)


def test_forward_and_derivative_forms_match_erf_gelu():
    fwd, bwd = _body("gelu_fast"), _body("gelu_grad_fast")
    cf = _floats(fwd)                     # c4, c3, c2, c1, c0 in Horner order
    cb = _floats(bwd)
    assert len(cf) == 5 and len(cb) == 11 and cb[:5] == cf       # the derivative reuses the forward exponent
    x = np.linspace(-30, 30, 1200001).astype(np.float32)
    ax = np.abs(x)
    q = _exponent(ax, cf)
    assert float(q.max()) <= 0.0 and np.all(np.diff(q[x >= 0]) <= 0)       # exponent <= 0 and decreasing: no overflow, no clamp
    e = np.exp2(q).astype(np.float32)
    g = (np.maximum(x, np.float32(0)) - np.float32(0.5) * ax * e).astype(np.float32)
    t = np.full_like(ax, cb[5])
    for cc in cb[6:]:
        t = (t * ax + cc).astype(np.float32)
    m = (t * e).astype(np.float32)
    d = np.where(x > 0, np.float32(1) - m, m)
    xd = x.astype(np.float64)
    cdf = 0.5 * (1 + erf(xd / np.sqrt(2)))
    ref_g, ref_d = xd * cdf, cdf + xd * np.exp(-xd * xd / 2) / np.sqrt(2 * np.pi)
    eg, ed = np.abs(g - ref_g).max(), np.abs(d - ref_d).max()
    assert eg < 1e-6 and ed < 3e-6, (eg, ed)
    # relative to what the 16-bit store keeps: far below half an fp16 ulp of values of order one
    big = np.abs(ref_g) > 1e-2
    assert (np.abs(g - ref_g)[big] / np.abs(ref_g)[big]).max() < 2.0 ** -13
    # exact limits
    assert g[0] == 0.0 and g[-1] == x[-1] and d[0] == 0.0 and d[-1] == 1.0
