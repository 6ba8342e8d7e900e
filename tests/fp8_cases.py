"""Shared helpers of the fp8 precision mode: e4m3 rounding as the hardware does it, the fp64 reference of a configuration-matrix row
(tests/tc_matrix_cases.py) with the fp8 mode's rounding, and the fp8 bars.

What the fp8 mode rounds (DESIGN.md section 4): the operands of every residual block's conv1 and conv2 are e4m3 -- the activations
act(GN(x)) unscaled, the weights scaled per output channel by s_n = 2^floor(log2(448 / max|w_n|)) and divided by s_n again after the
fp32 accumulation (exact: s_n is a power of two).  Every other convolution and linear layer takes fp16 operands, as on the fp16 path.
The reference keys this on the ``tower.<i>.conv1.weight`` / ``tower.<i>.conv2.weight`` tensors, not on shapes: the interaction conv
has the same shape and stays fp16.
"""
from __future__ import annotations

import functools

import torch

import tc_matrix_cases as M

E4M3_MAX = 448.0


def e4m3(t: torch.Tensor) -> torch.Tensor:
    """t rounded to the nearest e4m3 value (ties to even), saturating at +-448 like cvt.rn.satfinite: torch's cast rounds the same way
    but gives NaN past the largest finite value, so the input is clamped first.  Returns t's dtype."""
    return t.clamp(-E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn).to(t.dtype)


def weight_scale(w: torch.Tensor) -> torch.Tensor:
    """Per output channel power-of-two scale 2^floor(log2(448 / max|w_n|)) of a [n, ...] weight (1 for an all-zero row), computed the way
    the kernel does (exactly, from the binary exponent: max = f 2^k, f in [0.5, 1), 448 = 0.875 2^9)."""
    m = w.abs().reshape(w.shape[0], -1).amax(dim=1).to(torch.float32)
    f, k = torch.frexp(m)
    e = torch.where(f <= 0.875, 9 - k, 8 - k).clamp(-126, 126)
    e = torch.where(m > 0, e, torch.zeros_like(e))
    return torch.pow(2.0, e.to(torch.float64))


def quantize_weight(w: torch.Tensor) -> torch.Tensor:
    """The weights the e4m3 tensor cores multiply by, in w's dtype: e4m3(w s_n) / s_n."""
    s = weight_scale(w).to(w.dtype).reshape(-1, *([1] * (w.dim() - 1)))
    return e4m3(w * s) / s


class _Fp8F:
    """torch.nn.functional with fp16-rounded conv2d / linear operands, except for the tower convolutions listed by identity, whose
    operands are e4m3 (activations unscaled, weights per-channel scaled)."""

    def __init__(self, F, fp8_weights):
        self._F, self._ids = F, {id(t) for t in fp8_weights}

    def conv2d(self, x, w, *a, **k):
        if id(w) in self._ids:
            return self._F.conv2d(e4m3(x), quantize_weight(w), *a, **k)
        return self._F.conv2d(x.half().to(x.dtype), w.half().to(w.dtype), *a, **k)

    def linear(self, x, w, b=None):
        return self._F.linear(x.half().to(x.dtype), w.half().to(w.dtype), b)

    def __getattr__(self, n):
        return getattr(self._F, n)


def tower_conv_keys(sd):
    return [k for k in sd if k.startswith("tower.") and (k.endswith(".conv1.weight") or k.endswith(".conv2.weight"))]


def reference_fp8(name, sd=None, n=M.N_POSITIONS):
    """fp64 forward of a matrix row with the fp8 mode's rounding: (logits [n, 4672], values [n]) as float64 numpy."""
    if sd is None:
        return _reference_fp8_cached(name, n)
    return _reference_fp8(name, sd, n)


@functools.lru_cache(maxsize=None)
def _reference_fp8_cached(name, n):
    return _reference_fp8(name, None, n)


def _reference_fp8(name, sd, n):
    from oracle import nn_ref
    sd = M.state_dict(name) if sd is None else sd
    sd64 = {k: v.double() for k, v in sd.items()}
    F = nn_ref.F
    nn_ref.F = _Fp8F(F, [sd64[k] for k in tower_conv_keys(sd64)])
    try:
        with torch.no_grad():
            p, v = nn_ref.forward(sd64, M.net_config(name), M.positions()[:n].double())
    finally:
        nn_ref.F = F
    return p.numpy(), v.numpy()


def accepted(name):
    """Rows the fp8 mode runs: the fused CTA-pair tower (every row but the unfused SE path of se_hidden > 256)."""
    cfg = M.BY_NAME[name]["cfg"]
    hid = max(8, int(cfg["channels"] * cfg["se_ratio"]))
    return not (cfg["se"] and hid > 256)


ROWS = [r["name"] for r in M.ROWS if accepted(r["name"])]
REJECTED = [r["name"] for r in M.ROWS if not accepted(r["name"])]

# Bars of the fp8 mode against the plain fp64 reference (max |dlogit| / s, block RMS / s, max |dvalue|): they bound e4m3 quantisation
# noise only.  The emulated fp8 forward (reference_fp8) stays within half of them on every accepted row (tests/test_fp8_bars.py); the
# largest emulated metrics over the 34 rows at 24 positions were (0.486, 0.082) on w320_nose and |dvalue| 0.090 on w96_nose (w128:
# 0.067), so the value bar is 0.20 rather than the 0.11 a four-row sample suggested.  Kernel bugs are caught against reference_fp8
# with the fp16 bars instead (tests/test_fp8_gpu.py): at this width quantisation noise and the injected faults overlap.
BARS = {"fp8": (1.0, 0.17, 0.20)}


# Bars of the GPU fp8 forward against reference_fp8.  The fp16 bars cannot hold here: e4m3 rounding amplifies any difference in the
# values it rounds.  Perturbing the tower convolutions' inputs by 1e-4 relative (a fifth of an fp16 ulp) moves the emulated w288 forward
# by (0.044, 0.0089, 0.0080) -- twice the fp16 bars -- because operands cross e4m3 rounding boundaries; the GPU's inputs to those
# convolutions differ from the fp64 reference's by at least that much (fp32 GroupNorm, the fp16 tensors of the other layers).  Measured on
# one B200 (1000 W power limit) over the 34 accepted rows at 96 positions, the worst GPU rows against reference_fp8 were (0.143, 0.023)
# on w320_nose and |dvalue| 0.031 on w96_nose; these bars sit about 2x above that.  Only the zeroed 3x3 tap is large against them.
EMULATION_BARS = (0.3, 0.05, 0.065)


def within(m, bars):
    return all(a <= b for a, b in zip(m, bars))


def excess(m, bars):
    return max(a / b for a, b in zip(m, bars))

