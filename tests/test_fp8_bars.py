"""The fp8 precision mode checked on the CPU, in fp64, without a GPU (tests/fp8_cases.py):

- the e4m3 rounding helper does what cvt.rn.satfinite.e4m3x2.f32 does (ties to even, saturation instead of NaN, subnormals);
- the weight scale is the power of two of the quantisation rule;
- not too tight: the emulated fp8 forward stays within half the fp8 bars on every row the mode accepts;
- not vacuous: each injected fault exceeds the fp16 bars at least 3x when the faulted and the clean net are both emulated in fp8;
- the GPU's bars against reference_fp8 (EMULATION_BARS) hold the emulation's own sensitivity to a 1e-4 relative perturbation of the
  e4m3-rounded inputs within half of them, and the zeroed 3x3 tap -- the fault the GPU test loads -- exceeds them at least 2x.

These run over the first 24 of the matrix's 96 positions to stay fast; the GPU tests use all 96.
"""
import math

import pytest
import torch

import fp8_cases as F8
import tc_matrix_cases as M

N = 24
FAULT_ROWS = ("w96", "w288", "w320")


def test_e4m3_rounding_matches_the_hardware_conversion():
    t = torch.tensor([1000.0, -1000.0, 449.0, 448.0, 1.0625, 0.0011, 1.125 + 0.0625, 0.013671875, -0.0, 2.0 ** -10, 3 * 2.0 ** -11],
                     dtype=torch.float64)
    got = F8.e4m3(t)
    want = [448.0, -448.0, 448.0, 448.0, 1.0, 2.0 ** -9, 1.25, 0.013671875, -0.0, 0.0, 2.0 ** -9]
    # 1.0625 is the tie between 1.0 and 1.125 -> even mantissa 1.0; 1.1875 the tie between 1.125 and 1.25 -> 1.25;
    # 0.013671875 = 7 * 2^-9 is the largest subnormal; 2^-10 is the tie between 0 and 2^-9 -> 0; 3 * 2^-11 rounds up to 2^-9
    assert got.tolist() == want
    assert math.copysign(1.0, float(got[8])) < 0      # negative zero keeps its sign
    assert not torch.isnan(got).any()


def test_weight_scale_is_the_power_of_two_rule():
    g = torch.Generator().manual_seed(5)
    w = torch.randn(64, 32, 3, 3, generator=g, dtype=torch.float64) * torch.logspace(-6, 2, 64, dtype=torch.float64)[:, None, None, None]
    w[3] = 0.0
    w[7, 0, 0, 0] = 448.0 / 8                       # max exactly 448 / 2^3: scale 2^3
    s = F8.weight_scale(w)
    for n in range(64):
        m = float(w[n].abs().max())
        want = 1.0 if m == 0 else 2.0 ** math.floor(math.log2(448.0 / m))
        assert float(s[n]) == want, (n, m, float(s[n]), want)
    q = F8.quantize_weight(w)
    assert float((q[3]).abs().max()) == 0.0
    assert float((w * s[:, None, None, None]).abs().max()) <= 448.0


@pytest.mark.parametrize("name", F8.ROWS)
def test_fp8_rounding_noise_is_within_half_the_bars(name):
    m = M.metrics(*F8.reference_fp8(name, n=N), M.reference(name, n=N))
    assert F8.excess(m, F8.BARS["fp8"]) <= 0.5, (m, F8.BARS["fp8"])


@pytest.mark.parametrize("name", FAULT_ROWS)
@pytest.mark.parametrize("fault", sorted(M.FAULTS))
def test_injected_faults_exceed_the_fp16_bars_against_the_fp8_reference(name, fault):
    m = M.metrics(*F8.reference_fp8(name, sd=M.faulted_state_dict(name, fault), n=N), F8.reference_fp8(name, n=N))
    assert M.excess(m, "fp16") >= 3.0, (m, M.BARS["fp16"])


def _perturbed_reference_fp8(name, eps, n=N):
    """reference_fp8 with the inputs of the e4m3 convolutions scaled by 1 + eps * N(0, 1) before rounding."""
    from oracle import nn_ref
    g = torch.Generator().manual_seed(0)

    class Perturbed(F8._Fp8F):
        def conv2d(self, x, w, *a, **k):
            if id(w) in self._ids:
                x = x * (1 + eps * torch.randn(x.shape, generator=g, dtype=x.dtype))
            return super().conv2d(x, w, *a, **k)

    sd64 = {k: v.double() for k, v in M.state_dict(name).items()}
    F = nn_ref.F
    nn_ref.F = Perturbed(F, [sd64[k] for k in F8.tower_conv_keys(sd64)])
    try:
        with torch.no_grad():
            p, v = nn_ref.forward(sd64, M.net_config(name), M.positions()[:n].double())
    finally:
        nn_ref.F = F
    return p.numpy(), v.numpy()


@pytest.mark.parametrize("name", FAULT_ROWS)
def test_emulation_bars_cover_the_rounding_sensitivity(name):
    m = M.metrics(*_perturbed_reference_fp8(name, 1e-4), F8.reference_fp8(name, n=N))
    assert F8.excess(m, F8.EMULATION_BARS) <= 0.5, (m, F8.EMULATION_BARS)
    assert M.excess(m, "fp16") > 1.0, m        # why the fp16 bars cannot be used against reference_fp8


@pytest.mark.parametrize("name", FAULT_ROWS)
def test_zeroed_tap_exceeds_the_emulation_bars(name):
    m = M.metrics(*F8.reference_fp8(name, sd=M.faulted_state_dict(name, "conv_tap"), n=N), F8.reference_fp8(name, n=N))
    assert F8.excess(m, F8.EMULATION_BARS) >= 2.0, (m, F8.EMULATION_BARS)


def test_the_interaction_conv_stays_fp16():
    sd = M.state_dict("w64")
    keys = F8.tower_conv_keys(sd)
    assert "chess_features.interaction_conv.weight" not in keys
    assert len(keys) == 2 * M.net_config("w64").blocks
    assert sd["chess_features.interaction_conv.weight"].shape == sd["tower.0.conv1.weight"].shape


def test_rejected_rows():
    assert F8.REJECTED == ["w320_se085"]
