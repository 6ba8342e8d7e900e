"""The error bars of the 16-bit configuration matrix (tests/tc_matrix_cases.py) checked on the CPU, in fp64, without a GPU.

- Not too tight: the fp64 reference with every convolution and linear layer fed 16-bit-rounded inputs and weights (the rounding the
  tensor-core GEMMs cannot avoid) stays within half the bar on every row.
- Not vacuous: each injected fault (a gamma / beta tail read from the wrong channels, a dropped bias, a zeroed 3x3 tap) exceeds the fp16
  bar at least 3x.  bf16 keeps 8 mantissa bits and needs a bar about 8x wider, so only the faults that are large against that bar are
  required of it: the zeroed tap.

These run over the first 24 of the matrix's 96 positions to stay fast; the GPU tests use all 96.
"""
import pytest
import torch

import tc_matrix_cases as M

N = 24
FAULT_ROWS = ("w96", "w288", "w320")
BF16_FAULTS = ("conv_tap",)


@pytest.mark.parametrize("name", [r["name"] for r in M.ROWS])
def test_rounding_noise_is_within_half_the_bars(name):
    ref = M.reference(name, n=N)
    for fmt, dt in (("fp16", torch.float16), ("bf16", torch.bfloat16)):
        m = M.metrics(*M.reference(name, rounding=dt, n=N), ref)
        assert M.excess(m, fmt) <= 0.5, (fmt, m, M.BARS[fmt])


@pytest.mark.parametrize("name", FAULT_ROWS)
@pytest.mark.parametrize("fault", sorted(M.FAULTS))
def test_injected_faults_exceed_the_bars(name, fault):
    m = M.metrics(*M.reference(name, sd=M.faulted_state_dict(name, fault), n=N), M.reference(name, n=N))
    assert M.excess(m, "fp16") >= 3.0, (m, M.BARS["fp16"])
    if fault in BF16_FAULTS:
        assert M.excess(m, "bf16") >= 3.0, (m, M.BARS["bf16"])


def test_reference_runs_in_the_state_dict_dtype():
    from oracle import nn_ref
    sd = {k: v.double() for k, v in M.state_dict("w64").items()}
    p, v = nn_ref.forward(sd, M.net_config("w64"), M.positions()[:2])
    assert p.dtype == torch.float64 and v.dtype == torch.float64
