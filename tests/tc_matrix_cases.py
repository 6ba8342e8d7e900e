"""Shared helpers: the configuration matrix of the fp16 / bf16 tensor-core forward, its fp64 reference and its error bars.

Every row is a small network (2-4 blocks, attention after every block) that takes one branch of ``tc_net_prepare`` /
``tc_net_forward`` the other rows do not, with non-trivial weights (``nn_ref.make_state_dict``: norm gains 1 +- 0.2, biases 0.1 sigma,
relative-position biases 0.5 sigma), never the reference's init, whose unit gammas and zero betas / head biases hide a parameter read
from the wrong channel.  Callers compare logits and values only.
"""
from __future__ import annotations

import functools

import numpy as np
import torch

N_POSITIONS = 96

# launch sites of the 16-bit forward (nn_tc_kernels.cu, m0_profile_get) that the rows below are checked against
SITES = ("conv1+gn", "conv2+se+res+gn", "conv2+pool", "se_fc1", "se_tail", "se_gate", "se_apply_gn", "attention_tc", "attention_f32",
         "f32_to_bf16", "ln_res_gn", "gemm_pst", "groupnorm_f32", "gemm_pol_fc1", "gemm_val_fc2")

_BASE = dict(planes=19, blocks=2, attention=True, attention_every_k=1, infer_attention_stride=1, policy_size=4672, norm="group",
             activation="silu", value_activation="leaky_relu", preact=True, policy_factor_rank=160, se=True, se_ratio=0.25,
             chess_features=True, piece_square_tables=True, attention_relbias=True, attention_unmasked_mix=0.2, self_supervised=False,
             ssl_tasks=[])

# the path every width takes by default: fused SE pipeline, tensor-core attention (head dim 16), heads on tensor cores fed by ln_res_gn
_FUSED = ("conv1+gn", "conv2+se+res+gn", "se_fc1", "se_tail", "attention_tc", "ln_res_gn", "gemm_pst", "gemm_pol_fc1", "gemm_val_fc2")
_NOT_FUSED = ("conv2+pool", "se_gate", "attention_f32", "f32_to_bf16", "groupnorm_f32")


def _row(name, C, must=_FUSED, must_not=_NOT_FUSED, **over):
    cfg = dict(_BASE, channels=C, attention_heads=C // 16)
    cfg.update(over)
    return dict(name=name, cfg=cfg, must=tuple(must), must_not=tuple(must_not))


def _swap(seq, drop=(), add=()):
    return tuple(s for s in seq if s not in drop) + tuple(add)


_HEADS_F32 = dict(must=_swap(_FUSED, drop=("gemm_pol_fc1", "gemm_val_fc2")), must_not=_NOT_FUSED + ("gemm_pol_fc1", "gemm_val_fc2"))
_ATT_F32 = dict(must=_swap(_FUSED, drop=("attention_tc",), add=("attention_f32", "f32_to_bf16")),
                must_not=_swap(_NOT_FUSED, drop=("attention_f32", "f32_to_bf16"), add=("attention_tc",)))

ROWS = [
    # every accepted width, head dim 16 (C % 64 == 32 at 96, 160, 224, 288: half-populated last k-block / GN / LN slice)
    *[_row(f"w{C}", C) for C in range(64, 321, 32)],
    # policy_fc1 wider than 256 columns (zero-padded to two 160-column halves)
    _row("w288_r272", 288, policy_factor_rank=272),
    _row("w288_r288", 288, policy_factor_rank=288),
    _row("w288_r304", 288, policy_factor_rank=304),
    _row("w320_r288", 320, policy_factor_rank=288),
    # head dim 8 and 32: fp32 attention inside the 16-bit forward, then f32_to_bf16
    _row("w128_hd8", 128, attention_heads=16, **_ATT_F32),
    _row("w256_hd32", 256, attention_heads=8, **_ATT_F32),
    _row("w320_hd32", 320, attention_heads=10, **_ATT_F32),
    # stem without the chess-specific features / without the piece-square tables
    _row("w160_nochess", 160, chess_features=False, must=_swap(_FUSED, drop=("gemm_pst",), add=("groupnorm_f32",)),
         must_not=_swap(_NOT_FUSED, drop=("groupnorm_f32",), add=("gemm_pst",))),
    _row("w288_nopst", 288, piece_square_tables=False, must=_swap(_FUSED, drop=("gemm_pst",)), must_not=_NOT_FUSED + ("gemm_pst",)),
    # no SE: the fused conv2 epilogue without a gate
    _row("w96_nose", 96, se=False, must=_swap(_FUSED, drop=("se_fc1", "se_tail")), must_not=_NOT_FUSED + ("se_fc1", "se_tail")),
    _row("w320_nose", 320, se=False, must=_swap(_FUSED, drop=("se_fc1", "se_tail")), must_not=_NOT_FUSED + ("se_fc1", "se_tail")),
    # se_hidden 272 > 256 turns the fused SE pipeline off: conv2 + pool, se_gate, se_apply_gn
    _row("w320_se085", 320, se_ratio=0.85, must=_swap(_FUSED, drop=("conv2+se+res+gn", "se_fc1", "se_tail"), add=("conv2+pool", "se_gate", "se_apply_gn")),
         must_not=_swap(_NOT_FUSED, drop=("conv2+pool", "se_gate"), add=("conv2+se+res+gn", "se_fc1", "se_tail"))),
    # se_hidden 8: the first SE GEMM runs 16 columns
    _row("w64_se01", 64, se_ratio=0.1),
    # no attention at all: the heads convert the residual stream with f32_to_bf16
    _row("w192_noatt", 192, attention=False, must=_swap(_FUSED, drop=("attention_tc", "ln_res_gn"), add=("f32_to_bf16",)),
         must_not=_swap(_NOT_FUSED, drop=("f32_to_bf16",), add=("attention_tc", "ln_res_gn"))),
    _row("w224_norelbias", 224, attention_relbias=False),
    _row("w96_mix0", 96, attention_unmasked_mix=0.0),
    _row("w288_mix1", 288, attention_unmasked_mix=1.0),
    # policy heads on the fp32 fallback: dense policy_fc, a rank that is not a multiple of 16, a rank above 320
    _row("w128_r0", 128, policy_factor_rank=0, **_HEADS_F32),
    _row("w96_r40", 96, policy_factor_rank=40, **_HEADS_F32),
    _row("w64_r384", 64, policy_factor_rank=384, **_HEADS_F32),
    # narrow tensor-core policy ranks
    _row("w64_r16", 64, policy_factor_rank=16),
    _row("w160_r48", 160, policy_factor_rank=48),
    # activations: relu trunk with a silu value head, and a relu value head
    _row("w256_relu_silu", 256, activation="relu", value_activation="silu"),
    _row("w96_relu", 96, activation="relu", value_activation="relu"),
    # stride 2 over 3 blocks: the last block skips attention, so the heads take f32_to_bf16 instead of ln_res_gn's half copy
    _row("w288_stride2", 288, blocks=3, infer_attention_stride=2, must=_FUSED + ("f32_to_bf16",), must_not=_swap(_NOT_FUSED, drop=("f32_to_bf16",))),
    # 4 blocks, the last one with attention: the heads read the 16-bit copy ln_res_gn writes
    _row("w320_4blocks", 320, blocks=4),
]
BY_NAME = {r["name"]: r for r in ROWS}
assert len(BY_NAME) == len(ROWS)


def net_config(name):
    from matrix0_b200.model import NetConfig
    return NetConfig(**BY_NAME[name]["cfg"])


@functools.lru_cache(maxsize=None)
def state_dict(name, seed=3):
    """fp32 synthetic weights of a row (CPU)."""
    from matrix0_b200.model import parameter_shapes
    from oracle import nn_ref
    return nn_ref.make_state_dict(parameter_shapes(net_config(name)), seed)


@functools.lru_cache(maxsize=None)
def positions():
    """[96, 19, 8, 8] float32 planes of random-playout positions (oracle encoder)."""
    from conftest import random_playout_boards
    from oracle.encoding_ref import encode_board
    boards = random_playout_boards(16, 140, seed=41)[::5][:N_POSITIONS]
    assert len(boards) == N_POSITIONS
    return torch.from_numpy(np.stack([encode_board(b) for b in boards]))


def reference(name, sd=None, rounding=None, n=N_POSITIONS):
    """fp64 forward of a row over the first n positions: (logits [n, 4672], values [n]) as float64 numpy.  ``sd`` replaces the row's
    weights (injected faults); ``rounding`` in {None, torch.float16, torch.bfloat16} rounds the inputs and weights of every convolution
    and linear layer to that format first (what the tensor-core GEMMs consume)."""
    if sd is None and rounding is None:
        return _reference_cached(name, n)
    return _reference(name, sd, rounding, n)


@functools.lru_cache(maxsize=None)
def _reference_cached(name, n):
    return _reference(name, None, None, n)


class _RoundedF:
    """torch.nn.functional with the operands of conv2d / linear rounded to a 16-bit format."""

    def __init__(self, F, dt):
        self._F, self._dt = F, dt

    def _q(self, t):
        return t.to(self._dt).to(t.dtype)

    def conv2d(self, x, w, *a, **k):
        return self._F.conv2d(self._q(x), self._q(w), *a, **k)

    def linear(self, x, w, b=None):
        return self._F.linear(self._q(x), self._q(w), b)

    def __getattr__(self, n):
        return getattr(self._F, n)


def _reference(name, sd, rounding, n):
    from oracle import nn_ref
    sd = state_dict(name) if sd is None else sd
    sd64 = {k: v.double() for k, v in sd.items()}
    F = nn_ref.F
    if rounding is not None:
        nn_ref.F = _RoundedF(F, rounding)
    try:
        with torch.no_grad():
            p, v = nn_ref.forward(sd64, net_config(name), positions()[:n].double())
    finally:
        nn_ref.F = F
    return p.numpy(), v.numpy()


def metrics(logits, values, ref):
    """(max |dlogit| / s, largest RMS(dlogit) / s over the 73 blocks of 64 logit columns, max |dvalue|), s = std of the reference logits.
    The per-block RMS keeps an error confined to one column slice (a padded last slice, one policy_fc2 launch) from being diluted."""
    rl, rv = ref
    lg = np.asarray(logits, dtype=np.float64).reshape(rl.shape)
    s = float(rl.std())
    d = lg - rl
    blocks = np.sqrt((d.reshape(d.shape[0], -1, 64) ** 2).mean(axis=(0, 2)))
    return float(np.abs(d).max()) / s, float(blocks.max()) / s, float(np.abs(np.asarray(values, dtype=np.float64).reshape(rv.shape) - rv).max())


# Bars per output format, against the fp64 reference: (max |dlogit| / s, block RMS / s, max |dvalue|).  Measured on one B200
# (1000 W power limit) over the 34 rows at 96 positions, the worst row (w320_nose in all three metrics but fp16 max |dvalue|, w96_mix0)
# gave fp16 (9.2e-3, 1.5e-3, 2.2e-3) and bf16 (7.1e-2, 1.2e-2, 2.2e-2); the bars sit about 2x above that.  The smallest injected
# fault the format must catch (tests/test_tc_matrix_bars.py, fp64 on the CPU) is the dropped SE fc1 bias for fp16, (8.9e-2, 1.4e-2,
# 2.7e-2) at its least, and the zeroed 3x3 tap for bf16, (0.64, 0.12, 0.14): each bar is at most half of those.
BARS = {
    "fp16": (2.0e-2, 3.2e-3, 4.5e-3),
    "bf16": (1.5e-1, 2.5e-2, 4.5e-2),
}
# the fp32 CUDA path: the existing relative bar of the oracle comparisons
FP32_REL = 1e-4


def within(m, fmt):
    return all(a <= b for a, b in zip(m, BARS[fmt]))


def excess(m, fmt):
    """Largest ratio metric / bar: > 1 fails the bar."""
    return max(a / b for a, b in zip(m, BARS[fmt]))


# ---- injected faults (a parameter read from the wrong place, a dropped term) applied to a row's weights ----
def _last_block(name):
    from matrix0_b200.model import tower_layout
    return tower_layout(net_config(name))[-1]


def fault_gn_gamma_tail(name, sd):
    sd[f"tower.{_last_block(name)[0]}.bn2.weight"][-32:] = 1.0


def fault_ln_beta_tail(name, sd):
    sd[f"tower.{_last_block(name)[1]}.norm.bias"][-32:] = 0.0


def fault_se_fc1_bias(name, sd):
    sd["tower.0.se_fc1.bias"].zero_()


def fault_conv_tap(name, sd):
    sd["tower.0.conv2.weight"][:, :, 0, 2] = 0.0


def fault_value_fc2_bias(name, sd):
    sd["value_fc2.bias"].zero_()


def fault_policy_fc1_bias_tail(name, sd):
    sd["policy_fc1.bias"][-16:] = 0.0


FAULTS = {f.__name__[len("fault_"):]: f for f in (fault_gn_gamma_tail, fault_ln_beta_tail, fault_se_fc1_bias, fault_conv_tap,
                                                  fault_value_fc2_bias, fault_policy_fc1_bias_tail)}


def faulted_state_dict(name, fault):
    sd = {k: v.clone() for k, v in state_dict(name).items()}
    FAULTS[fault](name, sd)
    return sd
