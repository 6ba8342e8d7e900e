"""TEST INFRASTRUCTURE ONLY -- functional fp32 restatement of ``PolicyValueNet.forward`` (eval mode).

Plain PyTorch CPU ops on a reference-format ``state_dict`` (``azchess/model/resnet.py``), each step
citing the reference lines it follows.  ``infer_amp_tower`` is forced off: this is the fp32 oracle
(SURVEY Q11).  Pinned against the UNMODIFIED reference module (loaded with a stub ``chess``) in
tests/test_oracle_nn.py where the reference tree is present, and through tests/golden/nn_golden.npz.
``make_state_dict`` produces deterministic weights from the parameter names so that goldens need
to store outputs only.  Only tests/, smoke() and bench.py's CPU legs import this module.
"""
from __future__ import annotations

import math
import zlib
from typing import Dict

import numpy as np
import torch
import torch.nn.functional as F


def make_state_dict(shapes: Dict[str, tuple], seed: int = 0) -> Dict[str, torch.Tensor]:
    """Deterministic pseudo-random parameters keyed by name (numpy legacy RandomState: stable across versions)."""
    sd = {}
    for name, shape in shapes.items():
        rs = np.random.RandomState((zlib.crc32(name.encode()) + seed * 7919) & 0x7FFFFFFF)
        if name == "_policy_logit_scale_raw":
            v = np.array(math.log(math.expm1(0.8)), dtype=np.float32)
        elif len(shape) <= 1:
            if name.endswith("weight"):
                v = (1.0 + 0.2 * rs.standard_normal(shape)).astype(np.float32)   # norm gains
            else:
                v = (0.1 * rs.standard_normal(shape)).astype(np.float32)         # biases
        elif name.endswith("position_encoding"):
            v = (0.1 * rs.standard_normal(shape)).astype(np.float32)
        elif name.endswith("rel_bias"):
            v = (0.5 * rs.standard_normal(shape)).astype(np.float32)
        else:
            fan_in = int(np.prod(shape[1:]))
            v = (rs.standard_normal(shape) * math.sqrt(2.0 / fan_in)).astype(np.float32)
        sd[name] = torch.from_numpy(np.ascontiguousarray(v)).reshape(tuple(shape))
    return sd


def _gn(x, w, b):  # _norm(..., "group"): nn.GroupNorm(C // 16, C), resnet.py:18-24
    return F.group_norm(x, max(1, x.shape[1] // 16), w, b, eps=1e-5)


def _act(x, name):
    return F.silu(x) if name == "silu" else F.relu(x)


def _attn_mask() -> torch.Tensor:  # resnet.py:105-129
    n = 8
    rows = torch.arange(n).repeat_interleave(n)
    cols = torch.arange(n).repeat(n)
    dr = rows[:, None] - rows[None, :]
    dc = cols[:, None] - cols[None, :]
    knight = ((dr.abs() == 2) & (dc.abs() == 1)) | ((dr.abs() == 1) & (dc.abs() == 2))
    adjacent = (dr.abs() <= 1) & (dc.abs() <= 1)
    return ((dr == 0) | (dc == 0) | (dr.abs() == dc.abs()) | knight | adjacent).view(1, 1, 64, 64)


def _attention(x, sd, p, cfg):  # ChessAttention.forward, resnet.py:137-190
    B, C, H, W = x.shape
    heads = cfg.attention_heads
    d = C // heads
    qkv = F.conv2d(x, sd[p + "qkv.weight"]).reshape(B, 3, heads, d, 64).permute(1, 0, 2, 4, 3)
    q, k, v = qkv[0], qkv[1], qkv[2]
    scores = torch.matmul(q, k.transpose(-2, -1)) * (1.0 / math.sqrt(d))
    if cfg.attention_relbias:
        scores = scores + sd[p + "rel_bias"]
    scores = torch.clamp(scores, -50.0, 50.0)
    out_m = torch.matmul(F.softmax(scores.masked_fill(_attn_mask() == 0, -1e4), dim=-1), v)
    mix = float(cfg.attention_unmasked_mix)
    if 0.0 < mix < 1.0:
        out_u = torch.matmul(F.softmax(scores, dim=-1), v)
        blend = 1.0 - mix
        out = blend * out_m + (1.0 - blend) * out_u
    elif mix >= 1.0:
        out = out_m
    else:
        out = torch.matmul(F.softmax(scores, dim=-1), v)
    out = out.transpose(1, 2).reshape(B, 64, C).transpose(1, 2).reshape(B, C, H, W)
    out = F.conv2d(out, sd[p + "proj.weight"]) + x
    out = F.layer_norm(out.permute(0, 2, 3, 1), (C,), sd[p + "norm.weight"], sd[p + "norm.bias"], eps=1e-5)
    return out.permute(0, 3, 1, 2).contiguous()


def forward(sd: Dict[str, torch.Tensor], cfg, x: torch.Tensor, return_ssl: bool = False):
    """cfg: object with NetConfig attributes (matrix0_b200.model.NetConfig or the reference's)."""
    from matrix0_b200.model import SSL_ORDER, tower_layout
    act = cfg.activation
    x = x.float()
    # stem + chess-specific features (always fp32), resnet.py:662-668, :229-244
    x = _act(_gn(F.conv2d(x, sd["stem.0.weight"], padding=1), sd["stem.1.weight"], sd["stem.1.bias"]), act)
    if cfg.chess_features:
        x = x + sd["chess_features.position_encoding"]
        if cfg.piece_square_tables:
            x = x + _act(_gn(F.conv2d(x, sd["chess_features.pst_conv.weight"]), sd["chess_features.pst_norm.weight"], sd["chess_features.pst_norm.bias"]), act)
        x = x + _act(_gn(F.conv2d(x, sd["chess_features.interaction_conv.weight"], padding=1), sd["chess_features.interaction_norm.weight"],
                         sd["chess_features.interaction_norm.bias"]), act)
    # tower with inference attention stride, resnet.py:676-689; ResidualBlock (pre-activation) :44-84
    att_seen = 0
    stride = max(1, int(cfg.infer_attention_stride))
    for bi, ai in tower_layout(cfg):
        p = f"tower.{bi}."
        out = F.conv2d(_act(_gn(x, sd[p + "bn1.weight"], sd[p + "bn1.bias"]), act), sd[p + "conv1.weight"], padding=1)
        out = F.conv2d(_act(_gn(out, sd[p + "bn2.weight"], sd[p + "bn2.bias"]), act), sd[p + "conv2.weight"], padding=1)
        if cfg.se:
            w = F.adaptive_avg_pool2d(out, 1).reshape(out.shape[0], -1)
            w = _act(F.linear(w, sd[p + "se_fc1.weight"], sd[p + "se_fc1.bias"]), act)
            w = torch.sigmoid(F.linear(w, sd[p + "se_fc2.weight"], sd[p + "se_fc2.bias"]))
            out = out * w[:, :, None, None]
        x = x + out
        if ai is not None:
            att_seen += 1
            if att_seen % stride == 0:
                x = _attention(x, sd, f"tower.{ai}.", cfg)
    feats = x
    # heads, resnet.py:697-753
    p = _act(_gn(F.conv2d(feats, sd["policy_head.0.weight"]), sd["policy_head.1.weight"], sd["policy_head.1.bias"]), act).reshape(x.shape[0], -1)
    if cfg.policy_factor_rank > 0:
        p = F.linear(F.relu(F.linear(p, sd["policy_fc1.weight"], sd["policy_fc1.bias"])), sd["policy_fc2.weight"], sd["policy_fc2.bias"])
    else:
        p = F.linear(p, sd["policy_fc.weight"], sd["policy_fc.bias"])
    p = p * torch.clamp(F.softplus(sd["_policy_logit_scale_raw"]) + 1e-3, max=5.0)

    def vact(t):
        n = cfg.value_activation
        return F.silu(t) if n == "silu" else (F.leaky_relu(t, negative_slope=0.05) if n == "leaky_relu" else F.relu(t))
    v = _act(_gn(F.conv2d(feats, sd["value_head.0.weight"]), sd["value_head.1.weight"], sd["value_head.1.bias"]), act)
    v = _act(_gn(F.conv2d(v, sd["value_head.3.weight"]), sd["value_head.4.weight"], sd["value_head.4.bias"]), act).reshape(x.shape[0], -1)
    v = vact(F.linear(v, sd["value_fc1.weight"], sd["value_fc1.bias"]))
    v = vact(F.linear(v, sd["value_fc2.weight"], sd["value_fc2.bias"]))
    v = v * torch.sigmoid(F.linear(v, sd["value_gate.0.weight"], sd["value_gate.0.bias"]))
    v = torch.tanh(F.linear(v, sd["value_fc3.weight"], sd["value_fc3.bias"])).squeeze(-1)
    if not return_ssl:
        return p, v
    ssl = {}
    for t in SSL_ORDER:
        if cfg.self_supervised and t in cfg.ssl_tasks:
            q = f"ssl_heads.{t}."
            h = _act(_gn(F.conv2d(feats, sd[q + "0.weight"]), sd[q + "1.weight"], sd[q + "1.bias"]), act)
            ssl[t] = F.conv2d(h, sd[q + "3.weight"])
    return p, v, ssl


class OracleNet:
    """CPU fp32 evaluator with the inference-backend seam (``infer_np``) -- the CPU baseline's network."""

    def __init__(self, cfg, sd):
        self.cfg, self.sd = cfg, {k: v.float() for k, v in sd.items()}

    @torch.no_grad()
    def infer_np(self, arr):
        a = np.asarray(arr, dtype=np.float32)
        if a.ndim == 3:
            a = a[None]
        p, v = forward(self.sd, self.cfg, torch.from_numpy(np.ascontiguousarray(a)))
        return p.numpy(), v.numpy()
