"""Native evaluator: drop-in for the inference side of ``azchess/model/resnet.py``.

``PolicyValueNet`` keeps the reference's call surface (``from_config``, ``forward(x, return_ssl)``,
``load_state_dict(sd, strict=False)`` with the reference's key names, ``eval()``, ``to()``,
``count_parameters()``, ``cfg.policy_size``) but holds its parameters as plain CUDA tensors in the
layouts the kernels consume and runs the forward through the C ABI (``m0_net_forward``): fp32 SIMT
kernels (``precision="fp32"``) or the tcgen05 pipeline with 16-bit operands (``"fp16"``, ``"bf16"``) or with e4m3
operands for the residual tower's 3x3 convolutions (``"fp8"``, opt-in; DESIGN.md section 4).  There is no
``torch.nn`` forward and no CPU path.  Training-only members of the reference module (losses, SSRL /
WDL / aux heads, ``to_coreml``) are out of scope (SURVEY.md section 2.1 #3).
"""
from __future__ import annotations

import ctypes
import math
from dataclasses import dataclass, field
from typing import Any, Dict, List, Optional, Tuple

import numpy as np

from . import _native
from ._native import c_float, c_int, c_void_p

MAX_BLOCKS = 64
MAX_SSL = 8
ACT = {"none": 0, "relu": 1, "silu": 2, "leaky_relu": 3}
PRECISIONS = {"fp32": 0, "bf16": 1, "fp16": 2, "fp8": 3}   # m0_net_forward's precision argument
SSL_CHANNELS = {"piece": 13, "threat": 1, "pin": 1, "fork": 1, "control": 3, "pawn_structure": 8, "king_safety": 3}
SSL_ORDER = ["piece", "threat", "pin", "fork", "control", "pawn_structure", "king_safety"]  # ModuleDict insertion order, resnet.py:366-433


@dataclass
class NetConfig:
    """Mirror of ``resnet.py:247-282`` (field names and defaults are the API)."""
    planes: int = 19
    channels: int = 160
    blocks: int = 14
    policy_size: int = 4672
    se: bool = True
    se_ratio: float = 0.25
    attention: bool = True
    attention_heads: int = 8
    attention_unmasked_mix: float = 0.2
    attention_relbias: bool = True
    attention_every_k: int = 3
    chess_features: bool = True
    self_supervised: bool = True
    piece_square_tables: bool = True
    wdl: bool = False
    policy_factor_rank: int = 0
    norm: str = "batch"
    activation: str = "relu"
    value_activation: str = "silu"
    preact: bool = False
    droppath: float = 0.0
    aux_policy_from_square: bool = False
    aux_policy_move_type: bool = False
    enable_visual: bool = False
    visual_encoder_channels: int = 64
    ssl_tasks: List[str] = field(default_factory=lambda: ["piece"])
    ssl_curriculum: bool = False
    ssrl_tasks: List[str] = field(default_factory=list)
    enable_llm_tutor: bool = False
    llm_model_path: str = ""
    infer_attention_stride: int = 1
    infer_amp_tower: bool = False


class _BlockW(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in ("gn1_w", "gn1_b", "conv1_w", "gn2_w", "gn2_b", "conv2_w", "se_w1", "se_b1", "se_w2", "se_b2")] \
        + [("has_attention", c_int)] + [(n, c_void_p) for n in ("att_qkv_w", "att_proj_w", "att_ln_w", "att_ln_b", "att_rel_bias")]


class _NetW(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in ("stem_w", "stem_gn_w", "stem_gn_b", "pos_enc", "pst_w", "pst_gn_w", "pst_gn_b",
                                        "inter_w", "inter_gn_w", "inter_gn_b")] \
        + [("blocks", _BlockW * MAX_BLOCKS)] \
        + [(n, c_void_p) for n in ("pol_conv_w", "pol_gn_w", "pol_gn_b", "pol_fc1_w", "pol_fc1_b", "pol_fc2_w", "pol_fc2_b")] \
        + [("policy_logit_scale", c_float)] \
        + [(n, c_void_p) for n in ("val_conv1_w", "val_gn1_w", "val_gn1_b", "val_conv2_w", "val_gn2_w", "val_gn2_b", "val_fc1_w", "val_fc1_b",
                                   "val_fc2_w", "val_fc2_b", "val_gate_w", "val_gate_b", "val_fc3_w", "val_fc3_b")] \
        + [("ssl_conv1_w", c_void_p * MAX_SSL), ("ssl_gn_w", c_void_p * MAX_SSL), ("ssl_gn_b", c_void_p * MAX_SSL), ("ssl_conv2_w", c_void_p * MAX_SSL)]


class _NetCfg(ctypes.Structure):
    _fields_ = [(n, c_int) for n in ("planes", "channels", "blocks", "policy_size", "se", "se_hidden", "attention", "attention_heads",
                                     "attention_every_k", "attention_relbias", "infer_attention_stride")] \
        + [("attention_unmasked_mix", c_float)] \
        + [(n, c_int) for n in ("policy_factor_rank", "activation", "value_activation", "chess_features", "piece_square_tables", "n_ssl_heads")] \
        + [("ssl_out_channels", c_int * MAX_SSL)]


def tower_layout(cfg: NetConfig) -> List[Tuple[int, Optional[int]]]:
    """[(tower index of residual block i, tower index of the attention module after it or None)], resnet.py:346-356."""
    out, t = [], 0
    k = int(cfg.attention_every_k)
    for i in range(cfg.blocks):
        bi = t
        t += 1
        ai = None
        if cfg.attention and k > 0 and (i % k) == (k - 1):
            ai = t
            t += 1
        out.append((bi, ai))
    return out


def parameter_shapes(cfg: NetConfig) -> Dict[str, Tuple[int, ...]]:
    """Reference state_dict keys (inference-relevant subset) and their shapes."""
    C, P = cfg.channels, cfg.planes
    hid = max(8, int(C * cfg.se_ratio))
    sh: Dict[str, Tuple[int, ...]] = {"stem.0.weight": (C, P, 3, 3), "stem.1.weight": (C,), "stem.1.bias": (C,)}
    if cfg.chess_features:
        sh["chess_features.position_encoding"] = (1, C, 8, 8)
        if cfg.piece_square_tables:
            sh.update({"chess_features.pst_conv.weight": (C, C, 1, 1), "chess_features.pst_norm.weight": (C,), "chess_features.pst_norm.bias": (C,)})
        sh.update({"chess_features.interaction_conv.weight": (C, C, 3, 3), "chess_features.interaction_norm.weight": (C,),
                   "chess_features.interaction_norm.bias": (C,)})
    for bi, ai in tower_layout(cfg):
        p = f"tower.{bi}."
        sh.update({p + "conv1.weight": (C, C, 3, 3), p + "bn1.weight": (C,), p + "bn1.bias": (C,),
                   p + "conv2.weight": (C, C, 3, 3), p + "bn2.weight": (C,), p + "bn2.bias": (C,)})
        if cfg.se:
            sh.update({p + "se_fc1.weight": (hid, C), p + "se_fc1.bias": (hid,), p + "se_fc2.weight": (C, hid), p + "se_fc2.bias": (C,)})
        if ai is not None:
            a = f"tower.{ai}."
            sh.update({a + "qkv.weight": (3 * C, C, 1, 1), a + "proj.weight": (C, C, 1, 1), a + "norm.weight": (C,), a + "norm.bias": (C,)})
            if cfg.attention_relbias:
                sh[a + "rel_bias"] = (1, cfg.attention_heads, 64, 64)
    sh.update({"policy_head.0.weight": (64, C, 1, 1), "policy_head.1.weight": (64,), "policy_head.1.bias": (64,), "_policy_logit_scale_raw": ()})
    if cfg.policy_factor_rank > 0:
        r = cfg.policy_factor_rank
        sh.update({"policy_fc1.weight": (r, 4096), "policy_fc1.bias": (r,), "policy_fc2.weight": (cfg.policy_size, r), "policy_fc2.bias": (cfg.policy_size,)})
    else:
        sh.update({"policy_fc.weight": (cfg.policy_size, 4096), "policy_fc.bias": (cfg.policy_size,)})
    sh.update({"value_head.0.weight": (128, C, 1, 1), "value_head.1.weight": (128,), "value_head.1.bias": (128,),
               "value_head.3.weight": (128, 128, 1, 1), "value_head.4.weight": (128,), "value_head.4.bias": (128,),
               "value_fc1.weight": (2 * C, 8192), "value_fc1.bias": (2 * C,), "value_fc2.weight": (C, 2 * C), "value_fc2.bias": (C,),
               "value_gate.0.weight": (C, C), "value_gate.0.bias": (C,), "value_fc3.weight": (1, C), "value_fc3.bias": (1,)})
    if cfg.self_supervised:
        for t in SSL_ORDER:
            if t in cfg.ssl_tasks:
                p = f"ssl_heads.{t}."
                sh.update({p + "0.weight": (C // 2, C, 1, 1), p + "1.weight": (C // 2,), p + "1.bias": (C // 2,),
                           p + "3.weight": (SSL_CHANNELS[t], C // 2, 1, 1)})
    return sh


def reference_init(cfg: NetConfig) -> Dict[str, Any]:
    """Parameter values of a freshly constructed reference ``PolicyValueNet(cfg)``, drawn from torch's GLOBAL CPU generator in
    the order the reference's constructor consumes it, so that ``torch.manual_seed(s)`` gives the reference's weights.

    Construction order (``resnet.py:313-550``): stem conv -> ChessSpecificFeatures (pst_conv, interaction_conv, then
    ``torch.randn`` for the position encoding followed by ``normal_(0, 0.1)``, ``:217-235``) -> tower (per block conv1, conv2,
    se_fc1, se_fc2, ``:30-41``; ChessAttention qkv, proj, ``:97-98``, rel_bias zeros ``:135``) -> SSL heads in ModuleDict order
    -> policy_head conv -> aux heads -> policy_fc1/fc2 (or policy_fc) -> value head convs, value_fc1, value_fc2, value_gate,
    value_fc3 -> SSRL heads; PyTorch defaults: Conv2d / Linear weight ``kaiming_uniform_(a=sqrt(5))``, Linear bias
    ``U(-1/sqrt(fan_in), 1/sqrt(fan_in))``, norm weight 1 / bias 0.  Then ``_init_weights`` (``:591-654``) re-draws the head
    weights (kaiming_normal fan_out for the head convs, xavier_uniform for the fully connected layers, zero biases),
    scales ``policy_fc2`` (or ``policy_fc``) by 0.8 and gives the piece SSL head xavier_uniform(gain=0.1).
    Training-only modules that this engine does not hold (aux / SSRL heads) still consume the generator and are drawn and dropped."""
    import torch
    from torch.nn import init
    C, sd = cfg.channels, {}

    def conv(name, co, ci, k):
        w = torch.empty(co, ci, k, k)
        init.kaiming_uniform_(w, a=math.sqrt(5))
        if name:
            sd[name + ".weight"] = w
        return w

    def linear(name, fo, fi):
        w = torch.empty(fo, fi)
        init.kaiming_uniform_(w, a=math.sqrt(5))
        b = torch.empty(fo)
        bound = 1.0 / math.sqrt(fi) if fi > 0 else 0
        init.uniform_(b, -bound, bound)
        if name:
            sd[name + ".weight"], sd[name + ".bias"] = w, b
        return w, b

    def norm(name, c):
        sd[name + ".weight"], sd[name + ".bias"] = torch.ones(c), torch.zeros(c)

    conv("stem.0", C, cfg.planes, 3)
    norm("stem.1", C)
    if cfg.chess_features:
        if cfg.piece_square_tables:
            conv("chess_features.pst_conv", C, C, 1)
            norm("chess_features.pst_norm", C)
        conv("chess_features.interaction_conv", C, C, 3)
        norm("chess_features.interaction_norm", C)
        pe = torch.randn(1, C, 8, 8)
        init.normal_(pe, mean=0.0, std=0.1)
        sd["chess_features.position_encoding"] = pe
    hid = max(8, int(C * cfg.se_ratio))
    for bi, ai in tower_layout(cfg):
        p = f"tower.{bi}"
        conv(p + ".conv1", C, C, 3)
        norm(p + ".bn1", C)
        conv(p + ".conv2", C, C, 3)
        norm(p + ".bn2", C)
        if cfg.se:
            linear(p + ".se_fc1", hid, C)
            linear(p + ".se_fc2", C, hid)
        if ai is not None:
            a = f"tower.{ai}"
            conv(a + ".qkv", 3 * C, C, 1)
            conv(a + ".proj", C, C, 1)
            norm(a + ".norm", C)
            if cfg.attention_relbias:
                sd[a + ".rel_bias"] = torch.zeros(1, cfg.attention_heads, 64, 64)
    if cfg.self_supervised:
        for t in SSL_ORDER:
            if t in cfg.ssl_tasks:
                p = f"ssl_heads.{t}"
                conv(p + ".0", C // 2, C, 1)
                norm(p + ".1", C // 2)
                conv(p + ".3", SSL_CHANNELS[t], C // 2, 1)
    conv("policy_head.0", 64, C, 1)
    norm("policy_head.1", 64)
    if cfg.aux_policy_from_square:
        conv(None, 32, C, 1)
        conv(None, 64, 32, 1)
    if cfg.aux_policy_move_type:
        conv(None, 32, C, 1)
        conv(None, 12, 32, 1)
    safe_init = max(0.2 - 1e-3, 1e-6)  # policy_logit_init_scale is not a NetConfig field: getattr default, resnet.py:476-480
    sd["_policy_logit_scale_raw"] = torch.tensor(math.log(math.expm1(safe_init)), dtype=torch.float32)
    if cfg.policy_factor_rank > 0:
        linear("policy_fc1", cfg.policy_factor_rank, 4096)
        linear("policy_fc2", cfg.policy_size, cfg.policy_factor_rank)
    else:
        linear("policy_fc", cfg.policy_size, 4096)
    conv("value_head.0", 128, C, 1)
    norm("value_head.1", 128)
    conv("value_head.3", 128, 128, 1)
    norm("value_head.4", 128)
    linear("value_fc1", 2 * C, 8192)
    linear("value_fc2", C, 2 * C)
    linear("value_gate.0", C, C)
    linear("value_fc3", 1, C)
    ssrl = [(t, {"position": 64, "material": 12, "rotation": 4}[t]) for t in cfg.ssrl_tasks if t in ("position", "material", "rotation")]
    ssrl_w = []
    for _, n_out in ssrl:
        ssrl_w.append((linear(None, C // 2, C)[0], linear(None, n_out, C // 2)[0]))
    # ---- _init_weights, resnet.py:591-654 ----
    init.kaiming_normal_(sd["policy_head.0.weight"], mode="fan_out", nonlinearity="relu")
    for n in (("policy_fc1", "policy_fc2") if cfg.policy_factor_rank > 0 else ("policy_fc",)):
        init.xavier_uniform_(sd[n + ".weight"], gain=1.0)
        sd[n + ".bias"].zero_()
    init.kaiming_normal_(sd["value_head.0.weight"], mode="fan_out", nonlinearity="relu")
    init.kaiming_normal_(sd["value_head.3.weight"], mode="fan_out", nonlinearity="relu")
    for n in ("value_fc1", "value_fc2", "value_fc3", "value_gate.0"):
        init.xavier_uniform_(sd[n + ".weight"], gain=1.0)
    for n in ("value_fc1", "value_fc2", "value_fc3", "value_gate.0"):
        sd[n + ".bias"].zero_()
    sd["policy_fc2.weight" if cfg.policy_factor_rank > 0 else "policy_fc.weight"].mul_(0.8)
    if cfg.self_supervised and "piece" in cfg.ssl_tasks:
        init.xavier_uniform_(sd["ssl_heads.piece.0.weight"], gain=0.1)
        init.xavier_uniform_(sd["ssl_heads.piece.3.weight"], gain=0.1)
    for w1, w2 in ssrl_w:
        init.xavier_uniform_(w1, gain=1.0)
        init.xavier_uniform_(w2, gain=1.0)
    return sd


class PolicyValueNet:
    def __init__(self, cfg: NetConfig, device: Optional[str] = None, precision: str = "fp16", seed: Optional[int] = None):
        import torch
        if cfg.policy_size != 4672:
            raise ValueError(f"Unsupported policy_size={cfg.policy_size}. Matrix0 currently supports legacy 4672 only")  # resnet.py:302-306
        if cfg.norm != "group" or not cfg.preact:
            raise NotImplementedError("matrix0_b200 implements the shipped V2 architecture family (norm='group', preact=True)")
        if cfg.activation not in ("silu", "relu") or cfg.value_activation not in ("silu", "relu", "leaky_relu"):
            raise ValueError("unsupported activation")
        if cfg.enable_visual or cfg.wdl:
            raise NotImplementedError("visual encoder / WDL head are training-side options and not part of this engine")
        self.cfg = cfg
        self.precision = precision
        self.training = False
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._shapes = parameter_shapes(cfg)
        self._params: Dict[str, "torch.Tensor"] = {}
        self._handle = None
        self._keep: List[Any] = []
        self._init_parameters(seed)

    # ---- reference-compatible surface -----------------------------------------------------------
    @staticmethod
    def from_config(d: dict, **kw) -> "PolicyValueNet":
        known = set(NetConfig.__dataclass_fields__.keys())
        return PolicyValueNet(NetConfig(**{k: v for k, v in d.items() if k in known}), **kw)

    def eval(self):
        self.training = False
        return self

    def train(self, mode: bool = True):
        if mode:
            raise NotImplementedError("matrix0_b200.PolicyValueNet is inference-only; train with the reference module and load its state_dict")
        return self

    def to(self, device=None, *a, **k):
        import torch
        if device is not None and torch.device(device).type == "cuda" and torch.device(device) != self.device:
            self.device = torch.device(device)
            self._params = {n: t.to(self.device) for n, t in self._params.items()}
            self._release()
        return self

    def count_parameters(self) -> int:
        return int(sum(t.numel() for t in self._params.values()))

    def parameters(self):
        return iter(self._params.values())

    def state_dict(self) -> Dict[str, Any]:
        return {k: v.clone() for k, v in self._params.items()}

    def load_state_dict(self, state_dict, strict: bool = False):
        """Reference semantics (resnet.py:1402-1442): V1 ``policy_fc.*`` keys map to ``policy_fc1.*``; keys missing
        from the checkpoint keep their (re-)initialised values; unknown keys are ignored unless strict."""
        import torch
        mapping = {"policy_fc.weight": "policy_fc1.weight", "policy_fc.bias": "policy_fc1.bias"} if self.cfg.policy_factor_rank > 0 else {}
        missing, unexpected, seen = [], [], set()
        for k, v in state_dict.items():
            k = mapping.get(k, k)
            if k not in self._shapes:
                unexpected.append(k)
                continue
            t = torch.as_tensor(v).detach().to(device=self.device, dtype=torch.float32)
            if t.numel() == 1 and len(self._shapes[k]) == 0:
                t = t.reshape(())  # torch accepts a (1,) tensor for a 0-dim parameter
            if tuple(t.shape) != tuple(self._shapes[k]):
                raise RuntimeError(f"size mismatch for {k}: checkpoint {tuple(t.shape)} vs model {tuple(self._shapes[k])}")
            self._params[k] = t.contiguous().clone()
            seen.add(k)
        missing = [k for k in self._shapes if k not in seen]
        if strict and (missing or [u for u in unexpected if not u.startswith(("ssl_head.", "ssl_piece_head.", "aux_", "ssrl_heads.", "wdl_head."))]):
            raise RuntimeError(f"Error(s) in loading state_dict: missing={missing} unexpected={unexpected}")
        self._release()
        return missing, unexpected

    # ---- parameters --------------------------------------------------------------------------------
    def _init_parameters(self, seed: Optional[int]) -> None:
        """Random initialisation: the parameter values ``PolicyValueNet(cfg)`` of the reference holds after ``__init__``
        (``resnet.py:286-589`` module construction with the PyTorch layer defaults, then ``_init_weights`` ``:591-654``).
        ``seed=None`` draws from torch's global generator exactly like the reference (``torch.manual_seed(s)`` before
        ``from_config`` gives the same weights as the reference module under the same seed, pinned by per-tensor digests in
        tests/golden/refinit_digest.json); an integer seed does the same inside a forked generator state."""
        import torch
        if seed is None:
            sd = reference_init(self.cfg)
        else:
            with torch.random.fork_rng(devices=[]):
                torch.manual_seed(int(seed))
                sd = reference_init(self.cfg)
        for name in self._shapes:
            self._params[name] = sd[name].to(self.device, dtype=torch.float32).contiguous()

    def _release(self) -> None:
        # a captured CUDA graph of the old net (SelfPlayEngine._forward) must not be replayed against freed weights /
        # workspaces: bump the workspace epoch that is part of its cache key
        self._ws_epoch = getattr(self, "_ws_epoch", 0) + 1
        self._max_batch = 0
        self.__dict__.pop("_fwd_graphs", None)
        if self._handle is not None:
            _native.load_library().m0_net_destroy(self._handle)
            self._handle = None
        self._keep = []

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def _build(self) -> None:
        """Lay the parameters out for the kernels and create the native net."""
        import torch
        cfg, P = self.cfg, self._params
        C = cfg.channels
        keep: List[Any] = []

        def dev(t):
            t = t.to(self.device, dtype=torch.float32).contiguous()
            keep.append(t)
            return t.data_ptr()

        def conv3(name):  # [co][ci][3][3] -> W[co][(ky*3+kx)*ci_n + ci]
            return dev(P[name].permute(0, 2, 3, 1).reshape(P[name].shape[0], -1))

        def conv1(name):  # [co][ci][1][1] -> W[co][ci]
            return dev(P[name].reshape(P[name].shape[0], -1))

        def fc_nhwc(name, ch):  # columns c*64 + sq  ->  sq*ch + c
            w = P[name]
            return dev(w.reshape(w.shape[0], ch, 64).permute(0, 2, 1).reshape(w.shape[0], -1))

        w = _NetW()
        w.stem_w, w.stem_gn_w, w.stem_gn_b = conv3("stem.0.weight"), dev(P["stem.1.weight"]), dev(P["stem.1.bias"])
        if cfg.chess_features:
            w.pos_enc = dev(P["chess_features.position_encoding"].reshape(C, 64).t())
            if cfg.piece_square_tables:
                w.pst_w, w.pst_gn_w, w.pst_gn_b = conv1("chess_features.pst_conv.weight"), dev(P["chess_features.pst_norm.weight"]), dev(P["chess_features.pst_norm.bias"])
            w.inter_w = conv3("chess_features.interaction_conv.weight")
            w.inter_gn_w, w.inter_gn_b = dev(P["chess_features.interaction_norm.weight"]), dev(P["chess_features.interaction_norm.bias"])
        for i, (bi, ai) in enumerate(tower_layout(cfg)):
            b, p = w.blocks[i], f"tower.{bi}."
            b.gn1_w, b.gn1_b, b.conv1_w = dev(P[p + "bn1.weight"]), dev(P[p + "bn1.bias"]), conv3(p + "conv1.weight")
            b.gn2_w, b.gn2_b, b.conv2_w = dev(P[p + "bn2.weight"]), dev(P[p + "bn2.bias"]), conv3(p + "conv2.weight")
            if cfg.se:
                b.se_w1, b.se_b1 = dev(P[p + "se_fc1.weight"]), dev(P[p + "se_fc1.bias"])
                b.se_w2, b.se_b2 = dev(P[p + "se_fc2.weight"]), dev(P[p + "se_fc2.bias"])
            b.has_attention = 0 if ai is None else 1
            if ai is not None:
                a = f"tower.{ai}."
                b.att_qkv_w, b.att_proj_w = conv1(a + "qkv.weight"), conv1(a + "proj.weight")
                b.att_ln_w, b.att_ln_b = dev(P[a + "norm.weight"]), dev(P[a + "norm.bias"])
                if cfg.attention_relbias:
                    b.att_rel_bias = dev(P[a + "rel_bias"].reshape(cfg.attention_heads, 64, 64))
        w.pol_conv_w, w.pol_gn_w, w.pol_gn_b = conv1("policy_head.0.weight"), dev(P["policy_head.1.weight"]), dev(P["policy_head.1.bias"])
        if cfg.policy_factor_rank > 0:
            w.pol_fc1_w, w.pol_fc1_b = fc_nhwc("policy_fc1.weight", 64), dev(P["policy_fc1.bias"])
            w.pol_fc2_w, w.pol_fc2_b = dev(P["policy_fc2.weight"]), dev(P["policy_fc2.bias"])
        else:
            w.pol_fc1_w, w.pol_fc1_b = fc_nhwc("policy_fc.weight", 64), dev(P["policy_fc.bias"])
        raw = float(P["_policy_logit_scale_raw"].float().cpu())
        softplus = math.log1p(math.exp(raw)) if raw < 20 else raw
        w.policy_logit_scale = min(float(np.float32(softplus) + np.float32(1e-3)), 5.0)  # resnet.py:709-710
        w.val_conv1_w, w.val_gn1_w, w.val_gn1_b = conv1("value_head.0.weight"), dev(P["value_head.1.weight"]), dev(P["value_head.1.bias"])
        w.val_conv2_w, w.val_gn2_w, w.val_gn2_b = conv1("value_head.3.weight"), dev(P["value_head.4.weight"]), dev(P["value_head.4.bias"])
        w.val_fc1_w, w.val_fc1_b = fc_nhwc("value_fc1.weight", 128), dev(P["value_fc1.bias"])
        w.val_fc2_w, w.val_fc2_b = dev(P["value_fc2.weight"]), dev(P["value_fc2.bias"])
        w.val_gate_w, w.val_gate_b = dev(P["value_gate.0.weight"]), dev(P["value_gate.0.bias"])
        w.val_fc3_w, w.val_fc3_b = dev(P["value_fc3.weight"]), dev(P["value_fc3.bias"])
        self._ssl_names = [t for t in SSL_ORDER if cfg.self_supervised and t in cfg.ssl_tasks]
        for h, t in enumerate(self._ssl_names):
            p = f"ssl_heads.{t}."
            w.ssl_conv1_w[h], w.ssl_gn_w[h], w.ssl_gn_b[h], w.ssl_conv2_w[h] = conv1(p + "0.weight"), dev(P[p + "1.weight"]), dev(P[p + "1.bias"]), conv1(p + "3.weight")

        c = _NetCfg()
        c.planes, c.channels, c.blocks, c.policy_size = cfg.planes, C, cfg.blocks, cfg.policy_size
        c.se, c.se_hidden = int(bool(cfg.se)), max(8, int(C * cfg.se_ratio))
        c.attention, c.attention_heads, c.attention_every_k = int(bool(cfg.attention)), cfg.attention_heads, cfg.attention_every_k
        c.attention_relbias = int(bool(cfg.attention_relbias))
        c.infer_attention_stride = max(1, int(cfg.infer_attention_stride))
        c.attention_unmasked_mix = float(cfg.attention_unmasked_mix)
        c.policy_factor_rank = int(cfg.policy_factor_rank)
        c.activation, c.value_activation = ACT[cfg.activation], ACT[cfg.value_activation]
        c.chess_features, c.piece_square_tables = int(bool(cfg.chess_features)), int(bool(cfg.piece_square_tables))
        c.n_ssl_heads = len(self._ssl_names)
        for h, t in enumerate(self._ssl_names):
            c.ssl_out_channels[h] = SSL_CHANNELS[t]
        lib = _native.lib()
        h = c_void_p()
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        _native.check(lib.m0_net_create(idx, ctypes.byref(c), ctypes.byref(w), ctypes.byref(h)), "m0_net_create")
        self._handle, self._keep = h, keep

    # ---- forward -----------------------------------------------------------------------------------------
    def forward_planes(self, planes, precision: Optional[str] = None):
        """planes: float32 CUDA tensor [B, 19, 8, 8] -> (logits float32 [B, 4672], values float32 [B]) on the device."""
        import torch
        if self._handle is None:
            self._build()
        assert planes.is_cuda and planes.dtype == torch.float32
        planes = planes.contiguous()
        B = planes.shape[0]
        logits = torch.empty((B, self.cfg.policy_size), dtype=torch.float32, device=planes.device)
        values = torch.empty((B,), dtype=torch.float32, device=planes.device)
        prec = PRECISIONS[precision or self.precision]
        if B == 0:
            return logits, values
        if B > getattr(self, "_max_batch", 0):     # the library grows its workspaces: captured graphs of smaller batches are stale
            self._max_batch = B
            self._ws_epoch = getattr(self, "_ws_epoch", 0) + 1
        with torch.cuda.device(planes.device):
            rc = _native.lib().m0_net_forward(self._handle, planes.data_ptr(), B, logits.data_ptr(), values.data_ptr(), prec,
                                              _native.current_stream())
        if rc == _native.M0_ERR_ARG and prec == PRECISIONS["fp8"]:   # a configuration the fp8 pipeline does not cover
            raise ValueError(f"precision='fp8': {_native.load_library().m0_last_error().decode()}")
        _native.check(rc, "m0_net_forward")
        return logits, values

    def capture_forward(self, planes, precision: Optional[str] = None):
        """CUDA graph of one forward over a FIXED planes buffer (the ~100 kernel launches of the tensor-core pipeline replay as one
        graph launch: no per-launch host work and no launch gaps).  Returns ``(graph, logits, values)``; ``graph.replay()`` refreshes
        the two static output tensors from the current contents of ``planes``.  The capture is stale once ``ws_epoch`` changes
        (a larger batch made the library reallocate its workspaces)."""
        import torch
        assert planes.is_cuda and planes.dtype == torch.float32 and planes.is_contiguous()
        with torch.cuda.device(planes.device):
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):              # warm-up outside the capture: workspaces, tensor maps, kernel attributes
                for _ in range(2):
                    self.forward_planes(planes, precision)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                logits, values = self.forward_planes(planes, precision)
        return graph, logits, values

    def forward_planes_graphed(self, planes, precision: Optional[str] = None):
        """``forward_planes`` through a cached CUDA graph per (planes buffer, batch, precision): for callers that evaluate the SAME
        device buffer again and again with small batches (the drop-in ``MCTS`` object: ten evaluator calls of <= 96 rows per move),
        where an eager forward is bound by its ~230 kernel launches.  The outputs are the graph's static tensors (overwritten by the
        next replay).  fp32 (the SIMT path) runs eagerly."""
        prec = precision or self.precision
        if prec == "fp32":
            return self.forward_planes(planes, precision)
        cache = self.__dict__.setdefault("_fwd_graphs", {})
        key = (planes.data_ptr(), int(planes.shape[0]), prec, self.ws_epoch)
        if key not in cache:
            graph, logits, values = self.capture_forward(planes, precision)     # (its warm-up passes may grow the workspaces)
            for k in [k for k in cache if k[3] != self.ws_epoch]:               # captures of older weights / workspaces are stale
                del cache[k]
            while len(cache) >= 8:
                del cache[next(iter(cache))]
            key = (planes.data_ptr(), int(planes.shape[0]), prec, self.ws_epoch)
            cache[key] = (graph, logits, values)
        graph, logits, values = cache[key]
        graph.replay()
        return logits, values

    @property
    def ws_epoch(self) -> int:
        return getattr(self, "_ws_epoch", 0)

    def forward(self, x, return_ssl: bool = False, visual_input=None):
        """``resnet.py:755-760``: (logits [B,4672], value [B]) or (+ dict of SSL maps [B,k,8,8])."""
        import torch
        x = torch.as_tensor(x)
        if x.dim() == 3:
            x = x[None]
        xd = x.to(self.device, dtype=torch.float32).contiguous()
        if not return_ssl:
            return self.forward_planes(xd)
        if self._handle is None:
            self._build()
        B = xd.shape[0]
        logits = torch.empty((B, self.cfg.policy_size), dtype=torch.float32, device=self.device)
        values = torch.empty((B,), dtype=torch.float32, device=self.device)
        outs = {t: torch.empty((B, SSL_CHANNELS[t], 8, 8), dtype=torch.float32, device=self.device) for t in self._ssl_names}
        arr = (c_void_p * MAX_SSL)(*[outs[t].data_ptr() for t in self._ssl_names])
        with torch.cuda.device(self.device):
            _native.check(_native.lib().m0_net_forward_ssl(self._handle, xd.data_ptr(), B, logits.data_ptr(), values.data_ptr(), arr,
                                                           _native.current_stream()), "m0_net_forward_ssl")
        return logits, values, outs

    __call__ = forward

    def infer_np(self, arr) -> Tuple[np.ndarray, np.ndarray]:
        """The inference-backend seam (``selfplay/inference.py:585``): numpy in, numpy out."""
        import torch
        a = np.asarray(arr, dtype=np.float32)
        if a.ndim == 3:
            a = a[None]
        lg, v = self.forward_planes(torch.from_numpy(np.ascontiguousarray(a)).to(self.device))
        return lg.cpu().numpy(), v.cpu().numpy()
