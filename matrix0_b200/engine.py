"""Python handle of the device-resident search engine (C ABI: m0_engine_*, m0_games_*, m0_search_*).

Thin plumbing only: owns the torch tensors used as I/O buffers (planes, logits, results) and turns
Python arguments into device pointers.  All search work happens in the CUDA tree kernels.
"""
from __future__ import annotations

import ctypes
import math
from typing import Optional, Sequence

import numpy as np

from . import _native
from .boards import MAX_MOVES, PLANES, POLICY_SIZE, POSITION_WORDS, board_to_raw, move_to_code

COUNTER_NAMES = ["sims", "terminal_sims", "nn_evals", "expansions", "tt_hops", "children_scanned", "path_nodes",
                 "children_created", "games_finished", "positions_played", "noisy_expansions", "leaf_samples", "root_evals_reused"]
ST_NODE_OVERFLOW, ST_TT_OVERFLOW, ST_DEPTH_CAP, ST_HIST_OVERFLOW, ST_STREAM_EXHAUSTED = 1, 2, 4, 8, 16


def cpuct_table(cfg, length: int) -> np.ndarray:
    """MCTS._cpuct_at(depth) (azchess/mcts.py:927-944) evaluated on the host in Python floats, exactly
    as the reference does, for depth = 0..length-1 (base_ply is always 0, SURVEY M9)."""
    out = np.empty(length, dtype=np.float64)
    for ply in range(length):
        c_base = getattr(cfg, "cpuct_c_base", None)
        c_init = getattr(cfg, "cpuct_c_init", None)
        if c_base is not None and c_init is not None:
            N = max(1.0, float(ply + 1))
            out[ply] = float(c_init) + math.log((N + float(c_base)) / float(c_base))
            continue
        start, end, span = cfg.cpuct_start, cfg.cpuct_end, int(cfg.cpuct_plies)
        if start is None or end is None or span <= 0:
            out[ply] = float(cfg.cpuct)
        else:
            t = min(max(ply, 0), span) / float(span)
            out[ply] = float(start) + (float(end) - float(start)) * t
    return out


@_native.on_own_device
class SearchEngine:
    def __init__(self, max_games: int, max_nodes: int = 65536, tt_capacity: int = 0, max_depth: int = 256,
                 hist_cap: int = 1024, device: Optional[int] = None):
        import torch
        self._lib = _native.lib()
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        self.G, self.max_nodes, self.max_depth, self.hist_cap = int(max_games), int(max_nodes), int(max_depth), int(hist_cap)
        h = ctypes.c_void_p()
        _native.check(self._lib.m0_engine_create(self.device_index, self.G, self.max_nodes, int(tt_capacity), self.max_depth,
                                                 self.hist_cap, ctypes.byref(h)), "m0_engine_create")
        self._h = h
        dev = self.device
        G = self.G
        self.planes = torch.zeros((G, PLANES, 8, 8), dtype=torch.float32, device=dev)
        self.info = torch.zeros((G,), dtype=torch.int32, device=dev)
        self.term_value = torch.zeros((G,), dtype=torch.float64, device=dev)
        self.pending = torch.zeros((G,), dtype=torch.int32, device=dev)
        self.res_moves = torch.zeros((G, MAX_MOVES), dtype=torch.int16, device=dev)
        self.res_visits = torch.zeros((G, MAX_MOVES), dtype=torch.int32, device=dev)
        self.res_q = torch.zeros((G, MAX_MOVES), dtype=torch.float64, device=dev)
        self.res_prior = torch.zeros((G, MAX_MOVES), dtype=torch.float64, device=dev)
        self.res_count = torch.zeros((G,), dtype=torch.int32, device=dev)
        self.res_pi = torch.zeros((G, POLICY_SIZE), dtype=torch.float32, device=dev)
        self.res_root_q = torch.zeros((G,), dtype=torch.float64, device=dev)
        self.res_root_n = torch.zeros((G,), dtype=torch.int32, device=dev)
        self.reset()

    # ---- lifetime ------------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.m0_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def bytes(self) -> int:
        return int(self._lib.m0_engine_bytes(self._h))

    def _stream(self) -> int:
        return _native.current_stream()

    # ---- configuration ---------------------------------------------------------------------------
    def configure(self, cfg, deterministic: bool, seed: int = 0, raw_logit_priors: bool = False, virtual_loss: bool = False) -> None:
        """``raw_logit_priors``: SURVEY Q3 switch -- the reference's direct-model path (``MCTS(cfg, model)`` without an inference
        backend and ``legal_softmax``) expands non-root leaves from the raw legal logits (mcts.py:697-703)."""
        table = np.ascontiguousarray(cpuct_table(cfg, self.max_depth + 1))
        s = _native.SearchConfigStruct()
        s.fpu_reduction = float(cfg.fpu_reduction)
        s.draw_penalty = float(cfg.draw_penalty)
        s.selection_jitter = float(cfg.selection_jitter)
        s.dirichlet_alpha = float(cfg.dirichlet_alpha)
        s.dirichlet_frac = float(cfg.dirichlet_frac)
        s.deterministic = 1 if deterministic else 0
        s.no_instant_backtrack = 1 if cfg.no_instant_backtrack else 0
        s.legal_softmax = 1 if cfg.legal_softmax else 0
        s.enable_entropy_noise = 1 if getattr(cfg, "enable_entropy_noise", True) else 0
        s.value_from_white = 1 if getattr(cfg, "value_from_white", False) else 0
        s.cpuct_len = len(table)
        s.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        s.cpuct_by_depth = table.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        s.max_children = int(getattr(cfg, "max_children", 0) or 0)
        s.min_child_prior = float(getattr(cfg, "min_child_prior", 0.0) or 0.0)
        s.raw_logit_priors = 1 if raw_logit_priors else 0
        s.virtual_loss = float(getattr(cfg, "virtual_loss", 1.0))
        s.virtual_loss_on = 1 if virtual_loss else 0
        _native.check(self._lib.m0_engine_configure(self._h, ctypes.byref(s), self._stream()), "m0_engine_configure")

    # ---- games -----------------------------------------------------------------------------------
    def reset(self, games=None) -> None:
        import torch
        if games is None:
            _native.check(self._lib.m0_games_reset(self._h, None, self.G, self._stream()), "m0_games_reset")
        else:
            g = torch.as_tensor(list(games), dtype=torch.int32, device=self.device)
            _native.check(self._lib.m0_games_reset(self._h, g.data_ptr(), g.numel(), self._stream()), "m0_games_reset")

    def set_positions_packed(self, root_pos, games=None, hist_pos=None, hist_moves=None, hist_lens=None) -> None:
        """root_pos: int64/uint64 [n, 9] device tensor of packed positions."""
        n = root_pos.shape[0]
        stride = 0 if hist_pos is None else hist_pos.shape[1]
        _native.check(self._lib.m0_games_set_positions(self._h, _native.ptr(games), n, root_pos.data_ptr(), _native.ptr(hist_pos),
                                                       _native.ptr(hist_moves), _native.ptr(hist_lens), stride, self._stream()),
                      "m0_games_set_positions")

    def set_boards(self, boards: Sequence, games=None, with_history: bool = True) -> None:
        """Upload python-chess style boards (root + move-stack history) into game slots."""
        import torch
        n = len(boards)
        hists = [board_history(b, self.hist_cap) if with_history else ([], []) for b in boards]
        L = max((len(h[1]) for h in hists), default=0)
        raw = np.zeros((n * (L + 1), 10), dtype=np.uint64)
        moves = np.zeros((n, max(L, 1)), dtype=np.uint16)
        lens = np.zeros(n, dtype=np.int32)
        for i, (b, (hp, hm)) in enumerate(zip(boards, hists)):
            board_to_raw(b, raw[i])
            for k, (rp, m) in enumerate(zip(hp, hm)):
                raw[n + i * L + k] = rp
                moves[i, k] = m
            lens[i] = len(hm)
        raw_d = torch.from_numpy(raw.view(np.int64)).to(self.device)
        pos_d = torch.empty((raw.shape[0], POSITION_WORDS), dtype=torch.int64, device=self.device)
        _native.check(self._lib.m0_positions_pack(raw_d.data_ptr(), raw.shape[0], pos_d.data_ptr(), self._stream()), "m0_positions_pack")
        root = pos_d[:n]
        games_d = None if games is None else torch.as_tensor(list(games), dtype=torch.int32, device=self.device)
        if L > 0:
            hist = pos_d[n:].view(n, L, POSITION_WORDS)
            self.set_positions_packed(root, games_d, hist, torch.from_numpy(moves.view(np.int16)).to(self.device),
                                      torch.from_numpy(lens).to(self.device))
        else:
            self.set_positions_packed(root, games_d)

    # ---- search steps ----------------------------------------------------------------------------
    def begin(self) -> None:
        _native.check(self._lib.m0_search_begin(self._h, self.planes.data_ptr(), self.info.data_ptr(), self.term_value.data_ptr(),
                                                self._stream()), "m0_search_begin")

    def select(self, batch_n: int) -> None:
        _native.check(self._lib.m0_search_select(self._h, int(batch_n), self.planes.data_ptr(), self._stream()), "m0_search_select")

    def add_dirichlet(self, noise=None, apply=None) -> None:
        """noise: float64 [G, 256] device tensor or None (device RNG); apply: int32 [G] gate or None."""
        _native.check(self._lib.m0_search_add_dirichlet(self._h, _native.ptr(noise), _native.ptr(apply), self._stream()),
                      "m0_search_add_dirichlet")

    def pending_counts(self):
        _native.check(self._lib.m0_search_pending_counts(self._h, self.pending.data_ptr(), self._stream()), "m0_search_pending_counts")
        return self.pending

    def expand_backup(self, logits, values) -> None:
        assert logits.dtype.is_floating_point and logits.element_size() == 4 and logits.is_contiguous()
        assert values.element_size() == 4 and values.is_contiguous()
        _native.check(self._lib.m0_search_expand_backup(self._h, logits.data_ptr(), logits.shape[1], values.data_ptr(), self._stream()),
                      "m0_search_expand_backup")

    def result(self, with_pi: bool = True) -> None:
        _native.check(self._lib.m0_search_result(self._h, self.res_moves.data_ptr(), self.res_visits.data_ptr(), self.res_q.data_ptr(),
                                                 self.res_prior.data_ptr(), self.res_count.data_ptr(),
                                                 self.res_pi.data_ptr() if with_pi else None, self.res_root_q.data_ptr(),
                                                 self.res_root_n.data_ptr(), self._stream()), "m0_search_result")

    # ---- the mini-batch as shipped: per-simulation jitter, distinct leaves (csrc/tree_multi_kernels.cu) -------------
    def enable_multi(self, samples_per_batch: int, virtual_loss: bool = False) -> None:
        import torch
        _native.check(self._lib.m0_search_multi_enable(self._h, int(samples_per_batch), 1 if virtual_loss else 0), "m0_search_multi_enable")
        self.ml_cap = int(samples_per_batch)
        self.row_base = torch.zeros((self.G + 1,), dtype=torch.int32, device=self.device)
        self.n_samples = torch.zeros((self.G,), dtype=torch.int32, device=self.device)

    # ---- reuse of the root's evaluation across moves -------------------------------------------------------------------------
    def enable_reuse(self, slots: int) -> None:
        """Keep the network outputs of the root's children (``slots`` per game) for the next ``begin``.  Afterwards ``begin`` also
        writes the roots found in no entry to ``miss_planes`` in compact rows (``miss_count`` rows), and ``expand_backup`` of the root
        evaluation takes the evaluator's outputs for those rows."""
        import torch
        self.miss_planes = torch.zeros((self.G, PLANES, 8, 8), dtype=torch.float32, device=self.device)
        self.miss_count = torch.zeros((1,), dtype=torch.int32, device=self.device)
        _native.check(self._lib.m0_search_reuse_enable(self._h, int(slots), self.miss_planes.data_ptr(), self.miss_count.data_ptr()),
                      "m0_search_reuse_enable")

    def clear_reuse(self) -> None:
        _native.check(self._lib.m0_search_reuse_clear(self._h, self._stream()), "m0_search_reuse_clear")

    def set_streams(self, jitter=None, normal=None) -> None:
        """jitter / normal: float64 [G, n] device tensors holding the values ``random.random()`` / ``np.random.normal(0, 0.1)``
        would return, in the reference's consumption order; None = device generator.  The tensors must stay alive."""
        self._streams = (jitter, normal)
        for t in (jitter, normal):
            assert t is None or (t.dtype.is_floating_point and t.element_size() == 8 and t.is_contiguous() and t.shape[0] == self.G)
        _native.check(self._lib.m0_search_set_streams(self._h, _native.ptr(jitter), 0 if jitter is None else jitter.shape[1],
                                                      _native.ptr(normal), 0 if normal is None else normal.shape[1], self._stream()),
                      "m0_search_set_streams")

    def select_multi(self, batch_n: int, sims_left=None) -> None:
        _native.check(self._lib.m0_search_select_multi(self._h, int(batch_n), _native.ptr(sims_left), self.row_base.data_ptr(),
                                                       self.n_samples.data_ptr(), self._stream()), "m0_search_select_multi")

    def multi_encode(self, g0: int, g1: int, row0: int, mode: int, planes, row_cap: int = 0) -> None:
        _native.check(self._lib.m0_search_multi_encode(self._h, int(g0), int(g1), int(row0), int(mode), planes.data_ptr(), int(row_cap),
                                                       self._stream()), "m0_search_multi_encode")

    def expand_backup_multi(self, g0: int, g1: int, logits, values, row0: int, per_sample: bool, row_cap: int = 0) -> None:
        assert logits.dtype.is_floating_point and logits.element_size() == 4 and logits.is_contiguous()
        assert values.element_size() == 4 and values.is_contiguous()
        _native.check(self._lib.m0_search_expand_backup_multi(self._h, int(g0), int(g1), logits.data_ptr(), logits.shape[1], values.data_ptr(),
                                                              int(row0), 1 if per_sample else 0, int(row_cap), self._stream()),
                      "m0_search_expand_backup_multi")

    def counters(self) -> dict:
        buf = (ctypes.c_uint64 * 16)()
        _native.check(self._lib.m0_engine_counters(self._h, buf), "m0_engine_counters")
        return {name: int(buf[i]) for i, name in enumerate(COUNTER_NAMES)}

    def status(self):
        import torch
        st = torch.zeros((self.G,), dtype=torch.int32, device=self.device)
        nc = torch.zeros((self.G,), dtype=torch.int32, device=self.device)
        _native.check(self._lib.m0_engine_status(self._h, st.data_ptr(), nc.data_ptr(), self._stream()), "m0_engine_status")
        return st, nc


def board_history(board, cap: int):
    """Positions before `board` (oldest first) and the moves played from them: the part of
    board.move_stack / board._stack that Board.is_repetition can look at (public API only)."""
    if not getattr(board, "move_stack", None):
        return [], []
    b = board.copy()
    moves = []
    while b.move_stack and len(moves) < cap:
        moves.append(b.pop())
    moves.reverse()
    raws, codes = [], []
    for m in moves:
        raws.append(board_to_raw(b).copy())
        codes.append(move_to_code(m))
        b.push(m)
    return raws, codes
