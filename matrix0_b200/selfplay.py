"""Batched, device-resident self-play: the B200 replacement of ``azchess/selfplay/internal.py``.

``SelfPlayEngine`` keeps G games on one GPU and advances all of them in lock step:

    per move :  trees_clear -> search_begin -> NN(roots not kept) -> expand (MCTS.run prologue)
                [select -> NN(leaves) -> expand+backup]  x ceil(sims / inference_batch_size)
                selfplay_advance (sample move, resign, push, finish / restart games)

Every step is a CUDA kernel launched through the C ABI; planes and logits never leave the GPU.
Search semantics per move are those of the reference's ``MCTS.run`` on a fresh ``MCTS`` object
("reference-exact" accounting: one pending leaf per game and mini-batch, SURVEY Q1).  The reference
itself reuses one MCTS object across moves, which makes its self-play fail with "zero visits" on
the second move (DESIGN.md, quirk Q12), so per-move fresh trees are the only working reading.

The configuration is the reference's YAML dictionary (``mcts:`` / ``selfplay:`` sections), merged
exactly as ``selfplay_worker`` does (internal.py:269-304).
"""
from __future__ import annotations

import ctypes
import math
import os
import time
from typing import Any, Dict, List, Optional

import numpy as np

from . import _native
from .engine import SearchEngine
from .mcts import MCTSConfig

END_REASONS = {1: "checkmate", 2: "stalemate", 3: "insufficient_material", 4: "fifty_moves", 5: "repetition", 6: "max_game_len", 7: "resign",
               8: "draw_adjudicated"}


def resolve_draw_config(cfg_dict: Dict[str, Any]) -> Dict[str, Any]:
    """``Config.draw()`` (azchess/config.py:37-49): top-level ``draw:`` merged with ``selfplay.draw:``, the latter winning."""
    merged = dict(cfg_dict.get("draw", {}) or {})
    merged.update((cfg_dict.get("selfplay", {}) or {}).get("draw", {}) or {})
    return merged


class SelfPlayConfigStruct(ctypes.Structure):
    """struct m0_selfplay_config (include/matrix0_b200.h)."""
    _fields_ = [(n, ctypes.c_double) for n in ("temperature_start", "temperature_end", "resign_threshold", "resign_min_entropy",
                                               "resign_value_margin")] \
        + [(n, ctypes.c_int) for n in ("temperature_moves", "max_game_len", "min_resign_plies", "resign_window",
                                       "resign_consecutive_bad", "opening_random_plies")] \
        + [("seed", ctypes.c_uint64)] \
        + [(n, ctypes.c_int) for n in ("argmax_after_plies", "low_visit_threshold", "draw_enabled", "draw_min_plies", "draw_window",
                                       "draw_min_unique", "draw_halfmove_cap", "draw_material_threshold")]


class FinishedGameStruct(ctypes.Structure):
    _fields_ = [("game", ctypes.c_int), ("plies", ctypes.c_int), ("z", ctypes.c_float), ("reason", ctypes.c_int), ("avg_entropy", ctypes.c_float)]


def resolve_mcts_config(cfg_dict: Dict[str, Any]) -> MCTSConfig:
    """The MCTSConfig ``selfplay_worker`` builds (internal.py:269-304): selfplay keys override mcts keys."""
    sp = dict(cfg_dict.get("selfplay", {}) or {})
    base = dict(cfg_dict.get("mcts", {}) or {}) or dict(cfg_dict.get("mcts_defaults", {}) or {})
    base.setdefault("num_simulations", int(sp.get("num_simulations", 800)))
    base.setdefault("cpuct", float(sp.get("cpuct", 2.5)))
    base.setdefault("dirichlet_alpha", float(sp.get("dirichlet_alpha", 0.3)))
    base.setdefault("dirichlet_frac", float(sp.get("dirichlet_frac", 0.25)))
    base.setdefault("inference_batch_size", 96)
    base.setdefault("selection_jitter", float(sp.get("selection_jitter", 0.01)))
    m = dict(base)
    m.update({
        "num_simulations": int(sp.get("num_simulations", m.get("num_simulations", 800))),
        "cpuct": float(sp.get("cpuct", m.get("cpuct", 2.5))),
        "dirichlet_alpha": float(sp.get("dirichlet_alpha", m.get("dirichlet_alpha", 0.3))),
        "dirichlet_frac": float(sp.get("dirichlet_frac", m.get("dirichlet_frac", 0.25))),
        "tt_capacity": int(m.get("tt_capacity", 2000000)),
        "selection_jitter": float(sp.get("selection_jitter", m.get("selection_jitter", 0.01))),
        "inference_batch_size": int(m.get("inference_batch_size", 96)),
        "fpu": float(sp.get("fpu", m.get("fpu", 0.5))),
        "parent_q_init": bool(sp.get("parent_q_init", m.get("parent_q_init", True))),
        "tt_cleanup_frequency": int(m.get("tt_cleanup_frequency", 500)),
        "draw_penalty": float(m.get("draw_penalty", -0.1)),
        "value_from_white": bool(m.get("value_from_white", False)),
    })
    return MCTSConfig.from_dict(m)


MAX_LEGAL_MOVES = 218     # the most legal moves a chess position can have
GUMBEL_NODE_BYTES = 50    # per node slot: prior, w, q (float64), n, first child, creator, move (int32), child count (int16), logit, r (fp32)


def gumbel_max_nodes(num_simulations: int) -> int:
    """Node slots a Gumbel move can fill in one game: the root, then at most num_simulations + 1 expansions (the root's and one per
    simulation) of at most 218 children each.  The tree has no transpositions, so a position with 218 moves at every node fills it."""
    return 1 + (int(num_simulations) + 1) * MAX_LEGAL_MOVES


GUMBEL_DEFAULTS = {"num_simulations": 32, "max_considered_actions": 16, "maxvisit_init": 50.0, "value_scale": 0.1}


def resolve_gumbel_config(cfg_dict: Dict[str, Any]) -> Dict[str, Any]:
    """The optional ``gumbel:`` section: num_simulations (1..4096), max_considered_actions (1..256), maxvisit_init (c_visit >= 0) and
    value_scale (c_scale > 0); out-of-range values raise ValueError."""
    sec = cfg_dict.get("gumbel", {}) or {}
    unknown = set(sec) - set(GUMBEL_DEFAULTS)
    if unknown:
        raise ValueError(f"unknown gumbel option(s): {sorted(unknown)}")
    out = dict(GUMBEL_DEFAULTS)
    out.update(sec)
    for key, lo, hi in (("num_simulations", 1, 4096), ("max_considered_actions", 1, 256)):
        v = out[key]
        if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or not lo <= int(v) <= hi:
            raise ValueError(f"gumbel.{key} must be an integer in [{lo}, {hi}], got {v!r}")
        out[key] = int(v)
    for key, positive in (("maxvisit_init", False), ("value_scale", True)):
        v = out[key]
        if isinstance(v, bool) or not isinstance(v, (int, float, np.integer, np.floating)) or not math.isfinite(float(v)) \
                or (float(v) <= 0.0 if positive else float(v) < 0.0):
            raise ValueError(f"gumbel.{key} must be a finite number {'> 0' if positive else '>= 0'}, got {v!r}")
        out[key] = float(v)
    return out


@_native.on_own_device
class SelfPlayEngine:
    # The root of a move is the child played at the previous move, and that child was evaluated during the previous search (a child
    # with visits reached its position at least once; only a terminal child has no row, and then the game ends).  The engine keeps
    # the network outputs of the root's children and expands the next root from them instead of evaluating it again.
    reuse_root_evals = True

    def __init__(self, model, cfg_dict: Dict[str, Any], games: int = 4096, device: Optional[int] = None, deterministic: bool = False,
                 seed: int = 1234, precision: Optional[str] = None, max_nodes: Optional[int] = None, cuda_graph: bool = True,
                 search_mode: str = "collapsed", forward_rows: Optional[int] = None):
        """``search_mode``:
        ``"collapsed"``   one selection per game and mini-batch, backed up with the multiplicity of the batch: exactly the reference
                          when its jitter is neutralised (SURVEY Q1; ``deterministic=True`` is bit-exact), and the throughput mode;
        ``"as_shipped"``  the reference with ``selection_jitter`` in force (config.yaml:138): every simulation of a mini-batch
                          selects with its own jitter draws (mcts.py:893-897), the distinct leaves of all games are compacted into
                          evaluator batches of ``forward_rows`` rows, samples are expanded / backed up in collection order;
        ``"virtual_loss"`` throughput mode: ``as_shipped`` plus the reference's in-flight marking (``_select``'s ``inflight_counts``,
                          mcts.py:889-890 / :922-923 -- code the reference ships but never activates, SURVEY Q2b) inside every mini-batch,
                          so the simulations of a batch spread over distinct leaves and (almost) every simulation evaluates its own row;
        ``"gumbel"``      Gumbel AlphaZero (DESIGN.md §9): ``gumbel.num_simulations`` simulation steps of one network row per game,
                          sequential halving at the root, the recorded policy is the improved policy softmax(logits + sigma(completed Q)).
                          Dirichlet noise, selection jitter, entropy noise, playout-cap randomisation and the temperature schedule do
                          not apply in this mode: the Gumbel draw at the root is its exploration."""
        import torch
        if search_mode not in ("collapsed", "as_shipped", "virtual_loss", "gumbel"):
            raise ValueError(f"search_mode must be 'collapsed', 'as_shipped', 'virtual_loss' or 'gumbel', got {search_mode!r}")
        self.virtual_loss = search_mode == "virtual_loss"
        self.search_mode = search_mode = "as_shipped" if self.virtual_loss else search_mode
        self.gumbel = resolve_gumbel_config(cfg_dict) if search_mode == "gumbel" else None
        self.reuse_root_evals = self.reuse_root_evals and self.gumbel is None    # a Gumbel move evaluates its root (its draws are new)
        self.model = model
        self.cfg_dict = cfg_dict
        self.mcfg = resolve_mcts_config(cfg_dict)
        self.sp = dict(cfg_dict.get("selfplay", {}) or {})
        self.G = int(games)
        self.deterministic = bool(deterministic)
        self.precision = precision
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        bs = max(1, int(self.mcfg.inference_batch_size))
        tt_capacity = 0                 # the engine's default: 2 * max_nodes
        if self.gumbel:
            # the table only holds the root (m0_search_begin); the tree itself has no transpositions
            tt_capacity = 64
            if max_nodes is None:
                max_nodes = gumbel_max_nodes(self.gumbel["num_simulations"])
                # the pool must fit in what the device has free now (the network and its workspaces are already allocated); a pool
                # that fits but leaves too little for the rest fails in the engine's allocation instead
                free, _ = torch.cuda.mem_get_info(self.device)
                if self.G * max_nodes * GUMBEL_NODE_BYTES > free:
                    raise ValueError(f"the Gumbel node pool of {self.G} games x {max_nodes} nodes (1 + (num_simulations + 1) x 218) needs "
                                     f"{self.G * max_nodes * GUMBEL_NODE_BYTES / 2**30:.1f} GiB, more than the {free / 2**30:.1f} GiB free on the "
                                     f"device: pass max_nodes= (a pool that can overflow on positions with many moves), fewer games or fewer simulations")
        elif max_nodes is None:
            # a fresh tree per move: every evaluated leaf adds its children (<= ~40 on average, 218 at most)
            sims_hi = int(self.mcfg.num_simulations * (1.0 + max(0.0, float(self.mcfg.playout_random_frac)))) + 1
            leaves = (sims_hi if search_mode == "as_shipped" else (sims_hi + bs - 1) // bs) + 2
            max_nodes = max(4096, 1 << int(math.ceil(math.log2(leaves * 48 + 256))))
        opening = int(self.sp.get("opening_random_plies", cfg_dict.get("openings", {}).get("random_plies", 0)))
        with torch.cuda.device(self.device):
            depth = 128 if not self.gumbel else max(128, self.gumbel["num_simulations"] + 2)   # a Gumbel path grows by at most one per step
            self.engine = SearchEngine(self.G, max_nodes=max_nodes, tt_capacity=tt_capacity, max_depth=depth,
                                       hist_cap=int(self.sp.get("max_game_len", 200)) + opening + 64, device=self.device_index)
            self.engine.configure(self.mcfg, deterministic, seed, virtual_loss=self.virtual_loss)
            if self.gumbel:
                gb = self.gumbel
                self.engine.gumbel_configure(gb["num_simulations"], gb["max_considered_actions"], gb["maxvisit_init"], gb["value_scale"])
            if search_mode == "as_shipped":
                self.engine.enable_multi(bs, virtual_loss=self.virtual_loss)
                if forward_rows is None:
                    # as shipped a mini-batch holds ~1.1 distinct leaves per game (entropy noise makes the priors peaked): one evaluator
                    # call of G + G/8 rows takes them all in the common case; the virtual-loss mode fills whole 4096-row calls
                    # (measured 1.19 rows per game and mini-batch); sized in whole rounds of the convolution kernel: 74 CTA pairs x 4 boards
                    rnd = 4 * max(1, torch.cuda.get_device_properties(self.device).multi_processor_count // 2)
                    forward_rows = 4096 if self.virtual_loss else min(8192, max(rnd, -(-int(1.2 * self.G) // rnd) * rnd))
                self.forward_rows = max(bs, min(int(forward_rows), self.G * bs))
                self.forward_rows += self.forward_rows & 1
                # evaluator batch sizes: full chunks of forward_rows rows, the tail chunk in the smallest size that holds it
                self.forward_sizes = sorted({self.forward_rows} | {s for s in (256, 512, 1024, 2048) if bs <= s < self.forward_rows})
                self.ml_planes = torch.zeros((self.forward_rows, 19, 8, 8), dtype=torch.float32, device=self.device)
            if self.reuse_root_evals:
                # collapsed: one evaluated leaf per game and mini-batch, so at most batches_per_move() root children per move; the
                # multi-leaf modes evaluate ~12 rows per game and move at all depths together (a full store only makes a later miss)
                self.engine.enable_reuse(32 if search_mode == "as_shipped" else min(32, self.batches_per_move()))
                # evaluator batch sizes of the roots that are not kept (new games, a child the store had no room for)
                self.root_sizes = sorted({self.G} | {s for s in (256, 512, 1024, 2048) if s < self.G})
                self._no_rows = (torch.zeros((1, 4672), dtype=torch.float32, device=self.device),
                                 torch.zeros((1,), dtype=torch.float32, device=self.device))
                self._reuse_epoch = model.ws_epoch
            s = SelfPlayConfigStruct()
            s.temperature_start = float(self.sp.get("temperature_start", 1.0))
            s.temperature_end = float(self.sp.get("temperature_end", 0.1))
            s.temperature_moves = int(self.sp.get("temperature_moves", 20))
            s.resign_threshold = float(self.sp.get("resign_threshold", -0.98))
            s.resign_min_entropy = float(self.sp.get("resign_min_entropy", 0.3))
            s.resign_value_margin = float(self.sp.get("resign_value_margin", 0.05))
            s.max_game_len = int(self.sp.get("max_game_len", 200))
            s.min_resign_plies = int(self.sp.get("min_resign_plies", 24))
            s.resign_window = int(self.sp.get("resign_window", 4))
            s.resign_consecutive_bad = int(self.sp.get("resign_consecutive_bad", 5))
            s.opening_random_plies = int(self.sp.get("opening_random_plies", cfg_dict.get("openings", {}).get("random_plies", 0)))
            s.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
            s.argmax_after_plies = int(self.sp.get("argmax_after_plies", -1))
            s.low_visit_threshold = int(self.sp.get("low_visit_threshold", 0) or 0)
            draw = resolve_draw_config(cfg_dict)                 # should_adjudicate_draw(board, move_history, draw_cfg), internal.py:383
            s.draw_enabled = 1 if bool(draw.get("enabled", False)) else 0
            s.draw_min_plies = int(draw.get("min_plies", 30))
            s.draw_window = int(draw.get("window", 12))
            s.draw_min_unique = int(draw.get("min_unique", 3))
            s.draw_halfmove_cap = int(draw.get("halfmove_cap", 50))
            s.draw_material_threshold = int(draw.get("material_draw_threshold", 10))
            lib = _native.lib()
            _native.check(lib.m0_selfplay_configure(self.engine._h, ctypes.byref(s), _native.current_stream()), "m0_selfplay_configure")
        self._lib = lib
        self.sims_left = torch.zeros((self.G,), dtype=torch.int32, device=self.device)
        self.plies = torch.zeros((self.G,), dtype=torch.int32, device=self.device)
        self.moves_played = torch.zeros((self.G,), dtype=torch.int16, device=self.device)
        self._gen = torch.Generator(device=self.device)
        self._gen.manual_seed(int(seed))
        self.cuda_graph = bool(cuda_graph) and hasattr(model, "capture_forward")   # replay the evaluator's launches as one CUDA graph
        self._graphs: Dict[Any, Any] = {}
        self.graph_kernels = 0      # kernels inside the captured forward
        self.graph_replays = 0
        self.nn_evals = 0
        self.nn_rows = 0
        self.nn_rows_padded = 0
        self.tree_events = None     # set to a list to collect CUDA events around the tree kernels of every search step
        self.moves = 0
        self.steps = 0
        self._result_ready = False  # Gumbel mode: gumbel_result() ran for the current move

    # ---- step plan --------------------------------------------------------------------------------
    def sims_per_move(self) -> float:
        return float(self.gumbel["num_simulations"] if self.gumbel else self.mcfg.num_simulations)

    def batches_per_move(self) -> int:
        if self.gumbel:
            return self.gumbel["num_simulations"]     # one simulation (one network row per game) per step
        sims = int(self.mcfg.num_simulations)
        frac = 0.0 if self.deterministic else float(self.mcfg.playout_random_frac)
        hi = int(max(max(1, sims * (1.0 - frac)), sims * (1.0 + frac))) if frac > 0 else sims
        bs = max(1, int(self.mcfg.inference_batch_size))
        return (hi + bs - 1) // bs

    def start(self, games: Optional[int] = None) -> None:
        """New games in the slots.  ``games``: play exactly this many games in total (``selfplay_worker``'s argument, internal.py:326):
        slots restart finished games until that many have been started, then go idle, and every started game is played to its end."""
        st = _native.current_stream()
        _native.check(self._lib.m0_selfplay_set_start_budget(self.engine._h, -1 if games is None else int(games), st), "m0_selfplay_set_start_budget")
        _native.check(self._lib.m0_selfplay_start(self.engine._h, st), "m0_selfplay_start")

    def active_games(self) -> int:
        n = ctypes.c_int(0)
        _native.check(self._lib.m0_selfplay_active_games(self.engine._h, ctypes.byref(n), _native.current_stream()), "m0_selfplay_active_games")
        return n.value

    def set_sampling_uniforms(self, uniforms) -> None:
        """uniforms: float64 [G] device tensor (or None): the np.random.choice draw of sample_move_from_counts for the next plies."""
        self._uniforms = uniforms
        _native.check(self._lib.m0_selfplay_set_uniforms(self.engine._h, _native.ptr(uniforms)), "m0_selfplay_set_uniforms")

    def check_status(self) -> None:
        """Raise when a game ran out of tree nodes / table slots / history (the reference bounds its memory by cleanups instead)."""
        st, _ = self.engine.status()
        bits = int(st.max()) if st.numel() else 0
        if bits & 0b11011:
            bad = int((st != 0).sum())
            raise RuntimeError(f"search capacity exhausted in {bad} game(s) (status bits {bits:#x}: 1 nodes, 2 transposition table, 8 history, "
                               f"16 random stream): raise max_nodes / hist_cap")

    def _forward(self, planes):
        self.nn_evals += 1
        self.nn_rows += planes.shape[0]
        if self.cuda_graph and (self.precision or getattr(self.model, "precision", "fp32")) != "fp32":
            key = (planes.data_ptr(), planes.shape[0], self.model.ws_epoch)
            if key not in self._graphs:
                lib = _native.lib()
                self._graphs = {k: v for k, v in self._graphs.items() if k[2] == self.model.ws_epoch}   # stale captures (old weights / workspaces)
                g, lg, v = self.model.capture_forward(planes, self.precision)
                if self.model.ws_epoch != key[2]:                           # the capture grew the workspaces: earlier graphs are stale
                    self._graphs = {}
                    key = (planes.data_ptr(), planes.shape[0], self.model.ws_epoch)
                n0 = int(lib.m0_launch_count())
                self.model.forward_planes(planes, self.precision)          # one eager pass to count the kernels the graph replays
                self.graph_kernels = int(lib.m0_launch_count()) - n0
                self._graphs[key] = (g, lg, v)
            g, lg, v = self._graphs[key]
            g.replay()
            self.graph_replays += 1
            return lg, v
        return self.model.forward_planes(planes, self.precision) if self.precision else self.model.forward_planes(planes)

    def begin_move(self) -> None:
        """MCTS.run prologue for every game: fresh tree, root evaluation + expansion, Dirichlet noise, budgets."""
        import torch
        eng = self.engine
        _native.check(self._lib.m0_trees_clear(eng._h, _native.current_stream()), "m0_trees_clear")
        if self.gumbel:
            eng.begin()
            logits, values = self._forward(eng.planes)
            eng.gumbel_expand_backup(logits, values)           # the root: children, r, Gumbel draws, N = 1, W = r
            self._result_ready = False
            self.steps += 1
            return
        if not self.reuse_root_evals:
            eng.begin()
            logits, values = self._forward(eng.planes)
        else:
            if self.model.ws_epoch != self._reuse_epoch:       # new weights (or only new workspaces): the kept outputs may be stale
                eng.clear_reuse()
                self._reuse_epoch = self.model.ws_epoch
            eng.begin()
            n = int(eng.miss_count.item())
            if n:
                size = next(s for s in self.root_sizes if s >= n)
                logits, values = self._forward(eng.miss_planes[:size])
                self.nn_rows += n - size
            else:
                logits, values = self._no_rows                      # every root is expanded from a kept output
        eng.expand_backup(logits, values)
        if not self.deterministic and float(self.mcfg.dirichlet_frac) > 0:
            _native.check(self._lib.m0_selfplay_plies(eng._h, self.plies.data_ptr(), _native.current_stream()), "m0_selfplay_plies")
            dp = getattr(self.mcfg, "dirichlet_plies", None)
            apply = None if dp is None else (self.plies < int(dp)).to(torch.int32)
            eng.add_dirichlet(None, apply)
        sims = int(self.mcfg.num_simulations)
        frac = 0.0 if self.deterministic else float(self.mcfg.playout_random_frac)
        if frac > 0.0 and sims > 0:  # per-game budgets, mcts.py:380-385
            low = int(max(1, sims * (1.0 - frac)))
            high = int(max(low, sims * (1.0 + frac)))
            self.sims_left.copy_(torch.randint(low, high + 1, (self.G,), device=self.device, generator=self._gen, dtype=torch.int32))
        else:
            self.sims_left.fill_(sims)
        self.steps += 1

    def search_step(self) -> None:
        """One mini-batch: select -> evaluate the pending leaves of all games -> expand + backup."""
        eng = self.engine
        if self.search_mode == "as_shipped":
            return self._search_step_as_shipped()
        ev = self.tree_events
        if ev is not None:        # measurement aid (bench.py): CUDA events around the two tree kernels of this step
            import torch
            e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            e[0].record()
        if self.gumbel:
            eng.gumbel_select()
        else:
            _native.check(self._lib.m0_search_select_var(eng._h, int(self.mcfg.inference_batch_size), self.sims_left.data_ptr(),
                                                         eng.planes.data_ptr(), _native.current_stream()), "m0_search_select_var")
        if ev is not None:
            e[1].record()
        logits, values = self._forward(eng.planes)
        if ev is not None:
            e[2].record()
        if self.gumbel:
            eng.gumbel_expand_backup(logits, values)
        else:
            eng.expand_backup(logits, values)
        if ev is not None:
            e[3].record()
            ev.append(e)
        self.steps += 1

    def warm_up_forward(self) -> None:
        """Capture the evaluator graphs of every batch size this engine uses (one-off cost of ~1 s per size, otherwise paid inside the
        first move that needs the size)."""
        calls = [(self.ml_planes, s) for s in self.forward_sizes] if self.search_mode == "as_shipped" else []
        if self.reuse_root_evals:
            calls += [(self.engine.miss_planes, s) for s in self.root_sizes]
        for buf, size in sorted(calls, key=lambda c: -c[1]):
            self._forward(buf[:size])
        self.nn_evals = self.nn_rows = 0

    def _search_step_as_shipped(self) -> None:
        """mcts.py:535-740 with jitter in force: collect batch_n samples per game, evaluate the distinct leaves of all games in
        compact batches (a chunk = a run of consecutive games whose rows fit ``forward_rows``), then expand / back up per game in
        collection order.  One small D2H read (the row numbering) per mini-batch sizes the evaluator calls."""
        eng = self.engine
        eng.select_multi(int(self.mcfg.inference_batch_size), self.sims_left)
        G, cap = self.G, self.forward_rows
        # first evaluator batch WITHOUT waiting for the row numbering: the kernels take as many leading games as fit into `cap` rows
        # (device-side gate on row_base), so the host's read below overlaps the forward instead of idling the GPU
        planes = self.ml_planes[:cap]
        eng.multi_encode(0, G, 0, 0, planes, row_cap=cap)
        logits, values = self._forward(planes)
        eng.expand_backup_multi(0, G, logits, values, 0, per_sample=False, row_cap=cap)
        rb = eng.row_base.cpu().numpy()
        g0 = max(int(np.searchsorted(rb, cap, side="right")) - 1, 0)        # games [0, g0) were in that batch
        self.nn_rows += int(rb[g0]) - cap
        self.nn_rows_padded += cap
        while g0 < G:
            g1 = int(np.searchsorted(rb, rb[g0] + cap, side="right")) - 1   # largest g1 with rb[g1] - rb[g0] <= cap
            g1 = min(max(g1, g0 + 1), G)
            rows = int(rb[g1] - rb[g0])
            if rows > 0:
                size = next(s for s in self.forward_sizes if s >= rows)
                planes = self.ml_planes[:size]
                eng.multi_encode(g0, g1, int(rb[g0]), 0, planes)
                logits, values = self._forward(planes)
                self.nn_rows += rows - size                                 # count the rows that carry a leaf, not the padding
                self.nn_rows_padded += size
                eng.expand_backup_multi(g0, g1, logits, values, int(rb[g0]), per_sample=False)
            g0 = g1
        self.steps += 1

    def gumbel_result(self, with_pi: bool = False) -> None:
        """Gumbel mode, after the simulations of a move: the move to play, the search value and the policy target (engine.gb_*,
        engine.res_*); end_move() calls it when nobody did."""
        self.engine.gumbel_result(with_pi=with_pi)
        self._result_ready = True

    def end_move(self) -> None:
        if self.gumbel:
            if not self._result_ready:
                self.gumbel_result()
            self._result_ready = False
            _native.check(self._lib.m0_selfplay_advance_gumbel(self.engine._h, self.moves_played.data_ptr(), _native.current_stream()),
                          "m0_selfplay_advance_gumbel")
        else:
            _native.check(self._lib.m0_selfplay_advance(self.engine._h, self.moves_played.data_ptr(), _native.current_stream()), "m0_selfplay_advance")
        self.moves += 1

    def play_move(self) -> None:
        self.begin_move()
        for _ in range(self.batches_per_move()):
            self.search_step()
        self.end_move()

    # ---- results ----------------------------------------------------------------------------------
    def finished_games(self, max_records: int = 65536) -> List[Dict[str, Any]]:
        buf = (FinishedGameStruct * max_records)()
        n = ctypes.c_int(0)
        _native.check(self._lib.m0_selfplay_finished(self.engine._h, buf, max_records, ctypes.byref(n), _native.current_stream()), "m0_selfplay_finished")
        return [{"slot": buf[i].game, "moves": buf[i].plies, "result": float(buf[i].z), "reason": END_REASONS.get(buf[i].reason, "?"),
                 "resigned": buf[i].reason == 7, "draw": float(buf[i].z) == 0.0, "avg_policy_entropy": float(buf[i].avg_entropy)}
                for i in range(n.value)]

    def counters(self) -> Dict[str, int]:
        return self.engine.counters()


LAST_WORKER_STATS: Dict[str, Any] = {}    # where the last selfplay_worker call of this process spent its time (tools/worker_throughput.py)


def selfplay_worker(proc_id: int, cfg_dict: Dict[str, Any], ckpt_path: Optional[str], games: int, q=None, shared_memory_resource=None,
                    device: Optional[int] = None, concurrent_games: Optional[int] = None, precision: str = "fp16", data_manager=None,
                    search_mode: str = "as_shipped") -> int:
    """Drop-in for ``azchess.selfplay.internal.selfplay_worker`` (internal.py:94): plays ``games`` self-play games and emits the same
    artefacts -- one NPZ shard per game (internal.py:626-651) and the orchestrator's queue messages (``heartbeat`` :546-556,
    ``game`` :666-679).  One call drives a whole GPU: ``concurrent_games`` games (default min(games, 4096)) advance in lock step on
    ``device`` instead of one game per process; the evaluator is the native network (``shared_memory_resource`` -- the handle of the
    reference's inference server -- is accepted and ignored, nothing leaves the device).

    ``data_manager``: any object with ``add_selfplay_data(game_data, worker_id, game_id) -> path`` (the reference's DataManager);
    default writes ``{cfg.data_dir or 'data'}/selfplay/selfplay_w{proc}_g{game}_{ms}.npz`` with ``records.write_game_npz``.
    Returns the number of games written."""
    import torch
    dev = int(device if device is not None else (proc_id % max(1, torch.cuda.device_count())))
    with torch.cuda.device(dev):          # everything below (recorder streams, events, page-locked copies) belongs to this device
        return _selfplay_worker_on_device(proc_id, cfg_dict, ckpt_path, games, q, dev, concurrent_games, precision, data_manager, search_mode)


def _selfplay_worker_on_device(proc_id: int, cfg_dict: Dict[str, Any], ckpt_path: Optional[str], games: int, q, dev: int,
                               concurrent_games: Optional[int], precision: str, data_manager, search_mode: str) -> int:
    import torch
    from .model import PolicyValueNet
    from .records import GameRecorder, write_game_npz
    seed = int(cfg_dict.get("seed", 1234)) + int(proc_id)     # internal.py:111-113 seeds by worker
    model = PolicyValueNet.from_config(cfg_dict.get("model", {}), device=f"cuda:{dev}", precision=precision, seed=seed)
    if ckpt_path:
        state = torch.load(ckpt_path, map_location="cpu", weights_only=False)
        sd = state.get("model_ema", state.get("model", state)) if isinstance(state, dict) else state   # internal.py:172-174
        model.load_state_dict(sd, strict=False)
    G = int(concurrent_games or min(int(games), 4096))
    # "as_shipped": the reference's search with its configured selection jitter and entropy noise (distinct leaves per mini-batch);
    # "collapsed": one evaluated leaf per game and mini-batch (the throughput mode, exact when the jitter is neutralised);
    # "gumbel": Gumbel AlphaZero with the improved policy as the recorded target (the config's `gumbel:` section)
    sp = SelfPlayEngine(model, cfg_dict, games=G, device=dev, deterministic=False, seed=seed, precision=precision, search_mode=search_mode)
    sp.warm_up_forward()
    mcfg = cfg_dict.get("model", {}) or {}
    ssl_tasks = tuple(mcfg.get("ssl_tasks", ())) if mcfg.get("self_supervised", False) else ()      # internal.py:251-256
    rec = GameRecorder(sp, ssl_tasks=ssl_tasks)
    out_dir = os.path.join(str(cfg_dict.get("data_dir", "data")), "selfplay")
    # The shards are compressed (np.savez_compressed, ~60 ms per 200-ply game) by a small pool of writer threads (zlib releases the GIL)
    # while the GPU searches on; at most `writer_queue_games` finished games wait in host memory, and the "game" messages keep game order.
    import collections
    from concurrent.futures import ThreadPoolExecutor
    n_writers = int((cfg_dict.get("selfplay", {}) or {}).get("writer_threads", min(12, max(1, (os.cpu_count() or 2) - 2))))
    pool = ThreadPoolExecutor(max_workers=max(1, n_writers), thread_name_prefix="m0-npz")
    # ~6.5 MB per 200-ply game, and every 160 of them keep one 1 GiB page-locked block of the recorder alive (0.45 s to allocate the first time)
    pending, max_pending = collections.deque(), int((cfg_dict.get("selfplay", {}) or {}).get("writer_queue_games", 32 * max(1, n_writers)))
    npz_level = (cfg_dict.get("selfplay", {}) or {}).get("npz_compresslevel", None)   # None: np.savez_compressed, byte-for-byte the reference's writer
    submitted, written, last_hb, t_start = 0, 0, time.perf_counter(), time.perf_counter()

    def save(gd, game_id):
        if data_manager is not None:
            return data_manager.add_selfplay_data(gd, worker_id=proc_id, game_id=game_id)
        return write_game_npz(out_dir, gd, proc_id, game_id, compresslevel=npz_level)

    stats = LAST_WORKER_STATS
    stats.clear()
    stats.update(seconds_search=0.0, seconds_record_assembly=0.0, seconds_waiting_for_writers=0.0, writer_threads=n_writers)

    def drain(everything: bool) -> None:
        nonlocal written
        while pending and (everything or len(pending) > max_pending or pending[0][0].done()):
            fut, meta = pending.popleft()
            try:
                tw = time.perf_counter()
                path = fut.result()
                stats["seconds_waiting_for_writers"] += time.perf_counter() - tw
            except Exception:                 # a failed save does not stop the worker (internal.py:652-656)
                path = None
            if path is not None:
                written += 1
            if q is not None:
                q.put(dict(meta, file=path))

    def handle(gd) -> None:
        nonlocal submitted
        if submitted >= games:
            return
        T = int(gd["meta_moves"][0])
        z = float(gd["meta_result"][0])
        secs = time.perf_counter() - t_start
        meta = {"type": "game", "proc": proc_id, "file": None, "moves": T, "result": z, "secs": secs,
                "resigned": bool(gd["meta_resigned"][0]), "resigner": None, "draw": bool(z == 0.0),
                "avg_policy_entropy": float(gd["meta_avg_policy_entropy"][0]), "avg_ms_per_move": secs * 1000.0 / max(1, T),
                "avg_sims": float(gd["meta_avg_sims"][0])}
        pending.append((pool.submit(save, gd, submitted), meta))
        submitted += 1
        drain(False)

    def handle_all(games_iter) -> None:
        it = iter(games_iter)
        while True:
            ta = time.perf_counter()
            gd = next(it, None)              # the recorder waits for a group's device-to-host copies inside next()
            stats["seconds_record_assembly"] += time.perf_counter() - ta
            if gd is None:
                return
            handle(gd)

    sp.start(games)                      # exactly `games` games are started; every one of them is played to its end (internal.py:326)
    try:
        while submitted < games:
            ts = time.perf_counter()
            sp.begin_move()
            for _ in range(sp.batches_per_move()):
                sp.search_step()
            rec.after_search()
            sp.end_move()
            sp.check_status()
            stats["seconds_search"] += time.perf_counter() - ts
            # the records of the games that ended on this ply are assembled and copied on a side stream under the next ply's search
            # and come out of the next call; groups are bounded, so a ply on which every slot ends does not stage all games at once
            # while the shard writers are busy the finished games wait in the recorder's device ring (up to max_game_len plies) instead
            # of blocking the search on the writer queue
            drain(False)
            room = max(0, max_pending - len(pending) - rec.pending_games())
            handle_all(rec.iter_after_move(defer=True, max_games=room))
            drain(False)
            if sp.active_games() == 0:
                break                            # every started game is over (games that ended inside their opening plies leave no shard)
            if q is not None and time.perf_counter() - last_hb >= 2.0:
                q.put({"type": "heartbeat", "proc": proc_id, "game": submitted, "moves": sp.moves, "avg_sims": sp.sims_per_move(),
                       "resigned": False, "avg_policy_entropy": 0.0})
                last_hb = time.perf_counter()
        handle_all(rec.flush())
    finally:
        drain(True)
        pool.shutdown(wait=True)
        stats["seconds_play_and_write"] = time.perf_counter() - t_start
        stats["recorder_seconds_by_phase"] = dict(rec.timing)
    return written
