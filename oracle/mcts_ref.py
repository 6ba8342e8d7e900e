"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the search algorithm of ``azchess/mcts.py``.

A compact Python port (on the oracle ``chess`` shim) of what ``MCTS.run`` computes, each function
citing the reference lines it follows.  It keeps the reference's quirks that bit-exact parity drags
in (SURVEY section 8, Q1-Q10): batched leaf collection without virtual loss, edge-child statistics
vs. transposition-table nodes, sequential fp64 backups, last-writer-wins TT registration, float32
softmax / float32 renormalisation of priors.

Deterministic harness (SURVEY 7-0c): ``jitter_value=0.5`` plays the role of ``random.random()``
patched to 0.5; Dirichlet / entropy noise / playout randomisation off; memory cleanups (wall-clock
and RSS driven, Q6) are not modelled.  Pinned against the UNMODIFIED reference executed on the same
shim in tests/test_oracle_mcts.py (where the reference tree is present) and through tests/golden/mcts_golden.json.
Only tests/, smoke() and bench.py's CPU legs import this module.
"""
from __future__ import annotations

import math
import random
from collections import OrderedDict
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from . import chess_shim  # noqa: F401
import chess
from .encoding_ref import encode_board, move_to_index_unchecked


class RefConfig:
    """Subset of MCTSConfig (mcts.py:61-107) that influences the result."""

    def __init__(self, **kw):
        self.num_simulations = 800
        self.cpuct = 2.5
        self.dirichlet_alpha = 0.3
        self.dirichlet_frac = 0.25
        self.dirichlet_plies = 16
        self.selection_jitter = 0.01
        self.fpu_reduction = 0.15
        self.draw_penalty = -0.1
        self.cpuct_start = None
        self.cpuct_end = None
        self.cpuct_plies = 0
        self.cpuct_c_base = None
        self.cpuct_c_init = None
        self.value_from_white = False
        self.legal_softmax = False
        self.no_instant_backtrack = True
        self.inference_batch_size = 96
        self.playout_random_frac = 0.0
        self.enable_entropy_noise = True
        self.max_children = 0
        self.min_child_prior = 0.0
        self.virtual_loss = 1.0
        for k, v in kw.items():
            if hasattr(self, k):
                setattr(self, k, v)


class RefNode:
    """mcts.py:120-133."""
    __slots__ = ("parent", "prior", "n", "w", "q", "children", "move", "expanded", "move_idx")

    def __init__(self, prior=0.0, move=None, parent=None):
        self.parent, self.prior, self.n, self.w, self.q = parent, prior, 0, 0.0, 0.0
        self.children: Dict[chess.Move, "RefNode"] = {}
        self.move, self.expanded, self.move_idx = move, False, None


def expand_with_legal_priors(node: RefNode, board, legal, pri: np.ndarray) -> None:
    """Node._expand_with_legal_priors, mcts.py:227-256 (fed RAW logits by the direct-model path, SURVEY Q3)."""
    if node.expanded or not legal:
        return
    pri = pri.astype(np.float32, copy=False)
    total = float(pri.sum())
    if not np.isfinite(total) or total <= 0:
        pri = np.full(len(legal), 1.0 / len(legal), dtype=np.float32)
    else:
        pri = pri / total
    wtm = board.turn == chess.WHITE
    for i, m in enumerate(legal):
        c = RefNode(prior=float(pri[i]), move=m, parent=node)
        c.move_idx = int(move_to_index_unchecked(wtm, m.from_square, m.to_square, m.promotion))
        if node.parent and node.parent.q != 0.0:
            c.q = -node.parent.q
        node.children[m] = c
    node.expanded = True


def expand(node: RefNode, board, logits: np.ndarray, legal_only: bool, allow_noise: bool, normal=None) -> None:
    """Node._expand, mcts.py:135-225.  normal(shape) stands in for np.random.normal(0, 0.1, shape)."""
    if node.expanded:
        return
    legal = list(board.legal_moves)
    if not legal:
        return
    logits = logits.astype(np.float32, copy=False)
    wtm = board.turn == chess.WHITE
    idxs = [move_to_index_unchecked(wtm, m.from_square, m.to_square, m.promotion) for m in legal]
    if np.any(np.isnan(logits)) or np.any(np.isinf(logits)):  # :147-149
        lp = np.full(len(legal), 1.0 / len(legal), dtype=np.float32)
    else:
        if legal_only:  # :158-163
            dist = torch.softmax(torch.from_numpy(np.ascontiguousarray(logits[idxs])), dim=-1).numpy()
        else:  # :164-168
            dist = torch.softmax(torch.from_numpy(np.ascontiguousarray(logits)), dim=-1).numpy()
        ent = -np.sum(dist * np.log(dist + 1e-8))  # :171-176
        ratio = ent / max(1e-9, np.log(max(1, len(legal))))
        if allow_noise and ratio > 0.9:  # :179-186
            dist = dist + (normal(dist.shape) if normal is not None else np.random.normal(0, 0.1, dist.shape))
            dist = np.maximum(dist, 1e-8)
            dist = dist / dist.sum()
        pri = []
        for i in range(len(legal)):  # :188-203
            p = float(dist[i]) if legal_only else float(dist[idxs[i]])
            if np.isnan(p) or np.isinf(p) or p < 0:
                p = 0.0
            pri.append(p)
        lp = np.asarray(pri, dtype=np.float32)  # :205-212
        tot = lp.sum()
        if tot > 0 and not np.isnan(tot) and not np.isinf(tot):
            lp = lp / tot
        else:
            lp = np.full(len(legal), 1.0 / len(legal), dtype=np.float32)
    for m, i, p in zip(legal, idxs, lp):  # :214-223
        c = RefNode(prior=float(p), move=m, parent=node)
        c.move_idx = int(i)
        if node.parent and node.parent.q != 0.0:
            c.q = -node.parent.q
        node.children[m] = c
    node.expanded = True


class RefMCTS:
    def __init__(self, cfg: RefConfig, backend, jitter_value: Optional[float] = 0.5, jitter_stream=None, normal_stream=None,
                 direct_model: bool = False, virtual_loss: bool = False):
        """backend: object with infer_np; jitter_value: constant standing in for random.random()
        (None = call random.random() like the reference).  jitter_stream / normal_stream: 1-D arrays consumed in order
        instead of random.random() / np.random.normal(0, 0.1) (the draws a seeded reference run would make).
        direct_model: the reference WITHOUT an inference backend -- non-root leaves of a legal_softmax search are expanded by
        _expand_with_legal_priors on the raw legal logits (mcts.py:697-703, SURVEY Q3)."""
        self.cfg, self.backend, self.jv = cfg, backend, jitter_value
        self.jitter_stream, self.normal_stream, self.jit_used, self.nrm_used = jitter_stream, normal_stream, 0, 0
        self.direct_model = direct_model
        # True: _select is called with an inflight_counts dict per mini-batch (mcts.py:851, :889-890, :922-923).  The reference ships that
        # code but _collect_leaf_position never passes the dict (:745, SURVEY Q1 / Q2b): this is the engine's throughput mode, not reference behaviour
        self.virtual_loss = virtual_loss
        self.min_gap = float("inf")   # smallest top-2 score gap over all selections (diagnostic for tolerance-limited parity)
        self.tt: "OrderedDict[tuple, RefNode]" = OrderedDict()
        self.nn_cache: Dict[tuple, tuple] = {}
        self.unique_evals = 0
        self.sample_rows = 0      # rows the reference evaluates (one per collected sample, duplicates included)
        self.distinct_rows = 0    # distinct (leaf node, board incl. clocks) pairs among them: the rows the engine evaluates
        self._last_root = None
        self._last_sims_run = 0

    # -- helpers ---------------------------------------------------------------------------------
    def _rand(self) -> float:
        if self.jitter_stream is not None:
            self.jit_used += 1
            return float(self.jitter_stream[self.jit_used - 1])
        return self.jv if self.jv is not None else random.random()

    def _normal(self, shape):
        if self.normal_stream is None:
            return np.random.normal(0, 0.1, shape)
        n = int(np.prod(shape))
        self.nrm_used += n
        return np.asarray(self.normal_stream[self.nrm_used - n:self.nrm_used], dtype=np.float64).reshape(shape)

    def _prune_children(self, node: RefNode) -> None:  # mcts.py:806-826
        if not node.children:
            return
        items = list(node.children.items())
        if self.cfg.min_child_prior > 0.0:
            items = [(m, c) for (m, c) in items if float(c.prior) >= float(self.cfg.min_child_prior)]
        if self.cfg.max_children and self.cfg.max_children > 0 and len(items) > self.cfg.max_children:
            items.sort(key=lambda mc: float(mc[1].prior), reverse=True)
            items = items[: int(self.cfg.max_children)]
        node.children = {m: c for (m, c) in items}

    def _expand_leaf(self, node: RefNode, lb, pol, allow_noise: bool) -> None:
        """mcts.py:654-665 (backend path) / :690-712 (direct-model path)."""
        if self.direct_model and self.cfg.legal_softmax:
            legal = list(lb.legal_moves)
            if legal:
                wtm = lb.turn == chess.WHITE
                idxs = [move_to_index_unchecked(wtm, m.from_square, m.to_square, m.promotion) for m in legal]
                expand_with_legal_priors(node, lb, legal, np.asarray(pol)[idxs])
        else:
            expand(node, lb, np.asarray(pol), self.cfg.legal_softmax, allow_noise, self._normal)
        self._prune_children(node)
        self._register_children(node, lb)

    def _cpuct_at(self, ply: int) -> float:  # mcts.py:927-944
        c = self.cfg
        if c.cpuct_c_base is not None and c.cpuct_c_init is not None:
            return float(c.cpuct_c_init) + math.log((max(1.0, float(ply + 1)) + float(c.cpuct_c_base)) / float(c.cpuct_c_base))
        if c.cpuct_start is None or c.cpuct_end is None or int(c.cpuct_plies) <= 0:
            return float(c.cpuct)
        t = min(max(ply, 0), int(c.cpuct_plies)) / float(int(c.cpuct_plies))
        return float(c.cpuct_start) + (float(c.cpuct_end) - float(c.cpuct_start)) * t

    def _terminal_value(self, b) -> float:  # mcts.py:1223-1229
        if b.is_checkmate():
            return -1.0
        if b.is_stalemate() or b.is_insufficient_material() or b.is_seventyfive_moves() or b.is_fivefold_repetition():
            return float(self.cfg.draw_penalty)
        return 0.0

    def _infer(self, b) -> Tuple[np.ndarray, float]:  # mcts.py:995-1190 (backend branch)
        p, v = self.backend.infer_np(encode_board(b)[None])
        p = np.asarray(p, dtype=np.float32).reshape(1, -1)
        v = np.clip(np.asarray(v, dtype=np.float32).reshape(-1), -1.0, 1.0)
        if self.cfg.value_from_white and b.turn == chess.BLACK:
            v = -v
        return p[0], float(v[0])

    def _backprop(self, path: List[RefNode], value: float) -> None:  # mcts.py:946-953
        v = max(-1.0, min(1.0, float(value)))
        for node in reversed(path):
            node.n += 1
            node.w += v
            node.q = node.w / node.n
            v = -v

    def _register_children(self, node: RefNode, b) -> None:  # mcts.py:1330-1346
        for m, child in node.children.items():
            b2 = b.copy(stack=False)
            b2.push(m)
            self.tt[b2._transposition_key()] = child

    def _select(self, b, root: RefNode, inflight=None):  # mcts.py:851-925 (inflight_counts is never passed by the reference: Q1)
        cfg = self.cfg
        node, path = root, [root]
        while node.expanded:
            if not node.children:
                break
            pv = max(1, node.n)
            best, best_s, second_s = None, -1e9, -1e9
            cp = self._cpuct_at(max(0, len(path) - 1))
            for child in node.children.values():
                q = (float(node.q) - float(cfg.fpu_reduction)) if child.n == 0 else child.q
                s = q + cp * child.prior * (math.sqrt(pv) / (1.0 + child.n))
                if cfg.no_instant_backtrack and len(path) >= 2 and child.move is not None and path[-1].move is not None:
                    prev = path[-1].move
                    if child.move.from_square == prev.to_square and child.move.to_square == prev.from_square:
                        s -= 0.01
                if inflight is not None and cfg.virtual_loss > 0.0:  # :889-890
                    s -= float(inflight.get(child, 0)) * float(cfg.virtual_loss)
                s += (self._rand() - 0.5) * (cfg.selection_jitter if cfg.selection_jitter > 0 else 0.001)
                if s > best_s:
                    second_s, best_s, best = best_s, s, child
                elif s > second_s:
                    second_s = s
            if len(node.children) > 1:
                self.min_gap = min(self.min_gap, best_s - second_s)
            if best is None:
                best = next(iter(node.children.values()))
            b.push(best.move)
            node = self.tt.get(b._transposition_key()) or best
            path.append(node)
            if inflight is not None:  # :922-923
                inflight[best] = inflight.get(best, 0) + 1
        return node, path, b

    # -- MCTS.run: mcts.py:318-512 -----------------------------------------------------------------
    def run(self, board, num_simulations: Optional[int] = None, ply: Optional[int] = None):
        cfg = self.cfg
        if board.is_game_over():
            return {}, np.zeros(4672, dtype=np.float32), self._terminal_value(board)
        key = board._transposition_key()
        root = self.tt.get(key)
        v = 0.0
        allow_noise = bool(cfg.enable_entropy_noise)
        if root is None:
            root = RefNode()
            logits, v = self._infer(board)
            self.unique_evals += 1
            expand(root, board, logits, cfg.legal_softmax, allow_noise, self._normal)
            self._prune_children(root)
            self.tt[key] = root
        else:
            if key not in self.nn_cache:
                logits, v = self._infer(board)
                self.nn_cache[key] = (logits, v)
            else:
                v = self.nn_cache[key][1]
        if cfg.dirichlet_plies is None or ply is None or ply < int(cfg.dirichlet_plies):
            self._add_dirichlet(root)
        sims = num_simulations if num_simulations is not None else cfg.num_simulations
        if cfg.playout_random_frac > 0.0 and sims > 0:  # :380-385
            low = int(max(1, sims * (1.0 - cfg.playout_random_frac)))
            sims = random.randint(low, int(max(low, sims * (1.0 + cfg.playout_random_frac))))
        if not root.expanded:  # :399-413
            logits, v = self._infer(board)
            self.unique_evals += 1
            expand(root, board, logits, cfg.legal_softmax, allow_noise, self._normal)
            self._prune_children(root)
            self._register_children(root, board)
            v = float(np.clip(v, -1.0, 1.0))
            root.q = v
        # _run_simulations_parallel_batched, :514-740 (sequential collection, backend branch)
        done, bs = 0, int(cfg.inference_batch_size) if int(cfg.inference_batch_size) > 0 else 96
        while done < sims:
            batch_n = min(bs, sims - done)
            samples = []
            inflight = {} if self.virtual_loss else None
            for _ in range(batch_n):
                node, path, lb = self._select(board.copy(), root, inflight)
                if lb.is_game_over():
                    self._backprop(path, self._terminal_value(lb))
                else:
                    samples.append((lb, node, list(path)))
            if samples:
                batch = np.stack([encode_board(s[0]) for s in samples], axis=0)
                policies, values = self.backend.infer_np(batch)
                self.unique_evals += 1
                self.sample_rows += len(samples)
                self.distinct_rows += len({(id(s[1]), s[0].halfmove_clock, s[0].fullmove_number, s[0].ep_square) for s in samples})
                for (lb, node, path), pol, val in zip(samples, policies, values):
                    if not node.expanded:
                        self._expand_leaf(node, lb, pol, allow_noise)
                    self._backprop(path, float(np.clip(val, -1.0, 1.0)))
            done += batch_n
        counts = {m: c.n for m, c in root.children.items()}
        total = sum(counts.values())
        if total == 0:  # :433-463, re-raised by :509-512
            raise RuntimeError(f"MCTS run failed: MCTS search failed: zero visits after {sims} simulations. "
                               f"Root node has {len(root.children)} children but none were visited.")
        pi = np.zeros(4672, dtype=np.float32)  # _policy_from_root, :828-849
        if total > 0:
            for m, c in root.children.items():
                pi[c.move_idx] = c.n / total
        else:
            for c in root.children.values():
                pi[c.move_idx] = 1.0 / len(root.children)
        self._last_root, self._last_sims_run = root, sims
        return counts, pi, (float(root.q) if root.n > 0 else float(v))

    def _add_dirichlet(self, root: RefNode) -> None:  # mcts.py:955-992
        cfg = self.cfg
        if not root.children or cfg.dirichlet_frac <= 0:
            return
        noise = np.random.dirichlet([cfg.dirichlet_alpha] * len(root.children))
        for i, child in enumerate(root.children.values()):
            p = child.prior * (1 - cfg.dirichlet_frac) + noise[i] * cfg.dirichlet_frac
            child.prior = max(1e-8, min(1.0 - 1e-8, p))
