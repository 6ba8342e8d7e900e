"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the per-game loop of ``azchess/selfplay/internal.py:326-600`` and of
``azchess/draw.py`` around a search whose results are handed in (visit counts, pi, value), with the ``np.random`` draw of
``sample_move_from_counts`` supplied by the caller.  ``should_adjudicate_draw`` and ``sample_move_from_counts`` are pinned against
the UNMODIFIED reference functions in tests/test_oracle_selfplay.py (stored answers, and live where the reference tree is present).  Only tests/ import this module.
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional, Sequence

import numpy as np

from . import chess_shim  # noqa: F401
import chess


def should_adjudicate_draw(board, moves: Sequence, cfg: Dict[str, Any]) -> bool:
    """draw.py:8-84."""
    if board.is_insufficient_material():
        return True
    if board.can_claim_fifty_moves():
        return True
    if board.is_repetition(3) or board.can_claim_threefold_repetition():
        return True
    if bool(cfg.get("stalemate_draw", True)) and board.is_stalemate():
        return True
    if not bool(cfg.get("enabled", False)):
        return False
    if len(moves) < int(cfg.get("min_plies", 30)):
        return False
    window, min_unique = int(cfg.get("window", 12)), int(cfg.get("min_unique", 3))
    if window > 0 and min_unique > 0 and len(moves) >= window:
        if len(set(str(m) for m in moves[-window:])) < min_unique:
            return True
    cap = int(cfg.get("halfmove_cap", 50))
    if cap and board.halfmove_clock >= cap:
        return True
    thr = int(cfg.get("material_draw_threshold", 10))
    if thr > 0:
        total = 0
        for color in (chess.WHITE, chess.BLACK):
            total += (len(board.pieces(chess.PAWN, color)) + 3 * len(board.pieces(chess.KNIGHT, color)) + 3 * len(board.pieces(chess.BISHOP, color))
                      + 5 * len(board.pieces(chess.ROOK, color)) + 9 * len(board.pieces(chess.QUEEN, color)))
        if total <= thr:
            return True
    return False


def choice_index(p: np.ndarray, u: float) -> int:
    """np.random.choice(len(p), p=p) given its one uniform draw u (numpy/random/mtrand.pyx: p as float64, cdf = p.cumsum(),
    cdf /= cdf[-1], cdf.searchsorted(u, side='right'))."""
    cdf = np.asarray(p, dtype=np.float64).cumsum()
    cdf /= cdf[-1]
    return int(cdf.searchsorted(u, side="right"))


def sample_move_from_counts(moves: List, visits_in: Sequence[int], temperature: float, u: float):
    """internal.py:690-735 with the np.random draw replaced by `u`: returns the chosen index into `moves` (uniform fallbacks pick
    int(u * k), the device's convention for a draw the reference makes with np.random.choice(legal_moves))."""
    visits = np.array(list(visits_in), dtype=np.float32)
    k = len(moves)
    if np.any(np.isnan(visits)) or np.all(visits == 0):
        return min(int(u * k), k - 1)
    if temperature < 1e-3:
        return int(np.argmax(visits))
    with np.errstate(over="ignore", invalid="ignore"):
        dist = visits ** (1.0 / temperature)
        s = dist.sum()
        if s <= 0 or np.isnan(s):
            return min(int(u * k), k - 1)
        dist /= s
    if np.any(np.isnan(dist)):
        return min(int(u * k), k - 1)
    return choice_index(dist, u)


def game_result(board) -> float:
    """internal.py:738-750."""
    if board.is_checkmate():
        return -1.0 if board.turn == chess.WHITE else 1.0
    res = board.result(claim_draw=True)
    return 1.0 if res == "1-0" else (-1.0 if res == "0-1" else 0.0)


class GameLoopRef:
    """One game of selfplay_worker's loop (internal.py:334-600), driven from outside: call ``ended()`` before every search and
    ``play(visit_counts, pi, v, u)`` after it."""

    def __init__(self, sp_cfg: Dict[str, Any], draw_cfg: Dict[str, Any], board=None, move_history: Optional[List] = None):
        self.sp, self.draw = sp_cfg, draw_cfg
        self.board = board if board is not None else chess.Board()
        self.move_history = list(move_history or [])
        self.n_states = 0
        self.search_values: List[float] = []
        self.recent_values: List[float] = []
        self.recent_entropies: List[float] = []
        self.consec_bad = 0
        self.resigned = False
        self.z: Optional[float] = None
        self.window_k = int(sp_cfg.get("resign_window", 4))

    def temperature(self) -> float:  # :386-394
        t_moves = int(self.sp.get("temperature_moves", 20))
        t0, t1 = float(self.sp.get("temperature_start", 1.0)), float(self.sp.get("temperature_end", 0.1))
        if t_moves <= 0:
            return t1
        t = min(max(self.board.fullmove_number, 0), t_moves) / float(max(1, t_moves))
        return t0 + (t1 - t0) * t

    def ended(self) -> Optional[str]:
        """Loop condition :382-384; returns the reason the game stops before another search, and sets z (:587-599)."""
        b = self.board
        reason = None
        if b.is_game_over():
            reason = ("checkmate" if b.is_checkmate() else "stalemate" if b.is_stalemate() else "insufficient_material" if b.is_insufficient_material()
                      else "fifty_moves" if b.is_seventyfive_moves() else "repetition")
        elif should_adjudicate_draw(b, self.move_history, dict(self.draw, enabled=False)):
            # a claimable draw: reported under its own name even when the length cap holds too (z is the same: a draw)
            reason = ("insufficient_material" if b.is_insufficient_material() else "fifty_moves" if b.can_claim_fifty_moves() else "repetition")
        elif self.n_states >= int(self.sp.get("max_game_len", 200)):
            reason = "max_game_len"
        elif should_adjudicate_draw(b, self.move_history, self.draw):
            reason = "draw_adjudicated"
        if reason is None:
            return None
        if b.is_game_over(claim_draw=True):
            self.z = game_result(b)
        else:
            self.z = float(self.search_values[-1]) if self.search_values else 0.0
        return reason

    def play(self, moves: List, visits: Sequence[int], pi: np.ndarray, v: float, u: float):
        """:408-539: sample the move, track entropy / values, resign rule, push.  Returns (move index or None when resigned)."""
        temp = self.temperature()
        thr = int(self.sp.get("low_visit_threshold", 0) or 0)
        if thr > 0 and max(visits) < thr:
            temp = max(temp, 0.8)
        idx = sample_move_from_counts(moves, visits, temp, u)
        _pi = np.clip(pi.astype(np.float64, copy=False), 1e-12, 1.0)
        ent = float(-np.sum(_pi * np.log(_pi)))
        self.recent_entropies.append(ent)
        if len(self.recent_entropies) > self.window_k:
            self.recent_entropies.pop(0)
        self.n_states += 1
        self.search_values.append(v)
        resign_thr = float(self.sp.get("resign_threshold", -0.98))
        if resign_thr > -1.0 and self.n_states >= int(self.sp.get("min_resign_plies", 24)):  # :507-536
            self.recent_values.append(float(v))
            if len(self.recent_values) > self.window_k:
                self.recent_values.pop(0)
            self.consec_bad = self.consec_bad + 1 if v < resign_thr else 0
            need = max(2, self.window_k // 2)
            stable_bad = len(self.recent_values) >= need and (sum(self.recent_values) / len(self.recent_values)) < (resign_thr + float(self.sp.get("resign_value_margin", 0.05)))
            low_unc = len(self.recent_entropies) >= need and (sum(self.recent_entropies) / len(self.recent_entropies)) < float(self.sp.get("resign_min_entropy", 0.3))
            if self.consec_bad >= int(self.sp.get("resign_consecutive_bad", 5)) and (stable_bad or low_unc):
                self.resigned = True
                self.z = -1.0 if self.board.turn == chess.WHITE else 1.0
                return None
        self.move_history.append(moves[idx])
        self.board.push(moves[idx])
        return idx
