"""Arena on the device game loop (SURVEY 8f-4): the two-evaluator match of ``azchess/arena.py:59-126`` / ``:129-270``.

Game ``idx`` gives evaluator A the white pieces when ``idx`` is even (arena.py:66); the side to move searches with ITS evaluator
(arena.py:68-71: every leaf of that search is evaluated by the mover's network), the move is sampled from visits^(1/T) at
temperature ``temp`` for the first ``temp_plies`` plies and is the most-visited move afterwards (arena.py:75-116); a game is scored
1 / 0.5 / 0 from A's side (arena.py:118-126).  All games of a batch advance in lock step on one GPU: per search step the pending
leaves are split by evaluator, each network runs once on its rows, and the outputs are scattered back -- no host round trip
besides one index computation per move.  Search settings follow ``_arena_worker_init`` (arena.py:33-57): the ``mcts:`` section with
``num_simulations`` overridden and ``selection_jitter`` taken from the ``selfplay:`` section (default 0.0).
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional

import numpy as np

from . import _native
from .selfplay import SelfPlayEngine


@_native.on_own_device
class _TwoEvaluatorGames(SelfPlayEngine):
    reuse_root_evals = False      # the root's children were evaluated by the other player's network

    def __init__(self, model_a, model_b, *args, **kw):
        super().__init__(model_a, *args, **kw)
        import torch
        self.model_b = model_b
        self.a_is_white = torch.zeros((self.G,), dtype=torch.bool, device=self.device)
        self._pos = torch.empty((self.G, 9), dtype=torch.int64, device=self.device)
        self._ia = self._ib = None
        self.rows_a = self.rows_b = 0

    def begin_move(self) -> None:
        # which evaluator moves in each game: A when (white to move) == (A has white)
        _native.check(self._lib.m0_games_get_positions(self.engine._h, self._pos.data_ptr(), _native.current_stream()), "m0_games_get_positions")
        white_to_move = (self._pos[:, 8] & 1).to(self.a_is_white.dtype)
        a_moves = white_to_move == self.a_is_white
        self._ia = a_moves.nonzero().squeeze(1)
        self._ib = (~a_moves).nonzero().squeeze(1)
        super().begin_move()

    def _forward(self, planes):
        import torch
        self.nn_evals += 1
        self.nn_rows += planes.shape[0]
        logits = torch.empty((self.G, 4672), dtype=torch.float32, device=self.device)
        values = torch.empty((self.G,), dtype=torch.float32, device=self.device)
        for rows, net in ((self._ia, self.model), (self._ib, self.model_b)):
            if rows.numel() == 0:
                continue
            lg, v = net.forward_planes(planes.index_select(0, rows), self.precision) if self.precision else net.forward_planes(planes.index_select(0, rows))
            logits.index_copy_(0, rows, lg)
            values.index_copy_(0, rows, v)
        self.rows_a += int(self._ia.numel())
        self.rows_b += int(self._ib.numel())
        return logits, values


class ArenaEngine:
    def __init__(self, model_a, model_b, cfg_dict: Dict[str, Any], num_sims: int, temperature: float = 0.0, temp_plies: int = 0,
                 max_moves: int = 200, concurrent_games: int = 1024, device: Optional[int] = None, seed: int = 1234,
                 precision: Optional[str] = None, deterministic: bool = False):
        mcts = dict(cfg_dict.get("mcts", {}) or {})
        sp_in = dict(cfg_dict.get("selfplay", {}) or {})
        mcts.update({"num_simulations": int(num_sims), "selection_jitter": float(sp_in.get("selection_jitter", 0.0))})   # arena.py:40-43
        sp = {"num_simulations": int(num_sims), "selection_jitter": float(sp_in.get("selection_jitter", 0.0)), "opening_random_plies": 0,
              "max_game_len": int(max_moves), "temperature_start": float(temperature), "temperature_end": 0.0, "temperature_moves": 0,
              "argmax_after_plies": int(temp_plies) if temperature > 1e-3 else 0, "resign_threshold": -2.0}
        self.G = int(concurrent_games)
        self.games = _TwoEvaluatorGames(model_a, model_b, {"mcts": mcts, "selfplay": sp}, games=self.G, device=device, deterministic=deterministic,
                                        seed=seed, precision=precision)

    def play(self, n_games: int) -> Dict[str, Any]:
        """Plays games 0 .. n_games-1 (A is White in the even ones) and returns A's score and the per-game results."""
        import torch
        g = self.games
        slot_game = np.full((self.G,), -1, dtype=np.int64)
        first = min(self.G, n_games)
        slot_game[:first] = np.arange(first)
        next_idx = first
        g.a_is_white.copy_(torch.from_numpy((slot_game % 2 == 0) & (slot_game >= 0)).to(g.device))
        g.start()
        results: List[Optional[Dict[str, Any]]] = [None] * n_games
        done = 0
        while done < n_games:
            g.play_move()
            changed = False
            for fin in g.finished_games():
                slot = fin["slot"]
                idx = int(slot_game[slot])
                if idx >= 0:
                    a_white = idx % 2 == 0
                    # only a mate decides an arena game; a game cut at max_moves is a draw (arena.py:118-126) -- the self-play loop
                    # would score it with the last root value (internal.py:587-599)
                    z = float(fin["result"]) if fin["reason"] == "checkmate" else 0.0
                    score = (z + 1.0) / 2.0 if a_white else (1.0 - z) / 2.0            # arena.py:118-126
                    results[idx] = {"game": idx, "a_is_white": a_white, "moves": fin["moves"], "score": score,
                                    "result": "1-0" if z > 0 else "0-1" if z < 0 else "1/2-1/2", "reason": fin["reason"]}
                    done += 1
                slot_game[slot] = next_idx if next_idx < n_games else -1              # the slot's next game (restarted on the device)
                next_idx += 1 if next_idx < n_games else 0
                changed = True
            if changed:
                g.a_is_white.copy_(torch.from_numpy((slot_game % 2 == 0) & (slot_game >= 0)).to(g.device))
        scores = [r["score"] for r in results]
        return {"games": results, "score_a": float(np.sum(scores)), "wins": int(sum(s == 1.0 for s in scores)),
                "draws": int(sum(s == 0.5 for s in scores)), "losses": int(sum(s == 0.0 for s in scores)),
                "rows_a": g.rows_a, "rows_b": g.rows_b}
