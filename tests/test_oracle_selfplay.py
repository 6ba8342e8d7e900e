"""oracle/selfplay_ref.py (restatements of azchess/draw.py and of sample_move_from_counts, azchess/selfplay/internal.py:690-735)
against the reference's stored answers (tests/golden/selfplay_golden.json) and, where the unmodified reference tree is present,
against the reference code itself."""
import numpy as np
import pytest

import chess
import selfplay_cases as C
from oracle import refload, selfplay_ref as R

needs_ref = pytest.mark.skipif(not refload.reference_available(), reason=refload.MISSING)


def test_should_adjudicate_draw_matches_reference_goldens():
    g = C.load()["draw"]
    assert g["cfgs"] == C.DRAW_CFGS
    games = [[chess.Move.from_uci(u) for u in game] for game in g["games"]]
    got = "".join("1" if R.should_adjudicate_draw(b, moves, cfg) else "0" for b, moves, cfg in C.draw_cases(games))
    assert got == g["decisions"]
    assert len(got) > 5000 and 200 < got.count("1") < len(got) - 200


def test_sample_move_from_counts_matches_reference_goldens():
    g = C.load()["sample"]
    moves = list(chess.Board(g["fen"]).legal_moves)
    assert len(g["trials"]) == 400
    for t in g["trials"]:
        got = R.sample_move_from_counts(moves[:t["moves"]], t["counts"], t["temperature"], C.uniform(t["seed"]))
        assert got == t["choice"], t


@needs_ref
def test_should_adjudicate_draw_matches_reference():
    ref = refload.load_reference("draw").should_adjudicate_draw
    n = hits = 0
    for b, moves, cfg in C.draw_cases(C.draw_games()):
        want = ref(b, moves, cfg)
        assert R.should_adjudicate_draw(b, moves, cfg) == want, (b.fen(), cfg)
        n += 1
        hits += bool(want)
    assert n > 5000 and 200 < hits < n - 200


@needs_ref
def test_sample_move_from_counts_matches_reference():
    ref = C.reference_function("azchess/selfplay/internal.py", "sample_move_from_counts")
    b = chess.Board(C.SAMPLE_FEN)
    n = 0
    for counts, T, seed in C.sample_trials():
        u = C.uniform(seed)
        np.random.seed(seed)
        want = ref(b, counts, T)
        got = R.sample_move_from_counts(list(counts.keys()), list(counts.values()), T, u)
        assert list(counts.keys())[got] == want, (seed, T)
        n += 1
    assert n == 400


def test_game_loop_gumbel_variant_plays_the_chosen_move_and_resigns():
    """GameLoopRef.play_gumbel: the searched move is pushed as chosen (no temperature, no sampling), the entropy of pi' and the search
    value feed the same resign rule as play(), and play() with an argmax pick of the same move leaves the same state."""
    import math
    from oracle.selfplay_ref import GameLoopRef
    sp = {"resign_threshold": -0.5, "min_resign_plies": 2, "resign_window": 4, "resign_consecutive_bad": 2, "resign_min_entropy": 9.0,
          "resign_value_margin": 0.05, "temperature_start": 1e-4, "temperature_end": 1e-4}
    pi = np.zeros(4672, dtype=np.float32)
    pi[[7, 9]] = 0.5
    gum, vis = GameLoopRef(sp, {}), GameLoopRef(sp, {})
    for ply, (idx, v) in enumerate([(3, -0.9), (0, -0.9)]):
        moves = list(gum.board.legal_moves)
        assert gum.play_gumbel(moves, idx, pi, v) == idx
        counts = [0] * len(moves)
        counts[idx] = 5
        assert vis.play(moves, counts, pi, v, 0.5) == idx
        assert gum.board.fen() == vis.board.fen() and gum.entropies == vis.entropies and gum.consec_bad == vis.consec_bad
    assert gum.board.move_stack[0] == list(chess.Board().legal_moves)[3]
    assert gum.entropies[0] == pytest.approx(math.log(2.0) - 4670 * 1e-12 * math.log(1e-12), rel=1e-12)
    # third ply: two values below the threshold in a row at ply >= min_resign_plies, and a mean entropy below 9: White resigns
    assert gum.play_gumbel(list(gum.board.legal_moves), 0, pi, -0.9) is None
    assert gum.resigned and gum.z == -1.0 and gum.n_states == 3 and len(gum.board.move_stack) == 2
    assert gum.resign_checks == [(False, False, True), (True, True, True)]     # plies 2 and 3: (bad streak, stable_bad, low_unc)
