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
