"""The Gumbel AlphaZero oracle (oracle/gumbel_ref.py) against hand-checked values of DESIGN.md §9: the sequential-halving visit
schedule, v_mix / Q~ / sigma, a single legal move, and mate-in-one positions under a uniform evaluator (the negamax sign)."""
import numpy as np
import pytest

import chess
from oracle import gumbel_ref as GR


def uniform(planes):
    return np.zeros(4672, dtype=np.float32), 0.0


SCHEDULES = [
    (4, 8, [0, 0, 0, 0, 1, 1, 2, 2], [3, 3, 1, 1]),
    (5, 12, [0, 0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4], [5, 4, 1, 1, 1]),
    (16, 32, [0] * 16 + [1] * 8 + [2] * 4 + [3] * 4, [4, 4, 4, 4, 2, 2, 2, 2] + [1] * 8),
    (2, 8, [0, 0, 1, 1, 2, 2, 3, 3], [4, 4]),
    (1, 4, [0, 1, 2, 3], [4]),
]


@pytest.mark.parametrize("m,n,seq,final", SCHEDULES)
def test_schedule_and_final_root_visits(m, n, seq, final):
    assert GR.schedule(m, n) == seq
    # the start position has 20 legal moves (>= m): the search's sorted final root visits are the schedule's final counts
    draws = np.random.default_rng(m * 100 + n).gumbel(size=256)
    out = GR.search(chess.Board(), uniform, draws, n=n, m=m)
    visits = sorted((int(v) for v in out["visits"] if v > 0), reverse=True)
    assert visits == final
    assert int(out["visits"].sum()) == n
    assert [int(out["visits"][a] > 0) for a in range(len(out["moves"]))].count(1) == len(final)


def test_sigma_no_visits_and_equal_q_floor():
    # Nc = 0: v_mix = r, every Q^ equal -> the 1e-8 floor makes Q~ = 0 and sigma = 0
    s, v_mix, qt = GR.sigma([0.0, np.log(3.0)], [0, 0], [0.0, 0.0], 0.4, 50.0, 0.1)
    assert v_mix == 0.4
    assert qt.tolist() == [0.0, 0.0] and s.tolist() == [0.0, 0.0]
    # all moves visited with the same q: again Q~ = 0
    s, v_mix, qt = GR.sigma([0.0, 1.0], [1, 1], [-0.3, -0.3], 0.1, 50.0, 0.1)
    assert qt.tolist() == [0.0, 0.0] and s.tolist() == [0.0, 0.0]


def test_sigma_all_visited():
    # p = (1/4, 3/4); q = -W/N = (-0.5, 0.3); v_mix = (0.4 + 4 * 0.1) / 5 = 0.16; Q~ = (0, 1); sigma = (50 + 3) * 0.1 * Q~
    s, v_mix, qt = GR.sigma([0.0, np.log(3.0)], [1, 3], [0.5, -0.9], 0.4, 50.0, 0.1)
    assert v_mix == pytest.approx(0.16, abs=1e-15)
    assert qt == pytest.approx([0.0, 1.0], abs=1e-15)
    assert s == pytest.approx([0.0, 5.3], abs=1e-14)


def test_sigma_partly_visited():
    # p = 1/3 each, only move 0 visited (N = 2, q = 0.5): v_mix = (-0.2 + 2 * 0.5) / 3; Q^ = (0.5, v_mix, v_mix) -> Q~ = (1, 0, 0)
    s, v_mix, qt = GR.sigma([0.0, 0.0, 0.0], [2, 0, 0], [-1.0, 0.0, 0.0], -0.2, 50.0, 0.1)
    assert v_mix == pytest.approx(0.8 / 3, abs=1e-15)
    assert qt == pytest.approx([1.0, 0.0, 0.0], abs=1e-15)
    assert s == pytest.approx([5.2, 0.0, 0.0], abs=1e-14)
    # c_visit / c_scale enter as (c_visit + max N) * c_scale
    s2, _, _ = GR.sigma([0.0, 0.0, 0.0], [2, 0, 0], [-1.0, 0.0, 0.0], -0.2, 10.0, 0.5)
    assert s2 == pytest.approx([6.0, 0.0, 0.0], abs=1e-14)


def test_single_legal_move():
    b = chess.Board("k7/8/8/8/8/8/1q6/K7 w - - 0 1")
    assert len(list(b.legal_moves)) == 1
    out = GR.search(b, uniform, np.zeros(256), n=8, m=16)
    assert str(out["move"]) == "a1b2"
    assert out["pi_legal"].tolist() == [1.0]
    assert out["actions"] == [0] * 8 and out["visits"].tolist() == [8]


@pytest.mark.parametrize("fen", ["6k1/5ppp/8/8/8/8/5PPP/3R2K1 w - - 0 1", "3r2k1/5ppp/8/8/8/8/5PPP/6K1 b - - 0 1"])
def test_mate_in_one_under_uniform_evaluator(fen):
    b = chess.Board(fen)
    k = len(list(b.legal_moves))
    for seed in range(4):
        draws = np.random.default_rng(seed).gumbel(size=256)
        out = GR.search(b, uniform, draws, n=2 * k, m=k)
        mates = []
        for mv in out["moves"]:
            c = b.copy()
            c.push(mv)
            mates.append(c.is_checkmate())
        assert mates[out["chosen"]], (fen, seed, str(out["move"]))
        assert mates[int(np.argmax(out["pi_legal"]))]
        assert out["q"][out["chosen"]] == 1.0      # the mated side's -1, seen from the root


def test_policy_target_is_stored_at_policy_indices():
    b = chess.Board()
    out = GR.search(b, uniform, np.random.default_rng(5).gumbel(size=256), n=16, m=8)
    from oracle.encoding_ref import get_legal_actions
    mask = get_legal_actions(b)
    assert (out["pi"][~mask] == 0).all()
    assert abs(float(out["pi"].astype(np.float64).sum()) - 1.0) < 1e-6
    assert out["value"] == 0.0 and out["margin"] >= 0.0


def test_gumbel_config_is_validated():
    from matrix0_b200.selfplay import resolve_gumbel_config
    assert resolve_gumbel_config({}) == {"num_simulations": 32, "max_considered_actions": 16, "maxvisit_init": 50.0, "value_scale": 0.1}
    for bad in ({"num_simulations": 0}, {"num_simulations": 5000}, {"max_considered_actions": 0}, {"max_considered_actions": 257},
                {"maxvisit_init": -1.0}, {"value_scale": 0.0}, {"value_scale": float("nan")}, {"num_simulations": 1.5}, {"bogus": 1}):
        with pytest.raises(ValueError):
            resolve_gumbel_config({"gumbel": bad})
