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


def test_schedule_grid_reaches_every_branch():
    """The (n, m) grid of tests/test_gumbel_edges_gpu.py against the device's halving_schedule_at, restated branch by branch: equal
    to the oracle's schedule at every grid entry, and together the entries take every branch (the grid's boards have at least m
    legal moves, so m' = m)."""
    from gumbel_cases import SCHEDULE_BRANCHES, SCHEDULE_GRID, schedule_branches
    taken = {}
    for n, m in SCHEDULE_GRID:
        T, branches = schedule_branches(m, n)
        assert T == GR.schedule(m, n), (n, m)
        for b in branches:
            taken.setdefault(b, []).append((n, m))
    assert set(taken) == SCHEDULE_BRANCHES, sorted(SCHEDULE_BRANCHES - set(taken))


def test_schedule_branches_of_known_settings():
    from gumbel_cases import schedule_branches
    assert schedule_branches(1, 4) == ([0, 1, 2, 3], {"single_candidate"})
    assert schedule_branches(2, 8)[1] == {"one_halving_level", "repeats_above_one", "clamped_to_two"}
    assert schedule_branches(16, 32)[1] == {"repeats_clamped", "repeats_above_one"}
    assert schedule_branches(7, 50)[1] == {"repeats_above_one", "odd_halving", "clamped_to_two"}
    assert schedule_branches(16, 2)[1] == {"n_below_m", "repeats_clamped"}


def _small_net_evaluator(golden_dir):
    """The golden small network through the oracle's float32 forward on the CPU, one position per call (cached)."""
    import torch
    from oracle import nn_ref
    from test_oracle_nn import load_case
    _, cfg, sd = load_case(golden_dir, "small")
    sd = {k: v.float() for k, v in sd.items()}
    cache = {}

    def evaluate(planes):
        key = planes.tobytes()
        if key not in cache:
            with torch.no_grad():
                p, v = nn_ref.forward(sd, cfg, torch.from_numpy(planes[None]))
            cache[key] = (p[0].numpy().astype(np.float32), float(v.reshape(-1)[0]))
        return cache[key]
    return evaluate


@pytest.mark.parametrize("n", [64, 200])
def test_gumbel_node_pool_bound_holds_on_edge_boards(golden_dir, n):
    """SelfPlayEngine sizes a Gumbel game's node pool as gumbel_max_nodes(n) = 1 + (n + 1) * 218.  The oracle counts the nodes it
    creates as the device allocates them: on every constructed board the count stays within the bound, each board's tree reaches
    the terminal rule it was built for, and the five-queen board outgrows the 4096 slots the visit-count sizing gave at n = 64."""
    from gumbel_cases import EDGE_BOARDS, EDGE_DRAW_SEED, EDGE_M
    from matrix0_b200.selfplay import gumbel_max_nodes
    evaluate = _small_net_evaluator(golden_dir)
    draws = np.random.default_rng(EDGE_DRAW_SEED).gumbel(size=256)
    bound = gumbel_max_nodes(n)
    assert bound == 1 + (n + 1) * 218
    for name, make, kind, min_depth in EDGE_BOARDS:
        b = make()
        out = GR.search(b.copy(), evaluate, draws, n=n, m=EDGE_M, draw_penalty=-0.05)
        assert out["nodes"] <= bound, name
        if kind is not None and n == 200:
            assert out["terminals"][kind] > 0, (name, out["terminals"])
            assert out["terminal_depth"][kind] >= min_depth, (name, out["terminal_depth"])
        if name == "five_queens" and n == 64:
            assert out["nodes"] > 4096, out["nodes"]
