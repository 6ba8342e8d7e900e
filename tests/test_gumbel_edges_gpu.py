"""Gumbel search (csrc/gumbel_kernels.cu) against the float64 oracle oracle/gumbel_ref.py where it can go wrong: every branch of the
sequential-halving schedule, constructed boards whose trees reach each terminal rule through the game history and the path
bookkeeping of gumbel_select_kernel, the node pool under its default sizing, and whole games of the Gumbel game loop
(selfplay_advance_kernel<true>, GameRecorder) against oracle/selfplay_ref.GameLoopRef.  Every search runs with the pool sizing
SelfPlayEngine chooses, and the CUDA fp32 network evaluates both sides (rows are evaluated independently)."""
import collections

import numpy as np
import pytest
import torch

import chess
from conftest import random_playout_boards
from gumbel_cases import EDGE_BOARDS, EDGE_DRAW_SEED, EDGE_M, SCHEDULE_GRID
from oracle import gumbel_ref as GR
from oracle.selfplay_ref import GameLoopRef
from test_gumbel_gpu import CONSTRUCTED, DRAW_PENALTY, _cfg, _code, _evaluator, _search
from test_selfplay_gpu import small_net

pytestmark = pytest.mark.gpu

ST_NODE_OVERFLOW = 1


def _compare_with_oracle(got, boards, draws, n, m, evaluate):
    """The assertions of test_gumbel_gpu.py per game; returns the oracle's results and the number of games excluded for a decision
    margin at rounding level."""
    refs, excluded = [], 0
    for g, b in enumerate(boards):
        ref = GR.search(b.copy(), evaluate, draws[g], n=n, m=m, draw_penalty=DRAW_PENALTY)
        refs.append(ref)
        if ref["margin"] < 1e-9:
            excluded += 1
            continue
        k = len(ref["moves"])
        assert int(got["count"][g]) == k, b.fen()
        assert got["actions"][g] == ref["actions"], b.fen()
        assert got["visits"][g, :k].tolist() == ref["visits"].tolist(), b.fen()
        assert int(got["move"][g]) == _code(ref["move"]), b.fen()
        assert np.abs(got["pi_children"][g, :k] - ref["pi_legal"]).max() <= 1e-12, b.fen()
        assert abs(float(got["value"][g]) - ref["value"]) <= 1e-12, b.fen()
        assert np.abs(got["q"][g, :k] - ref["q"]).max() <= 1e-12, b.fen()
        assert np.array_equal(got["pi"][g], ref["pi"]) or np.abs(got["pi"][g] - ref["pi"]).max() <= 1e-7, b.fen()
    return refs, excluded


@pytest.mark.parametrize("n,m", SCHEDULE_GRID)
def test_gumbel_schedule_grid_matches_oracle(golden_dir, n, m):
    """Every branch of halving_schedule_at (tests/test_gumbel_ref.py names the branch each entry takes), on middlegame boards with at
    least m legal moves and on constructed boards with fewer (m' = the legal-move count, down to 1)."""
    from matrix0_b200.selfplay import gumbel_max_nodes
    net = small_net(golden_dir)
    boards = random_playout_boards(12, 80, seed=29)[::4][:56] + [chess.Board(f) for f in CONSTRUCTED]
    legal = [b.legal_moves.count() for b in boards]
    assert sum(k >= m for k in legal) >= 40 and min(legal) == 1
    draws = np.random.default_rng(n * 1000 + m + 7).gumbel(size=(len(boards), 256))
    got = _search(net, boards, n, m, draws)
    assert got["sp"].engine.max_nodes == gumbel_max_nodes(n)
    assert int(np.abs(got["status"]).sum()) == 0
    _, excluded = _compare_with_oracle(got, boards, draws, n, m, _evaluator(net))
    print(f"schedule grid n={n} m={m}: {excluded} of {len(boards)} games excluded (oracle decision margin < 1e-9)")
    assert excluded < 0.05 * len(boards)


@pytest.mark.parametrize("n", [64, 200])
def test_gumbel_edge_boards_match_oracle(golden_dir, n):
    """Constructed boards uploaded with their move stacks (gumbel_cases.EDGE_BOARDS): many moves for both sides, few-move endgames
    with deep paths, a root whose history makes a fivefold repetition one ply away, halfmove clocks of 148 and 149, a capture to
    bare kings, mate and stalemate several plies down.  The device allocates exactly the oracle's node count, within the default
    pool, and no status bit is set; at n = 200 the oracle's tree reaches the terminal rule each board was built for."""
    from matrix0_b200.selfplay import gumbel_max_nodes
    net = small_net(golden_dir)
    boards = [make() for _, make, _, _ in EDGE_BOARDS]
    draws = np.tile(np.random.default_rng(EDGE_DRAW_SEED).gumbel(size=256), (len(boards), 1))
    got = _search(net, boards, n, EDGE_M, draws)
    eng = got["sp"].engine
    assert eng.max_nodes == gumbel_max_nodes(n)
    assert got["status"].tolist() == [0] * len(boards)       # no ST_NODE_OVERFLOW (nor any other bit)
    _, nodes = eng.status()
    refs, excluded = _compare_with_oracle(got, boards, draws, n, EDGE_M, _evaluator(net))
    assert excluded == 0
    for g, ((name, _, kind, min_depth), ref) in enumerate(zip(EDGE_BOARDS, refs)):
        assert int(nodes[g]) == ref["nodes"] <= gumbel_max_nodes(n), name
        print(f"edge n={n} {name}: {ref['nodes']} nodes, depth {ref['depth']}, terminals {ref['terminals']}")
        if kind is not None and n == 200:
            assert ref["terminals"][kind] > 0 and ref["terminal_depth"][kind] >= min_depth, (name, ref["terminals"], ref["terminal_depth"])
    if n == 64:
        assert refs[0]["nodes"] > 4096          # five_queens: more than the pool the visit-count sizing gave this setting


def test_gumbel_pool_of_visit_count_sizing_overflows_on_five_queens(golden_dir):
    """The pool the visit-count formula gave a Gumbel move at n = 64 (4096 slots) runs out on the five-queen board: the expansion
    is refused with ST_NODE_OVERFLOW and check_status() raises -- what the default pool now prevents."""
    from matrix0_b200.selfplay import SelfPlayEngine
    net = small_net(golden_dir)
    n = 64
    sp = SelfPlayEngine(net, _cfg(n, EDGE_M), games=1, deterministic=True, seed=1, precision="fp32", search_mode="gumbel", max_nodes=4096)
    eng = sp.engine
    eng.set_boards([EDGE_BOARDS[0][1]()])
    d = torch.from_numpy(np.random.default_rng(EDGE_DRAW_SEED).gumbel(size=(1, 256))).to(eng.device)
    eng.gumbel_set_draws(d)
    sp.begin_move()
    for _ in range(n):
        sp.search_step()
    st, nodes = eng.status()
    assert int(st[0]) & ST_NODE_OVERFLOW and int(nodes[0]) <= 4096
    with pytest.raises(RuntimeError, match="capacity exhausted"):
        sp.check_status()


def test_gumbel_pool_larger_than_the_device_is_refused(golden_dir):
    from matrix0_b200.selfplay import SelfPlayEngine
    net = small_net(golden_dir)
    with pytest.raises(ValueError, match="max_nodes"):
        SelfPlayEngine(net, _cfg(4096, 16), games=8192, precision="fp32", search_mode="gumbel")


# whole games: every slot plays one game; slot 0 starts from a board whose single legal move captures the last piece (a natural end)
NATURAL_END = "k7/8/8/8/8/8/1q6/K7 w - - 0 1"
# The resign settings sit inside the range the games produce (search values mostly within +-0.16, window means of the entropy of pi'
# between ~1.8 and ~2.9), so each part of the rule decides something: plies with two bad values in a row where neither window holds
# and the game goes on, resignations that only the entropy window allows, and ones that only the value window allows.
GAME_SP = {"max_game_len": 30, "resign_threshold": -0.05, "min_resign_plies": 4, "resign_window": 4, "resign_consecutive_bad": 2,
           "resign_min_entropy": 2.0, "resign_value_margin": 0.01}
GAME_DRAW = {"enabled": True, "min_plies": 8, "window": 8, "min_unique": 3, "halfmove_cap": 10, "material_draw_threshold": 0}
NATURAL_REASONS = {"checkmate", "stalemate", "insufficient_material", "fifty_moves", "repetition"}


def test_gumbel_whole_games_match_reference_loop(golden_dir):
    """48 Gumbel games (n = 16, m = 8, fp32) with fresh caller-supplied draws before every move, replayed by GameLoopRef.play_gumbel
    on the oracle's search with the same draws: per ply the move and the search value; per finished game (m0_selfplay_finished)
    the reason, result (the resigner's side for a resignation), move count and average entropy; per recorded game (GameRecorder)
    pi' of every ply and z.  The settings end games by resignation, draw adjudication, max_game_len and a rule of the game, and make
    both windows of the resign rule (mean search value, mean entropy of pi') decide whether a game resigns."""
    from matrix0_b200.records import GameRecorder
    from matrix0_b200.selfplay import SelfPlayEngine, resolve_draw_config
    net = small_net(golden_dir)
    n, m, G = 16, 8, 48
    cfg = _cfg(n, m, **GAME_SP)
    cfg["draw"] = GAME_DRAW
    sp_cfg, draw_cfg = cfg["selfplay"], resolve_draw_config(cfg)
    sp = SelfPlayEngine(net, cfg, games=G, deterministic=False, seed=19, precision="fp32", search_mode="gumbel")
    eng = sp.engine
    seen = []
    finished_games = sp.finished_games

    def spy(*a, **k):       # the recorder reads the finished-game ring; keep what it read for the comparison
        out = finished_games(*a, **k)
        seen.extend(out)
        return out
    sp.finished_games = spy
    rec = GameRecorder(sp)
    sp.start(G)
    eng.set_boards([chess.Board(NATURAL_END)], games=[0])
    loops = [GameLoopRef(sp_cfg, draw_cfg, board=chess.Board(NATURAL_END) if g == 0 else None) for g in range(G)]
    plies = {g: [] for g in range(G)}             # per slot: (oracle pi' float32, White to move) of every searched ply
    lost = set()                                  # slots whose game left the oracle's at a tie (margin < 1e-9)
    decided = collections.Counter()               # resignations by (stable_bad, low_unc) of the deciding ply
    finished_loops = []
    evaluate = _evaluator(net)
    rng = np.random.default_rng(13)
    reasons, excluded, compared_plies, compared_records = collections.Counter(), 0, 0, 0
    for ply in range(GAME_SP["max_game_len"] + 2):
        if sp.active_games() == 0:
            break
        draws = rng.gumbel(size=(G, 256))
        d = torch.from_numpy(draws).to(eng.device)
        eng.gumbel_set_draws(d)
        sp.begin_move()
        for _ in range(sp.batches_per_move()):
            sp.search_step()
        rec.after_search()
        cnt = eng.res_count.cpu().numpy()
        gmove = eng.gb_move.cpu().numpy().view(np.uint16)
        gval = eng.gb_value.cpu().numpy()
        sp.end_move()
        sp.check_status()
        played = sp.moves_played.cpu().numpy().view(np.uint16)
        n_seen = len(seen)
        records = rec.after_move()
        fin_now = seen[n_seen:]
        fin = {f["slot"]: f for f in fin_now}
        for g in range(G):
            L = loops[g]
            if L is None or g in lost:
                continue
            ref = GR.search(L.board.copy(), evaluate, draws[g], n=n, m=m, draw_penalty=DRAW_PENALTY)
            if ref["margin"] < 1e-9:              # the device may break the tie the other way: follow this game no further
                excluded += 1
                lost.add(g)
                continue
            assert int(cnt[g]) == len(ref["moves"]), (ply, g)
            assert int(gmove[g]) == _code(ref["move"]), (ply, g, L.board.fen())
            assert abs(float(gval[g]) - ref["value"]) <= 1e-12, (ply, g)
            compared_plies += 1
            plies[g].append((ref["pi"], L.board.turn == chess.WHITE))
            idx = L.play_gumbel(ref["moves"], ref["chosen"], ref["pi"], ref["value"])
            reason = "resign" if idx is None else L.ended()
            if idx is not None:
                assert int(played[g]) == int(gmove[g]), (ply, g)
            if reason is None:
                assert g not in fin, (ply, g, fin.get(g))
                continue
            f = fin[g]
            assert f["reason"] == reason and f["moves"] == L.n_states, (ply, g, f, reason, L.n_states)
            assert f["resigned"] == (reason == "resign")
            assert abs(f["result"] - np.float32(L.z)) < 1e-6, (f, L.z)
            assert abs(f["avg_policy_entropy"] - float(np.mean(L.entropies))) <= 1e-5 * max(1.0, float(np.mean(L.entropies))), (f, L.entropies)
            reasons[reason] += 1
            if reason == "resign":
                _, stable_bad, low_unc = L.resign_checks[-1]
                decided[(stable_bad, low_unc)] += 1
            finished_loops.append(L)
            loops[g] = None                       # the start budget is spent: the slot goes idle
        assert len(records) == len(fin_now)       # every game searched at least one ply, delivered in ring order
        for f, gd in zip(fin_now, records):
            g = f["slot"]
            if g in lost:
                continue
            want = plies[g]
            assert int(gd["meta_moves"][0]) == len(want) == f["moves"]
            pi = np.stack([p for p, _ in want])
            assert np.array_equal(gd["pi"], pi) or np.abs(gd["pi"] - pi).max() <= 1e-7, g
            z = np.float32(f["result"])
            assert gd["z"].tolist() == [float(z if white else -z) for _, white in want], g
            compared_records += 1
    assert sp.active_games() == 0
    print(f"whole games: {dict(reasons)}; {compared_plies} plies and {compared_records} records compared; {excluded} plies at a tie, "
          f"{len(lost)} games left the oracle's")
    assert len(lost) <= 2
    # the resign rule's windows decided outcomes the comparison above checks: a streak of bad values that both windows vetoed, a
    # resignation only the entropy window allowed and one only the value window allowed
    vetoed = sum(streak and not (sb or lu) for L in finished_loops for streak, sb, lu in L.resign_checks)
    print(f"resign rule: {vetoed} plies with a bad streak vetoed by both windows; resignations by (stable_bad, low_unc): {dict(decided)}")
    assert vetoed > 0 and decided[(False, True)] > 0 and decided[(True, False)] > 0, (vetoed, decided)
    assert reasons["resign"] and reasons["draw_adjudicated"] and reasons["max_game_len"] and NATURAL_REASONS & set(reasons), reasons
