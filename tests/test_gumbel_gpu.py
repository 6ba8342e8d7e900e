"""Gumbel AlphaZero search on the GPU (csrc/gumbel_kernels.cu, SelfPlayEngine(search_mode="gumbel")) against the float64 oracle
oracle/gumbel_ref.py, fed by the same CUDA fp32 network (rows are evaluated independently), and its invariants in self-play."""
import numpy as np
import pytest
import torch

import chess
from conftest import random_playout_boards
from oracle import gumbel_ref as GR
from test_selfplay_gpu import MCTS_KW, small_net

pytestmark = pytest.mark.gpu

DRAW_PENALTY = -0.05

CONSTRUCTED = [
    "6k1/5ppp/8/8/8/8/5PPP/3R2K1 w - - 0 1",      # mate in one (a terminal root child)
    "3r2k1/5ppp/8/8/8/8/5PPP/6K1 b - - 0 1",      # mate in one, Black to move
    "7k/8/5Q2/8/8/8/8/K7 w - - 0 1",              # stalemate trap: Qg6 stalemates (a terminal child worth the draw penalty)
    "k7/8/8/8/8/8/1q6/K7 w - - 0 1",              # a single legal move
    "8/P6k/8/8/8/8/6p1/K7 w - - 0 1",             # promotions (and under-promotions) on both sides
    "1n2k3/P7/8/8/8/8/6p1/4K2R b K - 0 1",        # promotions with captures, castling rights
]


def _cfg(n, m, **sp):
    return {"mcts": dict(MCTS_KW, num_simulations=n, draw_penalty=DRAW_PENALTY),
            "selfplay": {"num_simulations": n, "opening_random_plies": 0, **sp},
            "gumbel": {"num_simulations": n, "max_considered_actions": m}}


def _search(net, boards, n, m, draws, precision="fp32"):
    """One Gumbel move on `boards` with caller-supplied draws; returns per game the root action sequence and the result arrays."""
    from matrix0_b200.selfplay import SelfPlayEngine
    G = len(boards)
    sp = SelfPlayEngine(net, _cfg(n, m), games=G, deterministic=True, seed=1, precision=precision, search_mode="gumbel")
    eng = sp.engine
    eng.set_boards(boards)
    d = torch.from_numpy(np.ascontiguousarray(draws, dtype=np.float64)).to(eng.device)
    eng.gumbel_set_draws(d)
    sp.begin_move()
    prev = np.zeros((G, 256), dtype=np.int64)
    actions = [[] for _ in range(G)]
    for _ in range(n):
        sp.search_step()
        eng.gumbel_result(with_pi=False)
        vis = eng.res_visits.cpu().numpy().astype(np.int64)
        for g in range(G):
            diff = np.nonzero(vis[g] != prev[g])[0]
            if len(diff):
                actions[g].append(int(diff[0]))
        prev = vis
    sp.gumbel_result(with_pi=True)
    st, _ = eng.status()
    out = {"actions": actions, "visits": eng.res_visits.cpu().numpy(), "q": eng.res_q.cpu().numpy(), "count": eng.res_count.cpu().numpy(),
           "pi_children": eng.gb_pi_children.cpu().numpy(), "pi": eng.res_pi.cpu().numpy(), "value": eng.gb_value.cpu().numpy(),
           "move": eng.gb_move.cpu().numpy().view(np.uint16), "status": st.cpu().numpy(), "sp": sp}
    return out


def _evaluator(net):
    cache = {}

    def evaluate(planes):
        key = planes.tobytes()
        if key not in cache:
            lg, v = net.infer_np(planes[None])
            cache[key] = (lg[0].copy(), float(v.reshape(-1)[0]))
        return cache[key]
    return evaluate


def _code(mv):
    return mv.from_square | (mv.to_square << 6) | ((mv.promotion or 0) << 12)


@pytest.mark.parametrize("n,m", [(16, 16), (32, 16), (32, 256)])
def test_gumbel_search_matches_oracle_per_game(golden_dir, n, m):
    net = small_net(golden_dir)
    boards = random_playout_boards(12, 80, seed=23)[::4][:56] + [chess.Board(f) for f in CONSTRUCTED]
    assert len(boards) >= 54
    draws = np.random.default_rng(n * 1000 + m).gumbel(size=(len(boards), 256))
    got = _search(net, boards, n, m, draws)
    assert int(np.abs(got["status"]).sum()) == 0
    evaluate = _evaluator(net)
    excluded = 0
    for g, b in enumerate(boards):
        ref = GR.search(b.copy(), evaluate, draws[g], n=n, m=m, draw_penalty=DRAW_PENALTY)
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
    print(f"n={n} m={m}: {excluded} of {len(boards)} games excluded (oracle decision margin < 1e-9)")
    assert excluded < 0.05 * len(boards)


def _final_counts(m, n):
    visits = [0] * m
    for t in GR.schedule(m, n):
        visits[visits.index(t)] += 1
    return sorted(visits, reverse=True)


def test_gumbel_invariants_with_device_draws(golden_dir):
    from matrix0_b200 import encoding
    net = small_net(golden_dir)
    n, m = 32, 16
    boards = random_playout_boards(40, 120, seed=5)
    boards = [boards[i] for i in np.random.default_rng(1).choice(len(boards), 512, replace=False)]
    from matrix0_b200.selfplay import SelfPlayEngine
    sp = SelfPlayEngine(net, _cfg(n, m), games=512, deterministic=False, seed=11, precision="fp32", search_mode="gumbel")
    eng = sp.engine
    eng.set_boards(boards)
    sp.begin_move()
    for _ in range(sp.batches_per_move()):
        sp.search_step()
    sp.gumbel_result(with_pi=True)
    vis = eng.res_visits.cpu().numpy()
    cnt = eng.res_count.cpu().numpy()
    pi = eng.res_pi.cpu().numpy().astype(np.float64)
    mv = eng.gb_move.cpu().numpy().view(np.uint16)
    st, _ = eng.status()
    assert int(st.abs().sum()) == 0
    _, mask = encoding.encode_boards(boards)
    full = _final_counts(m, n)
    for g, b in enumerate(boards):
        k = int(cnt[g])
        legal = list(b.legal_moves)
        assert k == len(legal)
        v = vis[g, :k]
        assert int(v.sum()) == n
        if k >= m:
            assert sorted(v.tolist(), reverse=True)[:m] == full and int((v > 0).sum()) == m
        assert abs(pi[g].sum() - 1.0) <= 1e-6
        assert (pi[g][~mask[g].astype(bool)] == 0).all()
        j = [_code(x) for x in legal].index(int(mv[g]))
        assert v[j] == v.max()


def test_gumbel_batch_independence(golden_dir):
    net = small_net(golden_dir)
    n, m = 32, 16
    boards = random_playout_boards(8, 60, seed=31)[:64]
    assert len(boards) == 64
    draws = np.random.default_rng(4).gumbel(size=(64, 256))
    many = _search(net, boards, n, m, draws)
    for g in (0, 17, 63):
        one = _search(net, [boards[g]], n, m, draws[g:g + 1])
        assert one["actions"][0] == many["actions"][g]
        for key in ("visits", "q", "pi_children", "pi", "value", "move"):
            assert one[key][0].tobytes() == many[key][g].tobytes(), key


def _play_fp16(golden_dir, seed):
    from matrix0_b200.selfplay import SelfPlayEngine
    net = small_net(golden_dir, precision="fp16")
    cfg = _cfg(16, 8, opening_random_plies=4, max_game_len=12, resign_threshold=-0.9, min_resign_plies=4)
    sp = SelfPlayEngine(net, cfg, games=64, deterministic=False, seed=seed, precision="fp16", cuda_graph=True,
                        search_mode="gumbel")
    sp.start()
    moves = []
    for _ in range(14):
        sp.play_move()
        moves.append(sp.moves_played.cpu().numpy().copy())
    fin = sp.finished_games()
    sp.check_status()
    assert sp.graph_replays > 0
    # the finished-game ring is filled in the order the slots' warps finish: compare it as a set
    return np.stack(moves), sorted((f["slot"], f["moves"], f["result"], f["reason"], f["avg_policy_entropy"]) for f in fin)


def test_gumbel_fp16_graph_replay_is_reproducible(golden_dir):
    a = _play_fp16(golden_dir, 77)
    b = _play_fp16(golden_dir, 77)
    assert np.array_equal(a[0], b[0])
    assert a[1] == b[1] and len(a[1]) >= 64


def test_selfplay_worker_gumbel_writes_shards(golden_dir, tmp_path):
    import queue
    from matrix0_b200.selfplay import selfplay_worker
    from test_oracle_nn import load_case
    g, ncfg, sd = load_case(golden_dir, "small")
    ckpt = tmp_path / "ckpt.pt"
    torch.save({"model": sd}, ckpt)
    n = 16
    cfg = {"model": {k: getattr(ncfg, k) for k in ncfg.__dataclass_fields__}, "data_dir": str(tmp_path / "data"), "seed": 3,
           "mcts": dict(MCTS_KW, num_simulations=64, inference_batch_size=16),
           "selfplay": {"num_simulations": 64, "opening_random_plies": 4, "max_game_len": 10, "resign_threshold": -0.85, "min_resign_plies": 50},
           "gumbel": {"num_simulations": n, "max_considered_actions": 8}}
    q = queue.Queue()
    assert selfplay_worker(0, cfg, str(ckpt), games=10, q=q, concurrent_games=8, precision="fp32", search_mode="gumbel") == 10
    files = sorted((tmp_path / "data" / "selfplay").glob("selfplay_w0_g*.npz"))
    assert len(files) == 10
    msgs = []
    while not q.empty():
        msgs.append(q.get())
    game_msgs = [m for m in msgs if m["type"] == "game"]
    assert len(game_msgs) == 10
    assert set(game_msgs[0]) == {"type", "proc", "file", "moves", "result", "secs", "resigned", "resigner", "draw", "avg_policy_entropy",
                                 "avg_ms_per_move", "avg_sims"}
    for f in files:
        with np.load(f) as d:
            T = int(d["meta_moves"][0])
            assert d["s"].shape == (T, 19, 8, 8) and d["pi"].shape == (T, 4672) and d["pi"].dtype == np.float32
            mask = d["legal_mask"].astype(bool)
            pi = d["pi"].astype(np.float64)
            assert (pi[~mask] == 0).all()
            assert np.abs(pi.sum(1) - 1.0).max() <= 1e-6
            assert float(d["meta_avg_sims"][0]) == n
            assert 0.0 < float(d["meta_avg_policy_entropy"][0])
    for m in game_msgs:
        assert m["avg_sims"] == n and m["moves"] <= 10
