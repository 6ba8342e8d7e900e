"""GPU parity of the search: matrix0_b200.mcts.MCTS (CUDA tree kernels through the C ABI) fed the
same evaluator outputs as the reference.  Bar (BASELINE north_star): visit counts bit-exact with
noise off and deterministic tie-break; root value, child Q (fp64 sequential backups) bit-exact;
priors within 1e-6 relative (float32 softmax: CUDA expf vs torch CPU exp differ by <= 2 ulp, the
same tolerance the reference's own prior test uses, tests/test_mcts_logits.py:32-79)."""
import numpy as np
import pytest

import chess
from mcts_cases import run_all
from oracle.backends import ConstantBackend, HashBackend
from oracle.mcts_ref import RefConfig, RefMCTS

pytestmark = pytest.mark.gpu


def make_gpu(cfg, backend, sims):
    from matrix0_b200.mcts import MCTS, MCTSConfig
    c = MCTSConfig(num_threads=1, enable_memory_cleanup=False, dirichlet_frac=0.0, enable_entropy_noise=False,
                   playout_random_frac=0.0, num_simulations=sims, **cfg)
    return MCTS(c, None, device="cuda", inference_backend=backend, deterministic=True, max_nodes=32768)


def test_reference_goldens_fresh():
    assert run_all(make_gpu, prior_rtol=1e-6, kinds=("fresh", "game_fresh")) >= 50


def test_reference_goldens_tree_reuse():
    """Persistent instances: tree reuse through the TT, including the reference's zero-visit failure."""
    assert run_all(make_gpu, prior_rtol=1e-6, kinds=("persistent", "alternating")) >= 20


def test_live_vs_oracle_random_positions():
    from conftest import random_playout_boards
    kw = dict(cpuct_start=3.0, cpuct_end=2.0, cpuct_plies=40, fpu_reduction=0.1, draw_penalty=-0.05, legal_softmax=True,
              selection_jitter=0.05, inference_batch_size=96)
    boards = random_playout_boards(10, 150, seed=2024)[::9][:24]
    for i, b in enumerate(boards):
        m_gpu = make_gpu(kw, HashBackend(1.0, seed=100 + i), 400)
        m_ref = RefMCTS(RefConfig(dirichlet_frac=0.0, enable_entropy_noise=False, num_simulations=400, **kw), HashBackend(1.0, seed=100 + i))
        vc1, pi1, v1 = m_gpu.run(b, ply=5)
        vc2, pi2, v2 = m_ref.run(b.copy(), ply=5)
        assert [(m.uci(), n) for m, n in vc1.items()] == [(m.uci(), n) for m, n in vc2.items()], b.fen()
        assert pi1.tobytes() == pi2.tobytes() and v1 == v2, b.fen()


def test_api_surface():
    """reference tests/test_integration.py:196-237 + test_error_handling.py:140-155 + test_mcts_logits.py."""
    from matrix0_b200.mcts import MCTS, MCTSConfig
    cfg = MCTSConfig.from_dict({"num_simulations": 50, "cpuct": 1.5, "bogus_key": 1, "legal_softmax": True})
    m = MCTS(cfg, None, device="cpu", inference_backend=ConstantBackend(0.25), deterministic=True)
    vc, pi, v = m.run(chess.Board())
    assert isinstance(vc, dict) and pi.shape == (4672,) and pi.dtype == np.float32 and isinstance(v, float)
    assert 0.9 <= pi.sum() <= 1.1 and -1.0 <= v <= 1.0 and sum(vc.values()) == 50
    assert m._last_sims_run == 50 and m._last_root is not None
    # (model, cfg) argument order and terminal root
    m2 = MCTS(None, cfg, inference_backend=ConstantBackend(0.0), deterministic=True)
    vc, pi, v = m2.run(chess.Board("rnb1kbnr/pppp1ppp/8/4p3/6Pq/5P2/PPPPP2P/RNBQKBNR w KQkq - 1 3"))
    assert vc == {} and not pi.any() and v == -1.0
    # priors == softmax(logits[legal_idx]) in legal-move order (reference tests/test_mcts_logits.py:32-79)
    rs = np.random.RandomState(0)
    logits = rs.standard_normal(4672).astype(np.float32)

    class Fixed:
        def infer_np(self, x):
            n = 1 if np.asarray(x).ndim == 3 else len(x)
            return np.repeat(logits[None], n, 0), np.zeros(n, np.float32)
    for legal_only in (True, False):
        mm = MCTS(MCTSConfig(num_simulations=1, legal_softmax=legal_only), None, inference_backend=Fixed(), deterministic=True)
        b = chess.Board()
        mm.run(b)
        from oracle.encoding_ref import legal_moves_and_indices
        idx = [i for _, i in legal_moves_and_indices(b)]
        import torch
        if legal_only:
            exp = torch.softmax(torch.from_numpy(logits[idx]), -1).numpy()
        else:
            exp = torch.softmax(torch.from_numpy(logits), -1).numpy()[idx]
            exp = exp / exp.sum()
        got = [c.prior for c in mm._last_root.children.values()]
        np.testing.assert_allclose(got, exp, rtol=1e-6, atol=1e-6)
    m.reset()
    assert m.get_memory_usage()["simulations_run"] == 0
    m.shutdown()


def test_root_children_follow_python_chess_order_on_edge_positions():
    """The warp-cooperative ordered move generator inside the tree kernels (csrc/movegen_warp.cuh; its lanes are simulated on the host
    by tests/test_hostcheck.py): root children of constructed edge positions -- kingless boards and several kings take the single-lane
    fallback, checks / double checks / pins / en passant / promotions / castling the one-piece-per-lane path -- and of 600 playout
    positions come out in list(board.legal_moves) order."""
    import torch
    from matrix0_b200.engine import SearchEngine
    from matrix0_b200.mcts import MCTSConfig
    from conftest import random_playout_boards
    from oracle.encoding_ref import legal_moves_and_indices
    from test_hostcheck import WEIRD_FENS
    boards = [chess.Board(f) for f in WEIRD_FENS] + random_playout_boards(12, 160, seed=5)[:600]
    G = len(boards)
    eng = SearchEngine(G, max_nodes=512, tt_capacity=1024, max_depth=16, hist_cap=4)
    eng.configure(MCTSConfig(num_simulations=1, legal_softmax=True, enable_entropy_noise=False), deterministic=True)
    eng.set_boards(boards, with_history=False)
    eng.begin()
    info = eng.info.cpu().numpy()
    eng.expand_backup(torch.zeros((G, 4672), dtype=torch.float32, device="cuda"), torch.zeros((G,), dtype=torch.float32, device="cuda"))
    eng.result(with_pi=False)
    cnt, mv = eng.res_count.cpu().numpy(), eng.res_moves.cpu().numpy().view(np.uint16)
    checked = 0
    for g, b in enumerate(boards):
        exp = [c for c, _ in legal_moves_and_indices(b)]
        if info[g] & 1:                      # terminal root: nothing expanded
            assert b.is_game_over() or not exp, b.fen()
            continue
        assert [int(x) for x in mv[g, :int(cnt[g])]] == exp[:256], b.fen()
        checked += 1
    assert checked > 500
    eng.close()


def test_configs0_single_game_through_the_dropin_search_object():
    """BASELINE configs[0] on the GPU: ONE game from the start position, 800 simulations per move, ResNet-24 random init, searched by
    `MCTS(cfg, model, device="cuda").run(board)` move after move -- the call `selfplay_worker` / `arena.py` / `cli_play.py` of the reference
    make (one board per call, host dictionaries back).  The latency case: ten evaluator calls of <= 96 rows per move and nothing to batch
    across games.  The numbers are printed as one JSON line (shown with `pytest -s`); the assertion is only a floor well above the
    reference's CPU rate on the same configuration (65 ... 450 sims/s, `bench.py --impl reference`)."""
    import json
    import time
    import torch
    from bench_selfplay import reference_cfg
    from matrix0_b200.mcts import MCTS, MCTSConfig
    from matrix0_b200.model import PolicyValueNet
    cfg = reference_cfg(800)
    net = PolicyValueNet.from_config(cfg["model"], device="cuda:0", precision="fp16", seed=0)
    out = {"workload": "BASELINE configs[0]: one game from the start position, 800 sims/move, ResNet-24 fp16 random init, MCTS.run per move"}
    for name, det in (("as_shipped", False), ("deterministic", True)):
        mcts = MCTS(MCTSConfig.from_dict(cfg["mcts"]), net, device="cuda", deterministic=det, seed=1234)
        board = chess.Board()
        for _ in range(2):                      # warm-up: workspaces, first launches, the evaluator's CUDA graphs
            mcts.reset()
            mcts.run(board, ply=0)
        per_move, sims = [], 0
        for ply in range(8):
            torch.cuda.synchronize()
            t = time.perf_counter()
            mcts.reset()                        # a fresh tree per move: the only working reading of the reference (DESIGN.md Q12 -- with
            visits, pi, v = mcts.run(board, ply=ply)   # a persistent object its second move raises "zero visits", and so does ours)
            torch.cuda.synchronize()
            per_move.append((time.perf_counter() - t) * 1e3)
            sims += int(mcts._last_sims_run)
            assert visits and abs(float(pi.sum()) - 1.0) < 1e-4 and -1.0 <= v <= 1.0
            board.push(max(visits.items(), key=lambda kv: kv[1])[0])
        total = sum(per_move) * 1e-3
        out[name] = {"moves": len(per_move), "ms_per_move": per_move, "ms_per_move_median": sorted(per_move)[len(per_move) // 2], "sims": sims,
                     "sims_per_s": sims / total, "positions_per_s": len(per_move) / total}
        mcts.shutdown()
        assert sims / total > 2000.0, out[name]
    print(json.dumps(out))
