"""Golden vectors for the search AS SHIPPED: the UNMODIFIED reference ``MCTS.run`` with ``selection_jitter`` in force
(per-child per-simulation ``random.random()``, mcts.py:893-897), entropy noise (``np.random.normal(0, 0.1)``, :170-186), child
pruning (:806-826) and the direct-model path (:697-703), fed SEEDED streams of random draws.

Needs the unmodified reference tree (oracle/_ref or MATRIX0_REFERENCE_ROOT):  python tests/golden/make_stochastic_golden.py
Output: tests/golden/mcts_stochastic_golden.json
        python tests/golden/make_stochastic_golden.py vl   ->  tests/golden/mcts_vl_golden.json: the same with the reference's
        in-flight marking switched ON inside every mini-batch (the engine's throughput mode).  The reference ships that code in
        ``MCTS._select`` (inflight_counts, mcts.py:889-890, :922-923) but ``_collect_leaf_position`` never passes the dict (:745); the
        generator subclasses the reference ``MCTS`` and overrides ONLY ``_collect_leaf_position`` to pass one dict per mini-batch, so the
        selection itself is still the unmodified ``_select``.

Streams (the GPU test regenerates them from the seeds): jitter = ``random.Random(seed).random()`` values, normal =
``np.random.RandomState(seed).normal(0, 0.1, n)``; the generator patches ``random.random`` / ``np.random.normal`` of the reference
to read them in order.  Every case is also run through oracle/mcts_ref.RefMCTS with the same streams and must agree exactly
(this pins the oracle's stochastic path); the oracle additionally reports the smallest top-2 PUCT score gap of the run.  float32
softmax priors differ by <= 2 ulp between torch CPU and CUDA ``expf`` (the tolerance of the reference's own prior test), which moves
scores by <= ~1e-7; candidate cases with a gap below ``MIN_GAP`` somewhere are therefore dropped, except the zero-logit cases
(softmax of equal logits is exact on both sides) which are kept unconditionally.
"""
from __future__ import annotations

import json
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import refload  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
MIN_GAP = 2e-6
N_JITTER, N_NORMAL = 600_000, 600_000

CFGS = {
    # config.yaml as self-play resolves it (SURVEY 8, "effective configuration")
    "selfplay": dict(cpuct=2.5, cpuct_start=3.0, cpuct_end=2.0, cpuct_plies=40, fpu_reduction=0.1, draw_penalty=-0.05, legal_softmax=True,
                     selection_jitter=0.05, inference_batch_size=96, no_instant_backtrack=True, enable_entropy_noise=True),
    "selfplay_b32": dict(cpuct=2.5, cpuct_start=3.0, cpuct_end=2.0, cpuct_plies=40, fpu_reduction=0.1, draw_penalty=-0.05, legal_softmax=True,
                         selection_jitter=0.05, inference_batch_size=32, no_instant_backtrack=True, enable_entropy_noise=True),
    # arena / tools: selection_jitter 0.0 -> the +-0.0005 branch (SURVEY Q2b); full-policy softmax, no entropy noise
    "arena_full": dict(cpuct=1.7, fpu_reduction=0.15, legal_softmax=False, selection_jitter=0.0, inference_batch_size=16,
                       enable_entropy_noise=False),
    # pruning on (mcts.py:806-826)
    "prune": dict(cpuct_c_base=19652.0, cpuct_c_init=1.25, fpu_reduction=0.2, legal_softmax=True, selection_jitter=0.02,
                  inference_batch_size=24, no_instant_backtrack=False, draw_penalty=-0.3, enable_entropy_noise=True,
                  max_children=7, min_child_prior=0.012),
    # MCTSConfig's own defaults: full-policy softmax WITH entropy noise -- N(0, 0.1) on all 4672 entries (mcts.py:164-186)
    "default_full": dict(cpuct=2.5, fpu_reduction=0.15, draw_penalty=-0.1, legal_softmax=False, selection_jitter=0.01, inference_batch_size=16,
                         enable_entropy_noise=True),
    # the reference without an inference backend: raw-logit priors below the root (SURVEY Q3)
    "direct": dict(cpuct=2.0, fpu_reduction=0.1, legal_softmax=True, selection_jitter=0.05, inference_batch_size=48, enable_entropy_noise=True),
}
FENS = [
    "rnbqkbnr/pppppppp/8/8/8/8/PPPPPPPP/RNBQKBNR w KQkq - 0 1",
    "r3k2r/p1ppqpb1/bn2pnp1/3PN3/1p2P3/2N2Q1p/PPPBBPPP/R3K2R w KQkq - 0 1",
    "8/2p5/3p4/KP5r/1R3p1k/8/4P1P1/8 w - - 0 1",
    "6k1/5ppp/8/8/8/8/5PPP/3R2K1 w - - 0 1",          # mate in one available: terminal leaves inside a batch
    "4k3/8/8/8/8/8/8/4K2R w K - 148 90",              # 75-move rule two plies away
    "r4rk1/1pp1qppp/p1np1n2/2b1p1B1/2B1P1b1/P1NP1N2/1PP1QPPP/R4RK1 w - - 0 10",
]


class Stream:
    def __init__(self, arr):
        self.a, self.i = arr, 0

    def next(self):
        self.i += 1
        return float(self.a[self.i - 1])

    def take(self, shape):
        n = int(np.prod(shape))
        self.i += n
        return np.asarray(self.a[self.i - n:self.i], dtype=np.float64).reshape(shape)


def streams(seed):
    rj = random.Random(seed)
    return (np.array([rj.random() for _ in range(N_JITTER)], dtype=np.float64),
            np.random.RandomState(seed).normal(0, 0.1, N_NORMAL))


def main():
    import logging
    import torch
    logging.disable(logging.CRITICAL)
    VL = len(sys.argv) > 1 and sys.argv[1] == "vl"
    ref = refload.load_reference("mcts")
    import chess
    from oracle.backends import HashBackend
    from oracle.mcts_ref import RefConfig, RefMCTS
    ref.psutil_available = False
    real_random, real_normal = random.random, np.random.normal

    class _Model:
        class cfg:
            policy_size = 4672

    class TorchBackendModel(torch.nn.Module):
        """The direct-model seam (mcts.py:679-686): a torch module whose forward evaluates the hash backend."""

        def __init__(self, be):
            super().__init__()
            self.be = be

            class cfg:
                policy_size = 4672
            self.cfg = cfg

        def forward(self, x):
            p, v = self.be.infer_np(x.numpy())
            return torch.from_numpy(p), torch.from_numpy(v)

    class VirtualLossMCTS(ref.MCTS):
        """Reference MCTS whose mini-batches call the UNMODIFIED _select with an inflight_counts dict (one per mini-batch)."""

        def _collect_leaf_position(self, board, root, leaf_samples, append_lock):
            if getattr(self, "_vl_list", None) is not leaf_samples:     # a new leaf_samples list = a new mini-batch (mcts.py:538)
                self._vl_list, self._vl = leaf_samples, {}
            node, path, leaf_board = self._select(board, root, self._vl)
            if leaf_board.is_game_over():                                 # mcts.py:747-751
                self._backpropagate(path, self._terminal_value(leaf_board))
                return
            leaf_samples.append({"board": leaf_board, "node": node, "path": list(path)})

    MCTSClass = VirtualLossMCTS if VL else ref.MCTS
    rng = random.Random(99)
    boards = [(f, []) for f in FENS]
    for _ in range(14):     # positions along random playouts (with their move stacks: repetition history)
        b = chess.Board()
        for _ in range(rng.randint(4, 90)):
            if b.is_game_over():
                break
            b.push(rng.choice(list(b.legal_moves)))
        if not b.is_game_over():
            boards.append((chess.STARTING_FEN, [m.uci() for m in b.move_stack]))

    plan = []
    if VL:
        CFGS["selfplay_vl"] = dict(CFGS["selfplay"], virtual_loss=1.0)
        CFGS["vl_small"] = dict(CFGS["selfplay_b32"], virtual_loss=0.3, enable_entropy_noise=False)
        for i, (fen, moves) in enumerate(boards):
            plan.append(("selfplay_vl", ("hash", 0.0 if i % 3 == 0 else 1.0, 700 + i), 300, fen, moves))
            if i % 2 == 1:
                plan.append(("vl_small", ("hash", 1.0, 800 + i), 160, fen, moves))
        boards = []
    for i, (fen, moves) in enumerate(boards):
        plan.append(("selfplay", ("hash", 0.0, 100 + i), 300, fen, moves))          # exact priors, noise on every expansion
        plan.append(("selfplay", ("hash", 0.02, 200 + i), 400, fen, moves))         # random-init-like logits
        if i % 2 == 0:
            plan.append(("selfplay_b32", ("hash", 1.0, 300 + i), 200, fen, moves))  # trained-like logits: entropy test both ways
        if i % 3 == 0:
            plan.append(("arena_full", ("hash", 1.5, 400 + i), 150, fen, moves))
            plan.append(("prune", ("hash", 1.0, 500 + i), 150, fen, moves))
        if i % 4 == 1:
            plan.append(("direct", ("hash", 1.0, 600 + i), 150, fen, moves))
    if not VL:   # appended last so that the seeds of the earlier cases stay what they were
        for i in (0, 2, 5, 9, 13):
            fen, moves = boards[i]
            plan.append(("default_full", ("hash", 0.02 if i % 2 else 1.0, 900 + i), 96, fen, moves))
    cases, dropped = [], 0
    for ci, (cfg_name, backend, sims, fen, moves) in enumerate(plan):
        kw = dict(CFGS[cfg_name])
        seed = 1000 + ci
        jit, nrm = streams(seed)
        b = chess.Board(fen)
        for u in moves:
            b.push(chess.Move.from_uci(u))
        # (1) the unmodified reference, sequential collection (num_threads=1 -> no executor, mcts.py:293-298)
        sj, sn = Stream(jit), Stream(nrm)
        random.random = sj.next
        np.random.normal = lambda loc, scale, shape: sn.take(shape)
        try:
            cfg = ref.MCTSConfig(num_threads=1, enable_memory_cleanup=False, dirichlet_frac=0.0, playout_random_frac=0.0, num_simulations=sims, **kw)
            be = HashBackend(scale=backend[1], seed=backend[2])
            if cfg_name == "direct":
                m = MCTSClass(cfg, TorchBackendModel(be), device="cpu", inference_backend=None)
            else:
                m = MCTSClass(cfg, _Model(), device="cpu", inference_backend=be)
            vc, pi, v = m.run(b.copy(), ply=len(moves))
            root = m._last_root
        finally:
            random.random, np.random.normal = real_random, real_normal
        exp = {"visits": [[mv.uci(), n] for mv, n in vc.items()], "value": v, "pi_nonzero": [[int(i), float(pi[i])] for i in np.nonzero(pi)[0]],
               "root_n": root.n, "child_q": [c.q for c in root.children.values()], "child_prior": [c.prior for c in root.children.values()],
               "jitter_used": sj.i, "normal_used": sn.i}
        # (2) the oracle restatement on the same streams: must agree exactly; reports the smallest top-2 gap
        o = RefMCTS(RefConfig(dirichlet_frac=0.0, playout_random_frac=0.0, num_simulations=sims, **kw), HashBackend(scale=backend[1], seed=backend[2]),
                    jitter_value=None, jitter_stream=jit, normal_stream=nrm, direct_model=(cfg_name == "direct"), virtual_loss=VL)
        vc2, pi2, v2 = o.run(b.copy(), ply=len(moves))
        assert [[mv.uci(), n] for mv, n in vc2.items()] == exp["visits"], ("oracle != reference", ci, cfg_name)
        assert v2 == v and pi2.tobytes() == pi.tobytes() and o.jit_used == sj.i and o.nrm_used == sn.i, ("oracle != reference", ci)
        assert [c.q for c in o._last_root.children.values()] == exp["child_q"]
        assert [c.prior for c in o._last_root.children.values()] == exp["child_prior"]
        exp["min_gap"] = o.min_gap
        exp["distinct_rows"] = o.distinct_rows
        if backend[1] != 0.0 and o.min_gap < MIN_GAP:
            dropped += 1
            continue
        cases.append({"cfg": cfg_name, "backend": list(backend), "sims": sims, "fen": fen, "moves": moves, "ply": len(moves), "seed": seed,
                      "expect": exp})
        print(ci, cfg_name, backend, "visits top", max(n for _, n in exp["visits"]), "jit", sj.i, "nrm", sn.i, "gap %.2e" % o.min_gap,
              "rows", o.distinct_rows, flush=True)
    json.dump({"configs": CFGS, "n_jitter": N_JITTER, "n_normal": N_NORMAL, "min_gap": MIN_GAP, "dropped_for_near_ties": dropped,
               "virtual_loss_batches": VL, "cases": cases}, open(os.path.join(HERE, "mcts_vl_golden.json" if VL else "mcts_stochastic_golden.json"), "w"))
    print("stochastic goldens:", len(cases), "cases kept,", dropped, "dropped (top-2 gap <", MIN_GAP, ")")


if __name__ == "__main__":
    main()
