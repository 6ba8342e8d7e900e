"""The oracle search restatement (oracle/mcts_ref.py) reproduces the committed golden vectors that
the UNMODIFIED reference MCTS produced (tests/golden/make_golden.py), and -- where the reference tree
exists -- is compared live with the reference on further seeds."""
import logging

import numpy as np
import pytest

import chess
from mcts_cases import run_all
from oracle import refload
from oracle.backends import HashBackend
from oracle.mcts_ref import RefConfig, RefMCTS


def make_ref(cfg, backend, sims):
    return RefMCTS(RefConfig(dirichlet_frac=0.0, enable_entropy_noise=False, num_simulations=sims, **cfg), backend, jitter_value=0.5)


def test_oracle_reproduces_reference_goldens():
    assert run_all(make_ref, prior_rtol=0.0) >= 80


@pytest.mark.skipif(not refload.reference_available(), reason=refload.MISSING)
def test_oracle_matches_unmodified_reference_live():
    logging.disable(logging.CRITICAL)
    try:
        ref = refload.load_reference("mcts")
        ref.random.random = lambda: 0.5
        ref.psutil_available = False

        class _Model:
            class cfg:
                policy_size = 4672
        kw = dict(cpuct_start=3.0, cpuct_end=2.0, cpuct_plies=40, fpu_reduction=0.1, draw_penalty=-0.05, legal_softmax=True,
                  selection_jitter=0.05, inference_batch_size=96)
        from conftest import random_playout_boards
        for i, b in enumerate(random_playout_boards(6, 80, seed=99)[::7][:12]):
            cfg = ref.MCTSConfig(num_threads=1, enable_memory_cleanup=False, dirichlet_frac=0.0, enable_entropy_noise=False,
                                 playout_random_frac=0.0, num_simulations=250, **kw)
            m1 = ref.MCTS(cfg, _Model(), device="cpu", inference_backend=HashBackend(1.0, seed=i))
            m2 = make_ref(kw, HashBackend(1.0, seed=i), 250)
            vc1, pi1, v1 = m1.run(b, ply=3)
            vc2, pi2, v2 = m2.run(b.copy(), ply=3)
            assert list(vc1.items()) == list(vc2.items()) and pi1.tobytes() == pi2.tobytes() and v1 == v2
    finally:
        logging.disable(logging.NOTSET)
