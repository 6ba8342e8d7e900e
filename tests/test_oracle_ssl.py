"""oracle/ssl_ref.py (numpy restatement of azchess/ssl_algorithms.py) against the golden vectors generated from the unmodified
reference module (tests/golden/make_ssl_golden.py), and -- where the reference tree is present -- against the module itself."""
import os

import numpy as np
import pytest

from oracle import ssl_ref


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "ssl_golden.npz"))


def test_ssl_oracle_matches_reference_goldens(golden):
    planes = golden["planes"]
    assert float(golden["pin"].sum()) == 0.0      # the reference's pin map is identically zero (oracle/ssl_ref.py docstring)
    for i in range(planes.shape[0]):
        t = ssl_ref.ssl_targets(planes[i])
        for k in ("piece", "threat", "pin", "fork", "control"):
            assert np.array_equal(t[k], golden[k][i]), (k, str(golden["fens"][i]))


def test_ssl_oracle_matches_live_reference():
    from oracle import refload
    if not refload.reference_available():
        pytest.skip(refload.MISSING)
    import torch
    enc, ssl = refload.load_reference("encoding", "ssl_algorithms")
    from conftest import random_playout_boards
    algo = ssl.get_ssl_algorithms()
    for b in random_playout_boards(12, 100, seed=5)[::9][:60]:
        planes = enc.encode_board(b).astype(np.float32)
        ref = algo.create_enhanced_ssl_targets(torch.from_numpy(planes[None]).float())
        got = ssl_ref.ssl_targets(planes)
        for k in got:
            assert np.array_equal(got[k], ref[k][0].numpy().astype(np.float32)), (k, b.fen())
