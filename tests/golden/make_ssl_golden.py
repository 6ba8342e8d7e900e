"""Generate tests/golden/ssl_golden.npz by running the UNMODIFIED reference `azchess/ssl_algorithms.py`
(`create_enhanced_ssl_targets`, called per played ply with a batch of ONE position by selfplay_worker, internal.py:460-466)
on top of the oracle chess shim.  Needs the reference tree (oracle/_ref or MATRIX0_REFERENCE_ROOT):  python tests/golden/make_ssl_golden.py
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import refload  # noqa: E402


def main():
    enc, ssl = refload.load_reference("encoding", "ssl_algorithms")
    import chess
    from conftest import random_playout_boards
    boards = random_playout_boards(48, 140, seed=77)[::7][:384]
    boards += [chess.Board(f) for f in [
        "4k3/8/8/8/4r3/8/4B3/4K3 w - - 0 1",            # pinned bishop on the e-file
        "4k3/8/8/b7/8/2N5/8/4K3 w - - 0 1",             # pinned knight on the diagonal
        "r3k2r/8/8/3N4/8/8/8/4K3 w kq - 0 1",           # knight forking
        "4k3/8/2q1r3/8/3N4/8/8/4K3 w - - 0 1",
        "4k3/8/8/8/8/8/8/R3K2R b KQ - 0 1",
        "R6R/3Q4/1Q4Q1/4Q3/2Q4Q/Q4Q2/pp1Q4/kBNN1KB1 w - - 0 1",
        "8/8/8/8/8/8/8/K6k w - - 0 1",
    ]]
    algo = ssl.get_ssl_algorithms()
    planes = np.stack([enc.encode_board(b) for b in boards]).astype(np.float32)
    out = {k: [] for k in ("piece", "threat", "pin", "fork", "control")}
    for i in range(len(boards)):
        t = algo.create_enhanced_ssl_targets(torch.from_numpy(planes[i:i + 1]).float())      # batch of one, as the worker does
        for k in out:
            out[k].append(t[k][0].cpu().numpy().astype(np.float32))
    arrays = {k: np.stack(v) for k, v in out.items()}
    np.savez_compressed(os.path.join(HERE, "ssl_golden.npz"), fens=np.array([b.fen(en_passant="fen") for b in boards]), planes=planes, **arrays)
    print("ssl goldens:", len(boards), {k: (v.shape, float(v.sum())) for k, v in arrays.items()})


if __name__ == "__main__":
    main()
