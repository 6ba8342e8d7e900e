"""Writes tests/golden/selfplay_golden.json: the answers of the reference's ``should_adjudicate_draw`` (azchess/draw.py) and
``sample_move_from_counts`` (azchess/selfplay/internal.py:690-735) on the inputs of tests/selfplay_cases.py.

    python tests/golden/make_selfplay_golden.py                     # with the unmodified reference tree (oracle/_ref or MATRIX0_REFERENCE_ROOT)
    python tests/golden/make_selfplay_golden.py --from-restatement  # from oracle/selfplay_ref.py

The committed file was written with ``--from-restatement``.  Those answers are the reference's: the live tests of
tests/test_oracle_selfplay.py compared the restatement with the unmodified reference on exactly these inputs when the game loop
was added, and neither oracle/selfplay_ref.py, the oracle chess module nor the input generation has changed since.
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))                     # tests/
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))    # repository root
from oracle import chess_shim  # noqa: E402,F401
from oracle import refload  # noqa: E402
import selfplay_cases as C  # noqa: E402


def main():
    if "--from-restatement" in sys.argv:
        from oracle import selfplay_ref as R
        draw, source = R.should_adjudicate_draw, "oracle/selfplay_ref.py (equal to the reference on these inputs, see make_selfplay_golden.py)"

        def sample(counts, T, seed):
            return R.sample_move_from_counts(list(counts), list(counts.values()), T, C.uniform(seed))
    else:
        draw = refload.load_reference("draw").should_adjudicate_draw
        ref_sample = C.reference_function("azchess/selfplay/internal.py", "sample_move_from_counts")
        source = "the unmodified reference"

        def sample(counts, T, seed):
            import numpy as np
            import chess
            np.random.seed(seed)
            return list(counts).index(ref_sample(chess.Board(C.SAMPLE_FEN), counts, T))

    games = C.draw_games()
    decisions = "".join("1" if draw(b, moves, cfg) else "0" for b, moves, cfg in C.draw_cases(games))
    trials = [{"moves": len(counts), "counts": list(counts.values()), "temperature": T, "seed": seed, "choice": sample(counts, T, seed)}
              for counts, T, seed in C.sample_trials()]
    out = {"source": source,
           "draw": {"cfgs": C.DRAW_CFGS, "games": [[m.uci() for m in g] for g in games], "decisions": decisions},
           "sample": {"fen": C.SAMPLE_FEN, "trials": trials}}
    with open(C.GOLDEN, "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print(f"{len(decisions)} draw decisions ({decisions.count('1')} draws), {len(trials)} sampling trials -> {C.GOLDEN}")


if __name__ == "__main__":
    main()
