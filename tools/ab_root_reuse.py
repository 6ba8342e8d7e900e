"""Alternating A/B of the default benchmark line between two trees (a baseline checkout and this tree), plus the evaluator rows one
move really costs now that the root's evaluation is reused across moves.

    python tools/ab_root_reuse.py --baseline DIR [--runs 3] [--out FILE.json]

First ``bench.py --no-extras --dump-outputs`` runs in both trees and the dumped arrays are compared byte for byte.  Then each run
executes ``python bench.py`` (default arguments) in the baseline tree and then in this tree, so both see the same box,
the same power cap and the same neighbours; the card name and power limit are read in the same call.  Afterwards one engine of the
default workload (4096 games, 800 simulations, ResNet-24 fp16) plays three moves in this tree and reports, per move, the rows the
evaluator ran (``nn_rows``), the roots expanded from kept outputs (counter ``root_evals_reused``) and G x (1 + mini-batches), the rows
the benchmark line's ``unique_nn_evals_per_s`` assumes.  Needs a GPU."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench_line(tree: str) -> dict:
    out = subprocess.run([sys.executable, "bench.py"], cwd=tree, check=True, capture_output=True, text=True).stdout
    line = [l for l in out.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    ash = d.get("as_shipped") or {}
    return {"value": d["value"], "ms_per_step": d["ms_per_step"], "clocks": d.get("clocks"), "forward_ms": d["forward"]["ms"],
            "conv_pair_frac": d["roofline"]["frac"], "conv_pair_kernel_us": d["roofline"]["kernel_us"],
            "encode_value": (d.get("encode") or {}).get("value"), "as_shipped_sims_per_s": ash.get("sims_per_s"),
            "as_shipped_rows_per_move_per_game": ash.get("rows_per_move_per_game")}


def dump_compare(baseline: str) -> dict:
    """``bench.py --no-extras --dump-outputs`` in both trees: every array the last timed step produced, compared byte for byte."""
    import numpy as np
    with tempfile.TemporaryDirectory() as tmp:
        dirs = {}
        for name, tree in (("baseline", baseline), ("this", ROOT)):
            dirs[name] = os.path.join(tmp, name)
            subprocess.run([sys.executable, "bench.py", "--no-extras", "--dump-outputs", dirs[name]], cwd=tree, check=True,
                           capture_output=True, text=True)
        files = sorted(set(os.listdir(dirs["baseline"])) | set(os.listdir(dirs["this"])))
        out = {}
        for f in files:
            a, b = (os.path.join(dirs[n], f) for n in ("baseline", "this"))
            if not (os.path.exists(a) and os.path.exists(b)):
                out[f] = "missing in one tree"
                continue
            x, y = np.load(a), np.load(b)
            out[f] = {"shape": list(x.shape), "dtype": str(x.dtype),
                      "identical": x.shape == y.shape and x.dtype == y.dtype and x.tobytes() == y.tobytes()}
        return out


def rows_per_move(moves: int = 3) -> dict:
    sys.path.insert(0, ROOT)
    import bench_selfplay
    from matrix0_b200.model import PolicyValueNet
    from matrix0_b200.selfplay import SelfPlayEngine
    cfg = bench_selfplay.reference_cfg(800)
    net = PolicyValueNet.from_config(cfg["model"], device="cuda:0", precision="fp16", seed=0)
    sp = SelfPlayEngine(net, cfg, games=4096, device=0, deterministic=False, seed=1234, precision="fp16", max_nodes=4096)
    sp.start()
    for _ in range(2):          # warm-up: the first moves evaluate every root (empty store, workspaces growing)
        sp.play_move()
    per_move = []
    for _ in range(moves):
        c0, r0 = sp.counters(), sp.nn_rows
        sp.play_move()
        c1 = sp.counters()
        per_move.append({"nn_rows": sp.nn_rows - r0, "root_evals_reused": c1["root_evals_reused"] - c0["root_evals_reused"],
                         "rows_assumed_by_bench_line": sp.G * (1 + sp.batches_per_move())})
    return {"games": sp.G, "engine_bytes": sp.engine.bytes, "moves": per_move}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline", required=True, help="tree of the commit to compare against (built)")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    dumps = dump_compare(os.path.abspath(args.baseline))
    print(json.dumps({"dump_outputs": dumps}), flush=True)
    runs = {"baseline": [], "this": []}
    for i in range(args.runs):
        for name, tree in (("baseline", os.path.abspath(args.baseline)), ("this", ROOT)):
            r = bench_line(tree)
            runs[name].append(r)
            print(json.dumps({"run": i, "tree": name, **r}), flush=True)
    summary = {}
    for key in ("value", "ms_per_step", "forward_ms", "conv_pair_frac", "encode_value", "as_shipped_sims_per_s"):
        a = [r[key] for r in runs["baseline"] if r[key] is not None]
        b = [r[key] for r in runs["this"] if r[key] is not None]
        if a and b:
            summary[key] = {"baseline_median": statistics.median(a), "this_median": statistics.median(b),
                            "ratio": statistics.median(b) / statistics.median(a)}
    result = {"gpu": smi, "dump_outputs": dumps, "runs": runs, "summary": summary, "rows_per_move": rows_per_move()}
    print(json.dumps({"summary": summary, "gpu": smi, "rows_per_move": result["rows_per_move"]}, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
