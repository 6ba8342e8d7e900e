"""Gumbel AlphaZero self-play (search_mode="gumbel", n simulations of one network row per game) next to collapsed self-play at 800
simulations, for ResNet-24 (bench.py's model) and the model config.yaml ships (288 channels), fp16, in one process:
    python tools/bench_gumbel.py [--games 4096] [--moves 3] [--sims 16 32 64] [--m 16] [--out profiles/r07_gumbel_bench.json]
Per model and mode, over --moves whole moves after one warm-up move (CUDA events around the moves):
* positions/s (plies played by all games per second) and ms per move;
* network rows per game and move (evaluator rows of the timed moves / positions played);
* the tree kernels' share of the time: CUDA events around select and expand+backup of every search step (SelfPlayEngine.tree_events),
  recorded in a second pass of --moves moves so the events do not perturb the first;
* the card's name, power limit and SM clocks before and after.  Needs a GPU."""
from __future__ import annotations

import argparse
import gc
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools")]

from bench_shipped_model import gpu_context, model_cfgs  # noqa: E402


def run_mode(net, model, mode, sims, m, games, moves):
    import torch
    from bench_selfplay import reference_cfg
    from matrix0_b200.selfplay import SelfPlayEngine
    cfg = dict(reference_cfg(800), model=model)
    if mode == "gumbel":
        cfg["gumbel"] = {"num_simulations": sims, "max_considered_actions": m}
    sp = SelfPlayEngine(net, cfg, games=games, device=0, deterministic=False, seed=1234, precision="fp16", search_mode=mode)
    sp.start()
    sp.play_move()                                   # warm-up: graph captures of every batch size this mode uses
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    c0, rows0 = sp.counters(), sp.nn_rows
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(moves):
        sp.play_move()
    b.record(stream)
    torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    c1 = sp.counters()
    positions = c1["positions_played"] - c0["positions_played"]
    rows = sp.nn_rows - rows0
    # second pass with events around the tree kernels of every search step
    sp.tree_events = []
    a.record(stream)
    for _ in range(moves):
        sp.play_move()
    b.record(stream)
    torch.cuda.synchronize()
    ms2 = a.elapsed_time(b)
    tree_ms = sum(e[0].elapsed_time(e[1]) + e[2].elapsed_time(e[3]) for e in sp.tree_events)
    st, _ = sp.engine.status()
    out = {"mode": mode, "simulations": sims, "max_considered_actions": m if mode == "gumbel" else None, "games": games, "moves": moves,
           "positions_per_s": positions / (ms * 1e-3), "ms_per_move": ms / moves, "network_rows_per_game_move": rows / max(1, positions),
           "tree_kernel_share": tree_ms / ms2, "status_bits": int(st.abs().sum())}
    del sp
    gc.collect()
    torch.cuda.empty_cache()
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--moves", type=int, default=3)
    ap.add_argument("--sims", type=int, nargs="+", default=[16, 32, 64])
    ap.add_argument("--m", type=int, default=16)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_gumbel_bench.json"))
    args = ap.parse_args()
    import torch
    from matrix0_b200.model import PolicyValueNet
    if not torch.cuda.is_available():
        raise SystemExit("bench_gumbel.py needs a GPU")
    torch.cuda.set_device(0)
    result = {"gpu_before": gpu_context(), "precision": "fp16", "runs": {}}
    for name, model in model_cfgs().items():
        net = PolicyValueNet.from_config(model, device="cuda:0", precision="fp16", seed=0)
        runs = [run_mode(net, model, "collapsed", 800, args.m, args.games, args.moves)]
        runs += [run_mode(net, model, "gumbel", n, args.m, args.games, args.moves) for n in args.sims]
        for r in runs:
            print(json.dumps(dict(r, model=name)), flush=True)
        result["runs"][name] = runs
        del net
        gc.collect()
        torch.cuda.empty_cache()
    result["gpu_after"] = gpu_context()
    print(json.dumps({"gpu_before": result["gpu_before"], "gpu_after": result["gpu_after"]}), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
