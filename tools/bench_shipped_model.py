"""The model config.yaml ships (288 channels, 22 blocks, 18 heads) against the ResNet-24 that bench.py measures (320 / 24 / 20), both
fp16 on the tensor-core path, in one process:

    python tools/bench_shipped_model.py [--batches 256,...,8192] [--iters 20] [--moves 3] [--out profiles/r04_shipped_model.json]

* forward: B = 256 ... 8192 random-playout positions generated on the device, the two models alternating batch size by batch size
  (warm-up, then CUDA events around --iters forwards on the launching stream), and the time ratio shipped / R24;
* FLOPs per position computed here from the layer shapes (3x3 and 1x1 convolutions, linear layers, attention matmuls; 2 x MAC);
* collapsed self-play (SelfPlayEngine, 4096 games x 800 simulations): sims/s, evaluated rows/s and ms per search step over --moves
  whole moves after two warm-up moves;
* the card's name, power limit and SM clocks, read in the same run.  Needs a GPU."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def model_cfgs():
    from bench_selfplay import reference_cfg
    r24 = reference_cfg(800)["model"]
    return {"shipped": dict(r24, channels=288, blocks=22, attention_heads=18), "r24": r24}


def flops_per_position(model: dict) -> dict:
    """Multiply-adds x 2 of one position's forward (policy + value heads, attention at the inference stride), by kind."""
    from matrix0_b200.model import NetConfig, tower_layout
    cfg = NetConfig(**{k: v for k, v in model.items() if k in NetConfig.__dataclass_fields__})
    C, hid = cfg.channels, max(8, int(cfg.channels * cfg.se_ratio))
    conv3 = lambda ci, co: 2 * 64 * 9 * ci * co        # noqa: E731
    conv1 = lambda ci, co: 2 * 64 * ci * co            # noqa: E731
    lin = lambda i, o: 2 * i * o                       # noqa: E731
    conv, mm, bmm = conv3(cfg.planes, C), 0, 0
    if cfg.chess_features:
        conv += conv3(C, C) + (conv1(C, C) if cfg.piece_square_tables else 0)
    seen, stride = 0, max(1, int(cfg.infer_attention_stride))
    mix = float(cfg.attention_unmasked_mix)
    for _, ai in tower_layout(cfg):
        conv += 2 * conv3(C, C)
        mm += lin(C, hid) + lin(hid, C) if cfg.se else 0
        if ai is not None:
            seen += 1
            if seen % stride == 0:
                conv += conv1(C, 3 * C) + conv1(C, C)
                bmm += (3 if 0.0 < mix < 1.0 else 2) * 2 * 64 * 64 * C   # q k^T, then softmax(.) v for the masked (and unmasked) scores
    r = cfg.policy_factor_rank
    conv += conv1(C, 64) + conv1(C, 128) + conv1(128, 128)
    mm += (lin(4096, r) + lin(r, cfg.policy_size)) if r > 0 else lin(4096, cfg.policy_size)
    mm += lin(8192, 2 * C) + lin(2 * C, C) + lin(C, C) + lin(C, 1)
    return {"conv": conv, "mm": mm, "bmm": bmm, "total": conv + mm + bmm}


def gpu_context() -> list:
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks_throttle_reasons.active",
                           "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()


def forward_sweep(nets, batches, warmup, iters):
    import torch
    from matrix0_b200 import _native
    lib = _native.lib()
    stream = torch.cuda.current_stream()
    out = []
    for B in batches:
        pos = torch.empty((B, 9), dtype=torch.int64, device="cuda")
        _native.check(lib.m0_random_playouts(pos.data_ptr(), B, 7, 80, stream.cuda_stream))
        planes = torch.empty((B, 19, 8, 8), dtype=torch.float32, device="cuda")
        _native.check(lib.m0_encode_planes(pos.data_ptr(), B, planes.data_ptr(), stream.cuda_stream))
        row = {"batch": B}
        for name, (net, flops) in nets.items():
            for _ in range(warmup):
                net.forward_planes(planes, "fp16")
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(iters):
                net.forward_planes(planes, "fp16")
            b.record(stream)
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / iters
            row[name] = {"ms": ms, "positions_per_s": B / (ms * 1e-3), "tflops": flops * B / (ms * 1e-3) / 1e12}
        row["time_ratio_shipped_over_r24"] = row["shipped"]["ms"] / row["r24"]["ms"]
        print(json.dumps(row), flush=True)
        out.append(row)
    return out


def selfplay(net, model, games, moves):
    """Collapsed self-play as bench.py runs it: `moves` whole moves after two warm-up moves, timed with CUDA events."""
    import torch
    from bench_selfplay import reference_cfg
    from matrix0_b200.selfplay import SelfPlayEngine
    cfg = dict(reference_cfg(800), model=model)
    sp = SelfPlayEngine(net, cfg, games=games, device=0, deterministic=False, seed=1234, precision="fp16", max_nodes=4096)
    sp.start()
    for _ in range(2):
        sp.play_move()
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    c0, r0 = sp.counters(), sp.nn_rows
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(moves):
        sp.play_move()
    b.record(stream)
    torch.cuda.synchronize()
    secs = a.elapsed_time(b) * 1e-3
    c1 = sp.counters()
    steps = moves * (1 + sp.batches_per_move())
    return {"games": sp.G, "moves": moves, "sims_per_s": (c1["sims"] - c0["sims"]) / secs, "evaluated_rows_per_s": (sp.nn_rows - r0) / secs,
            "ms_per_step": 1e3 * secs / steps, "steps": steps}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="256,512,1024,2048,4096,8192")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--moves", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_shipped_model.json"))
    args = ap.parse_args()
    cfgs = model_cfgs()
    flops = {name: flops_per_position(m) for name, m in cfgs.items()}
    print(json.dumps({"flops_per_position": flops}), flush=True)
    import torch
    from matrix0_b200.model import PolicyValueNet
    if not torch.cuda.is_available():
        raise SystemExit("bench_shipped_model.py needs a GPU")
    torch.cuda.set_device(0)
    result = {"gpu_before": gpu_context(), "flops_per_position": flops}
    nets = {name: (PolicyValueNet.from_config(m, device="cuda:0", precision="fp16", seed=0), flops[name]["total"]) for name, m in cfgs.items()}
    result["forward_fp16"] = forward_sweep(nets, [int(b) for b in args.batches.split(",")], args.warmup, args.iters)
    result["selfplay_collapsed"] = {}
    for name, m in cfgs.items():
        result["selfplay_collapsed"][name] = selfplay(nets[name][0], m, args.games, args.moves)
        print(json.dumps({name: result["selfplay_collapsed"][name]}), flush=True)
    result["gpu_after"] = gpu_context()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
