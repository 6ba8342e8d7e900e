"""precision="fp8" (e4m3 tower convolutions) against fp16 on the tensor-core path, for ResNet-24 (bench.py's model) and the model
config.yaml ships (288 channels), in one process:

    python tools/bench_fp8.py [--batch 4096] [--rounds 5] [--iters 20] [--moves 3] [--out profiles/r06_fp8_bench.json]

* forward: B = --batch random-playout positions, fp16 and fp8 alternating round by round (CUDA events around --iters forwards after a
  warm-up), per model; the fp8 / fp16 time ratio of the medians;
* the two tower launch sites (conv1+gn, conv2+se+res+gn) per precision from the per-launch-site event timing (m0_profile_enable, a
  run of its own), and the tower convolutions' achieved TFLOP/s counted with the algorithmic K (9 x C) and with the K the kernel runs
  (each tap padded to whole k-blocks: 64 channels at 16 bits, 128 at e4m3);
* collapsed self-play (SelfPlayEngine, --games games x 800 simulations) per precision and model: sims/s over --moves whole moves;
* the card's name, power limit and SM clocks before and after.  Needs a GPU."""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools")]

from bench_shipped_model import gpu_context, model_cfgs  # noqa: E402

PRECISIONS = ("fp16", "fp8")
SITES = ("conv1+gn", "conv2+se+res+gn")


def tower_conv_flops(model: dict, kb_channels: int = 0) -> float:
    """2 x MACs of one position's tower 3x3 convolutions (conv1 + conv2 of every block); kb_channels > 0 pads K per tap to whole
    k-blocks of that many channels (the MMA work the kernel issues)."""
    C, blocks = model["channels"], model["blocks"]
    k = (C + kb_channels - 1) // kb_channels * kb_channels if kb_channels else C
    return 2.0 * 64 * 9 * k * C * 2 * blocks


def planes_for(B, seed=7):
    import torch
    from matrix0_b200 import _native
    lib, s = _native.lib(), torch.cuda.current_stream().cuda_stream
    pos = torch.empty((B, 9), dtype=torch.int64, device="cuda")
    _native.check(lib.m0_random_playouts(pos.data_ptr(), B, seed, 80, s))
    planes = torch.empty((B, 19, 8, 8), dtype=torch.float32, device="cuda")
    _native.check(lib.m0_encode_planes(pos.data_ptr(), B, planes.data_ptr(), s))
    return planes


def time_forward(net, planes, prec, warmup, iters):
    import torch
    for _ in range(warmup):
        net.forward_planes(planes, prec)
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(iters):
        net.forward_planes(planes, prec)
    b.record(stream)
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def site_times(net, planes, prec, iters):
    import torch
    from matrix0_b200 import _native
    lib = _native.lib()
    net.forward_planes(planes, prec)
    torch.cuda.synchronize()
    _native.check(lib.m0_profile_enable(1))
    try:
        for _ in range(iters):
            net.forward_planes(planes, prec)
        torch.cuda.synchronize()
        out = {}
        for site in SITES:
            ms, cnt = ctypes.c_double(0), ctypes.c_longlong(0)
            _native.check(lib.m0_profile_get(site.encode(), ctypes.byref(ms), ctypes.byref(cnt)))
            out[site] = {"ms_per_forward": ms.value / iters, "launches_per_forward": cnt.value / iters}
    finally:
        _native.check(lib.m0_profile_enable(0))
    return out


def selfplay(net, model, prec, games, moves):
    import torch
    from bench_selfplay import reference_cfg
    from matrix0_b200.selfplay import SelfPlayEngine
    sp = SelfPlayEngine(net, dict(reference_cfg(800), model=model), games=games, device=0, deterministic=False, seed=1234, precision=prec,
                        max_nodes=4096)
    sp.start()
    for _ in range(2):
        sp.play_move()
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    c0 = sp.counters()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(moves):
        sp.play_move()
    b.record(stream)
    torch.cuda.synchronize()
    secs = a.elapsed_time(b) * 1e-3
    st, _ = sp.engine.status()
    return {"games": sp.G, "moves": moves, "sims_per_s": (sp.counters()["sims"] - c0["sims"]) / secs, "status_bits": int(st.abs().sum())}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--moves", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_fp8_bench.json"))
    args = ap.parse_args()
    cfgs = model_cfgs()
    flops = {name: {"algorithmic": tower_conv_flops(m), "padded_fp16": tower_conv_flops(m, 64), "padded_fp8": tower_conv_flops(m, 128)}
             for name, m in cfgs.items()}
    print(json.dumps({"tower_conv_flops_per_position": flops}), flush=True)
    import torch
    from matrix0_b200.model import PolicyValueNet
    if not torch.cuda.is_available():
        raise SystemExit("bench_fp8.py needs a GPU")
    torch.cuda.set_device(0)
    result = {"gpu_before": gpu_context(), "batch": args.batch, "tower_conv_flops_per_position": flops}
    nets = {name: PolicyValueNet.from_config(m, device="cuda:0", precision="fp16", seed=0) for name, m in cfgs.items()}
    planes = planes_for(args.batch)
    fwd = {name: {p: [] for p in PRECISIONS} for name in cfgs}
    for r in range(args.rounds):
        for name in cfgs:
            for p in (PRECISIONS if r % 2 == 0 else PRECISIONS[::-1]):
                fwd[name][p].append(time_forward(nets[name], planes, p, args.warmup, args.iters))
    result["forward"] = {}
    for name in cfgs:
        med = {p: statistics.median(fwd[name][p]) for p in PRECISIONS}
        result["forward"][name] = {"ms_rounds": fwd[name], "ms_median": med, "time_ratio_fp8_over_fp16": med["fp8"] / med["fp16"]}
        print(json.dumps({name: result["forward"][name]}), flush=True)
    result["sites"] = {}
    for name in cfgs:
        result["sites"][name] = {}
        for p in PRECISIONS:
            st = site_times(nets[name], planes, p, args.iters)
            ms = sum(v["ms_per_forward"] for v in st.values())
            kb = "padded_fp8" if p == "fp8" else "padded_fp16"
            st["tower_conv_tflops_algorithmic"] = flops[name]["algorithmic"] * args.batch / (ms * 1e-3) / 1e12
            st["tower_conv_tflops_padded"] = flops[name][kb] * args.batch / (ms * 1e-3) / 1e12
            result["sites"][name][p] = st
        print(json.dumps({name: result["sites"][name]}), flush=True)
    result["selfplay_collapsed"] = {}
    for name, m in cfgs.items():
        result["selfplay_collapsed"][name] = {p: selfplay(nets[name], m, p, args.games, args.moves) for p in PRECISIONS}
        print(json.dumps({name: result["selfplay_collapsed"][name]}), flush=True)
    result["gpu_after"] = gpu_context()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
