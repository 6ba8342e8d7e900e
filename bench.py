#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 self-play search engine (driver contract in the task).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload encode|selfplay] [--impl reference] [--dump-outputs DIR]

Workloads (BASELINE.json `configs`):
  selfplay  configs[3]/[4]: batched self-play, G concurrent games x 800 sims/move, ResNet-24 bf16;
            a step = one search step (select -> encode -> NN forward -> expand -> backup) over all games.
  encode    configs[1]: encode + legal-mask over 1M synthetic positions resident in HBM;
            a step = one pass of the fused kernel over the batch.
One process per GPU (torchrun for N > 1); games / positions are sharded across ranks, no data-path
collective (weak scaling).  `--impl reference` times the reference's CPU algorithm (oracle port:
the reference is pure Python on python-chess, restated under oracle/) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_tflops": float(p["bf16_tflops"]),
                "bf16_tflops_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(n_gpus: int):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def max_over_ranks(ms: float, world: int) -> float:
    if world == 1:
        return ms
    import torch
    import torch.distributed as dist
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(world: int):
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


DUMP_ROWS = 512          # --dump-outputs keeps at most this many rows of an array ...
DUMP_BYTES = 64 << 20    # ... and at most this many bytes in all


def dump_outputs(directory: str, arrays) -> None:
    """--dump-outputs: every array (torch or numpy) as DIR/<name>.npy.  Floating arrays keep float32 / float64, integer ones
    become float64 (exact).  An array of more than DUMP_ROWS rows is cut to a sample of rows drawn from a fixed seed, the same
    rows for every array of that length, so that two builds run with the same arguments can be compared output for output.
    The rows are picked where the array lives (on the device for a CUDA tensor) before anything is copied to the host."""
    import numpy as np
    out = {}
    for name, a in arrays.items():
        if not hasattr(a, "detach"):
            a = np.asarray(a)
        if a.ndim and a.shape[0] > DUMP_ROWS:
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], DUMP_ROWS, replace=False))
            if hasattr(a, "detach"):
                import torch
                rows = torch.from_numpy(rows).to(a.device)
            a = a[rows]
        if hasattr(a, "detach"):
            a = a.detach().cpu().numpy()
        out[name] = np.ascontiguousarray(a if a.dtype in (np.float32, np.float64) else a.astype(np.float64))
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes, more than {DUMP_BYTES}")
    os.makedirs(directory, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), a)


# ---- workload: encode (configs[1]) -------------------------------------------------------------
ENC_BYTES_PER_POS = 72 + 19 * 64 * 4 + 4672   # packed position read + float32 planes + uint8 mask written


def encode_traffic(n):
    """DRAM bytes of one launch from the committed `ncu --set full` capture (profiles/ncu_traffic.json), when that capture
    ran the same number of positions (the file stores bytes per launch of the 1 Mi-position default)."""
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")) as f:
            e = json.load(f).get("encode_mask_planes_kernel")
        return float(e["dram_bytes_per_launch"]) if e and n == 1 << 20 else None
    except (OSError, ValueError, KeyError):
        return None


def bench_encode(args, rank, world, local):
    import numpy as np
    import torch
    from matrix0_b200 import _native
    from matrix0_b200.boards import PLANES, POLICY_SIZE
    lib = _native.lib()
    n = args.positions
    stream = torch.cuda.current_stream()
    pos = torch.empty((n, 9), dtype=torch.int64, device="cuda")
    _native.check(lib.m0_random_playouts(pos.data_ptr(), n, 1234 + rank, 120, stream.cuda_stream), "m0_random_playouts")
    planes = torch.empty((n, PLANES, 8, 8), dtype=torch.float32, device="cuda")
    mask = torch.empty((n, POLICY_SIZE), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def step():
        _native.check(lib.m0_encode_positions(pos.data_ptr(), n, planes.data_ptr(), mask.data_ptr(), 0, 0, 0, stream.cuda_stream))

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local)
    barrier(world)
    sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for a, b in evs:
        a.record(stream)
        step()
        b.record(stream)
    t1.record(stream)
    barrier(world)
    clocks = sampler.stop()
    total_ms = max_over_ranks(t0.elapsed_time(t1), world)
    kern_ms = sum(a.elapsed_time(b) for a, b in evs) / len(evs)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"planes": planes, "legal_mask": mask})

    # end to end through the public Python API with HOST buffers: raw records in pinned memory ->
    # H2D -> pack + encode kernels -> D2H of planes and mask into pinned host buffers
    ne = min(n, args.e2e_positions)
    raw_host = torch.empty((ne, 10), dtype=torch.int64).pin_memory()
    # synthesize raw host records from the device positions (outside the timed region)
    p = pos[:ne].cpu().numpy().view(np.uint64)
    raw_np = raw_host.numpy().view(np.uint64)
    raw_np[:, :8] = p[:, :8]
    st = p[:, 8]
    cr = (st >> np.uint64(1)) & np.uint64(15)
    raw_np[:, 8] = ((cr & np.uint64(1)) << np.uint64(7)) | ((cr >> np.uint64(1)) & np.uint64(1)) \
        | (((cr >> np.uint64(2)) & np.uint64(1)) << np.uint64(63)) | (((cr >> np.uint64(3)) & np.uint64(1)) << np.uint64(56))
    ep = (st >> np.uint64(5)) & np.uint64(127)
    ep = np.where(ep > 63, np.uint64(255), ep)
    raw_np[:, 9] = (st & np.uint64(1)) | (ep << np.uint64(8)) | (((st >> np.uint64(16)) & np.uint64(0xFFFF)) << np.uint64(16)) \
        | (((st >> np.uint64(32)) & np.uint64(0xFFFF)) << np.uint64(32))
    planes_host = torch.empty((ne, PLANES, 8, 8), dtype=torch.float32).pin_memory()
    mask_host = torch.empty((ne, POLICY_SIZE), dtype=torch.uint8).pin_memory()
    raw_dev = torch.empty((ne, 10), dtype=torch.int64, device="cuda")
    pos_e = torch.empty((ne, 9), dtype=torch.int64, device="cuda")

    def e2e_step():
        raw_dev.copy_(raw_host, non_blocking=True)
        _native.check(lib.m0_positions_pack(raw_dev.data_ptr(), ne, pos_e.data_ptr(), stream.cuda_stream))
        _native.check(lib.m0_encode_positions(pos_e.data_ptr(), ne, planes.data_ptr(), mask.data_ptr(), 0, 0, 0, stream.cuda_stream))
        planes_host.copy_(planes[:ne], non_blocking=True)
        mask_host.copy_(mask[:ne], non_blocking=True)
        stream.synchronize()

    e2e_step()
    barrier(world)
    te = time.perf_counter()
    e2e_iters = max(1, min(args.steps, 5))
    for _ in range(e2e_iters):
        e2e_step()
    barrier(world)
    e2e_ms = max_over_ranks((time.perf_counter() - te) * 1e3 / e2e_iters, world)

    peaks = load_peaks()
    achieved = n * ENC_BYTES_PER_POS / (kern_ms * 1e-3) / 1e9
    out = {
        "metric": "encode+legal-mask positions/sec (BASELINE configs[1])", "value": n * world * args.steps / (total_ms * 1e-3),
        "unit": "positions/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64->f32/u8", "data": "synthetic",
        "config": {"workload": "encode+legal-mask microbench", "positions_per_gpu": n, "source": "device random playouts <=120 plies",
                   "outputs": "float32 planes [n,19,8,8] + uint8 mask [n,4672]", "l2": "outputs (9.5 GB/step) exceed the 126 MB L2"},
        "clocks": clocks,
        "e2e": {"value": ne * world / (e2e_ms * 1e-3), "unit": "positions/s", "h2d_bytes_per_step": ne * 80,
                "d2h_bytes_per_step": ne * (19 * 64 * 4 + 4672), "positions_per_step": ne},
        "gpu_launches": args.steps,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                     "traffic": encode_traffic(n), "peak_source": peaks["source"], "kernel": "encode_mask_planes_kernel",
                     "algorithmic_bytes_per_launch": n * ENC_BYTES_PER_POS, "kernel_ms": kern_ms},
    }
    if rank == 0:
        out["cpu_baseline"] = cpu_baseline_encode(args.cpu_seconds)
    return out


def cpu_baseline_encode(budget_s: float):
    """Oracle port of encode_board + get_legal_actions (single Python thread, like the reference)."""
    from oracle import chess_shim  # noqa: F401
    from oracle import encoding_ref as E
    import chess
    import random
    rng = random.Random(0)
    boards = []
    b = chess.Board()
    while len(boards) < 400:
        if b.is_game_over() or len(b.move_stack) > 120:
            b = chess.Board()
        boards.append(b.copy(stack=False))
        b.push(rng.choice(list(b.legal_moves)))
    t0 = time.perf_counter()
    n = 0
    while time.perf_counter() - t0 < budget_s:
        for bd in boards:
            E.encode_board(bd)
            E.get_legal_actions(bd)
        n += len(boards)
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "positions/s", "cores": 1, "kind": "port",
            "sample": f"{n} positions (400 distinct random-playout boards, repeated) in {dt:.1f}s, oracle/encoding_ref.py on oracle/chess"}


def reference_encode(args):
    base = cpu_baseline_encode(max(5.0, args.cpu_seconds))
    return {"impl": "reference", "metric": "encode+legal-mask positions/sec (BASELINE configs[1])", "value": base["value"],
            "unit": "positions/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": None,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64->f32/u8", "data": "synthetic",
            "config": {"workload": "encode+legal-mask microbench"}, "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "positions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default=os.environ.get("M0_BENCH_WORKLOAD", "auto"), choices=["auto", "encode", "selfplay"])
    ap.add_argument("--positions", type=int, default=1 << 20)
    ap.add_argument("--e2e-positions", type=int, default=1 << 16)
    ap.add_argument("--games", type=int, default=4096, help="concurrent games PER GPU (weak scaling, the default of the driver's 1..8 GPU runs)")
    ap.add_argument("--total-games", type=int, default=0,
                    help="BASELINE configs[4] as written: this many games in total, split evenly over the ranks (32768 -> 16384 / 8192 / 4096 per GPU at 2 / 4 / 8)")
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--leaf-batch", type=int, default=96,
                    help="mcts.inference_batch_size: 96 = the reference's accounting (one evaluated leaf per game stands for up to 96 "
                         "simulations, SURVEY Q1); 1 = distinct-leaf mode, every simulation evaluates its own leaf (SURVEY 8d row 4, second mode)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-extras", action="store_true", help="headline record only: skip the as_shipped / encode / forward_sweep sub-records")
    ap.add_argument("--precision", default=os.environ.get("M0_BENCH_PRECISION", "fp16"), choices=["fp16", "bf16", "fp32"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them computed as DIR/<name>.npy (rank 0; the same seeded sample "
                         f"of at most {DUMP_ROWS} rows of every array).  Equal arguments give equal inputs and, on one build, equal files.  "
                         "Self-play games reach the last step through moves the build itself searched and sampled, so the planes that step "
                         "evaluated are written too: between two builds, compare the rows whose planes agree")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup is not None and args.warmup < 0:
        ap.error("--warmup must not be negative")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the outputs of the native engine: it needs --impl native")
    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints "NCCL version ..." on the first
    # collective), so file descriptor 1 points at stderr while the run lasts and the line goes to the saved descriptor.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    if args.workload == "auto":
        try:
            import bench_selfplay  # noqa: F401
            args.workload = "selfplay"
        except ImportError:
            args.workload = "encode"
    if args.steps is None:
        args.steps = 20
    if args.warmup is None:
        args.warmup = 3

    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return
        if args.workload == "selfplay":
            import bench_selfplay
            out = bench_selfplay.reference_arm(args)
        else:
            out = reference_encode(args)
        emit(out)
        return

    rank, world, local = dist_setup(args.gpus)
    if args.total_games > 0:
        args.games = args.total_games // world
    if args.workload == "selfplay":
        import bench_selfplay
        dump = (lambda arrays: dump_outputs(args.dump_outputs, arrays)) if args.dump_outputs and rank == 0 else None
        out = bench_selfplay.run(args, rank, world, local, ClockSampler, load_peaks, barrier, max_over_ranks, dump=dump)
        if world == 1 and not args.no_extras:
            # BASELINE configs[1] beside the headline: the encode + legal-mask microbenchmark with its own roofline / e2e / cpu_baseline
            import torch
            torch.cuda.empty_cache()
            enc_args = argparse.Namespace(**vars(args))
            enc_args.steps, enc_args.warmup, enc_args.cpu_seconds = 10, 3, min(args.cpu_seconds, 5.0)
            enc_args.dump_outputs = None
            out["encode"] = bench_encode(enc_args, rank, world, local)
    else:
        out = bench_encode(args, rank, world, local)
    if rank == 0:
        emit(out)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
