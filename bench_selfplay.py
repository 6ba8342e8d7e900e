"""Helper module of bench.py (not part of the product package: its CPU legs run the oracle).  Workload "selfplay" (BASELINE configs[3] / [4]): batched self-play, G concurrent games x
`sims` simulations per move, ResNet-24 (320 channels, 24 blocks, 20 heads), one process per GPU.

A step = one search step over all games of the rank: select -> encode -> NN forward -> expand -> backup
(the first step of a move is the MCTS.run prologue: root evaluation + expansion; the last one is followed by
the move sampling / push kernel).  Reported separately, as SURVEY 8d demands: sims/s (reference accounting:
one evaluated leaf stands for up to inference_batch_size simulations, SURVEY Q1), unique NN evaluations/s and
self-play positions/s.
"""
from __future__ import annotations

import json
import os
import time

FLOP_PER_POSITION = 6.068e9  # SURVEY 6 [measured with FlopCounterMode]: conv 6020 + addmm 16 + bmm 31 MFLOP


def reference_cfg(sims: int, leaf_batch: int = 96):
    """config.yaml of the reference (mcts: / selfplay: / model: sections) with the BASELINE overrides:
    ResNet-24 = 320 channels / 24 blocks / 20 heads, num_simulations = sims."""
    model = dict(planes=19, channels=320, blocks=24, attention=True, attention_heads=20, policy_size=4672, norm="group", activation="silu",
                 value_activation="leaky_relu", preact=True, droppath=0.0, policy_factor_rank=160, infer_attention_stride=2,
                 infer_amp_tower=True, aux_policy_from_square=True, aux_policy_move_type=True, ssl_curriculum=True, self_supervised=True,
                 ssl_tasks=["piece", "threat", "pin", "fork", "control"])
    selfplay = dict(max_game_len=200, min_resign_plies=50, resign_threshold=-0.85, opening_random_plies=12, num_simulations=sims,
                    temperature_start=1.2, temperature_end=0.3, temperature_moves=40)
    mcts = dict(num_threads=4, num_simulations=sims, cpuct=2.5, cpuct_start=3.0, cpuct_end=2.0, cpuct_plies=40, dirichlet_alpha=0.3,
                dirichlet_frac=0.25, dirichlet_plies=30, selection_jitter=0.05, fpu=0.6, fpu_reduction=0.1, draw_penalty=-0.05,
                tt_capacity=1500000, tt_cleanup_frequency=5000, encoder_cache=True, legal_softmax=True, max_children=0, min_child_prior=0.0,
                no_instant_backtrack=True, parent_q_init=True, tt_cleanup_interval_s=5, value_from_white=False, virtual_loss=1.0,
                enable_memory_cleanup=True, inference_batch_size=int(leaf_batch), parallel_simulations=True, tree_parallelism=True,
                memory_cleanup_threshold_mb=512, max_tree_nodes=100000, playout_random_frac=0.05, enable_entropy_noise=True)
    return {"model": model, "selfplay": selfplay, "mcts": mcts}


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed `ncu --set full`
    capture (profiles/ncu_traffic.json, written from the .ncu-rep by tools/ncu_traffic.py); None when no capture is committed."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")
    try:
        with open(path) as f:
            return float(json.load(f)["conv_pair_kernel"]["dram_bytes_per_launch"])
    except (OSError, KeyError, ValueError):
        return None


def run(args, rank, world, local, ClockSampler, load_peaks, barrier, max_over_ranks, dump=None):
    """`dump`: None, or a callable that receives, by name, the arrays the last timed step produced (bench.py --dump-outputs)."""
    import numpy as np
    import torch
    from matrix0_b200 import _native
    from matrix0_b200.model import PolicyValueNet
    from matrix0_b200.selfplay import SelfPlayEngine
    lib = _native.lib()
    precision = os.environ.get("M0_BENCH_PRECISION", args.precision if hasattr(args, "precision") else "fp16")
    G = args.games
    leaf_batch = int(getattr(args, "leaf_batch", 96))
    cfg = reference_cfg(args.sims, leaf_batch)
    net = PolicyValueNet.from_config(cfg["model"], device=f"cuda:{local}", precision=precision, seed=0)
    from matrix0_b200 import distributed as D
    D.broadcast_parameters(net._params, src=0)  # identical weights everywhere: one NCCL broadcast per tensor (SURVEY 8e)
    sp = SelfPlayEngine(net, cfg, games=G, device=local, deterministic=False, seed=D.rank_seed(1234, rank), precision=precision,
                        max_nodes=4096 if leaf_batch >= 16 else 40960)   # distinct-leaf mode expands ~sims nodes of ~35 children per move
    stream = torch.cuda.current_stream()
    sp.start()
    per_move = 1 + sp.batches_per_move()

    class Cycle:
        i = 0

    def step():
        k = Cycle.i % per_move
        if k == 0:
            sp.begin_move()
        else:
            sp.search_step()
        if k == per_move - 1:
            sp.end_move()
        Cycle.i += 1

    # warm-up: one full move (buffers, workspaces) + the requested number of steps
    for _ in range(per_move + args.warmup):
        step()
    while Cycle.i % per_move:
        step()
    torch.cuda.synchronize()
    last = {}
    forward = sp._forward

    def keep_last(planes):     # the last timed step's evaluator call, for `dump`: its input planes and its outputs
        last["planes"] = planes.clone()
        last["policy_logits"], last["value"] = forward(planes)
        return last["policy_logits"], last["value"]
    c0 = sp.counters()
    l0 = int(lib.m0_launch_count())
    r0 = sp.graph_replays
    sampler = ClockSampler(local)
    barrier(world)
    sampler.start()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for i in range(args.steps):
        if dump is not None and i == args.steps - 1:
            sp._forward = keep_last
        step()
    t1.record(stream)
    barrier(world)
    clocks = sampler.stop()
    total_ms = max_over_ranks(t0.elapsed_time(t1), world)
    c1 = sp.counters()
    # kernels launched one by one + the kernels inside every CUDA-graph replay of the evaluator
    launches = int(lib.m0_launch_count()) - l0 + (sp.graph_replays - r0) * sp.graph_kernels
    d = {k: c1[k] - c0[k] for k in c1}
    nn_rows = args.steps * G
    if dump is not None:
        # what a caller of the search receives after that step: the root statistics of every game (m0_search_result) and the
        # move each game played last, beside the evaluator's input planes, policy logits and values of the step.  The games reach
        # that step through moves this build searched and sampled, so two builds' outputs compare row by row where the planes agree.
        sp._forward = forward
        eng = sp.engine
        eng.result(with_pi=True)
        dump(dict(last, root_moves=eng.res_moves, root_move_count=eng.res_count, root_visits=eng.res_visits, root_child_q=eng.res_q,
                  root_child_prior=eng.res_prior, root_pi=eng.res_pi, root_q=eng.res_root_q, root_n=eng.res_root_n,
                  moves_played=sp.moves_played))

    def allsum(x):
        if world == 1:
            return float(x)
        import torch.distributed as dist
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t)
        return float(t.item())
    sims_all = allsum(d["sims"])
    pos_all = allsum(d["positions_played"])
    evals_all = allsum(d["nn_evals"] + G * (args.steps // per_move + (1 if args.steps % per_move else 0)))
    secs = total_ms * 1e-3

    # dominant kernels in isolation: the NN forward over one step's batch, CUDA events on the launching stream
    planes = sp.engine.planes
    for _ in range(2):
        net.forward_planes(planes, precision)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(3)]
    for a, b in ev:
        a.record(stream)
        net.forward_planes(planes, precision)
        b.record(stream)
    torch.cuda.synchronize()
    nn_ms = sum(a.elapsed_time(b) for a, b in ev) / len(ev)
    peaks = load_peaks()
    achieved = FLOP_PER_POSITION * G / (nn_ms * 1e-3) / 1e12
    # the dominant kernel (CTA-pair 3x3 convolution C -> C, 2 launches per residual block) timed per launch inside the running
    # forward: CUDA events around every launch of its two sites
    import ctypes
    _native.check(lib.m0_profile_enable(1))
    for _ in range(3):
        net.forward_planes(planes, precision)
    torch.cuda.synchronize()
    conv_ms, conv_n, site_ms = 0.0, 0, {}
    for site in ("conv1+gn", "conv2+pool", "conv2+se+res+gn", "se_apply_gn", "se_gate", "se_fc1", "se_hidden", "se_fc2", "se_tail", "attention_tc", "gemm_qkv", "gemm_proj",
                 "layernorm_residual_f32", "ln_res_gn", "gn_act_res", "conv_other", "gemm_pst", "planes_to_nhwc_half", "f32_to_bf16", "gemm_pol_conv",
                 "gemm_pol_fc1", "gemm_pol_fc2", "gemm_val_conv1", "gemm_val_conv2", "gemm_val_fc1", "gemm_val_fc2", "gemm_val_gate", "value_tail", "gemm_f32"):
        ms, cnt = ctypes.c_double(0), ctypes.c_longlong(0)
        _native.check(lib.m0_profile_get(site.encode(), ctypes.byref(ms), ctypes.byref(cnt)))
        if cnt.value:
            site_ms[site] = {"launches_per_forward": cnt.value / 3, "us_per_launch": 1e3 * ms.value / cnt.value}
        if site.startswith("conv1") or site.startswith("conv2"):
            conv_ms += ms.value
            conv_n += cnt.value
    ms, cnt = ctypes.c_double(0), ctypes.c_longlong(0)
    _native.check(lib.m0_profile_get(None, ctypes.byref(ms), ctypes.byref(cnt)))
    fwd_profiled_ms = ms.value / 3
    _native.check(lib.m0_profile_enable(0))
    C = cfg["model"]["channels"]
    conv_flops = 2.0 * G * 64 * C * 9 * C
    conv_launch_ms = conv_ms / max(conv_n, 1)
    conv_tflops = conv_flops / (conv_launch_ms * 1e-3) / 1e12 if conv_n else 0.0
    traffic = load_traffic()

    # end to end with HOST buffers: root positions come from pinned host memory every move and the search
    # results (moves, visit counts, pi, root value) go back to pinned host memory
    eng = sp.engine
    root_host = torch.empty((G, 9), dtype=torch.int64).pin_memory()
    root_host.copy_(torch.from_numpy(np.zeros((G, 9), dtype=np.int64)))
    pos_dev = torch.empty((G, 9), dtype=torch.int64, device="cuda")
    _native.check(lib.m0_random_playouts(pos_dev.data_ptr(), G, 99 + rank, 60, stream.cuda_stream))
    root_host.copy_(pos_dev)
    h_moves = torch.empty((G, 256), dtype=torch.int16).pin_memory()
    h_visits = torch.empty((G, 256), dtype=torch.int32).pin_memory()
    h_pi = torch.empty((G, 4672), dtype=torch.float32).pin_memory()
    h_q = torch.empty((G,), dtype=torch.float64).pin_memory()

    def e2e_move():
        pos_dev.copy_(root_host, non_blocking=True)
        eng.set_positions_packed(pos_dev)
        sp.begin_move()
        for _ in range(per_move - 1):
            sp.search_step()
        eng.result(with_pi=True)
        h_moves.copy_(eng.res_moves, non_blocking=True)
        h_visits.copy_(eng.res_visits, non_blocking=True)
        h_pi.copy_(eng.res_pi, non_blocking=True)
        h_q.copy_(eng.res_root_q, non_blocking=True)
        stream.synchronize()

    e2e_move()
    ce0 = sp.counters()
    barrier(world)
    te = time.perf_counter()
    n_e2e = max(1, min(2, args.steps // per_move))
    for _ in range(n_e2e):
        e2e_move()
    barrier(world)
    e2e_s = max_over_ranks((time.perf_counter() - te) * 1e3, world) * 1e-3
    ce1 = sp.counters()
    e2e_sims = allsum(ce1["sims"] - ce0["sims"])

    # tree kernels in situ: CUDA events around search_select_kernel and search_expand_backup_kernel over one more move; algorithmic bytes
    # from the device counters of the same steps (+ the logits rows the expansion scans / gathers and the planes the selection writes)
    while Cycle.i % per_move:
        step()
    ct0 = sp.counters()
    sp.tree_events = []
    sp.begin_move()
    for _ in range(per_move - 1):
        sp.search_step()
    sp.end_move()
    torch.cuda.synchronize()
    evs, sp.tree_events = sp.tree_events, None
    ct1 = sp.counters()
    dt = {k: ct1[k] - ct0[k] for k in ct1}
    sel_us = 1e3 * sum(e[0].elapsed_time(e[1]) for e in evs) / len(evs)
    exp_us = 1e3 * sum(e[2].elapsed_time(e[3]) for e in evs) / len(evs)
    tree_bytes = (24 * dt["children_scanned"] + 24 * dt["path_nodes"] + 44 * dt["children_created"]
                  + (4 * 4672 + 72 + 19 * 64 * 4) * (dt["nn_evals"])) / len(evs)
    tree_gbs = tree_bytes / ((sel_us + exp_us) * 1e-6) / 1e9
    out = {
        "metric": "MCTS sims/sec, batched self-play, ResNet-24 (BASELINE configs[3])", "value": sims_all / secs, "unit": "sims/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "strong" if int(getattr(args, "total_games", 0)) > 0 else "weak", "vs_baseline": None, "dtype": precision, "data": "synthetic",
        "config": {"workload": f"batched self-play: {G} concurrent games/GPU x {args.sims} sims/move, ResNet-24 320ch/24 blocks/20 heads {precision}, random init",
                   "games_per_gpu": G, "total_games": G * world, "sims_per_move": args.sims, "inference_batch_size": leaf_batch, "steps_per_move": per_move,
                   "mode": ("reference-exact accounting (one evaluated leaf per game and mini-batch, SURVEY Q1), fresh tree per move" if leaf_batch > 1
                            else "distinct leaves: every simulation selects, evaluates and backs up its own leaf (inference_batch_size = 1), fresh tree per move"),
                   "openings": "start position + 12 random plies (device RNG)", "l2": "per-step activations (>1 GB) exceed the 126 MB L2"},
        "positions_per_s": pos_all / secs, "unique_nn_evals_per_s": allsum(nn_rows) / secs, "pending_leaf_evals_per_s": evals_all / secs,
        "clocks": clocks,
        "e2e": {"value": e2e_sims / e2e_s, "unit": "sims/s", "h2d_bytes_per_step": int(G * 72 / per_move),
                "d2h_bytes_per_step": int(G * (4672 * 4 + 256 * 6 + 8) / per_move), "moves_timed": n_e2e},
        "gpu_launches": launches,
        "roofline": {"bound": "tensor", "achieved": conv_tflops, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                     "frac": conv_tflops / peaks["bf16_tflops_sustained"], "traffic": traffic,
                     "peak_source": peaks["source"] + " (sustained bf16: the kernel is timed inside the running forward)",
                     "kernel": f"tc::conv_pair_kernel, 3x3 convolution {C}->{C} over {G} boards (tcgen05 cta_group::2 implicit GEMM, 2 launches per residual block)",
                     "algorithmic_flops_per_launch": conv_flops, "kernel_us": 1e3 * conv_launch_ms, "launches_timed": conv_n,
                     "share_of_step": (conv_ms / 3) / (total_ms / args.steps),
                     "timing": "CUDA events around each launch on the launching stream, 3 forwards after the timed region"},
        "forward": {"achieved": achieved, "unit": "TFLOP/s", "frac_of_sustained_peak": achieved / peaks["bf16_tflops_sustained"],
                    "algorithmic_flops": FLOP_PER_POSITION * G, "ms": nn_ms, "share_of_step": nn_ms / (total_ms / args.steps),
                    "launch_sites": site_ms, "sum_of_sites_ms": fwd_profiled_ms},
        "tree": {"children_scanned": d["children_scanned"], "path_nodes": d["path_nodes"], "children_created": d["children_created"],
                 "terminal_sims": d["terminal_sims"], "tt_hops": d["tt_hops"],
                 "algorithmic_bytes": 24 * d["children_scanned"] + 24 * d["path_nodes"] + 44 * d["children_created"],
                 "roofline": {"bound": "hbm (latency-bound in practice: one warp per game, dependent pointer chasing down the tree)",
                              "select_us_per_step": sel_us, "expand_backup_us_per_step": exp_us, "algorithmic_bytes_per_step": tree_bytes,
                              "achieved": tree_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": tree_gbs / peaks["hbm_gbs"],
                              "share_of_step": (sel_us + exp_us) * 1e-3 / (total_ms / args.steps),
                              "bytes": "24 B x children scanned + 24 B x path nodes + 44 B x children created + per evaluated leaf the logits row "
                                       "(18,688 B), the leaf position (72 B) and its planes (4,864 B)",
                              "timing": "CUDA events around the two kernels of every search step of one move, in the running loop"}},
    }
    out["accounting"] = ("value counts SIMULATIONS in the reference's accounting: with the jitter neutralised every simulation of a mini-batch reaches "
                         "the same leaf (SURVEY Q1), so one evaluated row stands for up to inference_batch_size simulations; the physical rate is "
                         "unique_nn_evals_per_s rows/s.  `as_shipped` is the same engine with the reference's per-simulation jitter and entropy noise: "
                         "compare its nn_rows_per_s with cpu_baseline.distinct_rows_per_s (like with like) or its sims_per_s with cpu_baseline.value")
    if not getattr(args, "no_extras", False) and leaf_batch > 1:
        del eng
        sp.engine.close()
        torch.cuda.empty_cache()
        out["as_shipped"] = bench_as_shipped(net, cfg, G, local, D.rank_seed(4321, rank), precision, stream)
        out["as_shipped"]["scope"] = "per GPU (rank 0's engine; every rank runs the same leg on its own games)"
        if world == 1:
            out["throughput_virtual_loss"] = bench_as_shipped(net, cfg, min(G, 512), local, D.rank_seed(999, rank), precision, stream, moves=1,
                                                              search_mode="virtual_loss")
            out["forward_sweep"] = forward_sweep(net, precision, stream, load_peaks)
            if precision != "bf16":   # BASELINE configs[2] names bf16: the same sweep with bf16 operands (same tensor-core rate)
                out["forward_sweep_bf16"] = forward_sweep(net, "bf16", stream, load_peaks, iters=5)
    if rank == 0:
        out["cpu_baseline"] = cpu_baseline(args.sims, args.cpu_seconds)
    return out


def bench_as_shipped(net, cfg, G, local, seed, precision, stream, moves=2, search_mode="as_shipped"):
    """The reference's search AS SHIPPED (selection_jitter 0.05 drawn per child per simulation, entropy noise on near-uniform priors,
    Dirichlet noise, playout-cap randomisation): every mini-batch collects up to 96 samples per game, the DISTINCT leaves of all games are
    evaluated in compact batches.  Timed with CUDA events over `moves` whole moves after one warm-up move."""
    import torch
    from matrix0_b200.selfplay import SelfPlayEngine
    sp = SelfPlayEngine(net, cfg, games=G, device=local, deterministic=False, seed=seed, precision=precision, search_mode=search_mode)
    sp.warm_up_forward()
    sp.start()
    sp.play_move()
    torch.cuda.synchronize()
    c0, r0, p0 = sp.counters(), sp.nn_rows, sp.nn_rows_padded
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for _ in range(moves):
        sp.play_move()
    t1.record(stream)
    torch.cuda.synchronize()
    secs = t0.elapsed_time(t1) * 1e-3
    c1 = sp.counters()
    d = {k: c1[k] - c0[k] for k in c1}
    sp.check_status()
    rows = d["nn_evals"] + G * moves          # distinct leaves + the root evaluation of every move
    label = ("as shipped: per-simulation selection jitter (mcts.py:893-897), entropy noise (:170-186), Dirichlet noise, playout-cap "
             "randomisation; one evaluator row per DISTINCT leaf of a mini-batch, fresh tree per move")
    if search_mode == "virtual_loss":
        label = ("throughput mode: as shipped PLUS the in-flight marking of MCTS._select (virtual loss, mcts.py:889-890 / :922-923, code the "
                 "reference ships but never activates) inside every mini-batch: the simulations of a batch spread over distinct leaves, "
                 "(almost) every simulation evaluates its own row")
    out = {"mode": label,
           "games_per_gpu": G, "moves_timed": moves, "seconds": secs, "sims_per_s": d["sims"] / secs, "positions_per_s": d["positions_played"] / secs,
           "nn_rows_per_s": rows / secs, "padded_rows_per_s": (sp.nn_rows_padded - p0 + G * moves) / secs,
           "samples_per_s": d["leaf_samples"] / secs, "distinct_rows_per_sample": d["nn_evals"] / max(1, d["leaf_samples"]),
           "rows_per_move_per_game": rows / (G * moves), "noisy_expansions_share": d["noisy_expansions"] / max(1, d["expansions"]),
           "engine_bytes": sp.engine.bytes, "max_nodes_per_game": sp.engine.max_nodes}
    sp.engine.close()
    return out


def forward_sweep(net, precision, stream, load_peaks, batches=(256, 512, 1024, 2048, 4096, 8192), warmup=3, iters=10):
    """BASELINE configs[2]: ResNet-24 inference forward alone over a batch sweep (real encoded positions, CUDA events)."""
    import torch
    from matrix0_b200 import _native
    lib = _native.lib()
    peaks = load_peaks()
    res = []
    for B in batches:
        pos = torch.empty((B, 9), dtype=torch.int64, device="cuda")
        _native.check(lib.m0_random_playouts(pos.data_ptr(), B, 7, 80, stream.cuda_stream))
        planes = torch.empty((B, 19, 8, 8), dtype=torch.float32, device="cuda")
        _native.check(lib.m0_encode_planes(pos.data_ptr(), B, planes.data_ptr(), stream.cuda_stream))
        for _ in range(warmup):
            net.forward_planes(planes, precision)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(iters):
            net.forward_planes(planes, precision)
        b.record(stream)
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / iters
        tf = FLOP_PER_POSITION * B / (ms * 1e-3) / 1e12
        res.append({"batch": B, "ms": ms, "positions_per_s": B / (ms * 1e-3), "tflops": tf, "frac_of_burst_peak": tf / peaks["bf16_tflops"],
                    "frac_of_sustained_peak": tf / peaks["bf16_tflops_sustained"]})
    return {"workload": "ResNet-24 inference forward alone (BASELINE configs[2]), real encoded positions, " + precision, "dtype": precision,
            "sweep": res}



def cpu_baseline(sims: int, budget_s: float, moves_cap: int = 1):
    """The reference's CPU self-play path restated (oracle port): RefMCTS on the oracle chess shim + the fp32 torch
    restatement of ResNet-24 on all host cores, one game from the start position, fresh MCTS per move."""
    import torch
    from oracle import chess_shim  # noqa: F401
    import chess
    from oracle import nn_ref
    from oracle.mcts_ref import RefConfig, RefMCTS
    from matrix0_b200.model import NetConfig, parameter_shapes
    cfg = reference_cfg(sims)
    known = set(NetConfig.__dataclass_fields__)
    ncfg = NetConfig(**{k: v for k, v in cfg["model"].items() if k in known})
    sd = nn_ref.make_state_dict(parameter_shapes(ncfg), seed=1)
    net = nn_ref.OracleNet(ncfg, sd)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    m = {k: v for k, v in cfg["mcts"].items()}
    b = chess.Board()
    t0 = time.perf_counter()
    done_sims = moves = 0
    evals = rows = distinct = 0
    while moves < moves_cap or time.perf_counter() - t0 < budget_s * 0.5:
        mc = RefMCTS(RefConfig(**m), net, jitter_value=None)     # as shipped: random.random() jitter, entropy / Dirichlet noise, playout cap
        vc, pi, v = mc.run(b, ply=moves)
        done_sims += mc._last_sims_run
        evals += mc.unique_evals
        rows += mc.sample_rows + 1
        distinct += mc.distinct_rows + 1
        moves += 1
        b.push(max(vc.items(), key=lambda kv: kv[1])[0])
        if b.is_game_over() or time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {"value": done_sims / dt, "unit": "sims/s", "cores": cores, "kind": "port",
            "sample": f"{moves} move(s) x ~{sims} sims of one game from the start position in {dt:.1f}s, as shipped (jitter, entropy / Dirichlet noise, "
                      f"playout cap): {evals} NN calls, {rows} rows evaluated (one per collected sample, duplicates included) of which {distinct} "
                      f"distinct leaves, fp32 torch CPU; positions/s = {moves / dt:.4f}",
            "positions_per_s": moves / dt, "nn_rows_per_s": rows / dt, "distinct_rows_per_s": distinct / dt}


def reference_arm(args):
    base = cpu_baseline(args.sims, max(20.0, args.cpu_seconds * 2), moves_cap=2)
    return {"impl": "reference", "metric": "MCTS sims/sec, batched self-play, ResNet-24 (BASELINE configs[3])", "value": base["value"],
            "unit": "sims/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"batched self-play: {args.games} concurrent games/GPU x {args.sims} sims/move, ResNet-24 320ch/24 blocks/20 heads, random init",
                       "games_per_gpu": args.games, "sims_per_move": args.sims, "inference_batch_size": int(getattr(args, "leaf_batch", 96)),
                       "sample": "the reference's CPU path (RefMCTS + fp32 torch forward on all host cores) on ONE game of that workload, "
                                 "bounded to a few moves; games are independent, so sims/s per game is the reference's rate for any number of games"},
            "positions_per_s": base["positions_per_s"], "nn_rows_per_s": base["nn_rows_per_s"], "distinct_rows_per_s": base["distinct_rows_per_s"],
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
