"""The network config.yaml ships (288 channels, 22 blocks, 18 heads: bench_selfplay.reference_cfg without the ResNet-24 overrides) on
the 16-bit tensor-core path.  288 = 4.5 k-blocks of 64 channels: the last k-block of every tap is half empty (zero-filled activations,
3x3 weights stored with each tap padded to whole k-blocks), the CTA-pair convolution runs two 144-column halves, and the first SE
layer runs 72 hidden units as 80 columns."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def shipped_model_cfg():
    from bench_selfplay import reference_cfg
    return dict(reference_cfg(800)["model"], channels=288, blocks=22, attention_heads=18)


_NETS = {}


def shipped_net(precision):
    """The shipped model with the reference's own initialisation (seed 0)."""
    if precision not in _NETS:
        from matrix0_b200.model import PolicyValueNet
        _NETS[precision] = PolicyValueNet.from_config(shipped_model_cfg(), device="cuda", precision=precision, seed=0)
    return _NETS[precision]


def _device_positions(n, seed):
    """Planes of n positions from random playouts (device)."""
    from matrix0_b200 import _native
    lib = _native.lib()
    pos = torch.empty((n, 9), dtype=torch.int64, device="cuda")
    _native.check(lib.m0_random_playouts(pos.data_ptr(), n, seed, 40, _native.current_stream()))
    planes = torch.empty((n, 19, 8, 8), dtype=torch.float32, device="cuda")
    _native.check(lib.m0_encode_planes(pos.data_ptr(), n, planes.data_ptr(), _native.current_stream()))
    return planes


def _run_tc(act, w, taps):
    from matrix0_b200 import _native
    lib = _native.lib()
    boards, cin, n = act.shape[0], act.shape[-1], w.shape[0]
    out = torch.empty((boards * 64, n), dtype=torch.float32, device="cuda")
    _native.check(lib.m0_tc_conv(act.data_ptr(), w.data_ptr(), boards, cin, n, taps, out.data_ptr(), _native.current_stream()), "m0_tc_conv")
    torch.cuda.synchronize()
    return out


# ---- 1. the kernels alone: K tail (cin % 64 == 32) and 144-column halves, against plain PyTorch fp32 on the same bf16 operands ----
@pytest.mark.parametrize("boards", [2, 298])
@pytest.mark.parametrize("cin,n", [(96, 96), (288, 288), (288, 144), (320, 288)])
def test_conv3x3_k_tail(boards, cin, n):
    g = torch.Generator(device="cuda").manual_seed(5 + boards + cin + n)
    act = torch.randn((boards, 8, 8, cin), device="cuda", generator=g).to(torch.bfloat16)
    wt = (torch.randn((n, cin, 3, 3), device="cuda", generator=g) / (9 * cin) ** 0.5).to(torch.bfloat16)
    w = wt.permute(0, 2, 3, 1).reshape(n, 9 * cin).contiguous()          # k = (ky*3+kx)*cin + ci
    out = _run_tc(act, w, 9)
    ref = torch.nn.functional.conv2d(act.float().permute(0, 3, 1, 2), wt.float(), padding=1)
    ref = ref.permute(0, 2, 3, 1).reshape(boards * 64, n)
    err = (out - ref).abs().max().item()
    assert err <= 2e-3 * max(1.0, ref.abs().max().item()), err


@pytest.mark.parametrize("boards", [2, 298])
@pytest.mark.parametrize("cin,n", [(96, 96), (288, 288), (288, 144), (320, 288), (288, 80)])
def test_gemm_k_tail(boards, cin, n):
    g = torch.Generator(device="cuda").manual_seed(9 + boards + cin + n)
    act = torch.randn((boards, 64, cin), device="cuda", generator=g).to(torch.bfloat16)
    w = (torch.randn((n, cin), device="cuda", generator=g) / cin ** 0.5).to(torch.bfloat16)
    out = _run_tc(act, w, 1)
    ref = act.float().reshape(-1, cin) @ w.float().t()
    err = (out - ref).abs().max().item()
    assert err <= 2e-3 * max(1.0, ref.abs().max().item()), err


# ---- 2. the yardstick: the fp32 CUDA path at 288 against the oracle ----
def test_fp32_path_matches_the_oracle_at_288():
    from conftest import random_playout_boards
    from oracle import nn_ref
    from oracle.encoding_ref import encode_board
    net = shipped_net("fp32")
    boards = random_playout_boards(8, 100, seed=17)[::2][:64]
    x = torch.from_numpy(np.stack([encode_board(b) for b in boards]))
    p, v = net.forward(x)
    sd = {k: t.cpu() for k, t in net.state_dict().items()}
    with torch.no_grad():
        pr, vr = nn_ref.forward(sd, net.cfg, x)
    for got, ref in ((p.cpu().numpy(), pr.numpy()), (v.cpu().numpy(), vr.numpy())):
        scale = float(np.abs(ref).max())
        assert float(np.abs(got - ref).max()) <= 1e-4 * max(scale, 1e-6), (float(np.abs(got - ref).max()), scale)


# ---- 3. the gate: 16-bit path against the fp32 CUDA path ----
def _agreement(net, f32, x, legal):
    ps, vs, prs, vrs = [], [], [], []
    for i in range(0, x.shape[0], 1152):
        p, v = net.forward(x[i:i + 1152])
        pr, vr = f32.forward(x[i:i + 1152])
        ps.append(p.float()); vs.append(v.float()); prs.append(pr); vrs.append(vr)
    p, v, pr, vr = torch.cat(ps), torch.cat(vs), torch.cat(prs), torch.cat(vrs)
    neg = torch.full_like(pr, -1e30)
    top1_all = (p.argmax(1) == pr.argmax(1)).float().mean().item()
    top1_legal = (torch.where(legal, p, neg).argmax(1) == torch.where(legal, pr, neg).argmax(1)).float().mean().item()
    return top1_all, top1_legal, (v - vr).abs().max().item()


def _check_gate(precision, a, al, dv, what):
    print(f"{what} {precision}: top-1 {a:.4f} legal top-1 {al:.4f} max|dv| {dv:.2e}")
    if precision == "fp16":
        assert a >= 0.99 and al >= 0.99 and dv <= 2e-2, (a, al, dv)
    else:   # bf16: the bars of the R24 reference-init gate on the legal policy
        assert al >= 0.99 and a >= 0.98 and dv <= 2e-2, (a, al, dv)


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_shipped_model_gate_on_refinit_positions(golden_dir, precision):
    """The 2,304 positions of refinit_golden.npz (FENs encoded by the oracle), shipped model with the reference's init (seed 0)."""
    from test_nn_gpu import _refinit
    r = _refinit(golden_dir)
    _check_gate(precision, *_agreement(shipped_net(precision), shipped_net("fp32"), r["x"], r["legal"].cuda()), "shipped model")


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_96_channel_net_gate(precision):
    """96 channels (1.5 k-blocks), 4 blocks, 6 heads of 16, seeded init, random-playout positions."""
    from conftest import random_playout_boards
    from matrix0_b200.model import PolicyValueNet
    from oracle.encoding_ref import encode_board, get_legal_actions
    cfg = dict(shipped_model_cfg(), channels=96, blocks=4, attention_heads=6, infer_attention_stride=1)
    net = PolicyValueNet.from_config(cfg, device="cuda", precision=precision, seed=5)
    f32 = PolicyValueNet.from_config(cfg, device="cuda", precision="fp32", seed=5)
    boards = random_playout_boards(24, 120, seed=29)[::2][:640]
    x = torch.from_numpy(np.stack([encode_board(b) for b in boards]))
    legal = torch.from_numpy(np.stack([get_legal_actions(b) for b in boards])).cuda()
    _check_gate(precision, *_agreement(net, f32, x, legal), "96-channel net")


# ---- 4. the pipeline: the same fused tensor-core stages as ResNet-24 ----
def test_shipped_model_runs_the_fused_tensor_core_pipeline():
    import ctypes
    from matrix0_b200 import _native
    lib = _native.lib()
    net = shipped_net("fp16")
    x = _device_positions(64, 3)
    net.forward_planes(x, "fp16")
    torch.cuda.synchronize()
    _native.check(lib.m0_profile_enable(1))
    try:
        net.forward_planes(x, "fp16")
        torch.cuda.synchronize()
        counts = {}
        for site in ("conv1+gn", "conv2+se+res+gn", "attention_tc", "attention_f32", "gemm_f32", "layernorm_residual_f32", "groupnorm_f32",
                     "se_gate", "conv2+pool"):
            ms, cnt = ctypes.c_double(0), ctypes.c_longlong(0)
            _native.check(lib.m0_profile_get(site.encode(), ctypes.byref(ms), ctypes.byref(cnt)))
            counts[site] = cnt.value
    finally:
        _native.check(lib.m0_profile_enable(0))
    assert counts["conv1+gn"] == 22 and counts["conv2+se+res+gn"] == 22 and counts["attention_tc"] == 3, counts
    assert all(counts[s] == 0 for s in ("attention_f32", "gemm_f32", "layernorm_residual_f32", "groupnorm_f32", "se_gate", "conv2+pool")), counts


# ---- 5. a row's output is a function of the row alone (root reuse in SelfPlayEngine relies on it) ----
@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_row_output_depends_on_the_row_alone_at_288(precision):
    net = shipped_net(precision)
    x = _device_positions(4096, 7)
    lg, v = (t.clone() for t in net.forward_planes(x, precision))
    for n in (1, 37, 256, 300, 2048):
        a, b = net.forward_planes(x[:n].contiguous(), precision)
        assert torch.equal(a, lg[:n]) and torch.equal(b, v[:n]), n
    perm = torch.randperm(4096, generator=torch.Generator().manual_seed(3)).cuda()
    a, b = net.forward_planes(x[perm].contiguous(), precision)
    assert torch.equal(a, lg[perm]) and torch.equal(b, v[perm])
    y = _device_positions(4096, 11)
    keep = torch.arange(0, 4096, 5, device="cuda")
    y[keep] = x[keep]
    a, b = net.forward_planes(y, precision)
    assert torch.equal(a[keep], lg[keep]) and torch.equal(b[keep], v[keep])
    z = y[:37].clone()
    z[20] = x[3]
    a, b = net.forward_planes(z, precision)
    assert torch.equal(a[20], lg[3]) and torch.equal(b[20], v[3])


# ---- 6. end to end: the orchestrator's worker entry with config.yaml's model section ----
def test_selfplay_worker_with_the_shipped_model(tmp_path):
    import queue
    from matrix0_b200.selfplay import selfplay_worker
    from test_selfplay_gpu import MCTS_KW
    cfg = {"model": shipped_model_cfg(), "data_dir": str(tmp_path / "data"), "seed": 3,
           "mcts": dict(MCTS_KW, num_simulations=32, inference_batch_size=16),
           "selfplay": {"num_simulations": 32, "opening_random_plies": 4, "max_game_len": 8, "temperature_start": 1.0, "temperature_end": 0.3,
                        "temperature_moves": 40, "resign_threshold": -0.85, "min_resign_plies": 50}}
    q = queue.Queue()
    n = selfplay_worker(0, cfg, None, games=6, q=q, concurrent_games=6, precision="fp16")
    assert n == 6
    files = sorted((tmp_path / "data" / "selfplay").glob("selfplay_w0_g*.npz"))
    assert len(files) == 6
    msgs = []
    while not q.empty():
        msgs.append(q.get())
    game_msgs = [m for m in msgs if m["type"] == "game"]
    assert len(game_msgs) == 6
    assert set(game_msgs[0]) >= {"type", "proc", "file", "moves", "result", "secs", "resigned", "resigner", "draw", "avg_policy_entropy",
                                 "avg_ms_per_move", "avg_sims"}
    for path in files:
        with np.load(path) as f:
            T = int(f["meta_moves"][0])
            assert T >= 1
            assert f["s"].shape == (T, 19, 8, 8) and f["pi"].shape == (T, 4672) and f["z"].shape == (T,)
            assert np.isfinite(f["pi"]).all()
