"""precision="fp8" on the GPU: the fp16 tensor-core forward with e4m3 operands for every residual block's conv1 / conv2 (DESIGN.md
section 4).  The kernel alone is checked exactly (e4m3 inputs, power-of-two scales); the network against the fp64 reference that
applies the same e4m3 rounding (fp8_cases.reference_fp8) with fp8_cases.EMULATION_BARS, and against the plain fp64 reference with the
fp8 bars.  ``-s`` prints the metrics."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import fp8_cases as F8
import tc_matrix_cases as M

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.abspath(os.path.dirname(__file__)))
_NETS = {}


def _net(name, sd=None):
    from matrix0_b200.model import PolicyValueNet
    net = PolicyValueNet(M.net_config(name), device="cuda", precision="fp8", seed=0)
    net.load_state_dict(M.state_dict(name) if sd is None else sd, strict=True)
    return net


def row_net(name):
    if name not in _NETS:
        _NETS[name] = _net(name)
    return _NETS[name]


def _x():
    return M.positions().cuda()


def _run(net, x, fmt="fp8"):
    lg, v = net.forward_planes(x, fmt)
    return lg.cpu().numpy(), v.cpu().numpy()


def _fmt(m):
    return "(" + ", ".join(f"{v:.2e}" for v in m) + ")"


# ---- 1. the e4m3 kernel alone: exact e4m3 operands and power-of-two scales, so only the accumulation order differs from fp64 ----
def _conv_fp8(act8, w8, scale, boards, cin, n):
    from matrix0_b200 import _native
    out = torch.empty((boards * 64, n), dtype=torch.float32, device="cuda")
    _native.check(_native.lib().m0_tc_conv_fp8(act8.data_ptr(), w8.data_ptr(), scale.data_ptr(), boards, cin, n, out.data_ptr(),
                                               _native.current_stream()), "m0_tc_conv_fp8")
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("boards", [2, 6, 302])           # 302 boards: the last 4-board tile holds two
@pytest.mark.parametrize("cin", [64, 96, 256, 288, 320])
@pytest.mark.parametrize("n", [64, 96, 288, 320])
def test_e4m3_conv_kernel_alone(boards, cin, n):
    g = torch.Generator(device="cuda").manual_seed(boards * 1000 + cin + n)
    act = F8.e4m3(torch.randn((boards, 8, 8, cin), device="cuda", generator=g) * 2.0)
    wt = F8.e4m3(torch.randn((n, cin, 3, 3), device="cuda", generator=g) * 8.0)
    scale = torch.pow(2.0, -(torch.arange(n, device="cuda") % 7 + 4).float())     # dequantisation factors 2^-4 .. 2^-10
    act8 = act.to(torch.float8_e4m3fn).view(torch.uint8).contiguous()
    w8 = wt.permute(0, 2, 3, 1).reshape(n, 9 * cin).to(torch.float8_e4m3fn).view(torch.uint8).contiguous()   # k = (ky*3+kx)*cin + ci
    out = _conv_fp8(act8, w8, scale, boards, cin, n).double()
    ref = torch.nn.functional.conv2d(act.double().permute(0, 3, 1, 2), wt.double(), padding=1) * scale.double()[None, :, None, None]
    ref = ref.permute(0, 2, 3, 1).reshape(boards * 64, n)
    err = (out - ref).abs().max().item()
    assert err <= 1e-5 * ref.abs().max().item(), err


def test_e4m3_conv_rejects_what_it_cannot_run():
    from matrix0_b200 import _native
    lib = _native.lib()
    buf = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    for boards, cin, n in ((3, 64, 64), (2, 48, 64), (2, 64, 80), (2, 64, 352), (2, 64, 32)):
        assert lib.m0_tc_conv_fp8(buf.data_ptr(), buf.data_ptr(), buf.data_ptr(), boards, cin, n, buf.data_ptr(), 0) == _native.M0_ERR_ARG


# ---- 2. every row the mode accepts: against the emulated-fp8 reference (EMULATION_BARS) and the plain reference (fp8 bars) ----
@pytest.mark.parametrize("name", F8.ROWS)
def test_row_matches_the_emulated_fp8_reference(name):
    lg, v = _run(row_net(name), _x())
    emu = M.metrics(lg, v, F8.reference_fp8(name))
    plain = M.metrics(lg, v, M.reference(name))
    print(f"\n[fp8] {name:16s} vs emulated {_fmt(emu)} vs fp64 {_fmt(plain)}")
    assert F8.within(emu, F8.EMULATION_BARS), (emu, F8.EMULATION_BARS)
    assert F8.within(plain, F8.BARS["fp8"]), (plain, F8.BARS["fp8"])


@pytest.mark.parametrize("name", F8.ROWS)
def test_row_reaches_its_launch_sites(name):
    from matrix0_b200 import _native
    lib = _native.lib()
    net, x = row_net(name), _x()
    net.forward_planes(x, "fp8")
    torch.cuda.synchronize()
    _native.check(lib.m0_profile_enable(1))
    try:
        net.forward_planes(x, "fp8")
        torch.cuda.synchronize()
        counts = {}
        for site in M.SITES:
            ms, cnt = ctypes.c_double(0), ctypes.c_longlong(0)
            _native.check(lib.m0_profile_get(site.encode(), ctypes.byref(ms), ctypes.byref(cnt)))
            counts[site] = cnt.value
    finally:
        _native.check(lib.m0_profile_enable(0))
    row = M.BY_NAME[name]
    assert all(counts[s] > 0 for s in row["must"]), ([s for s in row["must"] if counts[s] == 0], counts)
    assert all(counts[s] == 0 for s in row["must_not"]), ([s for s in row["must_not"] if counts[s]], counts)
    assert counts["conv1+gn"] == M.net_config(name).blocks and counts["conv2+se+res+gn"] == M.net_config(name).blocks, counts


# ---- 3. a fault loaded into the CUDA net fails the emulated-reference comparison (the smaller faults of tc_matrix_cases sit inside
#      the e4m3 rounding sensitivity, fp8_cases.EMULATION_BARS; they are caught on the CPU against the fp16 bars only) ----
@pytest.mark.parametrize("name", ["w96", "w288", "w320"])
def test_zeroed_tap_fails_the_emulated_reference(name):
    m = M.metrics(*_run(_net(name, M.faulted_state_dict(name, "conv_tap")), _x()), F8.reference_fp8(name))
    assert F8.excess(m, F8.EMULATION_BARS) >= 1.5, (m, F8.EMULATION_BARS)


# ---- 4. configurations outside the fused CTA-pair tower are refused; the net keeps working in fp16 ----
def test_unfused_se_row_is_refused():
    from matrix0_b200.model import PolicyValueNet
    name = "w320_se085"
    net = PolicyValueNet(M.net_config(name), device="cuda", precision="fp16", seed=0)
    net.load_state_dict(M.state_dict(name), strict=True)
    with pytest.raises(ValueError, match="se_hidden > 256"):
        net.forward_planes(_x(), "fp8")
    assert M.within(M.metrics(*_run(net, _x(), "fp16"), M.reference(name)), "fp16")


_SWITCH_SCRIPT = r"""
import os, sys
root = sys.argv[1]
sys.path[:0] = [root, os.path.join(root, "tests")]
from oracle import chess_shim  # noqa: F401
import torch
import tc_matrix_cases as M
from matrix0_b200.model import PolicyValueNet
net = PolicyValueNet(M.net_config("w96"), device="cuda", precision="fp8", seed=0)
try:
    net.forward_planes(M.positions()[:4].cuda(), "fp8")
except ValueError as e:
    print("REFUSED", e)
net.forward_planes(M.positions()[:4].cuda(), "fp16")
torch.cuda.synchronize()
print("FP16 OK")
"""


@pytest.mark.parametrize("env,reason", [({"M0_TC_PAIR": "0"}, "M0_TC_PAIR=0"), ({"M0_TC_FUSE_SE": "0"}, "M0_TC_FUSE_SE=0")])
def test_switches_that_leave_the_fused_tower_are_refused(env, reason):
    out = subprocess.run([sys.executable, "-c", _SWITCH_SCRIPT, ROOT], env={**os.environ, **env}, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "REFUSED" in out.stdout and reason in out.stdout and "FP16 OK" in out.stdout, out.stdout


# ---- 5. each position's output is independent of the batch ----
def test_batch_independence():
    net, x = row_net("w288"), _x()
    big = x[torch.from_numpy(np.arange(4096) % M.N_POSITIONS).cuda()].contiguous()
    lg_all, v_all = _run(net, big)
    for i in range(M.N_POSITIONS, 4096, 7):
        assert np.array_equal(lg_all[i], lg_all[i % M.N_POSITIONS]) and v_all[i] == v_all[i % M.N_POSITIONS], i
    for B in (1, 37, 1031):
        lg, v = _run(net, big[:B].contiguous())
        assert np.array_equal(lg, lg_all[:B]) and np.array_equal(v, v_all[:B]), B


# ---- 6. format switches, workspace regrowth and graph replay on one net object ----
def test_format_switches_and_graph_replay():
    name = "w288"
    x = _x()
    big = x[torch.from_numpy(np.arange(1031) % M.N_POSITIONS).cuda()].contiguous()
    net = _net(name)
    fp16_before = _run(net, big[:8].contiguous(), "fp16")
    for step, (B, fmt) in enumerate([(8, "fp8"), (1031, "fp16"), (3, "fp8"), (1031, "fp8"), (8, "bf16"), (8, "fp16")]):
        planes = big[:B].contiguous()
        got = _run(net, planes, fmt)
        fresh = _run(_net(name), planes, fmt)
        assert np.array_equal(got[0], fresh[0]) and np.array_equal(got[1], fresh[1]), (step, B, fmt)
        lg, v = net.forward_planes_graphed(planes, fmt)
        assert np.array_equal(lg.cpu().numpy(), got[0]) and np.array_equal(v.cpu().numpy(), got[1]), (step, B, fmt)
    fp16_after = _run(net, big[:8].contiguous(), "fp16")
    assert np.array_equal(fp16_before[0], fp16_after[0]) and np.array_equal(fp16_before[1], fp16_after[1])


# ---- 7. agreement with the fp32 path on the 2,304 reference-init positions: the shipped model and ResNet-24 ----
# Floors from one B200 run (1000 W power limit, profiles/r06_fp8_gpu.log): top-1 over all logits / over legal moves and max |dv| were
# 90.5 % / 94.6 % / 0.049 for the shipped model and 90.4 % / 94.6 % / 0.067 for ResNet-24; the floors sit 1.5 points and ~1.5x under
# that.  fp8 is not held to the fp16 gate (99 % top-1): e4m3 tower noise is 2-3x bf16's on the logits.
AGREEMENT_FLOORS = {"shipped": (0.89, 0.93, 0.10), "r24": (0.89, 0.93, 0.10)}


def _agreement_nets(which, golden_dir):
    from matrix0_b200.model import PolicyValueNet
    from test_nn_gpu import _refinit
    r = _refinit(golden_dir)
    if which == "r24":
        cfg = r["cfg"]
        return (PolicyValueNet(cfg, device="cuda", precision="fp8", seed=0), PolicyValueNet(cfg, device="cuda", precision="fp32", seed=0), r)
    from test_shipped_model_gpu import shipped_model_cfg
    return (PolicyValueNet.from_config(shipped_model_cfg(), device="cuda", precision="fp8", seed=0),
            PolicyValueNet.from_config(shipped_model_cfg(), device="cuda", precision="fp32", seed=0), r)


@pytest.mark.parametrize("which", ["shipped", "r24"])
def test_agreement_with_the_fp32_path(golden_dir, which):
    from test_shipped_model_gpu import _agreement
    net, f32, r = _agreement_nets(which, golden_dir)
    a, al, dv = _agreement(net, f32, r["x"], r["legal"].cuda())
    print(f"\n[fp8 agreement] {which}: top-1 {a:.4f} legal top-1 {al:.4f} max|dv| {dv:.2e}")
    fa, fal, fdv = AGREEMENT_FLOORS[which]
    assert a >= fa and al >= fal and dv <= fdv, (a, al, dv)


# ---- 8. self-play end to end: collapsed and as-shipped search with no status bits ----
@pytest.mark.parametrize("search_mode", ["collapsed", "as_shipped"])
def test_selfplay_engine_plays_in_fp8(search_mode):
    from matrix0_b200.model import PolicyValueNet
    from matrix0_b200.selfplay import SelfPlayEngine
    from test_selfplay_gpu import MCTS_KW
    from test_shipped_model_gpu import shipped_model_cfg
    net = PolicyValueNet.from_config(shipped_model_cfg(), device="cuda", precision="fp8", seed=0)
    G, sims = 64, 32
    cfg = {"mcts": dict(MCTS_KW, num_simulations=sims, inference_batch_size=16),
           "selfplay": {"num_simulations": sims, "opening_random_plies": 4, "max_game_len": 10, "temperature_start": 1.2, "temperature_end": 0.3,
                        "temperature_moves": 40, "resign_threshold": -0.85, "min_resign_plies": 50}}
    sp = SelfPlayEngine(net, cfg, games=G, deterministic=False, seed=7, precision="fp8", search_mode=search_mode)
    sp.start()
    for _ in range(6):
        sp.play_move()
    torch.cuda.synchronize()
    assert sp.counters()["positions_played"] == 6 * G
    st, _ = sp.engine.status()
    assert int(st.abs().sum()) == 0


def test_selfplay_worker_with_the_shipped_model_in_fp8(tmp_path):
    import queue
    from matrix0_b200.selfplay import selfplay_worker
    from test_selfplay_gpu import MCTS_KW
    from test_shipped_model_gpu import shipped_model_cfg
    cfg = {"model": shipped_model_cfg(), "data_dir": str(tmp_path / "data"), "seed": 3,
           "mcts": dict(MCTS_KW, num_simulations=32, inference_batch_size=16),
           "selfplay": {"num_simulations": 32, "opening_random_plies": 4, "max_game_len": 8, "temperature_start": 1.0, "temperature_end": 0.3,
                        "temperature_moves": 40, "resign_threshold": -0.85, "min_resign_plies": 50}}
    assert selfplay_worker(0, cfg, None, games=4, q=queue.Queue(), concurrent_games=4, precision="fp8") == 4
    assert len(sorted((tmp_path / "data" / "selfplay").glob("selfplay_w0_g*.npz"))) == 4
