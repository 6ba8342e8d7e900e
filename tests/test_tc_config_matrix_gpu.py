"""The fp16 / bf16 tensor-core forward against an fp64 reference on every row of the configuration matrix (tests/tc_matrix_cases.py):
every accepted width from 64 to 320, the head dims, the SE / attention / stem / policy-rank / activation branches, all with
non-unit gammas, non-zero betas and biases.  Only logits and values are compared, with the element-wise bars of tc_matrix_cases.BARS
(their calibration is checked without a GPU by tests/test_tc_matrix_bars.py).  ``-s`` prints one line of metrics per row."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import tc_matrix_cases as M

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_NETS = {}


def _net(name, sd=None):
    from matrix0_b200.model import PolicyValueNet
    net = PolicyValueNet(M.net_config(name), device="cuda", precision="fp16", seed=0)
    net.load_state_dict(M.state_dict(name) if sd is None else sd, strict=True)
    return net


def row_net(name):
    if name not in _NETS:
        _NETS[name] = _net(name)
    return _NETS[name]


def _x():
    return M.positions().cuda()


def _run(net, x, fmt):
    lg, v = net.forward_planes(x, fmt)
    return lg.cpu().numpy(), v.cpu().numpy()


def _fmt(m):
    return "(" + ", ".join(f"{v:.2e}" for v in m) + ")"


# ---- 1. every row, both 16-bit formats and the fp32 path, against the fp64 reference ----
@pytest.mark.parametrize("name", [r["name"] for r in M.ROWS])
def test_row_matches_fp64_reference(name):
    ref = M.reference(name)
    net, x = row_net(name), _x()
    got = {fmt: M.metrics(*_run(net, x, fmt), ref) for fmt in ("fp16", "bf16")}
    lg, v = _run(net, x, "fp32")
    rel = max(float(np.abs(lg - ref[0]).max()) / float(np.abs(ref[0]).max()), float(np.abs(v - ref[1]).max()) / float(np.abs(ref[1]).max()))
    print(f"\n[matrix] {name:16s} fp16 {_fmt(got['fp16'])} bf16 {_fmt(got['bf16'])} fp32 rel {rel:.2e}")
    assert rel <= M.FP32_REL, rel
    for fmt, m in got.items():
        assert M.within(m, fmt), (fmt, m, M.BARS[fmt])


# ---- 2. each row reaches the launch sites it is meant to cover, and not the others ----
@pytest.mark.parametrize("name", [r["name"] for r in M.ROWS])
def test_row_reaches_its_launch_sites(name):
    from matrix0_b200 import _native
    lib = _native.lib()
    net, x = row_net(name), _x()
    net.forward_planes(x, "fp16")
    torch.cuda.synchronize()
    _native.check(lib.m0_profile_enable(1))
    try:
        net.forward_planes(x, "fp16")
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


# ---- 3. the bars catch a wrong parameter end to end (faults loaded into the CUDA net, no kernel modified) ----
@pytest.mark.parametrize("name,fault,fmts", [("w288", "gn_gamma_tail", ("fp16",)), ("w288", "value_fc2_bias", ("fp16",)),
                                             ("w96", "conv_tap", ("fp16", "bf16"))])
def test_injected_fault_fails_the_bars(name, fault, fmts):
    net = _net(name, M.faulted_state_dict(name, fault))
    for fmt in fmts:
        m = M.metrics(*_run(net, _x(), fmt), M.reference(name))
        assert M.excess(m, fmt) >= 2.0, (fmt, m, M.BARS[fmt])


# ---- 4. batch edges: every batch size within the bars, and each position's output independent of the batch ----
@pytest.mark.parametrize("name", ["w256", "w288"])
@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
def test_batch_edges(name, fmt):
    net, x = row_net(name), _x()
    idx = np.arange(1031) % M.N_POSITIONS
    big = x[torch.from_numpy(idx).cuda()].contiguous()
    rl, rv = M.reference(name)
    lg_all, v_all = _run(net, big, fmt)
    for i in range(M.N_POSITIONS, 1031):          # the same position in another row of the batch
        assert np.array_equal(lg_all[i], lg_all[i % M.N_POSITIONS]) and v_all[i] == v_all[i % M.N_POSITIONS], i
    for B in (1, 2, 3, 63, 129, 257, 1031):
        lg, v = _run(net, big[:B].contiguous(), fmt)
        assert np.array_equal(lg, lg_all[:B]) and np.array_equal(v, v_all[:B]), B
        if B >= 2:
            m = M.metrics(lg, v, (rl[idx[:B]], rv[idx[:B]]))
            assert M.within(m, fmt), (B, m, M.BARS[fmt])


# ---- 5. workspace regrowth and format switches on one net object; graph replay equals the eager forward ----
def test_workspace_and_format_lifecycle():
    name = "w288"
    x = _x()
    big = x[torch.from_numpy(np.arange(1031) % M.N_POSITIONS).cuda()].contiguous()
    net = _net(name)
    for step, (B, fmt) in enumerate([(8, "fp16"), (1031, "bf16"), (3, "fp16"), (1031, "bf16"), (8, "fp16")]):
        planes = big[:B].contiguous()
        got = _run(net, planes, fmt)
        fresh = _run(_net(name), planes, fmt)
        assert np.array_equal(got[0], fresh[0]) and np.array_equal(got[1], fresh[1]), (step, B, fmt)
        lg, v = net.forward_planes_graphed(planes, fmt)
        assert np.array_equal(lg.cpu().numpy(), got[0]) and np.array_equal(v.cpu().numpy(), got[1]), (step, B, fmt)


# ---- nets of different widths in one process: each keeps running after the others have launched their kernels ----
def test_nets_of_every_width_take_turns_in_one_process():
    """The shared-memory limit of a kernel is one per device, not one per net: a narrow net that launched after a wide one must not
    leave the wide net's next launch without its shared memory."""
    names = [f"w{C}" for C in range(64, 321, 32)]
    x = _x()
    first = {n: _run(_net(n), x, "fp16") for n in names}
    nets = {n: _net(n) for n in names}
    for a in names:               # every ordered pair of widths back to back
        for n in (a, *names):
            got = _run(nets[n], x, "fp16")
            assert np.array_equal(got[0], first[n][0]) and np.array_equal(got[1], first[n][1]), (a, n)


# ---- 6. the A/B switches of the 16-bit forward compute the same network (one process per switch: they are read once) ----
SWITCHES = [{"M0_TC_FUSE_SE": "0"}, {"M0_SE_NOSPLIT": "1"}, {"M0_SE_TAIL": "0"}, {"M0_TC_PAIR": "0"}, {"M0_TC_PAIR_GEMM": "1"},
            {"M0_TC_ACC2": "0"}, {"M0_TC_PROJ_F32": "1"}, {"M0_TC_VALUE_TAIL": "0"}, {"M0_TC_SLICE_PROJ": "0"}, {"M0_TC_CLUSTER": "1"},
            {"M0_TC_STAGES": "2"}]
SWITCH_ROWS = ("w320", "w96")
_SWITCH_SCRIPT = r"""
import os, sys
import numpy as np
root, xpath, out = sys.argv[1:4]
sys.path[:0] = [root, os.path.join(root, "tests")]
from oracle import chess_shim  # noqa: F401
import torch
import tc_matrix_cases as M
from matrix0_b200.model import PolicyValueNet
x = torch.from_numpy(np.load(xpath)).cuda()
res = {}
for name in sys.argv[4:]:
    net = PolicyValueNet(M.net_config(name), device="cuda", precision="fp16", seed=0)
    net.load_state_dict(M.state_dict(name), strict=True)
    for fmt in ("fp16", "bf16"):
        lg, v = net.forward_planes(x, fmt)
        res[f"{name}/{fmt}/logits"], res[f"{name}/{fmt}/values"] = lg.cpu().numpy(), v.cpu().numpy()
np.savez(out, **res)
"""


def test_ab_switches_stay_within_the_bars(tmp_path):
    xpath = str(tmp_path / "x.npy")
    np.save(xpath, M.positions().numpy())
    procs = []
    for i, env in enumerate(SWITCHES):
        out = str(tmp_path / f"switch{i}.npz")
        log = open(tmp_path / f"switch{i}.log", "w")
        procs.append((env, out, log, subprocess.Popen([sys.executable, "-c", _SWITCH_SCRIPT, ROOT, xpath, out, *SWITCH_ROWS],
                                                      env={**os.environ, **env}, stdout=log, stderr=subprocess.STDOUT)))
    failures = []
    for env, out, log, p in procs:
        rc = p.wait(timeout=600)
        log.close()
        if rc != 0:
            failures.append((env, open(log.name).read()[-2000:]))
            continue
        with np.load(out) as r:
            for name in SWITCH_ROWS:
                for fmt in ("fp16", "bf16"):
                    m = M.metrics(r[f"{name}/{fmt}/logits"], r[f"{name}/{fmt}/values"], M.reference(name))
                    print(f"\n[switch] {env} {name} {fmt} {_fmt(m)}")
                    if not M.within(m, fmt):
                        failures.append((env, name, fmt, m))
    assert not failures, failures
