"""Host logic of the shared-memory evaluation seam (matrix0_b200/inference.py <-> azchess/selfplay/inference.py):
mailbox layout, client time-outs / errors, the server sweep with a test evaluator, interoperability with the UNMODIFIED
reference client and server where the reference tree is present (oracle/_ref or MATRIX0_REFERENCE_ROOT), and the loud failure
of the product entry point on a box without CUDA.  No compute of the product path runs here."""
import os
import sys
import threading

import numpy as np
import pytest
import torch

from matrix0_b200 import inference as m0inf
from matrix0_b200._native import NativeLibraryError
from oracle import refload

PLANES, POLICY = 19, 4672


def fake_rows(x: torch.Tensor):
    """A per-row function of the planes, so that any row mix-up between workers shows."""
    s = x.reshape(x.shape[0], -1)
    logits = (s[:, :64].sum(1, keepdim=True) + torch.arange(POLICY, dtype=torch.float32)[None] * 1e-3) * (1.0 + s[:, 100:101])
    values = torch.tanh(s.sum(1) * 1e-3)
    return logits, values


def fake_evaluate(resources, requests):
    total = requests[-1][1] + requests[-1][2]
    batch = torch.zeros((total, PLANES, 8, 8))
    for w, rows, first in requests:
        batch[first:first + rows] = resources[w]["request_tensor"][:rows]
    logits, values = fake_rows(batch)
    for w, rows, first in requests:
        resources[w]["response_policy_tensor"][:rows] = logits[first:first + rows]
        resources[w]["response_value_tensor"][:rows] = values[first:first + rows, None]


class ServerThread:
    def __init__(self, resources, evaluate=fake_evaluate):
        self.stop = threading.Event()
        self.sweeps = None
        self.t = threading.Thread(target=self._run, args=(resources, evaluate), daemon=True)

    def _run(self, resources, evaluate):
        self.sweeps = m0inf.serve_shared_memory(resources, evaluate, self.stop)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(10)
        assert not self.t.is_alive()


# the reference's mailbox keys in its order (inference.py:18-35), as test_reference_client_against_our_server compares them live
REFERENCE_KEYS = ("request_tensor", "response_policy_tensor", "response_value_tensor", "request_event", "response_event", "batch_size_tensor")


def test_mailbox_layout():
    """inference.py:18-35 -- keys, shapes, dtypes, shared memory."""
    res = m0inf.setup_shared_memory_for_worker(3, PLANES, POLICY, 96)
    assert tuple(res.keys()) == m0inf.RESOURCE_KEYS == REFERENCE_KEYS
    assert res["request_tensor"].shape == (96, PLANES, 8, 8) and res["request_tensor"].dtype == torch.float32
    assert res["response_policy_tensor"].shape == (96, POLICY) and res["response_policy_tensor"].dtype == torch.float32
    assert res["response_value_tensor"].shape == (96, 1) and res["response_value_tensor"].dtype == torch.float32
    assert res["batch_size_tensor"].shape == (1,) and res["batch_size_tensor"].dtype == torch.int32
    for k in ("request_tensor", "response_policy_tensor", "response_value_tensor", "batch_size_tensor"):
        assert res[k].is_shared() and not res[k].any()
    assert not res["request_event"].is_set() and not res["response_event"].is_set()


def test_timeout_table(monkeypatch):
    """inference.py:599-614."""
    monkeypatch.delenv("MATRIX0_FAST_TIMEOUTS", raising=False)
    t = m0inf.InferenceClient.request_timeout
    assert [t(1), t(8), t(9), t(32), t(64), t(96), t(4096)] == [10.0, 7.5, 5.0, 5.0, 10.0, 12.5, 15.0]
    monkeypatch.setenv("MATRIX0_FAST_TIMEOUTS", "0")
    assert [t(1), t(8), t(32), t(64), t(4096)] == [24.0, 18.0, 12.0, 24.0, 30.0]


def test_client_server_ragged_concurrent():
    """Three workers posting ragged batches concurrently (single position, (C,H,W) input, a full mailbox, float64 input):
    every worker gets exactly its own rows back."""
    caps = [96, 8, 32]
    resources = [m0inf.setup_shared_memory_for_worker(i, PLANES, POLICY, c) for i, c in enumerate(caps)]
    errors = []

    def worker(i):
        try:
            rng = np.random.default_rng(i)
            client = m0inf.InferenceClient(resources[i])
            for rows in [1, caps[i], 3, 0, caps[i] // 2]:
                if rows == 0:
                    x = rng.random((PLANES, 8, 8), dtype=np.float32)          # (C,H,W)
                    p, v = client.infer_np(x)
                    x = x[None]
                else:
                    x = rng.random((rows, PLANES, 8, 8)).astype(np.float64 if rows == 3 else np.float32)
                    p, v = client.infer_np(x)
                pr, vr = fake_rows(torch.from_numpy(x.astype(np.float32)))
                assert p.shape == (x.shape[0], POLICY) and v.shape == (x.shape[0],) and p.dtype == np.float32 and v.dtype == np.float32
                assert np.array_equal(p, pr.numpy()) and np.array_equal(v, vr.numpy())
        except Exception as e:  # surfaced in the main thread
            errors.append((i, repr(e)))

    with ServerThread(resources) as srv:
        ts = [threading.Thread(target=worker, args=(i,)) for i in range(3)]
        [t.start() for t in ts]
        [t.join(60) for t in ts]
    assert not errors, errors
    assert srv.sweeps >= 5
    assert all(not r["request_event"].is_set() and not r["response_event"].is_set() for r in resources)


def test_collect_requests_edge_cases():
    """inference.py:360-373: row count <= 0 is ignored, a row count above the capacity is clamped and written back;
    slices of one sweep are consecutive."""
    resources = [m0inf.setup_shared_memory_for_worker(i, PLANES, POLICY, 4) for i in range(4)]
    assert m0inf.collect_requests(resources) == []
    for i, n in enumerate([3, 0, 9, -2]):
        resources[i]["batch_size_tensor"][0] = n
        resources[i]["request_event"].set()
    assert m0inf.collect_requests(resources) == [(0, 3, 0), (2, 4, 3)]
    assert int(resources[2]["batch_size_tensor"][0]) == 4
    assert all(not r["request_event"].is_set() for r in resources)
    assert m0inf.collect_requests([]) == []


def test_client_errors(monkeypatch):
    """ValueError on a wrong rank (inference.py:589-591); no server -> 3 attempts, then RuntimeError chained to the
    TimeoutError (the reference's outermost handler wraps it, :676-681); a request larger than the mailbox fails the same way."""
    res = m0inf.setup_shared_memory_for_worker(0, PLANES, POLICY, 4)
    client = m0inf.InferenceClient(res)
    with pytest.raises(ValueError, match=r"expects \(B,C,H,W\) or \(C,H,W\)"):
        client.infer_np(np.zeros((8, 8), np.float32))
    monkeypatch.setattr(m0inf.InferenceClient, "_timeout_scale", 0.004)
    with pytest.raises(RuntimeError, match="Failed to copy data to shared memory: Inference timeout") as ei:
        client.infer_np(np.zeros((2, PLANES, 8, 8), np.float32))
    assert isinstance(ei.value.__cause__, TimeoutError) and "final attempt after 3 retries" in str(ei.value)
    assert not res["request_event"].is_set()                      # cleared by the retries, as in the reference
    with pytest.raises(RuntimeError, match="Failed to copy data to shared memory"):
        client.infer_np(np.zeros((5, PLANES, 8, 8), np.float32))


def test_server_survives_evaluator_error(monkeypatch):
    """inference.py:555-566: a failing batch clears the workers' events and the loop carries on; the client's retry
    does not re-post, so that request ends in the time-out error and the NEXT request is served."""
    res = [m0inf.setup_shared_memory_for_worker(0, PLANES, POLICY, 4)]
    calls = {"n": 0}

    def flaky(resources, requests):
        calls["n"] += 1
        if calls["n"] == 1:
            raise RuntimeError("boom")
        fake_evaluate(resources, requests)

    monkeypatch.setattr(m0inf.InferenceClient, "_timeout_scale", 0.02)
    client = m0inf.InferenceClient(res[0])
    x = np.ones((2, PLANES, 8, 8), np.float32)
    with ServerThread(res, flaky):
        with pytest.raises(RuntimeError, match="Inference timeout"):
            client.infer_np(x)
        p, v = client.infer_np(x)
    assert calls["n"] == 2 and np.array_equal(p, fake_rows(torch.from_numpy(x))[0].numpy())


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_product_server_fails_loudly_without_cuda():
    """No CPU evaluator behind the product entry point: the server raises and never reports ready."""
    res = [m0inf.setup_shared_memory_for_worker(0, PLANES, POLICY, 4)]
    stop, ready = threading.Event(), threading.Event()
    with pytest.raises(NativeLibraryError):
        m0inf.run_inference_server("cuda", {"planes": 19, "channels": 32, "blocks": 2}, None, stop, ready, res)
    assert not ready.is_set()


# ---- interoperability with the unmodified reference module (where the reference tree is present) --------------------
def _reference_inference():
    resnet = refload.load_reference("model.resnet")
    sys.modules["azchess.model"].PolicyValueNet = resnet.PolicyValueNet       # what azchess/model/__init__.py exports
    refload._stub_package("azchess.selfplay", os.path.join(refload.REFERENCE_ROOT, "azchess", "selfplay"))
    import importlib
    return importlib.import_module("azchess.selfplay.inference"), resnet


needs_reference = pytest.mark.skipif(not refload.reference_available(), reason=refload.MISSING)


@needs_reference
def test_reference_client_against_our_server():
    ref, _ = _reference_inference()
    ours = m0inf.setup_shared_memory_for_worker(0, PLANES, POLICY, 16)
    theirs = ref.setup_shared_memory_for_worker(1, PLANES, POLICY, 16)
    assert list(ours.keys()) == list(theirs.keys())
    for k in ours:
        if hasattr(ours[k], "shape"):
            assert ours[k].shape == theirs[k].shape and ours[k].dtype == theirs[k].dtype, k
    resources = [ours, theirs]                                     # our server serves a reference-made mailbox too
    x = np.random.default_rng(5).random((7, PLANES, 8, 8), dtype=np.float32)
    pr, vr = fake_rows(torch.from_numpy(x))
    with ServerThread(resources):
        for res in resources:
            p, v = ref.InferenceClient(res).infer_np(x)
            assert np.array_equal(p, pr.numpy()) and np.array_equal(v, vr.numpy())
            p1, v1 = m0inf.InferenceClient(res).infer_np(x[3])
            assert np.array_equal(p1[0], pr.numpy()[3]) and v1[0] == vr.numpy()[3]


@needs_reference
def test_reference_server_cannot_run_off_mps(caplog):
    """Why the opposite direction (our client against the reference server) has no live test: the unmodified
    ``run_inference_server`` dies before it reports ready on every device except "mps" -- the ``import torch.mps``
    statements inside the function (inference.py:147, :242) make ``torch`` a local name, so ``torch.cuda.is_available()``
    (:234) raises UnboundLocalError, which the outer handler only logs (:571-572).  Pinned here as a reference quirk."""
    ref, resnet = _reference_inference()
    cfg = dict(planes=19, channels=32, blocks=2, attention_heads=4, policy_size=POLICY, norm="group", preact=True,
               activation="silu", policy_factor_rank=0, ssl_tasks=["piece"])
    res = [m0inf.setup_shared_memory_for_worker(0, PLANES, POLICY, 8)]
    stop, ready = threading.Event(), threading.Event()
    t = threading.Thread(target=ref.run_inference_server, args=("cpu", cfg, None, stop, ready, res), daemon=True)
    with caplog.at_level("ERROR"):
        t.start()
        t.join(120)
    stop.set()
    assert not t.is_alive() and not ready.is_set()
    assert any("cannot access local variable 'torch'" in r.getMessage() for r in caplog.records)
