"""The functional fp32 NN restatement (oracle/nn_ref.py) reproduces the committed outputs of the
UNMODIFIED reference PolicyValueNet (tests/golden/nn_golden.npz) and, where the reference tree is present,
is compared live with the reference module."""
import json
import os

import numpy as np
import pytest
import torch

from matrix0_b200.model import NetConfig, parameter_shapes
from oracle import nn_ref, refload


def load_case(golden_dir, name):
    g = np.load(os.path.join(golden_dir, "nn_golden.npz"))
    d = json.loads(str(g[f"{name}_cfg"]))
    known = set(NetConfig.__dataclass_fields__)
    cfg = NetConfig(**{k: v for k, v in d.items() if k in known})
    sd = nn_ref.make_state_dict(parameter_shapes(cfg), seed=1)
    return g, cfg, sd


@pytest.mark.parametrize("name", ["small", "r24"])
def test_restatement_reproduces_reference_outputs(golden_dir, name):
    g, cfg, sd = load_case(golden_dir, name)
    with torch.no_grad():
        p, v, ssl = nn_ref.forward(sd, cfg, torch.from_numpy(g[f"{name}_x"]), return_ssl=True)
    assert np.abs(p.numpy() - g[f"{name}_logits"]).max() < 2e-5
    assert np.abs(v.numpy() - g[f"{name}_values"]).max() < 2e-5
    for t, s in ssl.items():
        assert np.abs(s.numpy() - g[f"{name}_ssl_{t}"]).max() < 2e-5


@pytest.mark.skipif(not refload.reference_available(), reason=refload.MISSING)
def test_restatement_matches_reference_module_live(golden_dir):
    resnet = refload.load_reference("model.resnet")
    g, cfg, sd = load_case(golden_dir, "small")
    d = json.loads(str(g["small_cfg"]))
    ref = resnet.PolicyValueNet.from_config(d).eval()
    ref.load_state_dict(sd, strict=False)
    x = torch.rand(5, 19, 8, 8, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        p1, v1 = ref(x)
        p2, v2 = nn_ref.forward(sd, cfg, x)
    assert (p1 - p2).abs().max() < 2e-5 and (v1 - v2).abs().max() < 2e-5
    assert sorted(k for k in ref.state_dict() if k in sd) == sorted(sd)  # every key we model exists in the reference


def _refinit_cfg(golden_dir):
    d = json.load(open(os.path.join(golden_dir, "refinit_digest.json")))
    known = set(NetConfig.__dataclass_fields__)
    return d, NetConfig(**{k: v for k, v in d["model"].items() if k in known})


def test_reference_init_matches_committed_digests(golden_dir):
    """matrix0_b200.model.reference_init under torch.manual_seed(0) == the unmodified reference PolicyValueNet's own random
    initialisation (resnet.py:286-654), tensor by tensor (SHA-256 committed by tests/golden/make_refinit_golden.py)."""
    import hashlib
    from matrix0_b200.model import reference_init
    d, cfg = _refinit_cfg(golden_dir)
    torch.manual_seed(int(d["seed"]))
    sd = reference_init(cfg)
    shapes = parameter_shapes(cfg)
    assert set(shapes) <= set(d["sha256"])
    for k in shapes:
        assert tuple(sd[k].shape) == tuple(shapes[k]), k
        assert hashlib.sha256(sd[k].contiguous().numpy().tobytes()).hexdigest() == d["sha256"][k], k


@pytest.mark.skipif(not refload.reference_available(), reason=refload.MISSING)
def test_reference_init_matches_reference_module_live(golden_dir):
    from matrix0_b200.model import reference_init
    resnet = refload.load_reference("model.resnet")
    for over, seed in ((dict(channels=64, blocks=6, attention_heads=4, policy_factor_rank=32), 3),
                       (dict(channels=48, blocks=4, attention_heads=3, policy_factor_rank=0, ssl_tasks=["piece", "control"],
                             aux_policy_move_type=False, ssrl_tasks=["position", "rotation"]), 11)):
        d, _ = _refinit_cfg(golden_dir)
        m = dict(d["model"])
        m.update(over)
        torch.manual_seed(seed)
        ref = resnet.PolicyValueNet.from_config(m)
        after_ref = torch.rand(1)
        known = set(NetConfig.__dataclass_fields__)
        cfg = NetConfig(**{k: v for k, v in m.items() if k in known})
        torch.manual_seed(seed)
        sd = reference_init(cfg)
        assert torch.equal(torch.rand(1), after_ref)          # the generator was consumed exactly as the reference does
        rsd = ref.state_dict()
        for k in parameter_shapes(cfg):
            assert torch.equal(sd[k], rsd[k]), k
