"""SHA-256 of the 16-bit forward's outputs (policy logits and values) for ResNet-24 and the 64-channel `small` net of
tests/golden/nn_golden.npz, fp16 and bf16, at B = 1, 37, 1031 and 4096 random-playout positions.  Run it once per tree in the same
GPU session to show that two builds compute bit-identical outputs:

    python tools/output_hashes.py [--root TREE] > hashes.json

--root imports the package of another (built) tree.  Needs a GPU."""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    import numpy as np
    import torch
    from matrix0_b200 import _native
    from matrix0_b200.model import NetConfig, PolicyValueNet
    from bench_selfplay import reference_cfg
    lib = _native.lib()
    g = np.load(os.path.join(args.root, "tests", "golden", "nn_golden.npz"))
    known = set(NetConfig.__dataclass_fields__)
    small = {k: v for k, v in json.loads(str(g["small_cfg"])).items() if k in known}
    pos = torch.empty((4096, 9), dtype=torch.int64, device="cuda")
    _native.check(lib.m0_random_playouts(pos.data_ptr(), 4096, 5, 60, _native.current_stream()))
    planes = torch.empty((4096, 19, 8, 8), dtype=torch.float32, device="cuda")
    _native.check(lib.m0_encode_planes(pos.data_ptr(), 4096, planes.data_ptr(), _native.current_stream()))
    out = {}
    for name, cfg in (("r24", reference_cfg(800)["model"]), ("small", small)):
        for prec in ("fp16", "bf16"):
            net = PolicyValueNet.from_config(cfg, device="cuda:0", precision=prec, seed=0)
            for n in (1, 37, 1031, 4096):
                p, v = net.forward_planes(planes[:n].contiguous(), prec)
                out[f"{name}/{prec}/{n}"] = hashlib.sha256(p.float().cpu().numpy().tobytes() + v.float().cpu().numpy().tobytes()).hexdigest()
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
