"""Golden vectors for the reduced-precision gate on the REFERENCE'S OWN random initialisation.

Needs the unmodified reference tree (oracle/_ref or MATRIX0_REFERENCE_ROOT):  python tests/golden/make_refinit_golden.py
  tests/golden/refinit_digest.json   SHA-256 of every parameter tensor of the UNMODIFIED reference
                                     ``PolicyValueNet.from_config(config.yaml model + R24 overrides)`` built under
                                     ``torch.manual_seed(0)`` (pins matrix0_b200.model.reference_init)
  tests/golden/refinit_golden.npz    fp32 outputs of that module (infer_amp_tower off, the fp32 oracle of SURVEY Q11) on
                                     N_POS real positions: FENs, argmax over all 4672 logits, argmax over the legal moves,
                                     values, the top-1/top-2 logit gaps and, for N_FP16 of them, the same quantities from the
                                     reference's OWN fp16 inference path (infer_amp_tower: true, resnet.py:676-677) -- the
                                     yardstick for what reduced precision costs in the reference itself.
"""
from __future__ import annotations

import hashlib
import json
import os
import random
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import refload  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
N_POS = 2304
N_FP16 = 384
R24 = dict(channels=320, blocks=24, attention_heads=20)


def positions(n, seed):
    """Distinct positions along seeded random playouts (0..100 plies), non-terminal."""
    import chess
    rng = random.Random(seed)
    out, seen = [], set()
    while len(out) < n:
        b = chess.Board()
        for _ in range(rng.randint(0, 100)):
            if b.is_game_over():
                break
            b.push(rng.choice(list(b.legal_moves)))
        if b.is_game_over():
            continue
        f = b.fen(en_passant="fen")
        if f not in seen:
            seen.add(f)
            out.append(b)
    return out


def summarise(p, v, legal):
    neg = np.where(legal, p, -np.inf)
    srt = np.sort(p, axis=1)
    srt_l = np.sort(neg, axis=1)
    return dict(top1=p.argmax(1).astype(np.int16), top1_legal=neg.argmax(1).astype(np.int16), value=v.astype(np.float32),
                gap=(srt[:, -1] - srt[:, -2]).astype(np.float32), gap_legal=(srt_l[:, -1] - srt_l[:, -2]).astype(np.float32),
                logit_std=p.std(axis=1).astype(np.float32))


def main():
    import torch
    import yaml
    import logging
    logging.disable(logging.CRITICAL)
    resnet = refload.load_reference("model.resnet")
    from oracle.encoding_ref import encode_board, get_legal_actions
    d = dict(yaml.safe_load(open(os.path.join(refload.REFERENCE_ROOT, "config.yaml")))["model"])
    d.update(R24)
    d32 = dict(d, infer_amp_tower=False)
    torch.manual_seed(0)
    ref = resnet.PolicyValueNet.from_config(d32).eval()
    digest = {k: hashlib.sha256(t.detach().contiguous().numpy().tobytes()).hexdigest() for k, t in ref.state_dict().items()}
    json.dump({"seed": 0, "model": d, "sha256": digest}, open(os.path.join(HERE, "refinit_digest.json"), "w"), indent=0)
    boards = positions(N_POS, seed=77)
    x = torch.from_numpy(np.stack([encode_board(b) for b in boards]))
    legal = np.stack([get_legal_actions(b) for b in boards])
    torch.set_num_threads(os.cpu_count() or 1)
    t0 = time.time()
    ps, vs = [], []
    with torch.no_grad():
        for i in range(0, N_POS, 128):
            p, v = ref(x[i:i + 128])
            ps.append(p.float().numpy())
            vs.append(v.float().numpy())
    p32, v32 = np.concatenate(ps), np.concatenate(vs).reshape(-1)
    print(f"fp32 reference forward: {N_POS} positions in {time.time() - t0:.1f}s; logit std {p32.std(axis=1).mean():.4f}")
    out = {"fens": np.array([b.fen(en_passant="fen") for b in boards]), "cfg": np.array(json.dumps(d))}
    out.update({k: a for k, a in summarise(p32, v32, legal).items()})
    # the reference's own fp16 inference path on a subset
    ref.cfg.infer_amp_tower = True
    t0 = time.time()
    ps, vs = [], []
    with torch.no_grad():
        for i in range(0, N_FP16, 128):
            p, v = ref(x[i:i + 128])
            ps.append(p.float().numpy())
            vs.append(v.float().numpy())
    p16, v16 = np.concatenate(ps), np.concatenate(vs).reshape(-1)
    s16 = summarise(p16, v16, legal[:N_FP16])
    out.update({"ref_fp16_" + k: a for k, a in s16.items()})
    agree = float((s16["top1"] == out["top1"][:N_FP16]).mean())
    agree_l = float((s16["top1_legal"] == out["top1_legal"][:N_FP16]).mean())
    dv = float(np.abs(v16 - v32[:N_FP16]).max())
    dl = float(np.abs(p16 - p32[:N_FP16]).max())
    print(f"reference fp16-autocast path vs its fp32 path ({N_FP16} positions, {time.time() - t0:.1f}s): top-1 {agree:.4f}, "
          f"legal top-1 {agree_l:.4f}, max|dv| {dv:.2e}, max|dlogit| {dl:.2e}")
    out["ref_fp16_summary"] = np.array(json.dumps({"n": N_FP16, "top1": agree, "top1_legal": agree_l, "max_dv": dv, "max_dlogit": dl}))
    np.savez_compressed(os.path.join(HERE, "refinit_golden.npz"), **out)
    print("median top-1 gap", float(np.median(out["gap"])), "median legal gap", float(np.median(out["gap_legal"])))


if __name__ == "__main__":
    main()
