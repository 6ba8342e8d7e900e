"""Generate the committed golden vectors by running the UNMODIFIED reference modules
(azchess/encoding.py, mcts.py of the reference tree) on top of the oracle chess shim.

Needs the unmodified reference tree (oracle/_ref or MATRIX0_REFERENCE_ROOT):  python tests/golden/make_golden.py
Outputs (small, committed):
  tests/golden/encoding_golden.npz   positions + reference planes / move lists / policy indices
  tests/golden/tactical_kat.json     FEN + legal-move count + a legal move, sampled from the
                                     reference's data/tactical/tactical_metadata.json
  tests/golden/mcts_golden.json      reference MCTS.run visit counts with deterministic backends
"""
from __future__ import annotations

import json
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import refload  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

SPECIAL_FENS = [
    "rnbqkbnr/pppppppp/8/8/8/8/PPPPPPPP/RNBQKBNR w KQkq - 0 1",
    "r3k2r/8/8/8/8/8/8/R3K2R w KQkq - 0 1",                                   # tests/test_encoding.py:23-30
    "8/8/8/3pP3/8/8/8/8 w - d6 0 2",                                          # kingless e.p., :32-37
    "8/P7/8/8/8/8/8/k6K w - - 0 1",                                           # promotions, :39-48
    "r3k2r/p1ppqpb1/bn2pnp1/3PN3/1p2P3/2N2Q1p/PPPBBPPP/R3K2R w KQkq - 0 1",   # Kiwipete, :64-71
    "rnbqkbnr/pppppppp/8/8/4P3/8/PPPP1PPP/RNBQKBNR b KQkq e3 0 1",            # tests/test_board_tensor.py
    "rnb1kbnr/pppp1ppp/8/4p3/6Pq/5PP1/PPPPP2P/RNBQKBNR w KQkq - 1 3",         # test_error_handling.py:146
    "8/2p5/3p4/KP5r/1R3p1k/8/4P1P1/8 w - - 0 1",
    "r3k2r/Pppp1ppp/1b3nbN/nP6/BBP1P3/q4N2/Pp1P2PP/R2Q1RK1 w kq - 0 1",
    "rnbq1k1r/pp1Pbppp/2p5/8/2B5/8/PPP1NnPP/RNBQK2R w KQ - 1 8",
    "r4rk1/1pp1qppp/p1np1n2/2b1p1B1/2B1P1b1/P1NP1N2/1PP1QPPP/R4RK1 w - - 0 10",
    "8/8/8/8/k2Pp2Q/8/8/3K4 b - d3 0 1",                                      # e.p. skewer on the rank
    "8/8/8/2k5/3Pp3/8/8/4K3 b - d3 0 1",                                      # e.p. capture of a checking pawn
    "4k3/8/8/8/8/8/8/R3K2R w KQkq - 0 1",                                     # dirty castling flags
    "7k/8/8/8/8/8/8/K7 w - - 120 80", "7k/8/8/8/8/8/8/K6N w - - 99 250",      # clock saturation
    "2r3k1/5ppp/8/8/8/8/5PPP/2R3K1 b - - 3 31",
    "R6R/3Q4/1Q4Q1/4Q3/2Q4Q/Q4Q2/pp1Q4/kBNN1KB1 w - - 0 1",                   # 218 legal moves
]


def board_raw(b):
    ep = b.ep_square
    misc = (1 if b.turn else 0) | ((255 if ep is None else ep) << 8) | (min(b.halfmove_clock, 0xFFFF) << 16) \
        | (min(b.fullmove_number, 0xFFFF) << 32)
    return [b.pawns, b.knights, b.bishops, b.rooks, b.queens, b.kings, b.occupied_co[True], b.occupied_co[False],
            b.castling_rights, misc]


def main():
    enc, mcts_mod = refload.load_reference("encoding", "mcts")
    import chess

    # ---- encoding goldens ------------------------------------------------------------------
    rng = random.Random(20251018)
    boards = [chess.Board(f) for f in SPECIAL_FENS]
    while len(boards) < 400:
        b = chess.Board()
        for _ in range(rng.randint(0, 140)):
            if b.is_game_over():
                break
            b.push(rng.choice(list(b.legal_moves)))
        boards.append(b)
    tact = json.load(open(os.path.join(refload.REFERENCE_ROOT, "data/tactical/tactical_metadata.json")))
    rng.shuffle(tact)
    for e in tact[:112]:
        boards.append(chess.Board(e["fen"]))
    n = len(boards)
    raw = np.array([board_raw(b) for b in boards], dtype=np.uint64)
    planes = np.stack([enc.encode_board(b) for b in boards])
    piece_bits = np.packbits(planes[:, :12].astype(np.uint8).reshape(n, -1), axis=1)
    const_planes = planes[:, 12:, 0, 0].copy()
    assert (planes[:, 12:] == const_planes[:, :, None, None]).all()
    moves = np.zeros((n, 256), dtype=np.uint16)
    idx = np.zeros((n, 256), dtype=np.uint16)
    counts = np.zeros(n, dtype=np.int32)
    for i, b in enumerate(boards):
        lm = list(b.legal_moves)
        counts[i] = len(lm)
        for k, m in enumerate(lm):
            moves[i, k] = m.from_square | (m.to_square << 6) | ((m.promotion or 0) << 12)
            idx[i, k] = enc.move_to_index(b, m)
        mask = enc.move_encoder.get_legal_actions(b)
        assert sorted(np.nonzero(mask)[0].tolist()) == sorted(set(idx[i, :len(lm)].tolist()))
    np.savez_compressed(os.path.join(HERE, "encoding_golden.npz"), fens=np.array([b.fen(en_passant="fen") for b in boards]),
                        raw=raw, piece_bits=piece_bits, const_planes=const_planes, moves=moves, idx=idx, counts=counts)
    print("encoding goldens:", n, "positions, max moves", counts.max())

    kat = [{"fen": e["fen"], "legal_moves": e["legal_moves"], "move": e["move"]} for e in tact[112:1112]]
    json.dump(kat, open(os.path.join(HERE, "tactical_kat.json"), "w"))
    print("tactical KAT:", len(kat))
    make_mcts_golden(mcts_mod, chess)
    make_nn_golden()


NN_CASES = {
    # name -> overrides of config.yaml's model: section (SURVEY headline fact 3: R24 = 320 / 24 / 20)
    "small": dict(channels=64, blocks=6, attention_heads=4, policy_factor_rank=32),
    "r24": dict(channels=320, blocks=24, attention_heads=20),
}


def nn_inputs(n, seed):
    """Real encoded positions (binary planes) from seeded random playouts."""
    import chess
    from oracle.encoding_ref import encode_board
    rng = random.Random(seed)
    out = []
    while len(out) < n:
        b = chess.Board()
        for _ in range(rng.randint(0, 100)):
            if b.is_game_over():
                break
            b.push(rng.choice(list(b.legal_moves)))
        out.append(encode_board(b))
    return np.stack(out)


def make_nn_golden():
    """Outputs of the UNMODIFIED reference PolicyValueNet (fp32: infer_amp_tower off) on deterministic weights."""
    import torch
    import yaml
    from oracle import nn_ref
    from matrix0_b200.model import NetConfig, parameter_shapes
    resnet = refload.load_reference("model.resnet")
    base = yaml.safe_load(open(os.path.join(refload.REFERENCE_ROOT, "config.yaml")))["model"]
    out = {}
    for name, over in NN_CASES.items():
        d = dict(base)
        d.update(over)
        d["infer_amp_tower"] = False
        ref = resnet.PolicyValueNet.from_config(d).eval()
        known = set(NetConfig.__dataclass_fields__)
        cfg = NetConfig(**{k: v for k, v in d.items() if k in known})
        sd = nn_ref.make_state_dict(parameter_shapes(cfg), seed=1)
        ref.load_state_dict(sd, strict=False)
        x = torch.from_numpy(nn_inputs(6, seed=5))
        with torch.no_grad():
            p, v, ssl = ref(x, return_ssl=True)
        out[f"{name}_x"] = x.numpy()
        out[f"{name}_logits"] = p.numpy()
        out[f"{name}_values"] = v.numpy()
        for t, s in ssl.items():
            out[f"{name}_ssl_{t}"] = s.numpy()
        out[f"{name}_cfg"] = np.array(json.dumps(d))
    np.savez_compressed(os.path.join(HERE, "nn_golden.npz"), **out)
    print("nn goldens:", list(NN_CASES))


MCTS_CFGS = {
    # config.yaml mcts: section as self-play resolves it (SURVEY 8 "effective configuration"), noise off
    "selfplay": dict(cpuct=2.5, cpuct_start=3.0, cpuct_end=2.0, cpuct_plies=40, fpu_reduction=0.1, draw_penalty=-0.05,
                     legal_softmax=True, selection_jitter=0.05, inference_batch_size=96, no_instant_backtrack=True),
    # MCTSConfig defaults with a small batch and full-policy softmax
    "defaults_b8": dict(cpuct=1.7, fpu_reduction=0.15, legal_softmax=False, selection_jitter=0.0, inference_batch_size=8),
    "cbase": dict(cpuct_c_base=19652.0, cpuct_c_init=1.25, fpu_reduction=0.2, legal_softmax=True, inference_batch_size=32,
                  no_instant_backtrack=False, draw_penalty=-0.3),
}
MCTS_FENS = [
    "rnbqkbnr/pppppppp/8/8/8/8/PPPPPPPP/RNBQKBNR w KQkq - 0 1",
    "r3k2r/p1ppqpb1/bn2pnp1/3PN3/1p2P3/2N2Q1p/PPPBBPPP/R3K2R w KQkq - 0 1",
    "8/2p5/3p4/KP5r/1R3p1k/8/4P1P1/8 w - - 0 1",
    "6k1/5ppp/8/8/8/8/5PPP/3R2K1 w - - 0 1",          # mate in one available: terminal leaves inside a batch
    "7k/5Q2/6K1/8/8/8/8/8 b - - 0 1",                 # stalemate root -> terminal return
    "8/8/8/8/8/5k2/6q1/7K w - - 0 1",                 # checkmated root
    "4k3/8/8/8/8/8/8/4K2R w K - 148 90",              # 75-move rule two plies away
    "8/5k2/8/8/8/8/2K5/6B1 w - - 0 1",                # insufficient material root
]


def make_mcts_golden(ref, chess):
    """Visit counts of the UNMODIFIED reference MCTS.run with random.random() == 0.5, noise off."""
    import logging
    logging.disable(logging.CRITICAL)
    from oracle.backends import ConstantBackend, HashBackend
    ref.random.random = lambda: 0.5
    ref.psutil_available = False

    class _Model:
        class cfg:
            policy_size = 4672

    def new(cfg_name, backend, sims):
        kw = dict(MCTS_CFGS[cfg_name])
        cfg = ref.MCTSConfig(num_threads=1, enable_memory_cleanup=False, dirichlet_frac=0.0, enable_entropy_noise=False,
                             playout_random_frac=0.0, num_simulations=sims, **kw)
        be = ConstantBackend(backend[1]) if backend[0] == "const" else HashBackend(scale=backend[1], seed=backend[2])
        return ref.MCTS(cfg, _Model(), device="cpu", inference_backend=be)

    def record(m, board, ply):
        try:
            vc, pi, v = m.run(board, ply=ply)
        except RuntimeError as e:
            return {"error": "zero visits" if "zero visits" in str(e) else str(e)[:80]}
        root = m._last_root
        out = {"visits": [[mv.uci(), n] for mv, n in vc.items()], "value": v, "pi_nonzero": [[int(i), float(pi[i])] for i in np.nonzero(pi)[0]]}
        if root is not None:
            out["root_n"] = root.n
            out["child_q"] = [c.q for c in root.children.values()]
            out["child_prior"] = [c.prior for c in root.children.values()]
        return out

    cases = []
    rng = random.Random(7)
    # (1) fresh MCTS per call on fixed positions
    for cfg_name, backend, sims in [("selfplay", ("hash", 1.0, 0), 800), ("selfplay", ("hash", 0.02, 1), 800),
                                    ("defaults_b8", ("hash", 2.0, 2), 200), ("cbase", ("hash", 1.0, 3), 300),
                                    ("selfplay", ("const", 0.1), 800)]:
        for fen in MCTS_FENS:
            m = new(cfg_name, backend, sims)
            b = chess.Board(fen)
            cases.append({"kind": "fresh", "cfg": cfg_name, "backend": backend, "sims": sims, "fen": fen, "moves": [], "ply": 0,
                          "expect": record(m, b, 0)})
    # (2) fresh MCTS per move along a game (board carries its move stack -> repetition history)
    for cfg_name, backend, sims, fen, plies in [("selfplay", ("hash", 1.0, 4), 300, MCTS_FENS[0], 10),
                                                ("defaults_b8", ("hash", 1.5, 5), 120, MCTS_FENS[2], 12)]:
        b = chess.Board(fen)
        for ply in range(plies):
            if b.is_game_over():
                break
            m = new(cfg_name, backend, sims)
            exp = record(m, b, ply)
            cases.append({"kind": "game_fresh", "cfg": cfg_name, "backend": backend, "sims": sims, "fen": fen,
                          "moves": [mv.uci() for mv in b.move_stack], "ply": ply, "expect": exp})
            if "visits" not in exp:
                break
            best = max(exp["visits"], key=lambda kv: kv[1])[0]
            b.push(chess.Move.from_uci(best))
    # (3) shuffling history: the root has occurred before, so repetition draws appear inside the tree
    b = chess.Board()
    for uci in ["g1f3", "g8f6", "f3g1", "f6g8", "g1f3", "g8f6", "f3g1", "f6g8", "g1f3", "g8f6", "f3g1"]:
        b.push(chess.Move.from_uci(uci))
    m = new("selfplay", ("hash", 0.5, 6), 400)
    cases.append({"kind": "fresh", "cfg": "selfplay", "backend": ("hash", 0.5, 6), "sims": 400, "fen": MCTS_FENS[0],
                  "moves": [mv.uci() for mv in b.move_stack], "ply": 11, "expect": record(m, b, 11)})
    # (4) ONE persistent MCTS over consecutive plies (self-play usage, internal.py:305-408): tree reuse through the
    #     transposition table; the reference raises "zero visits" on the second move (DESIGN.md, quirk Q12)
    for cfg_name, backend, sims, fen in [("selfplay", ("hash", 1.0, 7), 300, MCTS_FENS[0]), ("defaults_b8", ("hash", 1.0, 8), 100, MCTS_FENS[1])]:
        m = new(cfg_name, backend, sims)
        b = chess.Board(fen)
        seq = []
        for ply in range(4):
            exp = record(m, b, ply)
            seq.append({"moves": [mv.uci() for mv in b.move_stack], "ply": ply, "expect": exp})
            if "visits" not in exp:
                break
            b.push(chess.Move.from_uci(max(exp["visits"], key=lambda kv: kv[1])[0]))
        cases.append({"kind": "persistent", "cfg": cfg_name, "backend": backend, "sims": sims, "fen": fen, "sequence": seq})
    # (5) two persistent instances alternating (arena usage, arena.py:157-192): roots are found in the TT
    for cfg_name, backend, sims, fen in [("selfplay", ("hash", 1.0, 9), 300, MCTS_FENS[0]), ("cbase", ("hash", 1.0, 10), 150, MCTS_FENS[1])]:
        ms = [new(cfg_name, backend, sims), new(cfg_name, backend, sims)]
        b = chess.Board(fen)
        seq = []
        for ply in range(10):
            if b.is_game_over():
                break
            exp = record(ms[ply % 2], b, ply)
            seq.append({"moves": [mv.uci() for mv in b.move_stack], "ply": ply, "expect": exp})
            if "visits" not in exp:
                break
            b.push(chess.Move.from_uci(max(exp["visits"], key=lambda kv: kv[1])[0]))
        cases.append({"kind": "alternating", "cfg": cfg_name, "backend": backend, "sims": sims, "fen": fen, "sequence": seq})
    json.dump({"configs": MCTS_CFGS, "cases": cases}, open(os.path.join(HERE, "mcts_golden.json"), "w"))
    print("mcts goldens:", len(cases), "cases")


if __name__ == "__main__":
    main()
