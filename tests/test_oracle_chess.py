"""Pin the oracle python-chess restatement: public perft constants, the reference's tactical KAT
(legal-move counts), its encoding known-answer tests, and -- when the reference tree is present --
the full fixture sweep (10k/40k/5k FENs, 140 PGN games)."""
import glob
import json
import os

import numpy as np
import pytest

import chess
from oracle import encoding_ref as E
from oracle import refload

PERFT = [
    (chess.STARTING_FEN, [20, 400, 8902]),
    ("r3k2r/p1ppqpb1/bn2pnp1/3PN3/1p2P3/2N2Q1p/PPPBBPPP/R3K2R w KQkq - 0 1", [48, 2039, 97862]),
    ("8/2p5/3p4/KP5r/1R3p1k/8/4P1P1/8 w - - 0 1", [14, 191, 2812, 43238]),
    ("r3k2r/Pppp1ppp/1b3nbN/nP6/BBP1P3/q4N2/Pp1P2PP/R2Q1RK1 w kq - 0 1", [6, 264, 9467]),
    ("rnbq1k1r/pp1Pbppp/2p5/8/2B5/8/PPP1NnPP/RNBQK2R w KQ - 1 8", [44, 1486, 62379]),
    ("r4rk1/1pp1qppp/p1np1n2/2b1p1B1/2B1P1b1/P1NP1N2/1PP1QPPP/R4RK1 w - - 0 10", [46, 2079, 89890]),
]


def perft(b, d):
    if d == 1:
        return sum(1 for _ in b.generate_legal_moves())
    n = 0
    for m in list(b.generate_legal_moves()):
        b.push(m)
        n += perft(b, d - 1)
        b.pop()
    return n


@pytest.mark.parametrize("fen,expected", PERFT)
def test_perft(fen, expected):
    b = chess.Board(fen)
    assert [perft(b, d + 1) for d in range(len(expected))] == expected


def test_tactical_kat(golden_dir):
    kat = json.load(open(os.path.join(golden_dir, "tactical_kat.json")))
    assert len(kat) == 1000
    for e in kat:
        b = chess.Board(e["fen"])
        legal = list(b.legal_moves)
        assert len(legal) == e["legal_moves"], e["fen"]
        assert chess.Move.from_uci(e["move"]) in legal


def test_encoding_golden(golden_dir):
    """oracle/encoding_ref + oracle/chess reproduce what the unmodified reference produced."""
    g = np.load(os.path.join(golden_dir, "encoding_golden.npz"))
    for i, fen in enumerate(g["fens"]):
        b = chess.Board(str(fen))
        planes = E.encode_board(b)
        bits = np.packbits(planes[:12].astype(np.uint8).reshape(-1))
        assert (bits == g["piece_bits"][i]).all(), fen
        assert planes[12:, 0, 0].tobytes() == g["const_planes"][i].tobytes(), fen
        mi = E.legal_moves_and_indices(b)
        n = int(g["counts"][i])
        assert len(mi) == n, fen
        assert [c for c, _ in mi] == g["moves"][i, :n].tolist(), fen
        assert [x for _, x in mi] == g["idx"][i, :n].tolist(), fen


# ---- the reference's own known-answer tests for this path, restated ------------------------------
def test_ref_kat_castling_indices():  # reference tests/test_encoding.py:23-30
    b = chess.Board("r3k2r/8/8/8/8/8/8/R3K2R w KQkq - 0 1")
    k = E.move_to_index(b, chess.Move.from_uci("e1g1"))
    q = E.move_to_index(b, chess.Move.from_uci("e1c1"))
    assert k != q and 0 <= k < 4672 and 0 <= q < 4672


def test_ref_kat_en_passant_kingless():  # tests/test_encoding.py:32-37
    b = chess.Board("8/8/8/3pP3/8/8/8/8 w - d6 0 2")
    assert 0 <= E.move_to_index(b, chess.Move.from_uci("e5d6")) < 4672


def test_ref_kat_underpromotion():  # tests/test_encoding.py:39-48
    b = chess.Board("8/P7/8/8/8/8/8/k6K w - - 0 1")
    n = E.move_to_index(b, chess.Move.from_uci("a7a8n"))
    q = E.move_to_index(b, chess.Move.from_uci("a7a8q"))
    assert n != q


def test_ref_kat_legal_mask_counts():  # tests/test_encoding.py:73-84
    b = chess.Board()
    m = E.get_legal_actions(b)
    assert m.shape == (4672,) and m.dtype == bool and m.sum() == 20
    b.push_san("e4")
    assert E.get_legal_actions(b).sum() == 20


def test_ref_kat_start_planes():  # tests/test_encoding.py:100-118
    enc = E.encode_board(chess.Board())
    assert (enc[0][6, :] == 1).all() and (enc[6][1, :] == 1).all()
    assert (enc[12] == 1).all() and (enc[13:17] == 1).all()


def test_ref_kat_board_tensor():  # tests/test_board_tensor.py:7-30
    t = E.encode_board(chess.Board("rnbqkbnr/pppppppp/8/8/4P3/8/PPPP1PPP/RNBQKBNR b KQkq e3 0 1"))
    assert t[0, 4, 4] == 1 and t[6, 1, 0] == 1
    assert (t[12] == 0).all() and (t[13:17] == 1).all() and t[17].mean() == 0
    assert abs(t[18].mean() - 0.005025) < 1e-6


def test_ref_kat_illegal_move_raises():  # tests/test_encoding.py:120-130
    with pytest.raises(ValueError):
        E.move_to_index(chess.Board(), chess.Move.from_uci("a1a8"))


def test_ref_kat_fools_mate_fen():  # tests/test_error_handling.py:146
    # the reference's "fool's mate" FEN has a pawn on g3, so it is NOT terminal; the real one is
    b = chess.Board("rnb1kbnr/pppp1ppp/8/4p3/6Pq/5PP1/PPPPP2P/RNBQKBNR w KQkq - 1 3")
    assert not b.is_game_over() and not b.is_check()
    b = chess.Board("rnb1kbnr/pppp1ppp/8/4p3/6Pq/5P2/PPPPP2P/RNBQKBNR w KQkq - 1 3")
    assert b.is_checkmate() and b.is_game_over() and b.result() == "0-1"


# ---- full sweep against the reference's data fixtures (where the reference tree is present) ------
needs_ref = pytest.mark.skipif(not refload.reference_available(), reason=refload.MISSING)


@needs_ref
@pytest.mark.slow
def test_reference_fixture_sweep():
    import chess.pgn
    R = os.path.join(refload.REFERENCE_ROOT, "data")
    for e in json.load(open(os.path.join(R, "tactical/tactical_metadata.json"))):
        b = chess.Board(e["fen"])
        legal = list(b.legal_moves)
        assert len(legal) == e["legal_moves"]
        assert chess.Move.from_uci(e["move"]) in legal
    for f in glob.glob(os.path.join(R, "stockfish_games/**/*.json"), recursive=True):
        s = json.load(open(f))
        for v in s.values():
            if isinstance(v, list):
                for e in v:
                    if isinstance(e, dict) and "fen" in e and e.get("best_move"):
                        chess.Board(e["fen"]).parse_uci(e["best_move"])
    for e in json.load(open(os.path.join(R, "openings/openings_metadata.json"))):
        chess.Board(e["fen"]).parse_san(e["move_san"])
    files = glob.glob(os.path.join(R, "eval_games/*.pgn")) + glob.glob(
        os.path.join(refload.REFERENCE_ROOT, "benchmarks/results/pgns_*/*.pgn"))
    plies = checks = mates = 0
    for f in files:
        with open(f) as fh:
            while True:
                g = chess.pgn.read_game(fh)
                if g is None:
                    break
                b = g.board()
                for san in g.san_moves:
                    b.push(b.parse_san(san))
                    plies += 1
                    if san.endswith("+"):
                        checks += 1
                        assert b.is_check() and not b.is_checkmate()
                    elif san.endswith("#"):
                        mates += 1
                        assert b.is_checkmate() and b.is_game_over()
                    else:
                        assert not b.is_check()
    assert (len(files), plies, checks, mates) == (140, 8464, 498, 111)  # SURVEY 4.4 [measured]


@needs_ref
def test_restatement_matches_unmodified_reference():
    """oracle/encoding_ref == the reference tree's azchess/encoding.py executed on the same boards."""
    from conftest import random_playout_boards
    enc = refload.load_reference("encoding")
    for b in random_playout_boards(12, 120, seed=11):
        assert E.encode_board(b).tobytes() == enc.encode_board(b).tobytes()
        assert [i for _, i in E.legal_moves_and_indices(b)] == [enc.move_to_index(b, m) for m in b.legal_moves]
        assert (E.get_legal_actions(b) == enc.move_encoder.get_legal_actions(b)).all()
