"""TEST INFRASTRUCTURE ONLY -- CPU restatement of ``azchess/encoding.py`` (numpy + oracle/chess).

Every function cites the reference lines it follows.  Pinned (tests/test_oracle_chess.py, run
where the reference tree is present) against the unmodified reference module executed on the same shim,
and against the reference's own known-answer tests (tests/test_encoding.py, test_board_tensor.py)
restated in tests/test_oracle_encoding.py.  Only tests/, smoke() and bench.py's CPU legs import it.
"""
from __future__ import annotations

import numpy as np

from . import chess_shim  # noqa: F401  (installs oracle/chess as `chess` when python-chess is absent)
import chess

RAY_DIRS = ((1, 0), (-1, 0), (0, 1), (0, -1), (1, 1), (1, -1), (-1, 1), (-1, -1))  # encoding.py:60-69
KNIGHT_DELTAS = ((-2, -1), (-2, 1), (-1, -2), (-1, 2), (1, -2), (1, 2), (2, -1), (2, 1))  # encoding.py:70-72
UNDERPROMO_PIECES = (chess.KNIGHT, chess.BISHOP, chess.ROOK)  # encoding.py:73


def _bitboard_to_plane(squares) -> np.ndarray:
    """encoding.py:40-46: row = 7 - rank, col = file."""
    plane = np.zeros((8, 8), dtype=np.float32)
    for sq in squares:
        plane[7 - chess.square_rank(sq), chess.square_file(sq)] = 1.0
    return plane


def encode_board(board, planes: int = 19) -> np.ndarray:
    """encoding.py:11-37."""
    P = []
    for color in (chess.WHITE, chess.BLACK):
        for piece in (chess.PAWN, chess.KNIGHT, chess.BISHOP, chess.ROOK, chess.QUEEN, chess.KING):
            P.append(_bitboard_to_plane(board.pieces(piece, color)))
    P.append(np.full((8, 8), 1.0 if board.turn == chess.WHITE else 0.0, dtype=np.float32))
    P.append(np.full((8, 8), 1.0 if board.has_kingside_castling_rights(chess.WHITE) else 0.0, dtype=np.float32))
    P.append(np.full((8, 8), 1.0 if board.has_queenside_castling_rights(chess.WHITE) else 0.0, dtype=np.float32))
    P.append(np.full((8, 8), 1.0 if board.has_kingside_castling_rights(chess.BLACK) else 0.0, dtype=np.float32))
    P.append(np.full((8, 8), 1.0 if board.has_queenside_castling_rights(chess.BLACK) else 0.0, dtype=np.float32))
    P.append(np.full((8, 8), min(board.halfmove_clock, 99) / 99.0, dtype=np.float32))
    P.append(np.full((8, 8), min(board.fullmove_number, 199) / 199.0, dtype=np.float32))
    if len(P) != planes:
        raise ValueError(f"Expected {planes} planes, got {len(P)}")
    return np.stack(P, axis=0).astype(np.float32)


def move_to_index_unchecked(white_to_move: bool, from_sq: int, to_sq: int, promotion) -> int:
    """encoding.py:123-150 without the legality test of :121."""
    fr, ff = from_sq >> 3, from_sq & 7
    tr, tf = to_sq >> 3, to_sq & 7
    dr, df = tr - fr, tf - ff
    if (dr, df) in KNIGHT_DELTAS:  # :129-131
        return from_sq * 73 + 56 + KNIGHT_DELTAS.index((dr, df))
    if promotion in UNDERPROMO_PIECES:  # :134-137, dirs :97-110
        dirs = ((1, 0), (1, -1), (1, 1)) if white_to_move else ((-1, 0), (-1, 1), (-1, -1))
        if (dr, df) in dirs:
            return from_sq * 73 + 64 + UNDERPROMO_PIECES.index(promotion) * 3 + dirs.index((dr, df))
    if dr == 0 or df == 0 or abs(dr) == abs(df):  # :140-146
        step = max(abs(dr), abs(df))
        sdr = 0 if dr == 0 else (1 if dr > 0 else -1)
        sdf = 0 if df == 0 else (1 if df > 0 else -1)
        if (sdr, sdf) in RAY_DIRS and 1 <= step <= 7:
            return from_sq * 73 + RAY_DIRS.index((sdr, sdf)) * 7 + (step - 1)
    raise ValueError("Illegal move")


def move_to_index(board, move) -> int:
    """encoding.py:113-150."""
    if not board.is_legal(move):
        raise ValueError(f"Illegal move: {move}")
    return move_to_index_unchecked(board.turn == chess.WHITE, move.from_square, move.to_square, move.promotion)


def legal_moves_and_indices(board):
    """[(move_code, policy_index)] in generation order -- what Node._expand iterates (mcts.py:140,153-156)."""
    out = []
    wtm = board.turn == chess.WHITE
    for m in board.generate_legal_moves():
        code = m.from_square | (m.to_square << 6) | ((m.promotion or 0) << 12)
        out.append((code, move_to_index_unchecked(wtm, m.from_square, m.to_square, m.promotion)))
    return out


def get_legal_actions(board) -> np.ndarray:
    """encoding.py:243-253."""
    mask = np.zeros(4672, dtype=bool)
    for _, idx in legal_moves_and_indices(board):
        mask[idx] = True
    return mask
