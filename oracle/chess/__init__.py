"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the python-chess subset Matrix0's hot path calls.

Matrix0 depends on the third-party PyPI package ``python-chess`` (import name ``chess``;
``requirements.txt:4`` pins ``python-chess[syzygy]>=1.9.0``, no lock file).  It is not vendored in
the reference tree and not a dependency of this repository, so its *published* algorithm (python-chess
1.9 - 1.11, ``chess/__init__.py``: bitboard board, ``generate_legal_moves`` ordering,
``_transposition_key``, game-end predicates) is restated here from its documented behaviour.
The module is deliberately shaped as a drop-in ``chess`` module: with ``oracle/`` on ``sys.path``
the reference's ``azchess/encoding.py``, ``azchess/mcts.py``, ``azchess/draw.py``,
``azchess/utils/board.py`` import and run unmodified on top of it (see ``oracle/refload.py``).

Reference call sites this restatement serves (SURVEY.md section 8c):
  encoding.py:22-33,43-44,121-126,163-165,193-196,219-228,247-252
  mcts.py:140,336-342,558,699,747,918-919,1185,1224-1227,1338-1343
  selfplay/internal.py:51-60,68,206-208,372-382,386,403,530,539,589,739-745
  draw.py:32-40,67-80 ; utils/board.py:28-37

Parity status: pinned against the reference's own fixtures (10k tactical FENs with legal-move
counts, 40k Stockfish FENs with a best move, 5k opening FENs with SAN, 140 PGN games replayed by
SAN with +/# suffixes) and public perft constants; see tests/test_oracle_chess.py.  Move ORDER is
only pinned by python-chess's documented generator structure (SURVEY Appendix A).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline/reference legs may import this.
"""
from __future__ import annotations

import re
from typing import Dict, Iterator, List, Optional, Tuple

Color = bool
COLORS = [WHITE, BLACK] = [True, False]
COLOR_NAMES = ["black", "white"]

PieceType = int
PIECE_TYPES = [PAWN, KNIGHT, BISHOP, ROOK, QUEEN, KING] = range(1, 7)
PIECE_SYMBOLS = [None, "p", "n", "b", "r", "q", "k"]
PIECE_NAMES = [None, "pawn", "knight", "bishop", "rook", "queen", "king"]

FILE_NAMES = ["a", "b", "c", "d", "e", "f", "g", "h"]
RANK_NAMES = ["1", "2", "3", "4", "5", "6", "7", "8"]

STARTING_FEN = "rnbqkbnr/pppppppp/8/8/8/8/PPPPPPPP/RNBQKBNR w KQkq - 0 1"
STARTING_BOARD_FEN = "rnbqkbnr/pppppppp/8/8/8/8/PPPPPPPP/RNBQKBNR"

Square = int
SQUARES = [
    A1, B1, C1, D1, E1, F1, G1, H1,
    A2, B2, C2, D2, E2, F2, G2, H2,
    A3, B3, C3, D3, E3, F3, G3, H3,
    A4, B4, C4, D4, E4, F4, G4, H4,
    A5, B5, C5, D5, E5, F5, G5, H5,
    A6, B6, C6, D6, E6, F6, G6, H6,
    A7, B7, C7, D7, E7, F7, G7, H7,
    A8, B8, C8, D8, E8, F8, G8, H8,
] = range(64)

SQUARE_NAMES = [f + r for r in RANK_NAMES for f in FILE_NAMES]


def parse_square(name: str) -> Square:
    return SQUARE_NAMES.index(name)


def square_name(square: Square) -> str:
    return SQUARE_NAMES[square]


def square(file_index: int, rank_index: int) -> Square:
    return rank_index * 8 + file_index


def square_file(square: Square) -> int:
    return square & 7


def square_rank(square: Square) -> int:
    return square >> 3


def square_distance(a: Square, b: Square) -> int:
    return max(abs(square_file(a) - square_file(b)), abs(square_rank(a) - square_rank(b)))


def square_mirror(square: Square) -> Square:
    return square ^ 0x38


Bitboard = int
BB_EMPTY = 0
BB_ALL = 0xFFFF_FFFF_FFFF_FFFF

BB_SQUARES = [
    BB_A1, BB_B1, BB_C1, BB_D1, BB_E1, BB_F1, BB_G1, BB_H1,
    BB_A2, BB_B2, BB_C2, BB_D2, BB_E2, BB_F2, BB_G2, BB_H2,
    BB_A3, BB_B3, BB_C3, BB_D3, BB_E3, BB_F3, BB_G3, BB_H3,
    BB_A4, BB_B4, BB_C4, BB_D4, BB_E4, BB_F4, BB_G4, BB_H4,
    BB_A5, BB_B5, BB_C5, BB_D5, BB_E5, BB_F5, BB_G5, BB_H5,
    BB_A6, BB_B6, BB_C6, BB_D6, BB_E6, BB_F6, BB_G6, BB_H6,
    BB_A7, BB_B7, BB_C7, BB_D7, BB_E7, BB_F7, BB_G7, BB_H7,
    BB_A8, BB_B8, BB_C8, BB_D8, BB_E8, BB_F8, BB_G8, BB_H8,
] = [1 << sq for sq in SQUARES]

BB_CORNERS = BB_A1 | BB_H1 | BB_A8 | BB_H8
BB_LIGHT_SQUARES = 0x55AA_55AA_55AA_55AA
BB_DARK_SQUARES = 0xAA55_AA55_AA55_AA55

BB_FILES = [BB_FILE_A, BB_FILE_B, BB_FILE_C, BB_FILE_D, BB_FILE_E, BB_FILE_F, BB_FILE_G, BB_FILE_H] = [
    0x0101_0101_0101_0101 << i for i in range(8)
]
BB_RANKS = [BB_RANK_1, BB_RANK_2, BB_RANK_3, BB_RANK_4, BB_RANK_5, BB_RANK_6, BB_RANK_7, BB_RANK_8] = [
    0xFF << (8 * i) for i in range(8)
]
BB_BACKRANKS = BB_RANK_1 | BB_RANK_8


def lsb(bb: Bitboard) -> int:
    return (bb & -bb).bit_length() - 1


def scan_forward(bb: Bitboard) -> Iterator[Square]:
    while bb:
        r = bb & -bb
        yield r.bit_length() - 1
        bb ^= r


def msb(bb: Bitboard) -> int:
    return bb.bit_length() - 1


def scan_reversed(bb: Bitboard) -> Iterator[Square]:
    while bb:
        r = bb.bit_length() - 1
        yield r
        bb ^= BB_SQUARES[r]


def popcount(bb: Bitboard) -> int:
    return bin(bb).count("1")


def _sliding_attacks(square: Square, occupied: Bitboard, deltas) -> Bitboard:
    attacks = BB_EMPTY
    for delta in deltas:
        sq = square
        while True:
            sq += delta
            if not (0 <= sq < 64) or square_distance(sq, sq - delta) > 2:
                break
            attacks |= BB_SQUARES[sq]
            if occupied & BB_SQUARES[sq]:
                break
    return attacks


def _step_attacks(square: Square, deltas) -> Bitboard:
    return _sliding_attacks(square, BB_ALL, deltas)


BB_KNIGHT_ATTACKS = [_step_attacks(sq, [17, 15, 10, 6, -17, -15, -10, -6]) for sq in SQUARES]
BB_KING_ATTACKS = [_step_attacks(sq, [9, 8, 7, 1, -9, -8, -7, -1]) for sq in SQUARES]
BB_PAWN_ATTACKS = [[_step_attacks(sq, deltas) for sq in SQUARES] for deltas in [[-7, -9], [7, 9]]]


def _edges(square: Square) -> Bitboard:
    return (((BB_RANK_1 | BB_RANK_8) & ~BB_RANKS[square_rank(square)]) |
            ((BB_FILE_A | BB_FILE_H) & ~BB_FILES[square_file(square)]))


def _carry_rippler(mask: Bitboard) -> Iterator[Bitboard]:
    subset = BB_EMPTY
    while True:
        yield subset
        subset = (subset - mask) & mask
        if not subset:
            break


def _attack_table(deltas) -> Tuple[List[Bitboard], List[Dict[Bitboard, Bitboard]]]:
    mask_table = []
    attack_table = []
    for sq in SQUARES:
        attacks = {}
        mask = _sliding_attacks(sq, 0, deltas) & ~_edges(sq)
        for subset in _carry_rippler(mask):
            attacks[subset] = _sliding_attacks(sq, subset, deltas)
        attack_table.append(attacks)
        mask_table.append(mask)
    return mask_table, attack_table


BB_DIAG_MASKS, BB_DIAG_ATTACKS = _attack_table([-9, -7, 7, 9])
BB_FILE_MASKS, BB_FILE_ATTACKS = _attack_table([-8, 8])
BB_RANK_MASKS, BB_RANK_ATTACKS = _attack_table([-1, 1])


def _rays() -> List[List[Bitboard]]:
    rays = []
    for a, bb_a in enumerate(BB_SQUARES):
        rays_row = []
        for b, bb_b in enumerate(BB_SQUARES):
            if BB_DIAG_ATTACKS[a][0] & bb_b:
                rays_row.append((BB_DIAG_ATTACKS[a][0] & BB_DIAG_ATTACKS[b][0]) | bb_a | bb_b)
            elif BB_RANK_ATTACKS[a][0] & bb_b:
                rays_row.append(BB_RANK_ATTACKS[a][0] | bb_a)
            elif BB_FILE_ATTACKS[a][0] & bb_b:
                rays_row.append(BB_FILE_ATTACKS[a][0] | bb_a)
            else:
                rays_row.append(BB_EMPTY)
        rays.append(rays_row)
    return rays


BB_RAYS = _rays()


def ray(a: Square, b: Square) -> Bitboard:
    return BB_RAYS[a][b]


def between(a: Square, b: Square) -> Bitboard:
    bb = BB_RAYS[a][b] & ((BB_ALL << a) ^ (BB_ALL << b))
    return bb & (bb - 1)


SAN_REGEX = re.compile(r"^([NBKRQ])?([a-h])?([1-8])?[\-x]?([a-h][1-8])(=?[nbrqkNBRQK])?[\+#]?\Z")


class IllegalMoveError(ValueError):
    pass


class AmbiguousMoveError(ValueError):
    pass


class InvalidMoveError(ValueError):
    pass


class Piece:
    __slots__ = ("piece_type", "color")

    def __init__(self, piece_type: PieceType, color: Color) -> None:
        self.piece_type = piece_type
        self.color = color

    def symbol(self) -> str:
        s = PIECE_SYMBOLS[self.piece_type]
        return s.upper() if self.color else s

    def __eq__(self, other) -> bool:
        return isinstance(other, Piece) and self.piece_type == other.piece_type and self.color == other.color

    def __hash__(self) -> int:
        return self.piece_type + (-1 if self.color else 5)

    def __repr__(self) -> str:
        return f"Piece.from_symbol({self.symbol()!r})"

    @classmethod
    def from_symbol(cls, symbol: str) -> "Piece":
        return cls(PIECE_SYMBOLS.index(symbol.lower()), symbol.isupper())


class Move:
    """(from_square, to_square, promotion, drop) value object; equality/hash over all four."""

    __slots__ = ("from_square", "to_square", "promotion", "drop")

    def __init__(self, from_square: Square, to_square: Square, promotion: Optional[PieceType] = None,
                 drop: Optional[PieceType] = None) -> None:
        self.from_square = from_square
        self.to_square = to_square
        self.promotion = promotion
        self.drop = drop

    def uci(self) -> str:
        if self.promotion:
            return SQUARE_NAMES[self.from_square] + SQUARE_NAMES[self.to_square] + PIECE_SYMBOLS[self.promotion]
        elif self:
            return SQUARE_NAMES[self.from_square] + SQUARE_NAMES[self.to_square]
        else:
            return "0000"

    def __bool__(self) -> bool:
        return bool(self.from_square or self.to_square or self.promotion or self.drop)

    def __eq__(self, other) -> bool:
        return (isinstance(other, Move) and self.from_square == other.from_square and
                self.to_square == other.to_square and self.promotion == other.promotion and self.drop == other.drop)

    def __hash__(self) -> int:
        return hash((self.from_square, self.to_square, self.promotion, self.drop))

    def __repr__(self) -> str:
        return f"Move.from_uci({self.uci()!r})"

    def __str__(self) -> str:
        return self.uci()

    @classmethod
    def from_uci(cls, uci: str) -> "Move":
        if uci == "0000":
            return cls.null()
        if 4 <= len(uci) <= 5:
            try:
                from_square = SQUARE_NAMES.index(uci[0:2])
                to_square = SQUARE_NAMES.index(uci[2:4])
                promotion = PIECE_SYMBOLS.index(uci[4]) if len(uci) == 5 else None
            except ValueError:
                raise InvalidMoveError(f"invalid uci: {uci!r}")
            if from_square == to_square:
                raise InvalidMoveError(f"invalid uci (use 0000 for null moves): {uci!r}")
            return cls(from_square, to_square, promotion=promotion)
        raise InvalidMoveError(f"expected uci string to be of length 4 or 5: {uci!r}")

    @classmethod
    def null(cls) -> "Move":
        return cls(0, 0)


class SquareSet:
    """Ascending-iteration set of squares (what ``Board.pieces`` returns)."""

    def __init__(self, squares: int = BB_EMPTY) -> None:
        self.mask = int(squares) & BB_ALL

    def __iter__(self) -> Iterator[Square]:
        return scan_forward(self.mask)

    def __reversed__(self) -> Iterator[Square]:
        return scan_reversed(self.mask)

    def __len__(self) -> int:
        return popcount(self.mask)

    def __contains__(self, square: Square) -> bool:
        return bool(BB_SQUARES[square] & self.mask)

    def __bool__(self) -> bool:
        return bool(self.mask)

    def __int__(self) -> int:
        return self.mask

    def __and__(self, other) -> "SquareSet":
        return SquareSet(self.mask & int(other))

    def __or__(self, other) -> "SquareSet":
        return SquareSet(self.mask | int(other))

    def __eq__(self, other) -> bool:
        try:
            return self.mask == int(other)
        except (TypeError, ValueError):
            return NotImplemented

    def __repr__(self) -> str:
        return f"SquareSet({self.mask:#021_x})"


class _BoardState:
    __slots__ = ("pawns", "knights", "bishops", "rooks", "queens", "kings", "occupied_w", "occupied_b", "occupied",
                 "promoted", "turn", "castling_rights", "ep_square", "halfmove_clock", "fullmove_number")

    def __init__(self, board: "Board") -> None:
        self.pawns = board.pawns
        self.knights = board.knights
        self.bishops = board.bishops
        self.rooks = board.rooks
        self.queens = board.queens
        self.kings = board.kings
        self.occupied_w = board.occupied_co[WHITE]
        self.occupied_b = board.occupied_co[BLACK]
        self.occupied = board.occupied
        self.promoted = board.promoted
        self.turn = board.turn
        self.castling_rights = board.castling_rights
        self.ep_square = board.ep_square
        self.halfmove_clock = board.halfmove_clock
        self.fullmove_number = board.fullmove_number

    def restore(self, board: "Board") -> None:
        board.pawns = self.pawns
        board.knights = self.knights
        board.bishops = self.bishops
        board.rooks = self.rooks
        board.queens = self.queens
        board.kings = self.kings
        board.occupied_co[WHITE] = self.occupied_w
        board.occupied_co[BLACK] = self.occupied_b
        board.occupied = self.occupied
        board.promoted = self.promoted
        board.turn = self.turn
        board.castling_rights = self.castling_rights
        board.ep_square = self.ep_square
        board.halfmove_clock = self.halfmove_clock
        board.fullmove_number = self.fullmove_number


class Outcome:
    def __init__(self, termination: str, winner: Optional[Color]) -> None:
        self.termination = termination
        self.winner = winner

    def result(self) -> str:
        return "1/2-1/2" if self.winner is None else ("1-0" if self.winner else "0-1")


class Board:
    """Standard-chess bitboard board with a move stack (python-chess ``Board`` subset)."""

    chess960 = False

    def __init__(self, fen: Optional[str] = STARTING_FEN) -> None:
        self.occupied_co = [BB_EMPTY, BB_EMPTY]
        self.move_stack: List[Move] = []
        self._stack: List[_BoardState] = []
        self.ep_square: Optional[Square] = None
        if fen is None:
            self.clear()
        elif fen == STARTING_FEN:
            self.reset()
        else:
            self.set_fen(fen)

    # ---- setup ---------------------------------------------------------------------------
    def reset(self) -> None:
        self.turn = WHITE
        self.castling_rights = BB_CORNERS
        self.ep_square = None
        self.halfmove_clock = 0
        self.fullmove_number = 1
        self.pawns = BB_RANK_2 | BB_RANK_7
        self.knights = BB_B1 | BB_G1 | BB_B8 | BB_G8
        self.bishops = BB_C1 | BB_F1 | BB_C8 | BB_F8
        self.rooks = BB_CORNERS
        self.queens = BB_D1 | BB_D8
        self.kings = BB_E1 | BB_E8
        self.promoted = BB_EMPTY
        self.occupied_co[WHITE] = BB_RANK_1 | BB_RANK_2
        self.occupied_co[BLACK] = BB_RANK_7 | BB_RANK_8
        self.occupied = BB_RANK_1 | BB_RANK_2 | BB_RANK_7 | BB_RANK_8
        self.clear_stack()

    def clear(self) -> None:
        self.turn = WHITE
        self.castling_rights = BB_EMPTY
        self.ep_square = None
        self.halfmove_clock = 0
        self.fullmove_number = 1
        self._clear_board()
        self.clear_stack()

    def _clear_board(self) -> None:
        self.pawns = self.knights = self.bishops = self.rooks = self.queens = self.kings = BB_EMPTY
        self.promoted = BB_EMPTY
        self.occupied_co[WHITE] = BB_EMPTY
        self.occupied_co[BLACK] = BB_EMPTY
        self.occupied = BB_EMPTY

    def clear_stack(self) -> None:
        self.move_stack.clear()
        self._stack.clear()

    def set_fen(self, fen: str) -> None:
        parts = fen.split()
        try:
            board_part = parts.pop(0)
        except IndexError:
            raise ValueError("empty fen")
        turn_part = parts.pop(0) if parts else "w"
        if turn_part == "w":
            turn = WHITE
        elif turn_part == "b":
            turn = BLACK
        else:
            raise ValueError(f"expected 'w' or 'b' for turn part of fen: {fen!r}")
        castling_part = parts.pop(0) if parts else "-"
        ep_part = parts.pop(0) if parts else "-"
        ep_square = None if ep_part == "-" else SQUARE_NAMES.index(ep_part)
        halfmove_part = parts.pop(0) if parts else "0"
        halfmove_clock = int(halfmove_part)
        if halfmove_clock < 0:
            raise ValueError("halfmove clock cannot be negative")
        fullmove_part = parts.pop(0) if parts else "1"
        fullmove_number = max(int(fullmove_part), 1)
        if parts:
            raise ValueError(f"fen string has more parts than expected: {fen!r}")
        self._set_board_fen(board_part)
        self.turn = turn
        self._set_castling_fen(castling_part)
        self.ep_square = ep_square
        self.halfmove_clock = halfmove_clock
        self.fullmove_number = fullmove_number
        self.clear_stack()

    def _set_board_fen(self, fen: str) -> None:
        rows = fen.split("/")
        if len(rows) != 8:
            raise ValueError(f"expected 8 rows in position part of fen: {fen!r}")
        self._clear_board()
        square_index = 0
        for c in fen:
            if c in "12345678":
                square_index += int(c)
            elif c == "/":
                pass
            elif c == "~":
                self.promoted |= BB_SQUARES[(square_index - 1) ^ 0x38]
            elif c.lower() in "pnbrqk":
                piece = Piece.from_symbol(c)
                self._set_piece_at(square_index ^ 0x38, piece.piece_type, piece.color)
                square_index += 1
            else:
                raise ValueError(f"invalid character in position part of fen: {fen!r}")

    def _set_castling_fen(self, castling_fen: str) -> None:
        self.castling_rights = BB_EMPTY
        if not castling_fen or castling_fen == "-":
            return
        for flag in castling_fen:
            color = WHITE if flag.isupper() else BLACK
            flag = flag.lower()
            backrank = BB_RANK_1 if color == WHITE else BB_RANK_8
            rooks = self.occupied_co[color] & self.rooks & backrank
            king = self.king(color)
            if flag == "q":
                # Select the leftmost rook.
                if king is not None and rooks and lsb(rooks) < king:
                    self.castling_rights |= rooks & -rooks
                else:
                    self.castling_rights |= BB_FILE_A & backrank
            elif flag == "k":
                # Select the rightmost rook.
                rook = msb(rooks) if rooks else -1
                if king is not None and rooks and king < rook:
                    self.castling_rights |= BB_SQUARES[rook]
                else:
                    self.castling_rights |= BB_FILE_H & backrank
            else:
                self.castling_rights |= BB_FILES[FILE_NAMES.index(flag)] & backrank

    # ---- piece access --------------------------------------------------------------------
    def pieces_mask(self, piece_type: PieceType, color: Color) -> Bitboard:
        if piece_type == PAWN:
            bb = self.pawns
        elif piece_type == KNIGHT:
            bb = self.knights
        elif piece_type == BISHOP:
            bb = self.bishops
        elif piece_type == ROOK:
            bb = self.rooks
        elif piece_type == QUEEN:
            bb = self.queens
        elif piece_type == KING:
            bb = self.kings
        else:
            raise AssertionError(f"expected PieceType, got {piece_type!r}")
        return bb & self.occupied_co[color]

    def pieces(self, piece_type: PieceType, color: Color) -> SquareSet:
        return SquareSet(self.pieces_mask(piece_type, color))

    def piece_type_at(self, square: Square) -> Optional[PieceType]:
        mask = BB_SQUARES[square]
        if not self.occupied & mask:
            return None
        elif self.pawns & mask:
            return PAWN
        elif self.knights & mask:
            return KNIGHT
        elif self.bishops & mask:
            return BISHOP
        elif self.rooks & mask:
            return ROOK
        elif self.queens & mask:
            return QUEEN
        else:
            return KING

    def piece_at(self, square: Square) -> Optional[Piece]:
        piece_type = self.piece_type_at(square)
        if piece_type:
            return Piece(piece_type, bool(self.occupied_co[WHITE] & BB_SQUARES[square]))
        return None

    def color_at(self, square: Square) -> Optional[Color]:
        mask = BB_SQUARES[square]
        if self.occupied_co[WHITE] & mask:
            return WHITE
        elif self.occupied_co[BLACK] & mask:
            return BLACK
        return None

    def king(self, color: Color) -> Optional[Square]:
        king_mask = self.occupied_co[color] & self.kings & ~self.promoted
        return msb(king_mask) if king_mask else None

    def piece_map(self) -> Dict[Square, Piece]:
        return {sq: self.piece_at(sq) for sq in scan_reversed(self.occupied)}

    def _remove_piece_at(self, square: Square) -> Optional[PieceType]:
        piece_type = self.piece_type_at(square)
        mask = BB_SQUARES[square]
        if piece_type == PAWN:
            self.pawns ^= mask
        elif piece_type == KNIGHT:
            self.knights ^= mask
        elif piece_type == BISHOP:
            self.bishops ^= mask
        elif piece_type == ROOK:
            self.rooks ^= mask
        elif piece_type == QUEEN:
            self.queens ^= mask
        elif piece_type == KING:
            self.kings ^= mask
        else:
            return None
        self.occupied ^= mask
        self.occupied_co[WHITE] &= ~mask
        self.occupied_co[BLACK] &= ~mask
        self.promoted &= ~mask
        return piece_type

    def _set_piece_at(self, square: Square, piece_type: PieceType, color: Color, promoted: bool = False) -> None:
        self._remove_piece_at(square)
        mask = BB_SQUARES[square]
        if piece_type == PAWN:
            self.pawns |= mask
        elif piece_type == KNIGHT:
            self.knights |= mask
        elif piece_type == BISHOP:
            self.bishops |= mask
        elif piece_type == ROOK:
            self.rooks |= mask
        elif piece_type == QUEEN:
            self.queens |= mask
        elif piece_type == KING:
            self.kings |= mask
        else:
            return
        self.occupied ^= mask
        self.occupied_co[color] ^= mask
        if promoted:
            self.promoted ^= mask

    def set_piece_at(self, square: Square, piece: Optional[Piece], promoted: bool = False) -> None:
        if piece is None:
            self._remove_piece_at(square)
        else:
            self._set_piece_at(square, piece.piece_type, piece.color, promoted)

    # ---- attacks -------------------------------------------------------------------------
    def attacks_mask(self, square: Square) -> Bitboard:
        bb_square = BB_SQUARES[square]
        if bb_square & self.pawns:
            color = bool(bb_square & self.occupied_co[WHITE])
            return BB_PAWN_ATTACKS[color][square]
        elif bb_square & self.knights:
            return BB_KNIGHT_ATTACKS[square]
        elif bb_square & self.kings:
            return BB_KING_ATTACKS[square]
        else:
            attacks = 0
            if bb_square & self.bishops or bb_square & self.queens:
                attacks = BB_DIAG_ATTACKS[square][BB_DIAG_MASKS[square] & self.occupied]
            if bb_square & self.rooks or bb_square & self.queens:
                attacks |= (BB_RANK_ATTACKS[square][BB_RANK_MASKS[square] & self.occupied] |
                            BB_FILE_ATTACKS[square][BB_FILE_MASKS[square] & self.occupied])
            return attacks

    def _attackers_mask(self, color: Color, square: Square, occupied: Bitboard) -> Bitboard:
        rank_pieces = BB_RANK_MASKS[square] & occupied
        file_pieces = BB_FILE_MASKS[square] & occupied
        diag_pieces = BB_DIAG_MASKS[square] & occupied
        queens_and_rooks = self.queens | self.rooks
        queens_and_bishops = self.queens | self.bishops
        attackers = (
            (BB_KING_ATTACKS[square] & self.kings) |
            (BB_KNIGHT_ATTACKS[square] & self.knights) |
            (BB_RANK_ATTACKS[square][rank_pieces] & queens_and_rooks) |
            (BB_FILE_ATTACKS[square][file_pieces] & queens_and_rooks) |
            (BB_DIAG_ATTACKS[square][diag_pieces] & queens_and_bishops) |
            (BB_PAWN_ATTACKS[not color][square] & self.pawns))
        return attackers & self.occupied_co[color]

    def attackers_mask(self, color: Color, square: Square) -> Bitboard:
        return self._attackers_mask(color, square, self.occupied)

    def is_attacked_by(self, color: Color, square: Square) -> bool:
        return bool(self.attackers_mask(color, square))

    def attackers(self, color: Color, square: Square) -> SquareSet:
        return SquareSet(self.attackers_mask(color, square))

    def pin_mask(self, color: Color, square: Square) -> Bitboard:
        king = self.king(color)
        if king is None:
            return BB_ALL
        square_mask = BB_SQUARES[square]
        for attacks, sliders in [(BB_FILE_ATTACKS, self.rooks | self.queens),
                                 (BB_RANK_ATTACKS, self.rooks | self.queens),
                                 (BB_DIAG_ATTACKS, self.bishops | self.queens)]:
            rays = attacks[king][0]
            if rays & square_mask:
                snipers = rays & sliders & self.occupied_co[not color]
                for sniper in scan_reversed(snipers):
                    if between(sniper, king) & (self.occupied | square_mask) == square_mask:
                        return ray(king, sniper)
                break
        return BB_ALL

    def checkers_mask(self) -> Bitboard:
        king = self.king(self.turn)
        return BB_EMPTY if king is None else self.attackers_mask(not self.turn, king)

    def is_check(self) -> bool:
        return bool(self.checkers_mask())

    # ---- move generation (order defines Node.children order, SURVEY Appendix A) ----------
    def generate_pseudo_legal_moves(self, from_mask: Bitboard = BB_ALL, to_mask: Bitboard = BB_ALL) -> Iterator[Move]:
        our_pieces = self.occupied_co[self.turn]

        # Generate piece moves.
        non_pawns = our_pieces & ~self.pawns & from_mask
        for from_square in scan_reversed(non_pawns):
            moves = self.attacks_mask(from_square) & ~our_pieces & to_mask
            for to_square in scan_reversed(moves):
                yield Move(from_square, to_square)

        # Generate castling moves.
        if from_mask & self.kings:
            yield from self.generate_castling_moves(from_mask, to_mask)

        # The remaining moves are all pawn moves.
        pawns = self.pawns & self.occupied_co[self.turn] & from_mask
        if not pawns:
            return

        # Generate pawn captures.
        capturers = pawns
        for from_square in scan_reversed(capturers):
            targets = BB_PAWN_ATTACKS[self.turn][from_square] & self.occupied_co[not self.turn] & to_mask
            for to_square in scan_reversed(targets):
                if square_rank(to_square) in [0, 7]:
                    yield Move(from_square, to_square, QUEEN)
                    yield Move(from_square, to_square, ROOK)
                    yield Move(from_square, to_square, BISHOP)
                    yield Move(from_square, to_square, KNIGHT)
                else:
                    yield Move(from_square, to_square)

        # Prepare pawn advance generation.
        if self.turn == WHITE:
            single_moves = pawns << 8 & ~self.occupied
            double_moves = single_moves << 8 & ~self.occupied & (BB_RANK_3 | BB_RANK_4)
        else:
            single_moves = pawns >> 8 & ~self.occupied
            double_moves = single_moves >> 8 & ~self.occupied & (BB_RANK_6 | BB_RANK_5)

        single_moves &= to_mask
        double_moves &= to_mask

        # Generate single pawn moves.
        for to_square in scan_reversed(single_moves):
            from_square = to_square + (8 if self.turn == BLACK else -8)
            if square_rank(to_square) in [0, 7]:
                yield Move(from_square, to_square, QUEEN)
                yield Move(from_square, to_square, ROOK)
                yield Move(from_square, to_square, BISHOP)
                yield Move(from_square, to_square, KNIGHT)
            else:
                yield Move(from_square, to_square)

        # Generate double pawn moves.
        for to_square in scan_reversed(double_moves):
            from_square = to_square + (16 if self.turn == BLACK else -16)
            yield Move(from_square, to_square)

        # Generate en passant captures.
        if self.ep_square:
            yield from self.generate_pseudo_legal_ep(from_mask, to_mask)

    def generate_pseudo_legal_ep(self, from_mask: Bitboard = BB_ALL, to_mask: Bitboard = BB_ALL) -> Iterator[Move]:
        if not self.ep_square or not BB_SQUARES[self.ep_square] & to_mask:
            return
        if BB_SQUARES[self.ep_square] & self.occupied:
            return
        capturers = (
            self.pawns & self.occupied_co[self.turn] & from_mask &
            BB_PAWN_ATTACKS[not self.turn][self.ep_square] &
            BB_RANKS[4 if self.turn else 3])
        for capturer in scan_reversed(capturers):
            yield Move(capturer, self.ep_square)

    def _attacked_for_king(self, path: Bitboard, occupied: Bitboard) -> bool:
        return any(self._attackers_mask(not self.turn, sq, occupied) for sq in scan_reversed(path))

    def generate_castling_moves(self, from_mask: Bitboard = BB_ALL, to_mask: Bitboard = BB_ALL) -> Iterator[Move]:
        backrank = BB_RANK_1 if self.turn == WHITE else BB_RANK_8
        king = self.occupied_co[self.turn] & self.kings & ~self.promoted & backrank & from_mask
        king &= -king
        if not king:
            return
        bb_c = BB_FILE_C & backrank
        bb_d = BB_FILE_D & backrank
        bb_f = BB_FILE_F & backrank
        bb_g = BB_FILE_G & backrank
        for candidate in scan_reversed(self.clean_castling_rights() & backrank & to_mask):
            rook = BB_SQUARES[candidate]
            a_side = rook < king
            king_to = bb_c if a_side else bb_g
            rook_to = bb_d if a_side else bb_f
            king_path = between(msb(king), msb(king_to))
            rook_path = between(candidate, msb(rook_to))
            if not ((self.occupied ^ king ^ rook) & (king_path | rook_path | king_to | rook_to) or
                    self._attacked_for_king(king_path | king, self.occupied ^ king) or
                    self._attacked_for_king(king_to, self.occupied ^ king ^ rook ^ rook_to)):
                yield self._from_chess960(self.chess960, msb(king), candidate)

    def _from_chess960(self, chess960: bool, from_square: Square, to_square: Square,
                       promotion: Optional[PieceType] = None, drop: Optional[PieceType] = None) -> Move:
        if not chess960 and promotion is None and drop is None:
            if from_square == E1 and self.kings & BB_E1:
                if to_square == H1:
                    return Move(E1, G1)
                elif to_square == A1:
                    return Move(E1, C1)
            elif from_square == E8 and self.kings & BB_E8:
                if to_square == H8:
                    return Move(E8, G8)
                elif to_square == A8:
                    return Move(E8, C8)
        return Move(from_square, to_square, promotion, drop)

    def _to_chess960(self, move: Move) -> Move:
        if move.from_square == E1 and self.kings & BB_E1:
            if move.to_square == G1 and not self.rooks & BB_G1:
                return Move(E1, H1)
            elif move.to_square == C1 and not self.rooks & BB_C1:
                return Move(E1, A1)
        elif move.from_square == E8 and self.kings & BB_E8:
            if move.to_square == G8 and not self.rooks & BB_G8:
                return Move(E8, H8)
            elif move.to_square == C8 and not self.rooks & BB_C8:
                return Move(E8, A8)
        return move

    def _slider_blockers(self, king: Square) -> Bitboard:
        rooks_and_queens = self.rooks | self.queens
        bishops_and_queens = self.bishops | self.queens
        snipers = ((BB_RANK_ATTACKS[king][0] & rooks_and_queens) |
                   (BB_FILE_ATTACKS[king][0] & rooks_and_queens) |
                   (BB_DIAG_ATTACKS[king][0] & bishops_and_queens))
        blockers = 0
        for sniper in scan_reversed(snipers & self.occupied_co[not self.turn]):
            b = between(king, sniper) & self.occupied
            # Add to blockers if exactly one piece in-between.
            if b and BB_SQUARES[msb(b)] == b:
                blockers |= b
        return blockers & self.occupied_co[self.turn]

    def _ep_skewered(self, king: Square, capturer: Square) -> bool:
        assert self.ep_square is not None
        last_double = self.ep_square + (-8 if self.turn == WHITE else 8)
        occupancy = (self.occupied & ~BB_SQUARES[last_double] & ~BB_SQUARES[capturer] | BB_SQUARES[self.ep_square])
        horizontal_attackers = self.occupied_co[not self.turn] & (self.rooks | self.queens)
        if BB_RANK_ATTACKS[king][BB_RANK_MASKS[king] & occupancy] & horizontal_attackers:
            return True
        diagonal_attackers = self.occupied_co[not self.turn] & (self.bishops | self.queens)
        if BB_DIAG_ATTACKS[king][BB_DIAG_MASKS[king] & occupancy] & diagonal_attackers:
            return True
        return False

    def _is_safe(self, king: Square, blockers: Bitboard, move: Move) -> bool:
        if move.from_square == king:
            if self.is_castling(move):
                return True
            else:
                return not self.is_attacked_by(not self.turn, move.to_square)
        elif self.is_en_passant(move):
            return bool(self.pin_mask(self.turn, move.from_square) & BB_SQUARES[move.to_square] and
                        not self._ep_skewered(king, move.from_square))
        else:
            return bool(not blockers & BB_SQUARES[move.from_square] or
                        ray(move.from_square, move.to_square) & BB_SQUARES[king])

    def _generate_evasions(self, king: Square, checkers: Bitboard, from_mask: Bitboard = BB_ALL,
                           to_mask: Bitboard = BB_ALL) -> Iterator[Move]:
        sliders = checkers & (self.bishops | self.rooks | self.queens)
        attacked = 0
        for checker in scan_reversed(sliders):
            attacked |= ray(king, checker) & ~BB_SQUARES[checker]
        if BB_SQUARES[king] & from_mask:
            for to_square in scan_reversed(BB_KING_ATTACKS[king] & ~self.occupied_co[self.turn] & ~attacked & to_mask):
                yield Move(king, to_square)
        checker = msb(checkers)
        if BB_SQUARES[checker] == checkers:
            # Capture or block a single checker.
            target = between(king, checker) | checkers
            yield from self.generate_pseudo_legal_moves(~self.kings & from_mask, target & to_mask)
            # Capture the checking pawn en passant (but avoid yielding duplicate moves).
            if self.ep_square and not BB_SQUARES[self.ep_square] & target:
                last_double = self.ep_square + (-8 if self.turn == WHITE else 8)
                if last_double == checker:
                    yield from self.generate_pseudo_legal_ep(from_mask, to_mask)

    def generate_legal_moves(self, from_mask: Bitboard = BB_ALL, to_mask: Bitboard = BB_ALL) -> Iterator[Move]:
        king_mask = self.kings & self.occupied_co[self.turn]
        if king_mask:
            king = msb(king_mask)
            blockers = self._slider_blockers(king)
            checkers = self.attackers_mask(not self.turn, king)
            if checkers:
                for move in self._generate_evasions(king, checkers, from_mask, to_mask):
                    if self._is_safe(king, blockers, move):
                        yield move
            else:
                for move in self.generate_pseudo_legal_moves(from_mask, to_mask):
                    if self._is_safe(king, blockers, move):
                        yield move
        else:
            yield from self.generate_pseudo_legal_moves(from_mask, to_mask)

    def generate_legal_ep(self, from_mask: Bitboard = BB_ALL, to_mask: Bitboard = BB_ALL) -> Iterator[Move]:
        for move in self.generate_pseudo_legal_ep(from_mask, to_mask):
            if not self.is_into_check(move):
                yield move

    @property
    def legal_moves(self) -> "LegalMoveGenerator":
        return LegalMoveGenerator(self)

    # ---- predicates ----------------------------------------------------------------------
    def is_en_passant(self, move: Move) -> bool:
        return (self.ep_square == move.to_square and
                bool(self.pawns & BB_SQUARES[move.from_square]) and
                abs(move.to_square - move.from_square) in [7, 9] and
                not self.occupied & BB_SQUARES[move.to_square])

    def is_capture(self, move: Move) -> bool:
        touched = BB_SQUARES[move.from_square] ^ BB_SQUARES[move.to_square]
        return bool(touched & self.occupied_co[not self.turn]) or self.is_en_passant(move)

    def is_zeroing(self, move: Move) -> bool:
        touched = BB_SQUARES[move.from_square] ^ BB_SQUARES[move.to_square]
        return bool(touched & self.pawns or touched & self.occupied_co[not self.turn] or move.drop == PAWN)

    def is_castling(self, move: Move) -> bool:
        if self.kings & BB_SQUARES[move.from_square]:
            diff = square_file(move.from_square) - square_file(move.to_square)
            return abs(diff) > 1 or bool(self.rooks & self.occupied_co[self.turn] & BB_SQUARES[move.to_square])
        return False

    def is_kingside_castling(self, move: Move) -> bool:
        return self.is_castling(move) and square_file(move.to_square) > square_file(move.from_square)

    def is_queenside_castling(self, move: Move) -> bool:
        return self.is_castling(move) and square_file(move.to_square) < square_file(move.from_square)

    def _reduces_castling_rights(self, move: Move) -> bool:
        cr = self.clean_castling_rights()
        touched = BB_SQUARES[move.from_square] ^ BB_SQUARES[move.to_square]
        return bool(touched & cr or
                    cr & BB_RANK_1 and touched & self.kings & self.occupied_co[WHITE] & ~self.promoted or
                    cr & BB_RANK_8 and touched & self.kings & self.occupied_co[BLACK] & ~self.promoted)

    def is_irreversible(self, move: Move) -> bool:
        return self.is_zeroing(move) or self._reduces_castling_rights(move) or self.has_legal_en_passant()

    def is_into_check(self, move: Move) -> bool:
        king = self.king(self.turn)
        if king is None:
            return False
        checkers = self.attackers_mask(not self.turn, king)
        if checkers and move not in self._generate_evasions(king, checkers, BB_SQUARES[move.from_square],
                                                            BB_SQUARES[move.to_square]):
            return True
        return not self._is_safe(king, self._slider_blockers(king), move)

    def is_pseudo_legal(self, move: Move) -> bool:
        # Null moves are not pseudo-legal.
        if not move:
            return False
        # Drops are not pseudo-legal.
        if move.drop:
            return False
        # Source square must not be vacant.
        piece = self.piece_type_at(move.from_square)
        if not piece:
            return False
        from_mask = BB_SQUARES[move.from_square]
        to_mask = BB_SQUARES[move.to_square]
        # Check turn.
        if not self.occupied_co[self.turn] & from_mask:
            return False
        # Only pawns can promote and only on the backrank.
        if move.promotion:
            if piece != PAWN:
                return False
            if self.turn == WHITE and square_rank(move.to_square) != 7:
                return False
            elif self.turn == BLACK and square_rank(move.to_square) != 0:
                return False
        # Handle castling.
        if piece == KING:
            move = self._from_chess960(self.chess960, move.from_square, move.to_square)
            if move in self.generate_castling_moves():
                return True
        # Destination square can not be occupied.
        if self.occupied_co[self.turn] & to_mask:
            return False
        # Handle pawn moves.
        if piece == PAWN:
            return move in self.generate_pseudo_legal_moves(from_mask, to_mask)
        # Handle all other pieces.
        return bool(self.attacks_mask(move.from_square) & to_mask)

    def is_legal(self, move: Move) -> bool:
        return self.is_pseudo_legal(move) and not self.is_into_check(move)

    def has_kingside_castling_rights(self, color: Color) -> bool:
        backrank = BB_RANK_1 if color == WHITE else BB_RANK_8
        king_mask = self.kings & self.occupied_co[color] & backrank & ~self.promoted
        if not king_mask:
            return False
        castling_rights = self.clean_castling_rights() & backrank
        while castling_rights:
            rook = castling_rights & -castling_rights
            if rook > king_mask:
                return True
            castling_rights &= castling_rights - 1
        return False

    def has_queenside_castling_rights(self, color: Color) -> bool:
        backrank = BB_RANK_1 if color == WHITE else BB_RANK_8
        king_mask = self.kings & self.occupied_co[color] & backrank & ~self.promoted
        if not king_mask:
            return False
        castling_rights = self.clean_castling_rights() & backrank
        while castling_rights:
            rook = castling_rights & -castling_rights
            if rook < king_mask:
                return True
            castling_rights &= castling_rights - 1
        return False

    def has_castling_rights(self, color: Color) -> bool:
        backrank = BB_RANK_1 if color == WHITE else BB_RANK_8
        return bool(self.clean_castling_rights() & backrank)

    def clean_castling_rights(self) -> Bitboard:
        if self._stack:
            # No new castling rights are assigned in a game, so they were filtered already.
            return self.castling_rights
        castling = self.castling_rights & self.rooks
        white_castling = castling & BB_RANK_1 & self.occupied_co[WHITE]
        black_castling = castling & BB_RANK_8 & self.occupied_co[BLACK]
        # The rooks must be on a1, h1, a8 or h8.
        white_castling &= (BB_A1 | BB_H1)
        black_castling &= (BB_A8 | BB_H8)
        # The kings must be on e1 or e8.
        if not self.occupied_co[WHITE] & self.kings & ~self.promoted & BB_E1:
            white_castling = 0
        if not self.occupied_co[BLACK] & self.kings & ~self.promoted & BB_E8:
            black_castling = 0
        return white_castling | black_castling

    def has_pseudo_legal_en_passant(self) -> bool:
        return self.ep_square is not None and any(self.generate_pseudo_legal_ep())

    def has_legal_en_passant(self) -> bool:
        return self.ep_square is not None and any(self.generate_legal_ep())

    def is_checkmate(self) -> bool:
        if not self.is_check():
            return False
        return not any(self.generate_legal_moves())

    def is_stalemate(self) -> bool:
        if self.is_check():
            return False
        return not any(self.generate_legal_moves())

    def has_insufficient_material(self, color: Color) -> bool:
        if self.occupied_co[color] & (self.pawns | self.rooks | self.queens):
            return False
        if self.occupied_co[color] & self.knights:
            return (popcount(self.occupied_co[color]) <= 2 and
                    not (self.occupied_co[not color] & ~self.kings & ~self.queens))
        if self.occupied_co[color] & self.bishops:
            same_color = (not self.bishops & BB_DARK_SQUARES) or (not self.bishops & BB_LIGHT_SQUARES)
            return same_color and not self.pawns and not self.knights
        return True

    def is_insufficient_material(self) -> bool:
        return all(self.has_insufficient_material(color) for color in COLORS)

    def _is_halfmoves(self, n: int) -> bool:
        return self.halfmove_clock >= n and any(self.generate_legal_moves())

    def is_seventyfive_moves(self) -> bool:
        return self._is_halfmoves(150)

    def is_fifty_moves(self) -> bool:
        return self._is_halfmoves(100)

    def is_fivefold_repetition(self) -> bool:
        return self.is_repetition(5)

    def can_claim_draw(self) -> bool:
        return self.can_claim_fifty_moves() or self.can_claim_threefold_repetition()

    def can_claim_fifty_moves(self) -> bool:
        if self.is_fifty_moves():
            return True
        if self.halfmove_clock >= 99:
            for move in self.generate_legal_moves():
                if not self.is_zeroing(move):
                    self.push(move)
                    try:
                        if self.is_fifty_moves():
                            return True
                    finally:
                        self.pop()
        return False

    def can_claim_threefold_repetition(self) -> bool:
        transposition_key = self._transposition_key()
        transpositions: Dict[object, int] = {}
        transpositions[transposition_key] = 1
        # Count positions.
        switchyard = []
        while self.move_stack:
            move = self.pop()
            switchyard.append(move)
            if self.is_irreversible(move):
                break
            k = self._transposition_key()
            transpositions[k] = transpositions.get(k, 0) + 1
        while switchyard:
            self.push(switchyard.pop())
        # Threefold repetition occurred.
        if transpositions[transposition_key] >= 3:
            return True
        # The next legal move is a threefold repetition.
        for move in self.generate_legal_moves():
            self.push(move)
            try:
                if transpositions.get(self._transposition_key(), 0) >= 2:
                    return True
            finally:
                self.pop()
        return False

    def is_repetition(self, count: int = 3) -> bool:
        # Fast check, based on occupancy only.
        maybe_repetitions = 1
        for state in reversed(self._stack):
            if state.occupied == self.occupied:
                maybe_repetitions += 1
                if maybe_repetitions >= count:
                    break
        if maybe_repetitions < count:
            return False
        # Check full replay.
        transposition_key = self._transposition_key()
        switchyard = []
        try:
            while True:
                if count <= 1:
                    return True
                if len(self.move_stack) < count - 1:
                    break
                move = self.pop()
                switchyard.append(move)
                if self.is_irreversible(move):
                    break
                if self._transposition_key() == transposition_key:
                    count -= 1
        finally:
            while switchyard:
                self.push(switchyard.pop())
        return False

    def outcome(self, *, claim_draw: bool = False) -> Optional[Outcome]:
        # Normal game end.
        if self.is_checkmate():
            return Outcome("checkmate", not self.turn)
        if self.is_insufficient_material():
            return Outcome("insufficient_material", None)
        if not any(self.generate_legal_moves()):
            return Outcome("stalemate", None)
        # Automatic draws.
        if self.is_seventyfive_moves():
            return Outcome("seventyfive_moves", None)
        if self.is_fivefold_repetition():
            return Outcome("fivefold_repetition", None)
        # Claimable draws.
        if claim_draw:
            if self.can_claim_fifty_moves():
                return Outcome("fifty_moves", None)
            if self.can_claim_threefold_repetition():
                return Outcome("threefold_repetition", None)
        return None

    def is_game_over(self, *, claim_draw: bool = False) -> bool:
        return self.outcome(claim_draw=claim_draw) is not None

    def result(self, *, claim_draw: bool = False) -> str:
        outcome = self.outcome(claim_draw=claim_draw)
        return outcome.result() if outcome else "*"

    def is_variant_end(self) -> bool:
        return False

    # ---- make / unmake -------------------------------------------------------------------
    def push(self, move: Move) -> None:
        # Push move and remember board state.
        move = self._to_chess960(move)
        board_state = _BoardState(self)
        self.castling_rights = self.clean_castling_rights()  # Before pushing stack
        self.move_stack.append(self._from_chess960(self.chess960, move.from_square, move.to_square,
                                                   move.promotion, move.drop))
        self._stack.append(board_state)

        # Reset en passant square.
        ep_square = self.ep_square
        self.ep_square = None

        # Increment move counters.
        self.halfmove_clock += 1
        if self.turn == BLACK:
            self.fullmove_number += 1

        # On a null move, simply swap turns and reset the en passant square.
        if not move:
            self.turn = not self.turn
            return

        # Zero the half-move clock.
        if self.is_zeroing(move):
            self.halfmove_clock = 0

        from_bb = BB_SQUARES[move.from_square]
        to_bb = BB_SQUARES[move.to_square]

        promoted = bool(self.promoted & from_bb)
        piece_type = self._remove_piece_at(move.from_square)
        assert piece_type is not None, f"push() expects move to be pseudo-legal, but got {move} in {self.board_fen()}"
        capture_square = move.to_square
        captured_piece_type = self.piece_type_at(capture_square)

        # Update castling rights.
        self.castling_rights &= ~to_bb & ~from_bb
        if piece_type == KING and not promoted:
            if self.turn == WHITE:
                self.castling_rights &= ~BB_RANK_1
            else:
                self.castling_rights &= ~BB_RANK_8
        elif captured_piece_type == KING and not self.promoted & to_bb:
            if self.turn == WHITE and square_rank(move.to_square) == 7:
                self.castling_rights &= ~BB_RANK_8
            elif self.turn == BLACK and square_rank(move.to_square) == 0:
                self.castling_rights &= ~BB_RANK_1

        # Handle special pawn moves.
        if piece_type == PAWN:
            diff = move.to_square - move.from_square
            if diff == 16 and square_rank(move.from_square) == 1:
                self.ep_square = move.from_square + 8
            elif diff == -16 and square_rank(move.from_square) == 6:
                self.ep_square = move.from_square - 8
            elif move.to_square == ep_square and abs(diff) in [7, 9] and not captured_piece_type:
                # Remove pawns captured en passant.
                down = -8 if self.turn == WHITE else 8
                capture_square = ep_square + down
                captured_piece_type = self._remove_piece_at(capture_square)

        # Promotion.
        if move.promotion:
            promoted = True
            piece_type = move.promotion

        # Castling.
        castling = piece_type == KING and self.occupied_co[self.turn] & to_bb
        if castling:
            a_side = square_file(move.to_square) < square_file(move.from_square)
            self._remove_piece_at(move.from_square)
            self._remove_piece_at(move.to_square)
            if a_side:
                self._set_piece_at(C1 if self.turn == WHITE else C8, KING, self.turn)
                self._set_piece_at(D1 if self.turn == WHITE else D8, ROOK, self.turn)
            else:
                self._set_piece_at(G1 if self.turn == WHITE else G8, KING, self.turn)
                self._set_piece_at(F1 if self.turn == WHITE else F8, ROOK, self.turn)

        # Put the piece on the target square.
        if not castling:
            self._set_piece_at(move.to_square, piece_type, self.turn, promoted)

        # Swap turn.
        self.turn = not self.turn

    def pop(self) -> Move:
        move = self.move_stack.pop()
        self._stack.pop().restore(self)
        return move

    def peek(self) -> Move:
        return self.move_stack[-1]

    def ply(self) -> int:
        return 2 * (self.fullmove_number - 1) + (self.turn == BLACK)

    def copy(self, *, stack=True) -> "Board":
        board = type(self)(None)
        board.pawns = self.pawns
        board.knights = self.knights
        board.bishops = self.bishops
        board.rooks = self.rooks
        board.queens = self.queens
        board.kings = self.kings
        board.occupied_co[WHITE] = self.occupied_co[WHITE]
        board.occupied_co[BLACK] = self.occupied_co[BLACK]
        board.occupied = self.occupied
        board.promoted = self.promoted
        board.ep_square = self.ep_square
        board.castling_rights = self.castling_rights
        board.turn = self.turn
        board.fullmove_number = self.fullmove_number
        board.halfmove_clock = self.halfmove_clock
        if stack:
            stack = len(self.move_stack) if stack is True else stack
            board.move_stack = [Move(m.from_square, m.to_square, m.promotion, m.drop) for m in self.move_stack[-stack:]]
            board._stack = self._stack[-stack:]
        return board

    def __copy__(self) -> "Board":
        return self.copy(stack=False)

    def __deepcopy__(self, memo) -> "Board":
        board = self.copy()
        memo[id(self)] = board
        return board

    def _transposition_key(self):
        return (self.pawns, self.knights, self.bishops, self.rooks, self.queens, self.kings,
                self.occupied_co[WHITE], self.occupied_co[BLACK],
                self.turn, self.clean_castling_rights(),
                self.ep_square if self.has_legal_en_passant() else None)

    def __eq__(self, other) -> bool:
        if isinstance(other, Board):
            return (self.halfmove_clock == other.halfmove_clock and
                    self.fullmove_number == other.fullmove_number and
                    self._transposition_key() == other._transposition_key())
        return NotImplemented

    # ---- text ----------------------------------------------------------------------------
    def board_fen(self) -> str:
        builder = []
        empty = 0
        for sq in [s ^ 0x38 for s in SQUARES]:
            piece = self.piece_at(sq)
            if not piece:
                empty += 1
            else:
                if empty:
                    builder.append(str(empty))
                    empty = 0
                builder.append(piece.symbol())
            if BB_SQUARES[sq] & BB_FILE_H:
                if empty:
                    builder.append(str(empty))
                    empty = 0
                if sq != H1:
                    builder.append("/")
        return "".join(builder)

    def castling_xfen(self) -> str:
        builder = []
        for color in COLORS:
            king = self.king(color)
            if king is None:
                continue
            king_file = square_file(king)
            backrank = BB_RANK_1 if color == WHITE else BB_RANK_8
            for rook_square in scan_reversed(self.clean_castling_rights() & backrank):
                rook_file = square_file(rook_square)
                a_side = rook_file < king_file
                ch = "q" if a_side else "k"
                builder.append(ch.upper() if color == WHITE else ch)
        return "".join(builder) if builder else "-"

    def fen(self, *, en_passant: str = "legal") -> str:
        if en_passant == "fen":
            ep = self.ep_square
        elif en_passant == "xfen":
            ep = self.ep_square if self.has_pseudo_legal_en_passant() else None
        else:
            ep = self.ep_square if self.has_legal_en_passant() else None
        return " ".join([
            self.board_fen(),
            "w" if self.turn == WHITE else "b",
            self.castling_xfen(),
            SQUARE_NAMES[ep] if ep is not None else "-",
            str(self.halfmove_clock),
            str(self.fullmove_number),
        ])

    def __repr__(self) -> str:
        return f"Board({self.fen()!r})"

    def uci(self, move: Move) -> str:
        return move.uci()

    def parse_uci(self, uci: str) -> Move:
        move = Move.from_uci(uci)
        if not move:
            return move
        move = self._to_chess960(move)
        move = self._from_chess960(self.chess960, move.from_square, move.to_square, move.promotion, move.drop)
        if not self.is_legal(move):
            raise IllegalMoveError(f"illegal uci: {uci!r} in {self.fen()}")
        return move

    def push_uci(self, uci: str) -> Move:
        move = self.parse_uci(uci)
        self.push(move)
        return move

    def parse_san(self, san: str) -> Move:
        # Castling.
        try:
            if san in ["O-O", "O-O+", "O-O#", "0-0", "0-0+", "0-0#"]:
                return next(move for move in self.generate_castling_moves() if self.is_kingside_castling(move))
            elif san in ["O-O-O", "O-O-O+", "O-O-O#", "0-0-0", "0-0-0+", "0-0-0#"]:
                return next(move for move in self.generate_castling_moves() if self.is_queenside_castling(move))
        except StopIteration:
            raise IllegalMoveError(f"illegal san: {san!r} in {self.fen()}")
        # Match normal moves.
        match = SAN_REGEX.match(san)
        if not match:
            if san in ["--", "Z0", "0000", "@@@@"]:
                return Move.null()
            raise InvalidMoveError(f"invalid san: {san!r}")
        # Get target square.
        to_square = SQUARE_NAMES.index(match.group(4))
        to_mask = BB_SQUARES[to_square] & ~self.occupied_co[self.turn]
        # Get the promotion piece type.
        p = match.group(5)
        promotion = PIECE_SYMBOLS.index(p[-1].lower()) if p else None
        # Filter by original square.
        from_mask = BB_ALL
        if match.group(2):
            from_mask &= BB_FILES[FILE_NAMES.index(match.group(2))]
        if match.group(3):
            from_mask &= BB_RANKS[int(match.group(3)) - 1]
        # Filter by piece type.
        if match.group(1):
            piece_type = PIECE_SYMBOLS.index(match.group(1).lower())
            from_mask &= self.pieces_mask(piece_type, self.turn)
        elif match.group(2) and match.group(3):
            # Allow fully specified moves, even if they are not pawn moves.
            move = self.find_move(SQUARE_NAMES.index(match.group(2) + match.group(3)), to_square, promotion)
            if move.promotion == promotion:
                return move
            raise IllegalMoveError(f"missing promotion piece type: {san!r} in {self.fen()}")
        else:
            from_mask &= self.pawns
            # Do not allow pawn captures if file is not specified.
            if not match.group(2):
                from_mask &= BB_FILES[square_file(to_square)]
        # Match legal moves.
        matched_move = None
        for move in self.generate_legal_moves(from_mask, to_mask):
            if move.promotion != promotion:
                continue
            if matched_move:
                raise AmbiguousMoveError(f"ambiguous san: {san!r} in {self.fen()}")
            matched_move = move
        if not matched_move:
            raise IllegalMoveError(f"illegal san: {san!r} in {self.fen()}")
        return matched_move

    def push_san(self, san: str) -> Move:
        move = self.parse_san(san)
        self.push(move)
        return move

    def find_move(self, from_square: Square, to_square: Square, promotion: Optional[PieceType] = None) -> Move:
        if promotion is None and self.pawns & BB_SQUARES[from_square] and BB_SQUARES[to_square] & BB_BACKRANKS:
            promotion = QUEEN
        move = self._from_chess960(self.chess960, from_square, to_square, promotion)
        if not self.is_legal(move):
            raise IllegalMoveError(f"no matching legal move for {move.uci()} in {self.fen()}")
        return move

    def gives_check(self, move: Move) -> bool:
        self.push(move)
        try:
            return self.is_check()
        finally:
            self.pop()


class LegalMoveGenerator:
    def __init__(self, board: Board) -> None:
        self.board = board

    def __bool__(self) -> bool:
        return any(self.board.generate_legal_moves())

    def count(self) -> int:
        return sum(1 for _ in self.board.generate_legal_moves())

    def __len__(self) -> int:
        return self.count()

    def __iter__(self) -> Iterator[Move]:
        return self.board.generate_legal_moves()

    def __contains__(self, move: Move) -> bool:
        return self.board.is_legal(move)

    def __repr__(self) -> str:
        return f"<LegalMoveGenerator ({', '.join(m.uci() for m in self)})>"
