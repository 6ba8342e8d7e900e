"""Cases shared by the Gumbel search tests: the (n, m) grid that reaches every branch of the device's sequential-halving schedule
(csrc/gumbel_kernels.cu, halving_schedule_at), and constructed boards, with their history, whose trees reach a given terminal rule."""
import chess

# (n simulations, m root candidates)
SCHEDULE_GRID = [(1, 16), (2, 16), (3, 3), (5, 2), (7, 5), (16, 1), (16, 2), (24, 3), (50, 7), (64, 16), (200, 4)]

# every branch of halving_schedule_at, named as schedule_branches() reports them
SCHEDULE_BRANCHES = {
    "single_candidate",        # m' = 1: T(k) = k
    "one_halving_level",       # m' = 2: L = 1
    "odd_halving",             # a phase of an odd number of candidates: kk / 2 rounds down
    "clamped_to_two",          # kk / 2 < 2 is clamped to 2 (m' = 3, or a halving that ends at 3)
    "repeats_clamped",         # n < L * kk in a phase: one round (covers n < m')
    "repeats_above_one",       # n / (L * kk) > 1: the phase repeats its round
    "n_below_m",               # fewer simulations than candidates: the schedule stops inside the first round
}


def schedule_branches(m: int, n: int):
    """halving_schedule_at(m, n, k) for k < n, written as the kernel writes it, and the branches it took: (T, set of branch names)."""
    taken = set()
    if m <= 1:
        return list(range(n)), {"single_candidate"}
    L = 0
    while (1 << L) < m:
        L += 1
    if L == 1:
        taken.add("one_halving_level")
    if n < m:
        taken.add("n_below_m")
    T, v, kk = [], 0, m
    while len(T) < n:
        d = L * kk
        reps = n // d if n // d > 1 else 1
        taken.add("repeats_above_one" if n // d > 1 else "repeats_clamped")
        for _ in range(reps):
            T += [v] * kk
            v += 1
        if kk // 2 < 2:
            taken.add("clamped_to_two")
        elif kk % 2:
            taken.add("odd_halving")
        kk = kk // 2 if kk // 2 > 2 else 2
    return T[:n], taken


def _repetition_board():
    """Black to move in a position that stood on the board three times before (3 knight shuffles, then Nf3 Nf6 Ng1): its history
    holds the start position four times, so ...Ng8 reaches a fivefold repetition one ply into the tree."""
    b = chess.Board()
    for _ in range(3):
        for u in ("g1f3", "g8f6", "f3g1", "f6g8"):
            b.push_uci(u)
    for u in ("g1f3", "g8f6", "f3g1"):
        b.push_uci(u)
    return b


# (name, board, terminal kind the oracle's tree reaches at n = 200 -- None: the board is there for its width or its depth, and a lower
# bound on the moves from the root at which the tree first reaches that kind: a board built to reach a rule only a few moves down
# says so here).  The same draws go to every board: EDGE_DRAW_SEED's first 256 Gumbel draws; the kinds hold for them under the golden
# small network.  The deepest paths these boards build at n = 200 are 12 moves: well inside the selection cap of max(128, n + 2).
EDGE_BOARDS = [
    # 77 legal moves and queens on both sides: more than 4096 nodes at n = 64
    ("five_queens", lambda: chess.Board("k7/pp2q1q1/8/q1q1q3/8/3Q1Q1Q/1Q1Q2PP/7K w - - 0 1"), None, 0),
    ("six_queens", lambda: chess.Board("k1q1q3/pp6/q1q1q3/8/8/3Q1Q1Q/6PP/3Q1Q1K w - - 0 1"), None, 0),
    # few-move endgames with the longest paths (11 moves at n = 200); K+R vs K first captures the rook 8 moves down
    ("k_rook_vs_k", lambda: chess.Board("8/8/4k3/8/8/8/8/4K2R w - - 0 1"), "insufficient_material", 2),
    ("k_queen_vs_k_pawn", lambda: chess.Board("8/8/8/8/8/5k2/1p6/1K5Q w - - 0 1"), "stalemate", 1),
    ("fivefold", _repetition_board, "fivefold_repetition", 1),
    ("halfmove_148", lambda: chess.Board("r3k3/8/8/8/8/8/8/R3K3 w - - 148 120"), "seventyfive_moves", 2),
    ("halfmove_149", lambda: chess.Board("r3k3/8/8/8/8/8/8/R3K3 w - - 149 120"), "seventyfive_moves", 1),
    ("capture_to_bare_kings", lambda: chess.Board("8/8/4k3/8/3p4/8/5B2/4K3 w - - 0 1"), "insufficient_material", 1),
    ("mate_deep", lambda: chess.Board("7k/8/5K2/8/8/8/8/R7 w - - 0 1"), "checkmate", 2),
    ("stalemate_deep", lambda: chess.Board("7k/5K2/8/8/8/8/8/6R1 b - - 0 1"), "stalemate", 2),
]
EDGE_DRAW_SEED = 7
EDGE_M = 16
