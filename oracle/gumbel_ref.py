"""TEST INFRASTRUCTURE ONLY -- float64 restatement of the Gumbel AlphaZero search of the batched self-play engine
(``SelfPlayEngine(search_mode="gumbel")``, csrc/gumbel_kernels.cu), one game at a time, on the oracle ``chess`` shim.

Danihelka, Guez, Schrittwieser, Silver, *Policy improvement by planning with Gumbel* (ICLR 2022), as DESIGN.md §9 defines it:
one leaf per simulation, a plain tree (children are reached only through their parent), sequential halving at the root as a
visit schedule, interior selection by ``argmax softmax(l + sigma) - N / (1 + Nc)``, and the policy target ``softmax(l + sigma)``
at the root.  Every node holds N and W from the view of its side to move; a child's value for its parent is ``-W / N``.

``search`` also returns the smallest decision margin (best minus second-best score over every argmax the search took): a test
that compares the device search against this one may drop games whose margin is at rounding level.  It counts the nodes it creates
as the device allocates them (the root, then every child of every expansion) and the simulations that ended on a terminal leaf, by
kind, so a test built around a terminal rule can check that the tree reaches it.
"""
from __future__ import annotations

import math
from typing import Callable, List, Optional, Tuple

import numpy as np

from . import chess_shim  # noqa: F401
import chess
from .encoding_ref import encode_board, move_to_index_unchecked


def schedule(m: int, n: int) -> List[int]:
    """T(m, n): the visit count a root candidate must have to be chosen at simulation k (sequential halving)."""
    if m <= 1:
        return list(range(n))
    L = math.ceil(math.log2(m))
    seq: List[int] = []
    visits = [0] * m
    k = m
    while len(seq) < n:
        for _ in range(max(1, int(n / (L * k)))):
            seq += visits[:k]
            visits[:k] = [v + 1 for v in visits[:k]]
        k = max(2, k // 2)
    return seq[:n]


def sigma(logits: np.ndarray, N: np.ndarray, W: np.ndarray, r: float, c_visit: float, c_scale: float):
    """sigma(completed Q) at a node: logits of its legal moves (float64), children's N and W (children's view), its own r.
    Returns (sigma, v_mix, q_tilde)."""
    logits = np.asarray(logits, dtype=np.float64)
    N = np.asarray(N, dtype=np.int64)
    W = np.asarray(W, dtype=np.float64)
    vis = N > 0
    q = np.where(vis, -W / np.maximum(N, 1), 0.0)
    p = np.exp(logits - logits.max())
    p /= p.sum()
    Nc = int(N.sum())
    if Nc == 0:
        v_mix = float(r)
    else:
        v_mix = (float(r) + Nc * float((p[vis] * q[vis]).sum()) / float(p[vis].sum())) / (1 + Nc)
    qhat = np.where(vis, q, v_mix)
    lo, hi = float(qhat.min()), float(qhat.max())
    qt = (qhat - lo) / max(hi - lo, 1e-8)
    return (c_visit + int(N.max())) * c_scale * qt, v_mix, qt


def softmax(x: np.ndarray) -> np.ndarray:
    e = np.exp(x - x.max())
    return e / e.sum()


class _Node:
    __slots__ = ("n", "w", "r", "moves", "logits", "children")

    def __init__(self):
        self.n, self.w, self.r = 0, 0.0, 0.0
        self.moves, self.logits, self.children = None, None, None   # set when expanded


def terminal_value(b, draw_penalty: float) -> Optional[float]:
    """None for a live position; checkmate -1, any other end of game draw_penalty (side to move's view)."""
    if not b.is_game_over():
        return None
    return -1.0 if b.is_checkmate() else float(draw_penalty)


TERMINAL_KINDS = ("checkmate", "stalemate", "insufficient_material", "seventyfive_moves", "fivefold_repetition")


def terminal_kind(b) -> str:
    """Which rule ends a position that is_game_over() calls over (checkmate first: its value is -1, every other kind is a draw)."""
    if b.is_checkmate():
        return "checkmate"
    if b.is_stalemate():
        return "stalemate"
    if b.is_insufficient_material():
        return "insufficient_material"
    return "seventyfive_moves" if b.is_seventyfive_moves() else "fivefold_repetition"


def _argmax(scores: np.ndarray) -> Tuple[int, float]:
    """First maximum and the margin to the second-best finite score (inf when there is no second)."""
    j = int(np.argmax(scores))
    rest = np.delete(scores, j)
    rest = rest[np.isfinite(rest)]
    return j, (float(scores[j] - rest.max()) if rest.size else math.inf)


def search(board, evaluate: Callable, gumbel: np.ndarray, n: int, m: int, c_visit: float = 50.0, c_scale: float = 0.1,
           draw_penalty: float = -0.1) -> dict:
    """One Gumbel search from `board` (history included).  evaluate(planes float32[19, 8, 8]) -> (logits float32[4672], value);
    gumbel: float64 draws, one per legal move in generation order."""
    margin = [math.inf]
    nodes = [1]                                   # the root
    max_depth = [0]                               # longest selection path, in moves from the root
    terminals = dict.fromkeys(TERMINAL_KINDS, 0)
    terminal_depth = {}                           # kind -> shallowest depth (moves from the root) it was reached at

    def expand(node: _Node, b) -> None:
        lg, v = evaluate(encode_board(b))
        lg = np.asarray(lg, dtype=np.float32).reshape(-1)
        wtm = b.turn == chess.WHITE
        node.moves = list(b.generate_legal_moves())
        node.logits = np.array([float(lg[move_to_index_unchecked(wtm, mv.from_square, mv.to_square, mv.promotion)]) for mv in node.moves],
                               dtype=np.float64)
        node.children = [_Node() for _ in node.moves]
        nodes[0] += len(node.moves)
        node.r = max(-1.0, min(1.0, float(np.float32(v))))

    def stats(node: _Node):
        return (np.array([c.n for c in node.children], dtype=np.int64), np.array([c.w for c in node.children], dtype=np.float64))

    def root_scores(node: _Node, allowed: np.ndarray) -> np.ndarray:
        N, W = stats(node)
        s, _, _ = sigma(node.logits, N, W, node.r, c_visit, c_scale)
        sc = g + node.logits - node.logits.max() + s
        return np.where(allowed, sc, -np.inf)

    if terminal_value(board, draw_penalty) is not None:
        raise ValueError("the root is terminal")
    root = _Node()
    expand(root, board)
    root.n, root.w = 1, root.r
    k_legal = len(root.moves)
    g = np.asarray(gumbel, dtype=np.float64)[:k_legal]
    mp = min(int(m), k_legal)
    T = schedule(mp, int(n))
    actions = []
    for k in range(int(n)):
        b = board.copy()
        N, _ = stats(root)
        a, mg = _argmax(root_scores(root, N == T[k]))
        margin[0] = min(margin[0], mg)
        actions.append(a)
        path = [root, root.children[a]]
        b.push(root.moves[a])
        node = path[-1]
        while node.children is not None:
            N, W = stats(node)
            s, _, _ = sigma(node.logits, N, W, node.r, c_visit, c_scale)
            j, mg = _argmax(softmax(node.logits + s) - N / (1.0 + N.sum()))
            margin[0] = min(margin[0], mg)
            b.push(node.moves[j])
            node = node.children[j]
            path.append(node)
        max_depth[0] = max(max_depth[0], len(path) - 1)
        v = terminal_value(b, draw_penalty)
        if v is None:
            expand(node, b)
            v = node.r
        else:
            kind = terminal_kind(b)
            terminals[kind] += 1
            terminal_depth[kind] = min(terminal_depth.get(kind, len(path)), len(path) - 1)
        v = max(-1.0, min(1.0, v))
        for nd in reversed(path):
            nd.n += 1
            nd.w += v
            v = -v
    N, W = stats(root)
    s, _, _ = sigma(root.logits, N, W, root.r, c_visit, c_scale)
    pi_legal = softmax(root.logits + s)
    chosen, mg = _argmax(root_scores(root, N == N.max()))
    margin[0] = min(margin[0], mg)
    wtm = board.turn == chess.WHITE
    pi = np.zeros(4672, dtype=np.float32)
    for mv, p in zip(root.moves, pi_legal):
        pi[move_to_index_unchecked(wtm, mv.from_square, mv.to_square, mv.promotion)] = np.float32(p)
    return {"moves": root.moves, "actions": actions, "visits": N, "q": np.where(N > 0, -W / np.maximum(N, 1), 0.0),
            "pi_legal": pi_legal, "pi": pi, "chosen": chosen, "move": root.moves[chosen], "value": root.w / root.n,
            "margin": margin[0], "nodes": nodes[0], "terminals": terminals, "terminal_depth": terminal_depth, "depth": max_depth[0]}
