"""Inputs of the draw-adjudication and move-sampling comparisons (tests/test_oracle_selfplay.py) and the stored reference answers
for them (tests/golden/selfplay_golden.json, written by tests/golden/make_selfplay_golden.py)."""
import ast
import json
import os
import random

import numpy as np

import chess

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "selfplay_golden.json")

DRAW_CFGS = [
    {}, {"enabled": True},
    {"enabled": True, "min_plies": 6, "window": 6, "min_unique": 5, "halfmove_cap": 5, "material_draw_threshold": 76},
    {"enabled": True, "min_plies": 0, "window": 4, "min_unique": 3, "halfmove_cap": 0, "material_draw_threshold": 0},
    {"enabled": True, "min_plies": 10, "window": 0, "min_unique": 3, "halfmove_cap": 8, "material_draw_threshold": 60, "stalemate_draw": False},
]

SAMPLE_FEN = "r3k2r/p1ppqpb1/bn2pnp1/3PN3/1p2P3/2N2Q1p/PPPBBPPP/R3K2R w KQkq - 0 1"
SAMPLE_TEMPERATURES = [1.2, 1.0, 0.75, 0.3, 0.1, 0.0005]


def draw_games():
    """40 seeded playouts (moves as chess.Move) in which knight shuffles make repetitions and low-uniqueness windows likely."""
    rng = random.Random(5)
    games = []
    for game in range(40):
        b = chess.Board()
        moves = []
        for ply in range(rng.randint(5, 120)):
            if b.is_game_over():
                break
            legal = list(b.legal_moves)
            back = [m for m in legal if moves and m.from_square == moves[-2].to_square and m.to_square == moves[-2].from_square] if len(moves) >= 2 else []
            m = back[0] if back and rng.random() < 0.5 else rng.choice(legal)
            b.push(m)
            moves.append(m)
        games.append(moves)
    return games


def draw_cases(games):
    """(board, moves so far, cfg) after every ply of every game, for every cfg of DRAW_CFGS, in a fixed order."""
    for game in games:
        b = chess.Board()
        moves = []
        for m in game:
            b.push(m)
            moves.append(m)
            for cfg in DRAW_CFGS:
                yield b, moves, cfg


def sample_trials():
    """400 seeded trials of sample_move_from_counts on SAMPLE_FEN: (counts keyed by move in insertion order, temperature, seed)."""
    rng = random.Random(9)
    moves = list(chess.Board(SAMPLE_FEN).legal_moves)
    out = []
    for trial in range(400):
        k = rng.randint(1, len(moves))
        counts = {m: (rng.randint(0, 300) if rng.random() < 0.8 else 0) for m in moves[:k]}
        if not any(counts.values()):
            counts[moves[0]] = 1
        out.append((counts, rng.choice(SAMPLE_TEMPERATURES), 1000 + trial))
    return out


def uniform(seed):
    """The draw np.random.choice makes inside sample_move_from_counts after np.random.seed(seed)."""
    np.random.seed(seed)
    return np.random.random_sample()


def reference_function(rel_path, name):
    """Compile ONE top-level function of a reference file unmodified (selfplay/internal.py cannot be imported as a module: its
    imports pull in the data manager / orchestrator stack)."""
    from typing import Dict
    from oracle import refload
    src = open(os.path.join(refload.REFERENCE_ROOT, rel_path)).read()
    fn = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == name)
    ns = {"np": np, "chess": chess, "Dict": Dict}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), rel_path, "exec"), ns)
    return ns[name]


def load():
    return json.load(open(GOLDEN))
