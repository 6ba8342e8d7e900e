"""Reuse of the root's evaluation across moves (SelfPlayEngine, m0_search_reuse_*): the root of a move is expanded from the network
output its position got as a child of the previous root, which must be exactly what a second evaluation returns.  That needs a row's
output to be a function of the row alone -- not of the other rows, its index or the batch size -- in the 16-bit paths too (the roots
that are not kept are evaluated in compact rows of a smaller batch)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _model_cfg():
    return dict(planes=19, channels=320, blocks=24, attention=True, attention_heads=20, policy_size=4672, norm="group", activation="silu",
                value_activation="leaky_relu", preact=True, droppath=0.0, policy_factor_rank=160, infer_attention_stride=2,
                infer_amp_tower=True, aux_policy_from_square=True, aux_policy_move_type=True, ssl_curriculum=True, self_supervised=True,
                ssl_tasks=["piece", "threat", "pin", "fork", "control"])


def _selfplay_cfg(sims=800, max_game_len=200):
    selfplay = dict(max_game_len=max_game_len, min_resign_plies=50, resign_threshold=-0.85, opening_random_plies=12, num_simulations=sims,
                    temperature_start=1.2, temperature_end=0.3, temperature_moves=40)
    mcts = dict(num_simulations=sims, cpuct=2.5, cpuct_start=3.0, cpuct_end=2.0, cpuct_plies=40, dirichlet_alpha=0.3, dirichlet_frac=0.25,
                dirichlet_plies=30, selection_jitter=0.05, fpu=0.6, fpu_reduction=0.1, draw_penalty=-0.05, legal_softmax=True,
                no_instant_backtrack=True, parent_q_init=True, value_from_white=False, virtual_loss=1.0, inference_batch_size=96,
                playout_random_frac=0.05, enable_entropy_noise=True)
    return {"model": _model_cfg(), "selfplay": selfplay, "mcts": mcts}


_NETS = {}


def _net(precision):
    """ResNet-24 with the reference's own initialisation (seed 0), as the benchmark runs it."""
    if precision not in _NETS:
        from matrix0_b200.model import PolicyValueNet
        _NETS[precision] = PolicyValueNet.from_config(_model_cfg(), device="cuda", precision=precision, seed=0)
    return _NETS[precision]


def _positions(n, seed):
    """Planes of n positions from random playouts (device)."""
    from matrix0_b200 import _native
    lib = _native.lib()
    pos = torch.empty((n, 9), dtype=torch.int64, device="cuda")
    _native.check(lib.m0_random_playouts(pos.data_ptr(), n, seed, 40, _native.current_stream()))
    planes = torch.empty((n, 19, 8, 8), dtype=torch.float32, device="cuda")
    _native.check(lib.m0_encode_planes(pos.data_ptr(), n, planes.data_ptr(), _native.current_stream()))
    return planes


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_row_output_depends_on_the_row_alone(precision):
    net = _net(precision)
    x = _positions(4096, 7)
    lg, v = (t.clone() for t in net.forward_planes(x, precision))
    # batch size: the leading rows of smaller batches
    for n in (1, 37, 256, 300, 2048):
        a, b = net.forward_planes(x[:n].contiguous(), precision)
        assert torch.equal(a, lg[:n]) and torch.equal(b, v[:n]), n
    # row index: a permutation of the batch permutes the outputs
    perm = torch.randperm(4096, generator=torch.Generator().manual_seed(3)).cuda()
    a, b = net.forward_planes(x[perm].contiguous(), precision)
    assert torch.equal(a, lg[perm]) and torch.equal(b, v[perm])
    # neighbours: every other row replaced by another position
    y = _positions(4096, 11)
    keep = torch.arange(0, 4096, 5, device="cuda")
    y[keep] = x[keep]
    a, b = net.forward_planes(y, precision)
    assert torch.equal(a[keep], lg[keep]) and torch.equal(b[keep], v[keep])
    # a row alone at another index of a small batch
    z = y[:37].clone()
    z[20] = x[3]
    a, b = net.forward_planes(z, precision)
    assert torch.equal(a[20], lg[3]) and torch.equal(b[20], v[3])


def _play(search_mode, max_game_len, clear_every_move, moves=6, games=256):
    """Per move: the search results, the roots expanded from kept outputs and the games that continue from the previous move."""
    from matrix0_b200 import _native
    from matrix0_b200.selfplay import SelfPlayEngine
    sp = SelfPlayEngine(_net("fp16"), _selfplay_cfg(max_game_len=max_game_len), games=games, deterministic=False, seed=5, precision="fp16",
                        search_mode=search_mode)
    sp.warm_up_forward()
    sp.start()
    eng = sp.engine
    out = []
    prev_plies = None
    for _ in range(moves):
        _native.check(sp._lib.m0_selfplay_plies(eng._h, sp.plies.data_ptr(), _native.current_stream()))
        plies = sp.plies.cpu().numpy().copy()
        c0 = sp.counters()["root_evals_reused"]
        if clear_every_move:
            eng.clear_reuse()
        sp.begin_move()
        info = eng.info.cpu().numpy()
        reused = sp.counters()["root_evals_reused"] - c0
        for _ in range(sp.batches_per_move()):
            sp.search_step()
        eng.result(with_pi=True)
        rec = {k: getattr(eng, k).cpu().numpy().copy() for k in ("res_moves", "res_visits", "res_q", "res_prior", "res_count", "res_pi",
                                                                    "res_root_q", "res_root_n")}
        sp.end_move()
        rec["moves_played"] = sp.moves_played.cpu().numpy().copy()
        # a game continues when it made one more ply since the last move and its root needed an evaluation (not terminal)
        evaluated = int(((info & 2) != 0).sum())
        cont = 0 if prev_plies is None else int(((plies == prev_plies + 1) & ((info & 2) != 0)).sum())
        out.append((rec, reused, cont, evaluated))
        prev_plies = plies
    return out


@pytest.mark.parametrize("search_mode", ["collapsed", "as_shipped"])
@pytest.mark.parametrize("max_game_len", [200, 3])
def test_reused_root_evaluations_give_identical_searches(search_mode, max_game_len):
    """Six moves with the store against six moves with the store cleared before every move.  The cleared run sends every root
    through the compact miss rows, not through row g of a G-row forward as an engine without the store does; that the reused
    outputs also equal that older path rests on the row invariance above and on the byte comparison of `bench.py --dump-outputs`
    against the previous code (profiles/r03_ab_root_reuse.json)."""
    reuse = _play(search_mode, max_game_len, clear_every_move=False)
    fresh = _play(search_mode, max_game_len, clear_every_move=True)
    for m, ((ra, na, ca, _), (rb, nb, _, _)) in enumerate(zip(reuse, fresh)):
        for k in ra:
            assert ra[k].tobytes() == rb[k].tobytes(), (m, k)
        assert nb == 0, m
        assert na == ca, (m, na, ca)
    assert sum(n for _, n, _, _ in reuse) > 0
    if max_game_len == 3:   # games restart inside the window: their roots go through the compact rows next to reused ones
        assert sum(e - c for _, _, c, e in reuse[1:]) > 0


def test_arena_does_not_reuse():
    """In the arena the root's children were evaluated by the other player's network: nothing is kept."""
    from matrix0_b200.arena import ArenaEngine
    net = _net("fp16")
    ar = ArenaEngine(net, net, _selfplay_cfg(), num_sims=192, temperature=1.0, temp_plies=4, max_moves=4, concurrent_games=64, seed=3,
                     precision="fp16")
    ar.play(64)
    c = ar.games.counters()
    assert c["root_evals_reused"] == 0 and c["positions_played"] > 0
