"""oth_alphabeta's exact endgames from 12 empties, which the split search (k_alphabeta_split) solves: bit for bit
against the CPU oracle, the other roots of a mixed launch unchanged node for node, D4 invariance, launch-geometry
independence, and arena matches with exact play from 12 empties replayed through the oracle."""
import numpy as np
import pytest

import alphabeta_oracle as ABO
import oracle as O
from test_alphabeta_cpu import forced_pass, forced_pass_positions, random_positions
from test_alphabeta_gpu import _POOL, O_NONE, _check, _kernel

pytestmark = pytest.mark.gpu


def _empties(positions):
    return np.array([(s == 0).sum() for s, _ in positions])


def _forced_pass_between(seed, n, lo, hi):
    """n positions with lo..hi empty squares where the side to move must pass, from seeded random games."""
    g, rng, out = O.OracleGame(), np.random.default_rng(seed), []
    while len(out) < n:
        s, pl = g.get_initial_state(), 1
        while not g.get_value_and_terminated(s, 0, pl)[1] and (s == 0).sum() >= lo:
            if (s == 0).sum() <= hi and forced_pass(s, pl):
                out.append((s.copy(), pl))
                break
            s = g.get_next_state(s, int(rng.choice(np.nonzero(g.get_valid_moves(s, pl))[0])), pl)
            pl = -pl
    return out


def test_exact_12_matches_oracle():
    pos = random_positions(310, 60, (12, 12))
    assert set(_empties(pos)) == {12}
    _check(pos, 1, 12)
    _check(pos[:20], 5, 12)
    fp = _forced_pass_between(311, 5, 12, 12)
    v, b, _ = _check(fp, 1, 12)
    assert (b == 64).all() and (v[:, :64] == O_NONE).all()
    # with exact_empties = 12 the roots of 13+ empties take the depth limit
    _check(random_positions(312, 30, (13, 20)), 4, 12)


def test_mixed_launch_keeps_the_other_roots_node_for_node():
    """Roots of <= 11 and >= 13 empties in a launch at (7, 12) are k_alphabeta's: values, best and node counts equal
    a launch at (7, 11).  The 12-empty roots in between are solved exactly (oracle)."""
    pos = random_positions(320, 400, (4, 50))
    e = _empties(pos)
    mid = e == 12
    assert mid.sum() >= 5 and (e <= 11).sum() >= 20 and (e >= 13).sum() >= 100
    v, b, n = _kernel(pos, 7, 12)
    v0, b0, n0 = _kernel(pos, 7, 11)
    old = ~mid
    assert np.array_equal(v[old], v0[old]) and np.array_equal(b[old], b0[old]) and np.array_equal(n[old], n0[old])
    ov, ob = _oracle_rows([p for p, m in zip(pos, mid) if m], 7, 12)
    assert np.array_equal(v[mid], ov) and np.array_equal(b[mid], ob)


def _oracle_rows(positions, depth, exact):
    ABO.lib()
    res = list(_POOL.map(lambda p: ABO.alphabeta(p[0], p[1], depth, exact), positions))
    return np.stack([r[0] for r in res]), np.array([r[1] for r in res], np.int32)


def test_d4_images_give_permuted_values_exact_12():
    import ctypes as C
    from alphazero_othello_b200 import _lib
    pos = random_positions(330, 150, (8, 30))
    v, _, _ = _kernel(pos, 3, 12)
    L = _lib.lib()
    n = len(pos)
    states = np.ascontiguousarray(np.stack([s.reshape(64) for s, _ in pos]).astype(np.int8))
    pis = np.ascontiguousarray(v.astype(np.float32))
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    for k in range(4):
        for flip in (0, 1):
            ks, fl = np.full(n, k, np.int32), np.full(n, flip, np.uint8)
            os_, op = np.zeros((n, 64), np.float32), np.zeros((n, 65), np.float32)
            _lib.check(L.oth_host_symmetry(p(states), p(pis), p(ks), p(fl), p(os_), p(op), n))
            img = [(os_[i].astype(np.int8).reshape(8, 8), pl) for i, (_, pl) in enumerate(pos)]
            vi, _, _ = _kernel(img, 3, 12)
            assert np.array_equal(vi, op.astype(np.int64).astype(np.int32)), (k, flip)


def test_launch_geometry_independence_exact_12():
    pos = random_positions(340, 4097, (10, 14))
    assert (_empties(pos) == 12).sum() >= 500
    v, b, nd = _kernel(pos, 3, 12)
    assert ((nd > 0) == (v != O_NONE)).all()
    for sl in (slice(0, 1), slice(1000, 1031)):
        vs, bs, ns = _kernel(pos[sl], 3, 12)
        assert np.array_equal(vs, v[sl]) and np.array_equal(bs, b[sl]) and np.array_equal(ns, nd[sl])
    perm = np.random.default_rng(0).permutation(len(pos))
    vp, bp, npn = _kernel([pos[i] for i in perm], 3, 12)
    assert np.array_equal(vp, v[perm]) and np.array_equal(bp, b[perm]) and np.array_equal(npn, nd[perm])


def test_terminal_roots_on_the_split_path():
    """Positions where neither side can move with 12 empty squares (one colour only on the board), among live ones."""
    term = []
    for pl in (1, -1):
        s = np.full(64, pl, np.int8)
        s[:12] = 0
        term.append((s.reshape(8, 8), pl))
    live = forced_pass_positions(350, 2) + random_positions(351, 2, (12, 12))
    for depth, exact in ((1, 12), (7, 12)):
        v, b, nodes = _kernel(term + live, depth, exact)
        assert (b[:2] == -1).all() and (v[:2] == O_NONE).all() and (nodes[:2] == 0).all()
        assert (b[2:] >= 0).all() and ((nodes[2:] > 0) == (v[2:] != O_NONE)).all()


def test_evaluate_vs_alphabeta_at_the_caps():
    import torch
    from alphazero_othello_b200.Models import FastOthelloNet
    from alphazero_othello_b200.alphabeta import AlphaBetaPlayer
    from alphazero_othello_b200.eval import evaluate_vs_alphabeta
    torch.manual_seed(0)
    np.random.seed(0)
    rates, log = evaluate_vs_alphabeta(FastOthelloNet(8, 65).eval(), {"c_puct": 2.0, "num_simulations": 6}, 2,
                                       player=AlphaBetaPlayer(depth=7, exact_empties=12, margin=10))
    assert set(rates) == {"win", "draw", "loss"} and abs(sum(rates.values()) - 1.0) < 1e-12
    assert (log["plies"] > 0).all()


def test_caps_vs_depth1_is_reproduced_by_the_oracle():
    """Every move of both sides is the oracle's values run through the player's pick.  The plies are first walked
    with the logged actions, then all searched by the oracle in parallel."""
    from alphazero_othello_b200.alphabeta import AlphaBetaPlayer, pick
    from alphazero_othello_b200.eval import play_matches_batched
    a, b = AlphaBetaPlayer(depth=7, exact_empties=12), AlphaBetaPlayer(depth=1, exact_empties=4)
    np.random.seed(5)
    results, log = play_matches_batched(a, b, {"num_simulations": 0}, 2)
    g = O.OracleGame()
    plies = []  # (match, ply, state, player, mover)
    for i in range(len(results)):
        first, second = (a, b) if i % 2 == 0 else (b, a)
        s, pl, res = g.get_initial_state(), 1, None
        for ply in range(128):
            plies.append((i, ply, s, pl, first if pl == 1 else second))
            act = int(log["actions"][i, ply])
            s = g.get_next_state(s, act, pl)
            rew, done = g.get_value_and_terminated(s, act, pl)
            if done:
                res = "Draw" if rew == 0 else ("A" if (rew == 1) == (pl == 1) else "B")
                break
            pl = -pl
        if i % 2 == 1 and res != "Draw":
            res = "B" if res == "A" else "A"
        assert res == results[i] and log["plies"][i] == ply + 1, i
    assert any(m is a and (s == 0).sum() == 12 for _, _, s, _, m in plies)  # an exact ply of the split search
    ABO.lib()
    vals = list(_POOL.map(lambda q: ABO.alphabeta(q[2], q[3], q[4].depth, q[4].exact_empties)[0], plies))
    for (i, ply, _, _, m), v in zip(plies, vals):
        assert pick(v, m.margin, log["u_tie"][i, ply]) == log["actions"][i, ply], (i, ply)
