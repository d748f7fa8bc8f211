"""oth_solve_wld on the GPU: bit for bit against the CPU oracle's win/draw/loss (itself checked against the alpha-beta
oracle's exact values in test_endgame_cpu.py) from 1 empty square to the cap, agreement with the alpha-beta player's
exact values, D4 invariance, launch-geometry independence, and relabelled self-play outputs."""
import numpy as np
import pytest

import oracle as O
import wld_oracle as WO
from test_alphabeta_cpu import random_positions
from test_alphabeta_deep_gpu import _forced_pass_between
from test_alphabeta_gpu import _POOL, _bits

pytestmark = pytest.mark.gpu


def _solve(positions, max_empties=None):
    import torch
    from alphazero_othello_b200 import endgame
    own, opp = _bits(positions)
    w, n = endgame.solve_wld(torch.from_numpy(own).cuda(), torch.from_numpy(opp).cuda(),
                             endgame.MAX_EMPTIES if max_empties is None else max_empties)
    return w.cpu().numpy(), n.cpu().numpy()


def _oracle(positions):
    WO.lib()  # compiled once, before the worker threads call it
    return np.array(list(_POOL.map(lambda p: WO.wld(p[0], p[1])[0], positions)), np.int8)


def _check(positions):
    w, nodes = _solve(positions)
    ow = _oracle(positions)
    bad = np.nonzero(w != ow)[0]
    assert len(bad) == 0, (bad[:5], w[bad[:5]], ow[bad[:5]])
    assert (nodes >= 1).all()
    return w


def _band(seed, n, lo, hi):
    """n positions with lo..hi empties, plus, if the band has none, a draw found in further seeded random games."""
    pos = random_positions(seed, n, (lo, hi))
    w, _ = _solve(pos)
    k = 1
    while not (w == 0).any():
        more = random_positions(seed + 1000 * k, 200, (lo, hi))
        mw, _ = _solve(more)
        pos += [more[i] for i in np.nonzero(mw == 0)[0][:1]]
        w = np.append(w, mw[mw == 0][:1])
        k += 1
    return pos


def test_solver_matches_oracle_up_to_10_empties():
    w = _check(_band(600, 2000, 1, 10) + _forced_pass_between(601, 40, 1, 10))
    assert set(w) == {-1, 0, 1}


def test_solver_matches_oracle_11_to_13_empties():
    w = _check(_band(610, 300, 11, 13) + _forced_pass_between(611, 10, 11, 13))
    assert set(w) == {-1, 0, 1}


def test_solver_matches_oracle_from_14_empties_to_the_cap():
    from alphazero_othello_b200.endgame import MAX_EMPTIES as cap
    at_cap = _band(620, 30, cap, cap)
    assert all((s == 0).sum() == cap for s, _ in at_cap)
    w = _check(_band(621, 70, 14, cap) + at_cap + _forced_pass_between(622, 3, 14, cap))
    assert set(w) == {-1, 0, 1}


def test_terminal_roots_and_roots_above_the_limit():
    g, rng, term = O.OracleGame(), np.random.default_rng(630), []
    while len(term) < 20:
        s, pl = g.get_initial_state(), 1
        while not g.get_value_and_terminated(s, 0, pl)[1]:
            s = g.get_next_state(s, int(rng.choice(np.nonzero(g.get_valid_moves(s, pl))[0])), pl)
            pl = -pl
        term.append((s, pl))
    for pl in (1, -1):  # one colour wiped out, 13 empty squares left
        s = np.full(64, pl, np.int8)
        s[:13] = 0
        term += [(s.reshape(8, 8), pl), (s.reshape(8, 8), -pl)]
    w, nodes = _solve(term)
    for (s, pl), x in zip(term, w):
        d = int((s == pl).sum()) - int((s == -pl).sum())
        assert x == (d > 0) - (d < 0)
    assert (nodes == 1).all()
    from alphazero_othello_b200.endgame import UNSOLVED
    pos = random_positions(631, 200, (4, 30))
    e = np.array([(s == 0).sum() for s, _ in pos])
    w8, n8 = _solve(pos, 8)
    w_all, n_all = _solve(pos)
    assert (e > 8).sum() >= 50 and (e <= 8).sum() >= 20
    assert (w8[e > 8] == UNSOLVED).all() and (n8[e > 8] == 0).all()
    assert np.array_equal(w8[e <= 8], w_all[e <= 8]) and np.array_equal(n8[e <= 8], n_all[e <= 8])
    w0, n0 = _solve(term[:20] + pos, 0)
    assert np.array_equal(w0[:20], w[:20]) and (w0[20:] == UNSOLVED).all() and (n0[20:] == 0).all()


def test_agrees_with_the_alphabeta_players_exact_values():
    import torch
    from alphazero_othello_b200.alphabeta import NONE, search
    pos = random_positions(640, 4097, (1, 12))
    w, _ = _solve(pos)
    own, opp = _bits(pos)
    v, _, _ = search(torch.from_numpy(own).cuda(), torch.from_numpy(opp).cuda(), 1, 12)
    v = v.cpu().numpy().astype(np.int64)
    best = np.where(v != NONE, v, -2**40).max(1)
    assert np.array_equal(w, np.sign(best)) and set(w) == {-1, 0, 1}


def test_d4_images_give_the_same_result():
    import ctypes as C
    from alphazero_othello_b200 import _lib
    pos = random_positions(650, 160, (4, 14))
    w, _ = _solve(pos)
    L = _lib.lib()
    n = len(pos)
    states = np.ascontiguousarray(np.stack([s.reshape(64) for s, _ in pos]).astype(np.int8))
    pis = np.zeros((n, 65), np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    for k in range(4):
        for flip in (0, 1):
            ks, fl = np.full(n, k, np.int32), np.full(n, flip, np.uint8)
            os_, op = np.zeros((n, 64), np.float32), np.zeros((n, 65), np.float32)
            _lib.check(L.oth_host_symmetry(p(states), p(pis), p(ks), p(fl), p(os_), p(op), n))
            img = [(os_[i].astype(np.int8).reshape(8, 8), pl) for i, (_, pl) in enumerate(pos)]
            assert np.array_equal(_solve(img)[0], w), (k, flip)


def test_launch_geometry_independence():
    pos = random_positions(660, 4097, (2, 14))
    w, nd = _solve(pos)
    for sl in (slice(0, 1), slice(1000, 1031)):
        ws, ns = _solve(pos[sl])
        assert np.array_equal(ws, w[sl]) and np.array_equal(ns, nd[sl])
    perm = np.random.default_rng(0).permutation(len(pos))
    wp, npn = _solve([pos[i] for i in perm])
    assert np.array_equal(wp, w[perm]) and np.array_equal(npn, nd[perm])
    # the host-buffer form
    import ctypes as C
    from alphazero_othello_b200 import _lib
    own, opp = _bits(pos[:300])
    hw, hn = np.zeros(300, np.int8), np.zeros(300, np.uint64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    _lib.check(_lib.lib().oth_host_solve_wld(p(own), p(opp), 300, _lib.SOLVE_MAX_EMPTIES, p(hw), p(hn)))
    assert np.array_equal(hw, w[:300]) and np.array_equal(hn.astype(np.int64), nd[:300])


ARGS = {"c_puct": 2.0, "num_simulations": 6, "dirichlet_alpha": 1.0, "dirichlet_epsilon": 0.3, "mcts_temperature": 1.0,
        "num_exploratory_moves": 35}


def _self_play(lam, **kw):
    import torch
    from alphazero_othello_b200.Models import FastOthelloNet
    from alphazero_othello_b200.self_play_worker import collect_self_play_games
    torch.manual_seed(0)
    return collect_self_play_games(FastOthelloNet(8, 65).eval(), dict(ARGS, **{"lambda": lam}), 16, n_slots=16, seed=7,
                                   return_raw=True, **kw)


def _positions(out):
    own, opp = out["boards"][:, 0].cpu().numpy().view(np.uint64), out["boards"][:, 1].cpu().numpy().view(np.uint64)
    bits = lambda x: ((x[:, None] >> np.arange(64, dtype=np.uint64)) & np.uint64(1)).astype(np.int8)
    states = bits(own) - bits(opp)
    return [(s.reshape(8, 8), 1) for s in states], (states == 0).sum(1)


def test_relabel_a_self_play_output():
    import torch
    from alphazero_othello_b200 import endgame
    out = _self_play(0.98)
    cap = endgame.MAX_EMPTIES
    pos, e = _positions(out)
    low = e <= cap
    assert low.sum() >= 48 and (~low).sum() >= 48
    want = _oracle([p for p, m in zip(pos, low) if m]).astype(np.float64)
    for src in (out, {k: v.cuda() for k, v in out.items()}):
        r = endgame.relabel(src, cap)
        assert set(r) == set(src) | {"solved"}
        for k in src:
            assert r[k].device == src[k].device
            if k != "values":
                assert r[k] is src[k]
        solved = r["solved"].cpu().numpy()
        assert np.array_equal(solved, low)
        vals, old = r["values"].cpu().numpy(), src["values"].cpu().numpy()
        assert vals.dtype == old.dtype and np.array_equal(vals[~low].view(np.int64), old[~low].view(np.int64))
        assert np.array_equal(vals[low], want)
    assert torch.equal(endgame.relabel(out, 14)["solved"], torch.from_numpy(e <= 14))


def test_collect_self_play_games_solve_empties():
    from alphazero_othello_b200 import endgame
    cap = endgame.MAX_EMPTIES
    out = _self_play(1.0, solve_empties=cap)
    pos, e = _positions(out)
    solved = out["solved"].cpu().numpy()
    assert np.array_equal(solved, e <= cap) and solved.sum() >= 48
    vals = out["values"].cpu().numpy()
    assert np.array_equal(vals[solved], _oracle([p for p, m in zip(pos, solved) if m]).astype(np.float64))
    # with lambda = 1 every other target is the game's outcome from its mover's side
    games = out["games"].cpu().numpy()
    player = (out["meta"].cpu().numpy() & 0xFF).astype(np.uint8).view(np.int8).astype(np.int64)
    outcome = np.zeros(len(vals))
    for _gid, first, n, winner in games:
        sl = slice(first, first + n)
        outcome[sl] = 0.0 if winner == 0 else np.where(player[sl] == winner, 1.0, -1.0)
    assert np.array_equal(vals[~solved], outcome[~solved])


def test_solve_empties_zero_never_relabels(monkeypatch):
    from alphazero_othello_b200 import endgame

    def fail(*a, **k):
        raise AssertionError("relabel called")
    monkeypatch.setattr(endgame, "relabel", fail)
    out = _self_play(0.98)
    assert "solved" not in out and out["values"].numel() > 0
