"""oth_alphabeta on the GPU: bit for bit against the CPU oracle's alpha-beta (itself checked against plain negamax in
test_alphabeta_cpu.py), D4 invariance, launch-geometry independence, and arena matches with AlphaBetaPlayer sides
replayed move by move through the oracle."""
import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import alphabeta_oracle as ABO
import oracle as O
from test_alphabeta_cpu import forced_pass_positions, random_positions

pytestmark = pytest.mark.gpu

_POOL = ThreadPoolExecutor(max(1, min(16, os.cpu_count() or 1)))  # the oracle's ctypes calls release the GIL


def _bits(positions):
    w = np.uint64(1) << np.arange(64, dtype=np.uint64)
    own = np.array([((s.reshape(64) == pl) * w).sum(dtype=np.uint64) for s, pl in positions], np.uint64)
    opp = np.array([((s.reshape(64) == -pl) * w).sum(dtype=np.uint64) for s, pl in positions], np.uint64)
    return own.view(np.int64), opp.view(np.int64)


def _kernel(positions, depth, exact=0):
    import torch
    from alphazero_othello_b200.alphabeta import search
    own, opp = _bits(positions)
    v, b, n = search(torch.from_numpy(own).cuda(), torch.from_numpy(opp).cuda(), depth, exact)
    return v.cpu().numpy(), b.cpu().numpy(), n.cpu().numpy()


def _oracle(positions, depth, exact=0):
    ABO.lib()  # compiled once, before the worker threads call it
    res =list(_POOL.map(lambda p: ABO.alphabeta(p[0], p[1], depth, exact), positions))
    return np.stack([r[0] for r in res]), np.array([r[1] for r in res], np.int32)


def _check(positions, depth, exact=0):
    v, b, nodes = _kernel(positions, depth, exact)
    ov, ob = _oracle(positions, depth, exact)
    bad = np.nonzero((v != ov).any(1) | (b != ob))[0]
    assert len(bad) == 0, (depth, exact, bad[:5], v[bad[:1]], ov[bad[:1]])
    legal = v != O_NONE
    assert ((nodes > 0) == legal).all()
    return v, b, nodes


O_NONE = -2**31


def test_kernel_matches_oracle_depths_1_to_4():
    for depth in (1, 2, 3, 4):
        _check(random_positions(200 + depth, 500, (4, 59)), depth)


def test_kernel_matches_oracle_depths_5_and_6():
    _check(random_positions(205, 130, (14, 56)), 5)
    _check(random_positions(206, 80, (18, 52)), 6)


def test_kernel_matches_oracle_exact_endgames():
    from alphazero_othello_b200 import _lib
    _check(random_positions(210, 110, (10, 11)), 2, 11)
    cap = _lib.AB_MAX_EXACT
    at_cap = random_positions(214, 12, (cap, cap))
    assert all((s == 0).sum() == cap for s, _ in at_cap)
    _check(at_cap, 1, cap)
    # below the threshold the depth limit applies: the same roots searched 3 plies deep
    _check(random_positions(211, 60, (10, 12)), 3, 9)


def test_kernel_forced_pass_and_terminal_roots():
    fp = forced_pass_positions(220, 40)
    v, b, _ = _check(fp, 3)
    assert (b == 64).all() and (v[:, :64] == O_NONE).all()
    _check([p for p in fp if (p[0] == 0).sum() <= 11], 1, 11)
    g, rng, term = O.OracleGame(), np.random.default_rng(221), []
    while len(term) < 20:
        s, pl = g.get_initial_state(), 1
        while not g.get_value_and_terminated(s, 0, pl)[1]:
            s = g.get_next_state(s, int(rng.choice(np.nonzero(g.get_valid_moves(s, pl))[0])), pl)
            pl = -pl
        term.append((s, pl))
    for depth, exact in ((1, 0), (4, 11)):
        v, b, nodes = _kernel(term + fp[:3], depth, exact)
        assert (b[:20] == -1).all() and (v[:20] == O_NONE).all() and (nodes[:20] == 0).all()
        assert (b[20:] == 64).all()


def test_d4_images_give_permuted_values():
    """The eight images of a position (oth_symmetry's mapping, applied to the board and to the value row) search to
    the image of the value row.  No oracle involved."""
    from alphazero_othello_b200 import _lib
    pos = random_positions(230, 150, (8, 56))
    v, b, _ = _kernel(pos, 3, 10)
    L = _lib.lib()
    for k in range(4):
        for flip in (0, 1):
            n = len(pos)
            states = np.ascontiguousarray(np.stack([s.reshape(64) for s, _ in pos]).astype(np.int8))
            pis = np.ascontiguousarray(v.astype(np.float32))
            ks, fl = np.full(n, k, np.int32), np.full(n, flip, np.uint8)
            os_, op = np.zeros((n, 64), np.float32), np.zeros((n, 65), np.float32)
            p = lambda a: a.ctypes.data_as(C.c_void_p)
            _lib.check(L.oth_host_symmetry(p(states), p(pis), p(ks), p(fl), p(os_), p(op), n))
            img = [(os_[i].astype(np.int8).reshape(8, 8), pl) for i, (_, pl) in enumerate(pos)]
            vi, _, _ = _kernel(img, 3, 10)
            assert np.array_equal(vi, op.astype(np.int64).astype(np.int32)), (k, flip)


def test_launch_geometry_independence():
    pos = random_positions(240, 4097, (6, 58))
    v, b, nd = _kernel(pos, 3, 8)
    v1, b1, n1 = _kernel(pos[:1], 3, 8)
    assert np.array_equal(v1, v[:1]) and np.array_equal(b1, b[:1]) and np.array_equal(n1, nd[:1])
    v31, b31, n31 = _kernel(pos[1000:1031], 3, 8)
    assert np.array_equal(v31, v[1000:1031]) and np.array_equal(b31, b[1000:1031]) and np.array_equal(n31, nd[1000:1031])
    perm = np.random.default_rng(0).permutation(len(pos))
    vp, bp, npn = _kernel([pos[i] for i in perm], 3, 8)
    assert np.array_equal(vp, v[perm]) and np.array_equal(bp, b[perm]) and np.array_equal(npn, nd[perm])


def _replay(log, results, sides, args):
    """Replay every match of an arena log on the CPU.  ``sides`` = (policy_a, policy_b): a salt (hash-stub MCTS) or an
    AlphaBetaPlayer.  The oracle MCTS is fed the logged tie uniforms; alpha-beta moves are the oracle's values run
    through the same pick."""
    from alphazero_othello_b200.alphabeta import AlphaBetaPlayer, pick
    g = O.OracleGame()
    games = set()
    for i in range(len(results)):
        first, second = sides if i % 2 == 0 else sides[::-1]
        movers = {}
        for colour, pol in ((1, first), (-1, second)):
            movers[colour] = pol if isinstance(pol, AlphaBetaPlayer) else \
                O.OracleMCTS(args["c_puct"], args["num_simulations"], O.Evaluator(stub=O.STUB_H, salt=pol))
        searched = {1: False, -1: False}
        s, pl, res = g.get_initial_state(), 1, None
        for ply in range(128):
            u = log["u_tie"][i, ply]
            m = movers[pl]
            if isinstance(m, AlphaBetaPlayer):
                vals, _, _ = ABO.alphabeta(s, pl, m.depth, m.exact_empties)
                a = pick(vals, m.margin, u)
            else:
                a = int(np.argmax(m.policy_improve_step(s, pl, 0.0, None, u)))
                searched[pl] = True
            assert a == log["actions"][i, ply], (i, ply, a, log["actions"][i, ply])
            s = g.get_next_state(s, a, pl)
            rew, done = g.get_value_and_terminated(s, a, pl)
            if done:
                res = "Draw" if rew == 0 else ("A" if (rew == 1) == (pl == 1) else "B")
                break
            for p2 in (1, -1):
                if searched[p2]:
                    movers[p2].make_move(a)
            pl = -pl
        if i % 2 == 1 and res != "Draw":
            res = "B" if res == "A" else "A"
        assert res == results[i] and log["plies"][i] == ply + 1, i
        games.add(tuple(log["actions"][i, :ply + 1]))
    return games


@pytest.mark.parametrize("margin", [0, 40])
def test_arena_stub_mcts_vs_alphabeta_replays_through_oracle(margin):
    from alphazero_othello_b200.alphabeta import AlphaBetaPlayer
    from alphazero_othello_b200.eval import DeviceStubPolicy, play_matches_batched
    args = {"c_puct": 2.0, "num_simulations": 12}
    ab = AlphaBetaPlayer(depth=2, exact_empties=8, margin=margin)
    np.random.seed(11 + margin)
    for sides in ((DeviceStubPolicy("H", 5), ab), (ab, DeviceStubPolicy("H", 6))):
        results, log = play_matches_batched(*sides, args, 6)
        salts = tuple(s if isinstance(s, AlphaBetaPlayer) else s.salt for s in sides)
        games = _replay(log, results, salts, args)
        if margin > 0:
            assert len(games) >= 2


def test_evaluate_vs_alphabeta_with_a_network():
    import torch
    from alphazero_othello_b200.Models import FastOthelloNet
    from alphazero_othello_b200.alphabeta import AlphaBetaPlayer
    from alphazero_othello_b200.eval import evaluate_vs_alphabeta
    torch.manual_seed(0)
    np.random.seed(0)
    rates, log = evaluate_vs_alphabeta(FastOthelloNet(8, 65).eval(), {"c_puct": 2.0, "num_simulations": 6}, 6,
                                       player=AlphaBetaPlayer(depth=2, exact_empties=6, margin=10))
    assert set(rates) == {"win", "draw", "loss"} and abs(sum(rates.values()) - 1.0) < 1e-12
    assert all(0.0 <= r <= 1.0 for r in rates.values()) and (log["plies"] > 0).all()


def test_alphabeta_vs_alphabeta_is_reproduced_by_the_oracle():
    from alphazero_othello_b200.alphabeta import AlphaBetaPlayer
    from alphazero_othello_b200.eval import play_matches_batched
    a, b = AlphaBetaPlayer(depth=3, exact_empties=8), AlphaBetaPlayer(depth=1, exact_empties=4)
    np.random.seed(3)
    results, log = play_matches_batched(a, b, {"num_simulations": 0}, 2)
    _replay(log, results, (a, b), {})
    again, log2 = play_matches_batched(a, b, {"num_simulations": 0}, 2, u_tie=log["u_tie"])
    assert again == results and np.array_equal(log2["actions"], log["actions"])
