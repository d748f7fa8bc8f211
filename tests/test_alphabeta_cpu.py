"""The alpha-beta player without a GPU: the CPU oracle's alpha-beta against its plain negamax, known answers, argument
validation of the library entry points, and the arena's move pick among the root values."""
import numpy as np
import pytest

import alphabeta_oracle as ABO
import oracle as O
from alphazero_othello_b200 import _lib
from alphazero_othello_b200.alphabeta import NONE, AlphaBetaPlayer, pick

W = np.array([[100, -20, 10, 5, 5, 10, -20, 100], [-20, -50, -2, -2, -2, -2, -50, -20], [10, -2, -1, -1, -1, -1, -2, 10],
              [5, -2, -1, -1, -1, -1, -2, 5]])
W = np.concatenate([W, W[::-1]])


def random_positions(seed, n, empties_range, want=None):
    """n (state, player) pairs from seeded uniform-random games, taken where the number of empty squares falls in
    ``empties_range`` (inclusive) and ``want(state, player)`` holds; terminal positions are never taken."""
    g, rng, out = O.OracleGame(), np.random.default_rng(seed), []
    lo, hi = empties_range
    while len(out) < n:
        s, pl = g.get_initial_state(), 1
        target = int(rng.integers(lo, hi + 1))
        while not g.get_value_and_terminated(s, 0, pl)[1]:
            if (s == 0).sum() <= target:
                if want is None or want(s, pl):
                    out.append((s.copy(), pl))
                break
            acts = np.nonzero(g.get_valid_moves(s, pl))[0]
            s = g.get_next_state(s, int(rng.choice(acts)), pl)
            pl = -pl
    return out


def forced_pass(s, pl):
    g = O.OracleGame()
    return g.get_valid_moves(s, pl)[64] == 1 and not g.get_value_and_terminated(s, 0, pl)[1]


def forced_pass_positions(seed, n):
    """Positions where the side to move must pass, from seeded random games."""
    g, rng, out = O.OracleGame(), np.random.default_rng(seed), []
    while len(out) < n:
        s, pl = g.get_initial_state(), 1
        while not g.get_value_and_terminated(s, 0, pl)[1]:
            if forced_pass(s, pl):
                out.append((s.copy(), pl))
                break
            acts = np.nonzero(g.get_valid_moves(s, pl))[0]
            s = g.get_next_state(s, int(rng.choice(acts)), pl)
            pl = -pl
    return out


def heuristic(s, pl):
    """The depth-0 score of include/othello_b200.h, from the definition."""
    g = O.OracleGame()
    mob = lambda p: 0 if g.get_valid_moves(s, p)[64] else int(g.get_valid_moves(s, p)[:64].sum())
    return int((W * ((s == pl).astype(int) - (s == -pl).astype(int))).sum()) + 10 * (mob(pl) - mob(-pl))


def exhaustive(s, pl):
    """Exact negamax on the Game API, for a handful of empty squares."""
    g = O.OracleGame()
    if g.get_value_and_terminated(s, 0, pl)[1]:
        return 10000 * g.get_score(s, pl)
    return max(-exhaustive(g.get_next_state(s, int(a), pl), -pl) for a in np.nonzero(g.get_valid_moves(s, pl))[0])


def _agree(s, pl, depth, exact):
    v1, b1, n1 = ABO.negamax(s, pl, depth, exact)
    v2, b2, n2 = ABO.alphabeta(s, pl, depth, exact)
    assert np.array_equal(v1, v2) and b1 == b2, (s, pl, depth, exact)
    assert n2 <= n1
    legal = v1 != NONE
    assert b1 == int(np.nonzero(legal & (v1 == v1[legal].max()))[0][0])
    return v1


@pytest.mark.parametrize("depth", [1, 2, 3, 4])
def test_oracle_alphabeta_equals_negamax_midgame(depth):
    for s, pl in random_positions(100 + depth, 12, (20, 56)):
        _agree(s, pl, depth, 0)


def test_oracle_alphabeta_equals_negamax_exact_endgames():
    for s, pl in random_positions(7, 25, (1, 8)):
        _agree(s, pl, 1, 8)
    # one move from the end, forced-pass roots (searched both depth-limited and exactly)
    for s, pl in random_positions(8, 10, (1, 1)):
        v = _agree(s, pl, 2, 0)
        assert np.array_equal(v, _agree(s, pl, 1, 1))
    for s, pl in forced_pass_positions(9, 8):
        v = _agree(s, pl, 3, 0)
        assert list(np.nonzero(v != NONE)[0]) == [64]
        if (s == 0).sum() <= 8:
            _agree(s, pl, 1, 8)


def test_depth_one_values_are_the_heuristic_of_the_children():
    g = O.OracleGame()
    s0 = g.get_initial_state()
    assert heuristic(s0, 1) == 0
    for s, pl in [(s0, 1)] + random_positions(3, 8, (10, 50)) + forced_pass_positions(4, 2):
        v, _, _ = ABO.alphabeta(s, pl, 1, 0)
        for a in np.nonzero(v != NONE)[0]:
            c = g.get_next_state(s, int(a), pl)
            want = 10000 * g.get_score(c, pl) if g.get_value_and_terminated(c, 0, -pl)[1] else -heuristic(c, -pl)
            assert v[a] == want, (a, v[a], want)


def test_initial_position_moves_are_equal_by_symmetry():
    s0 = O.OracleGame().get_initial_state()
    for depth in range(1, 6):
        v, best, _ = ABO.alphabeta(s0, 1, depth, 0)
        assert list(np.nonzero(v != NONE)[0]) == [19, 26, 37, 44]
        assert len(set(v[[19, 26, 37, 44]])) == 1 and best == 19


def test_last_empties_are_disc_difference_times_win_scale():
    s = -np.ones(64, np.int8)
    s[0], s[2] = 0, 1                    # +1 plays 0 and flips 1: a full board, 3 discs against 61
    v, best, _ = ABO.alphabeta(s, 1, 1, 2)
    assert best == 0 and v[0] == 10000 * (3 - 61) and (v[1:] == NONE).all()
    s[63], s[61] = 0, 1                  # a second empty: after 0, -1 must pass and +1 plays 63
    for depth, exact in ((1, 2), (3, 0), (7, 11)):
        v, best, _ = ABO.alphabeta(s, 1, depth, exact)
        legal = np.nonzero(v != NONE)[0]
        assert list(legal) == [0, 63]
        g = O.OracleGame()
        for a in legal:
            c = g.get_next_state(s.reshape(8, 8), int(a), 1)
            assert v[a] == -exhaustive(c, -1) and v[a] % 10000 == 0
        assert np.array_equal(v, ABO.negamax(s, 1, depth, exact)[0])


def test_terminal_root_has_no_action():
    s = np.ones(64, np.int8)
    s[:10] = -1
    for f in (ABO.negamax, ABO.alphabeta):
        v, best, nodes = f(s, 1, 3, 11)
        assert best == -1 and (v == NONE).all() and nodes == 0


def test_argument_validation_without_device():
    L = _lib.lib()
    E = _lib.OTH_E_ARG
    for fn, tail in ((L.oth_alphabeta, (None, None, None, None)), (L.oth_host_alphabeta, (None, None, None))):
        assert fn(None, None, 1, 0, 0, *tail) == E                        # depth 0
        assert fn(None, None, 1, _lib.AB_MAX_DEPTH + 1, 0, *tail) == E    # depth above the cap
        assert fn(None, None, 1, 4, _lib.AB_MAX_EXACT + 1, *tail) == E    # exact_empties above the cap
        assert fn(None, None, 1, 4, -1, *tail) == E
        assert fn(None, None, -1, 4, 0, *tail) == E                       # n < 0
        assert fn(None, None, 1, 4, 0, *tail) == E                        # missing buffers
        assert fn(None, None, 0, _lib.AB_MAX_DEPTH, _lib.AB_MAX_EXACT, *tail) == _lib.OTH_OK
    with pytest.raises(ValueError):
        AlphaBetaPlayer(depth=0)
    with pytest.raises(ValueError):
        AlphaBetaPlayer(exact_empties=_lib.AB_MAX_EXACT + 1)
    with pytest.raises(ValueError):
        AlphaBetaPlayer(margin=-1)


def test_pick_among_values_within_margin():
    row = np.full(65, NONE, np.int32)
    row[[3, 10, 20, 40]] = [50, 70, 70, 65]
    assert pick(row, 0, 0.0) == 10 and pick(row, 0, 0.49) == 10 and pick(row, 0, 0.5) == 20
    assert pick(row, 0, 1.0) == 20                           # u = 1 cannot index past the candidates
    assert [pick(row, 5, u) for u in (0.0, 0.34, 0.67, 0.99)] == [10, 20, 40, 40]
    assert [pick(row, 20, u) for u in (0.0, 0.25, 0.5, 0.75)] == [3, 10, 20, 40]
    neg = np.full(65, NONE, np.int32)
    neg[64] = -30000                                          # a forced pass is the only move
    assert pick(neg, 100, 0.9) == 64
    with pytest.raises(ValueError):
        pick(np.full(65, NONE, np.int32), 0, 0.5)
