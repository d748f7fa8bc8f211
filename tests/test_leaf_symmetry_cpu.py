"""The leaf-symmetry contract restated in numpy (tests/symmetry_reference.py), checked without a GPU: the symmetry id
is the documented Philox block, the eight ids are equally likely, the square permutation is the oracle's
get_random_symmetry mapping, and every consumer rejects a mode it does not support before touching a device."""
import numpy as np
import pytest
from scipy import stats

import symmetry_reference as R

# Random123's known-answer vectors of Philox4x32-10: (counter words c0..c3, key words k0, k1) -> x (first output word)
KAT = [((0, 0, 0, 0), (0, 0), 0x6627E8D5),
       ((0xFFFFFFFF,) * 4, (0xFFFFFFFF, 0xFFFFFFFF), 0x408F276D),
       ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), 0xD16CFE09)]


@pytest.mark.parametrize("ctr,key,x", KAT)
def test_symmetry_id_is_the_documented_philox_block(ctr, key, x):
    """own = (c1 << 32 | c0), opp = (c3 << 32 | c2), seed ^ OTH_SYM_SALT = (k1 << 32 | k0): the id is x & 7."""
    own = np.uint64(ctr[1] << 32 | ctr[0])
    opp = np.uint64(ctr[3] << 32 | ctr[2])
    seed = (key[1] << 32 | key[0]) ^ R.SYM_SALT
    assert int(R.sym_ids(seed, own, opp)) == x & 7


def test_symmetry_id_depends_on_the_position_and_the_seed():
    rng = np.random.default_rng(1)
    own = rng.integers(0, 2**63, 4096, dtype=np.uint64)
    opp = rng.integers(0, 2**63, 4096, dtype=np.uint64) & ~own
    a, b = R.sym_ids(7, own, opp), R.sym_ids(8, own, opp)
    assert np.array_equal(a, R.sym_ids(7, own.copy(), opp.copy()))
    assert (a != b).mean() > 0.8 and (a != R.sym_ids(7, opp, own)).mean() > 0.8


def test_eight_ids_are_equally_likely():
    rng = np.random.default_rng(2024)
    n = 100_000
    cells = rng.integers(-1, 2, (n, 64))  # random disc placements: own / empty / opponent per square
    ids = R.plane_ids(12345, cells.astype(np.float32))
    counts = np.bincount(ids, minlength=8)
    assert counts.sum() == n and len(counts) == 8
    assert stats.chisquare(counts).pvalue > 1e-3, counts


@pytest.mark.parametrize("s", range(8))
def test_transform_and_unsymmetrise_are_the_oracles_symmetry(s):
    import oracle as O
    rng = np.random.default_rng(s)
    for _ in range(4):
        board = rng.integers(-1, 2, (8, 8)).astype(np.int8)
        pi = rng.random(65).astype(np.float32)
        ref_s, ref_pi = O.symmetry(board, pi, s & 3, s >> 2)
        assert np.array_equal(R.transform(board.reshape(1, 64).astype(np.float32), s)[0], ref_s.reshape(64))
        assert np.array_equal(R.transform(pi[None], s)[0], ref_pi)
        # unsymmetrise undoes the transform on the squares and keeps the pass entry and any padding
        row = np.concatenate([pi, [7.0, 8.0]]).astype(np.float32)[None]
        u = R.unsymmetrise(row, s)
        assert np.array_equal(R.transform(u, s), row) and np.array_equal(u[0, 64:], row[0, 64:])
        assert np.array_equal(R.unsymmetrise(R.transform(row, s), s), row)


def test_mean_of_a_symmetric_network_is_its_own_output():
    """If every image's logits are the transform of one row, the mean of the unsymmetrised priors is that row's softmax."""
    rng = np.random.default_rng(3)
    row = rng.normal(size=(1, 65))
    logits = np.concatenate([R.transform(row, j) for j in range(8)])
    pri, val = R.mean(logits, np.full(8, 0.25))
    assert np.allclose(pri[0], R.softmax64(row)[0], atol=1e-15) and val[0] == 0.25


def test_every_consumer_rejects_a_mode_it_does_not_support():
    from alphazero_othello_b200 import symmetry
    from alphazero_othello_b200.MCTS_model import MCTS
    from alphazero_othello_b200.engine import SelfPlayRunner
    from alphazero_othello_b200.eval import play_matches_batched
    from alphazero_othello_b200.self_play_worker import collect_self_play_games, collect_self_play_games_distributed

    class HostPolicy:
        def inference(self, state, player):
            return np.full(65, 1 / 65, np.float32), 0.0

    assert symmetry.check_mode(None) is None and symmetry.check_mode("mean") == "mean"
    for bad in ("sideways", "Random", "", 1, ["random"]):
        for call in (lambda: SelfPlayRunner(None, None, leaf_symmetry=bad),
                     lambda: collect_self_play_games(None, {}, 1, leaf_symmetry=bad),
                     lambda: collect_self_play_games_distributed(None, {}, 1, leaf_symmetry=bad),
                     lambda: play_matches_batched(None, None, {}, 2, leaf_symmetry=bad),
                     lambda: MCTS(None, {}, None, leaf_symmetry=bad)):
            with pytest.raises(ValueError):
                call()
    # self-play offers "random" only: "mean" costs eight network rows per leaf
    for call in (lambda: SelfPlayRunner(None, None, leaf_symmetry="mean"),
                 lambda: collect_self_play_games(None, {}, 1, leaf_symmetry="mean"),
                 lambda: collect_self_play_games_distributed(None, {}, 1, leaf_symmetry="mean")):
        with pytest.raises(ValueError, match="not supported"):
            call()
    # MCTS: only a torch module policy is evaluated on the device; a host inference policy or rollouts have no network rows
    for mode in ("random", "mean"):
        for policy in (HostPolicy(), None):
            with pytest.raises(ValueError, match="torch module"):
                MCTS(None, {"num_simulations": 2, "c_puct": 1.0}, policy, leaf_symmetry=mode)
