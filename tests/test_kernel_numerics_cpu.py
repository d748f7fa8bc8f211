"""The float64 restatement of the engine's Dirichlet root noise (tests/noise_reference.py), checked before the kernel is
compared with it: its Philox against the CPU oracle's and the published known answers, its keys and counters against a
scalar transcription of ``make_noise``, and its output against the Dirichlet law it is meant to sample."""
import numpy as np
import pytest
from scipy import stats

import noise_reference as NR


def test_philox_restatement_matches_the_oracle_and_the_known_answers():
    import oracle as O
    # Random123's kat_vectors for philox4x32_10: (counter words, key words, output)
    kat = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
           ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for (c0, c1, c2, c3), (k0, k1), want in kat:
        seed, lo = k0 | (k1 << 32), c0 | (c1 << 32)
        assert tuple(int(v) for v in NR.philox4x32_10(seed, lo, c2, c3)) == want
        assert tuple(int(v) for v in O.philox(seed, lo, c2, c3)) == want
    rng = np.random.default_rng(5)
    seeds = rng.integers(0, 2**63, 64, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, 64, dtype=np.uint64)
    lo = rng.integers(0, 2**63, 64, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, 64, dtype=np.uint64)
    h0 = rng.integers(0, 2**32, 64, dtype=np.uint64).astype(np.uint32)
    h1 = rng.integers(0, 2**32, 64, dtype=np.uint64).astype(np.uint32)
    for i in range(64):
        got = NR.philox4x32_10(int(seeds[i]), lo[i], h0[i], h1[i])
        assert [int(v) for v in got] == [int(v) for v in O.philox(int(seeds[i]), int(lo[i]), int(h0[i]), int(h1[i]))]
    # vectorised over counters = one block at a time
    vec = NR.philox4x32_10(int(seeds[0]), lo, h0, h1)
    for i in range(64):
        assert [int(v[i]) for v in vec] == [int(v) for v in NR.philox4x32_10(int(seeds[0]), lo[i], h0[i], h1[i])]


def _scalar_gamma(seed, game_id, e, alpha, ply):
    """One entry of make_noise, transcribed line by line with the oracle's Philox (the counter argument order of
    ``orc_philox4x32_10`` / ``philox4x32_10(seed, ctr_lo, ctr_hi0, ctr_hi1)``)."""
    import math
    import oracle as O
    a = alpha + 1.0 if alpha < 1.0 else alpha
    d = a - 1.0 / 3.0
    cc = 1.0 / math.sqrt(9.0 * d)
    for k in range(256):
        r = [int(v) for v in O.philox(seed ^ 0x6E6F697365, game_id, e, k | (ply << 16))]
        u1 = (r[0] + 1.0) * (1.0 / 4294967296.0)
        u2 = r[1] * (1.0 / 4294967296.0)
        x = math.sqrt(-2.0 * math.log(u1)) * float(NR.cospi(np.float64(2.0 * u2)))
        v = 1.0 + cc * x
        if v <= 0.0:
            continue
        v = v * v * v
        u = (r[2] + 0.5) * (1.0 / 4294967296.0)
        if math.log(u) < 0.5 * x * x + d - d * v + d * math.log(v):
            g = d * v
            if alpha < 1.0:
                g *= float(np.power((r[3] + 0.5) * (1.0 / 4294967296.0), 1.0 / alpha))  # numpy's pow, as the restatement
            return g
    return d


@pytest.mark.parametrize("alpha", [0.03, 0.3, 1.0, 2.5, 10.0])
def test_noise_restatement_follows_the_documented_stream(alpha):
    """Key seed ^ 0x6e6f697365, counter (game_id, e, k | ply << 16): the vectorised restatement against a scalar
    transcription, for several seeds, game ids (one above 2^32) and plies."""
    for seed, gids, ply in ((0, [0, 1, 77], 0), (2024, [5, 2**33 + 9], 0), (123456789, [3, 40], 1), (9, [1], 17)):
        g = NR.gammas(seed, gids, alpha, ply)
        for i, gid in enumerate(gids):
            for e in (0, 1, 31, 63, 64):
                assert g[i, e] == _scalar_gamma(seed, gid, e, alpha, ply), (seed, gid, e, ply)
    # the ply is part of the counter: a fresh root at a later ply draws other noise
    assert not np.array_equal(NR.gammas(7, [3], alpha, 0), NR.gammas(7, [3], alpha, 1))
    nz = NR.dirichlet_noise(7, np.arange(64), alpha)
    assert (nz >= 0).all() and np.abs(nz.sum(1) - 1.0).max() < 1e-12


@pytest.mark.parametrize("alpha", [0.03, 0.3, 1.0, 2.5])
def test_noise_restatement_has_dirichlet_marginals(alpha):
    """Every marginal of Dirichlet(alpha 1_65) is Beta(alpha, 64 alpha): a Kolmogorov-Smirnov test per column on
    4 096 games, Bonferroni-corrected over the 65 columns (family-wise level 1e-3)."""
    n = 4096
    nz = NR.dirichlet_noise(31, np.arange(1000, 1000 + n), alpha)
    dist = stats.beta(alpha, 64 * alpha)
    worst = min((stats.kstest(nz[:, e], dist.cdf) for e in range(65)), key=lambda r: r.pvalue)
    assert worst.pvalue > 1e-3 / 65, (alpha, worst)
    # the whole table at once (columns are exchangeable): the mean and variance of the law
    a0 = 65 * alpha
    var = alpha * (a0 - alpha) / (a0 * a0 * (a0 + 1))
    assert abs(nz.var() / var - 1) < 0.05
    assert np.abs(nz.sum(1) - 1.0).max() < 1e-12


def _softmax_like_the_kernel(x32, lanes):
    """The fused tail's float32 softmax in numpy: max, expf(x - max), per-lane sums in index order, a shuffle-down
    tree over the lanes, one correctly rounded division (numpy's float32 exp stands in for expf)."""
    with np.errstate(over="ignore", invalid="ignore"):
        d = (x32 - x32.max()).astype(np.float32)
        e = np.exp(d).astype(np.float32)
    part = np.zeros(lanes, np.float32)
    for lane in range(lanes):
        for a in range(lane, 65, lanes):
            part[lane] = np.float32(part[lane] + e[a])
    o = lanes // 2
    while o:
        part[:lanes - o] = part[:lanes - o] + part[o:]
        o //= 2
    return (e / part[0]).astype(np.float32)


def test_fused_softmax_bound_holds_for_a_float32_model_of_the_kernel():
    """The per-prior bound of test_kernel_numerics_gpu.py, (26 + |x - max|) 2^-24 relative plus 3 x 2^-149, checked
    on a float32 model of the kernel's arithmetic over every row kind, root and lane width of that test.  A flat 2e-6
    relative bound leaves out the rounded subtraction x - max, which alone costs up to |x - max| 2^-24."""
    import torch
    import test_kernel_numerics_gpu as G
    rng = np.random.default_rng(0)
    for _ in range(40):
        for lanes in (8, 16, 32):
            for root in G.ROOT_ORDER:
                legal = G._mask(G._legal(*G.ROOTS[root]))
                for kind in range(8):
                    x = G._row(kind, rng, legal)
                    for xx in (x, torch.from_numpy(x).to(torch.bfloat16).float().numpy()):
                        p = _softmax_like_the_kernel(xx, lanes)
                        p64, d = G._softmax64(xx.astype(np.float64))
                        err = np.abs(p.astype(np.float64) - p64)
                        assert (err <= G._prior_tol(p64, d)).all(), (kind, lanes, root)
