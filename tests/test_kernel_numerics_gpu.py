"""The floating-point quantities the oracle takes as given, against float64 references.

The parity suite replays every game from what the engine recorded: the priors / values the fused step kernel applied,
the root noise and the move uniforms.  This file checks how those records are computed:

* the fused network tail (``run_slot<..., FUSED>``): softmax and tanh of raw float32 / bf16 head outputs, at 8, 16 and
  32 lanes per slot, through strided views and the ``eval_map`` indirection, on rows chosen so that neighbouring slots
  of one warp differ wildly; and the masked, renormalised priors that enter the tree;
* the Dirichlet root noise (``make_noise``) against its float64 restatement (tests/noise_reference.py), entry by entry,
  and against the Dirichlet law;
* the network-boundary kernels ``oth_nn_stem_im2col_bf16`` and ``oth_nn_bias_add_relu_bf16``, bit for bit.

Observed error maxima are printed with the prefix ``numerics:`` (``pytest -s``).
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

U = 2.0 ** -24            # float32 unit roundoff
TINY = 2.0 ** -149        # smallest float32 subnormal
BF16_MAX = 3.3895313892515355e38
ROOTS = {  # (own, opp) of the side to move; bit i = square i
    "opening": (0x810000000, 0x1008000000),
    "mid": (0x40406800141000, 0x10101E080400),            # ply 12, 12 legal moves
    "single": (0x7E665F5D754D5B3F, 0x8198A0A28A92A4C0),   # exactly one legal move
    "pass": (0x9E9E8EB4AAD43830, 0x6061714B552BC7CF),     # no legal move, the opponent has one: action 64 only
}
ROOT_ORDER = ["opening", "mid", "single", "pass"]
VPRE = [0.0, -0.0, 1e-8, -1e-8, 0.5, -0.5, 9.0, -9.0, 20.0, -20.0, BF16_MAX, -BF16_MAX]


def _legal(own, opp):
    moves = 0
    for sq in range(64):
        if ((own | opp) >> sq) & 1:
            continue
        r, c = divmod(sq, 8)
        for dr, dc in ((-1, -1), (-1, 0), (-1, 1), (0, -1), (0, 1), (1, -1), (1, 0), (1, 1)):
            rr, cc, n = r + dr, c + dc, 0
            while 0 <= rr < 8 and 0 <= cc < 8 and (opp >> (rr * 8 + cc)) & 1:
                rr, cc, n = rr + dr, cc + dc, n + 1
            if n and 0 <= rr < 8 and 0 <= cc < 8 and (own >> (rr * 8 + cc)) & 1:
                moves |= 1 << sq
                break
    return moves


def _mask(moves):
    m = np.array([(moves >> a) & 1 for a in range(64)] + [moves == 0], dtype=bool)
    return m


def test_root_positions_are_what_they_claim():
    assert [a for a in range(64) if (_legal(*ROOTS["opening"]) >> a) & 1] == [19, 26, 37, 44]
    assert bin(_legal(*ROOTS["mid"])).count("1") >= 12
    assert bin(_legal(*ROOTS["single"])).count("1") == 1
    own, opp = ROOTS["pass"]
    assert _legal(own, opp) == 0 and _legal(opp, own) != 0


# --------------------------------------------------------------------------------------- A. fused network tail --
def _softmax64(x):
    """float64 softmax of the exact values the kernel read; also returns d = x - max (float64)."""
    mx = x.max()
    d = x - mx
    e = np.exp(d)
    return e / e.sum(), d


def _prior_tol(p64, d):
    """|kernel - p64| allowed for one prior (derivation in ``test_fused_tail_matches_a_float64_softmax_and_tanh``)."""
    ad = np.where(np.isfinite(d), np.abs(d), 0.0)
    return (26.0 + ad) * U * p64 + 3 * TINY


def _row(kind, rng, legal):
    """One row of 65 logits.  Kinds: 0 ordinary N(0, 3); 1 / 2 the same around +1000 / -1000; 3 all equal; 4 one
    logit 50 above the rest; 5 illegal actions at -inf; 6 legal logits 90-100 below an illegal maximum (subnormal
    priors, masked sum < 1e-12); 7 values near +-3.38e38 (x - max overflows to -inf) among ordinary ones."""
    if kind == 0:
        x = rng.normal(0, 3, 65)
    elif kind == 1:
        x = 1000 + rng.normal(0, 3, 65)
    elif kind == 2:
        x = -1000 + rng.normal(0, 3, 65)
    elif kind == 3:
        x = np.full(65, 7.25)
    elif kind == 4:
        x = rng.normal(0, 1, 65)
        x[rng.integers(65)] = x.max() + 50
    elif kind == 5:
        x = rng.normal(0, 3, 65)
        x[~legal] = -np.inf
    elif kind == 6:
        x = rng.uniform(-5, 0, 65)
        x[rng.choice(np.nonzero(~legal)[0])] = 0.0
        x[legal] = rng.uniform(-100, -90, legal.sum())
    else:
        x = rng.normal(0, 3, 65)
        big = rng.random(65) < 0.5
        x[big] = rng.choice([-1.0, 1.0], big.sum()) * rng.uniform(0.995, 1.0, big.sum()) * BF16_MAX
    return x.astype(np.float32)


def _layout(kind, R, dtype, dev):
    """(logits view [R,65], value view [R,1]) in one of the layouts the kernel must read; the unused columns hold NaN."""
    import torch
    nan = lambda *s: torch.full(s, float("nan"), dtype=dtype, device=dev)
    if kind == "c65":
        return nan(R, 65), nan(R, 1)
    if kind == "s128":
        b = nan(R, 128)
        return b[:, :65], b[:, 100:101]
    if kind == "s67":
        b = nan(R, 67)
        return b[:, :65], b[:, 66:67]
    return nan(R, 65), nan(R, 7)[:, 3:4]  # "vstride": the value pre-activation has a stride of its own


def _manual_external(n, lanes, sims=8, eps=0.0, alpha=0.3, seed=0, roots=None):
    """Manual-mode engine whose slots all wait for a network evaluation of their root."""
    import torch
    from alphazero_othello_b200 import _lib
    from alphazero_othello_b200.engine import MctsEngine
    args = {"c_puct": 2.0, "num_simulations": sims, "dirichlet_alpha": alpha, "dirichlet_epsilon": eps}
    e = MctsEngine(n, args, self_play=False, eval_kind=_lib.EVAL_EXTERNAL, lanes=lanes, seed=seed, max_inline_sims=1000)
    roots = roots or [ROOT_ORDER[s % 4] for s in range(n)]
    own = np.array([ROOTS[r][0] for r in roots], np.uint64).view(np.int64)
    opp = np.array([ROOTS[r][1] for r in roots], np.uint64).view(np.int64)
    e.set_roots(torch.from_numpy(own).cuda(), torch.from_numpy(opp).cuda(), torch.ones(n, dtype=torch.int8, device="cuda"))
    e.begin_search()
    if (e.ctl()["phase"] == _lib.PH_RUN).any():
        e.step()
    e.raise_on_error()
    assert (e.ctl()["phase"] == _lib.PH_WAIT_EVAL).all()
    return e, [_mask(_legal(*ROOTS[r])) for r in roots]


def _tree_rule32(p32, legal):
    """MCTS_model.py:346-349 in float32: priors *= mask; priors /= sum (numpy's pairwise sum) if sum > 1e-12."""
    m = np.where(legal, p32, p32 * np.float32(0.0))
    s = m.sum(dtype=np.float32)
    return (m / s if s > np.float32(1e-12) else m), s


@pytest.mark.parametrize("mapped", [False, True], ids=["direct", "eval_map"])
@pytest.mark.parametrize("layout", ["c65", "s128", "s67", "vstride"])
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("lanes", [8, 16, 32])
def test_fused_tail_matches_a_float64_softmax_and_tanh(lanes, dtype, layout, mapped):
    """Priors and values the fused step kernel records, against a float64 softmax / tanh of the values it read.

    Bound on a prior (u = 2^-24, d_i = x_i - max in float64):
    * fl(x_i - m) = d_i (1 + delta), |delta| <= u, so exp() of it is off by |d_i| u relatively; expf is within 2 ulp
      (4u).  Each exponential: (4 + |d_i|) u.
    * The sum S adds positive terms in a fixed order, at most 12 deep (9 terms per lane at 8 lanes, then 3 shuffle
      levels; 5 + 4 at 16, 3 + 5 at 32): 12u, plus the terms' own errors weighted by their shares w_j,
      sum_j w_j (4 + |d_j|) u <= (4 + ln 65) u, since sum_j w_j |d_j| is at most the entropy of w.  S: <= 21 u.
    * __fdiv_rn rounds once: u.
    So |p_i - p64_i| <= (26 + |d_i|) u p64_i, plus 3 x 2^-149 where the result or e_i is subnormal (expf within 2 ulp
    of 2^-149 there, the division rounds to half of it; the library is built without flush-to-zero).  For |d_i| <= 7.5
    this is the 2e-6 relative of a plain derivation that leaves out the rounded subtraction.
    The value: tanhf is within 2 float32 ulp of tanh.

    Rows change kind from slot to slot, so the slots sharing a warp (4 at 8 lanes, 2 at 16) see +-1000, -inf and
    +-3.38e38 next to ordinary rows.  With eval_map, rows are permuted, some are read by two slots and some slots get
    -1: those must stay waiting, untouched, and be served on a later launch.
    """
    import torch
    from alphazero_othello_b200 import _lib
    n = 64
    tdt = torch.float32 if dtype == "f32" else torch.bfloat16
    e, legal = _manual_external(n, lanes)
    rng = np.random.default_rng(1000 * lanes + 10 * len(layout) + mapped + (dtype == "bf16"))
    root_p32, root_x = {}, {}
    worst_p, worst_v = 0.0, 0.0
    skipped = set()
    for launch in range(3):
        pre = e.ctl()
        waiting = pre["phase"] == _lib.PH_WAIT_EVAL
        rows = np.stack([_row((s + s // 8 + launch) % 8, rng, legal[s]) for s in range(n)])
        vals = np.array([VPRE[(s + launch) % len(VPRE)] for s in range(n)], np.float32)
        L, V = _layout(layout, n, tdt, "cuda")
        emap = None
        if mapped:
            perm = rng.permutation(n)
            m = perm.copy()
            for t in range(4, n):
                if t % 7 == 3:
                    m[t] = m[t - 4]  # same root, read twice
            if launch != 1:
                m[np.arange(n) % 5 == (2 if launch == 0 else 4)] = -1
            L[torch.from_numpy(perm).cuda()] = torch.from_numpy(rows).cuda().to(tdt)
            V[torch.from_numpy(perm).cuda(), 0] = torch.from_numpy(vals).cuda().to(tdt)
            emap = torch.from_numpy(m.astype(np.int32)).cuda()
        else:
            m = np.arange(n)
            L.copy_(torch.from_numpy(rows).to(tdt))
            V[:, 0] = torch.from_numpy(vals).to(tdt)
        X = L.float().cpu().numpy().astype(np.float64)  # exactly what the kernel reads (bf16 -> float64 is exact)
        XV = V[:, 0].float().cpu().numpy().astype(np.float64)
        e.priors.fill_(float("nan"))
        e.values.fill_(float("nan"))
        e.step_fused(L, V, record=True, eval_map=emap)
        e.raise_on_error()
        post = e.ctl()
        pr, va = e.priors.cpu().numpy(), e.values.cpu().numpy()
        for s in np.nonzero(waiting)[0]:
            r = int(m[s])
            if r < 0:
                assert post["phase"][s] == _lib.PH_WAIT_EVAL and post["pending"][s] == pre["pending"][s], s
                assert np.isnan(pr[s]).all() and np.isnan(va[s]), s
                skipped.add(s)
                continue
            p64, d = _softmax64(X[r])
            err = np.abs(pr[s].astype(np.float64) - p64)
            assert (err <= _prior_tol(p64, d)).all(), (s, launch, np.nonzero(err > _prior_tol(p64, d))[0], X[r], pr[s])
            big = p64 >= np.finfo(np.float32).tiny
            if big.any():
                worst_p = max(worst_p, float((err[big] / p64[big]).max()))
            t64 = np.tanh(XV[r])
            ulp = abs(float(va[s]) - t64) / float(np.spacing(np.abs(np.float32(t64))))
            assert ulp <= 2.0, (s, XV[r], va[s], t64)
            worst_v = max(worst_v, ulp)
            if s not in root_p32:
                root_p32[s], root_x[s] = pr[s].copy(), X[r].copy()
    if mapped:
        assert skipped and all(s in root_p32 for s in skipped)  # the slots left out were served later
    assert len(root_p32) == n
    # the priors that entered the tree, two ways
    cp = e.root_stats()["child_prior"].cpu().numpy()
    worst_t = 0.0
    for s in range(n):
        rule, s32 = _tree_rule32(root_p32[s], legal[s])
        assert np.array_equal(cp[s], np.where(legal[s], rule, 0.0).astype(np.float64)), s
        p64, d = _softmax64(root_x[s])
        q = np.where(legal[s], p64, 0.0)
        S = q.sum()
        assert (S > 1e-12) == (s32 > np.float32(1e-12)), (s, S, s32)
        ad = np.where(np.isfinite(d), np.abs(d), 0.0)
        if S > 1e-12:
            q = q / S
            DL = float((q * ad).sum())
            tol = (2 * 26 + ad + DL + 12 + 1) * U * q + (3 * TINY / S + TINY)  # p_i, the masked sum (11 deep), /
        else:
            tol = _prior_tol(q, d)
        err = np.abs(cp[s] - q)
        assert (err <= tol).all(), (s, np.nonzero(err > tol)[0])
        big = q >= np.finfo(np.float32).tiny
        if big.any():
            worst_t = max(worst_t, float((err[big] / q[big]).max()))
    print(f"numerics: fused lanes={lanes} {dtype} {layout} map={mapped}: max rel prior err {worst_p:.3e}, "
          f"max tanh err {worst_v:.2f} ulp, max rel tree-prior err {worst_t:.3e}")


def test_noised_root_priors_follow_the_float64_mix():
    """With epsilon > 0 the root priors are float64: f64(f32(1 - eps) p) + eps noise, masked, divided by numpy's
    pairwise sum (MCTS_model.py:339-349), on the kernel's own priors and the recorded noise: within 1e-15 relative."""
    import torch
    n, eps = 32, 0.25
    e, legal = _manual_external(n, 8, eps=eps, alpha=0.3, seed=11)
    rng = np.random.default_rng(4)
    nz = e.noise.cpu().numpy().copy()
    rows = np.stack([_row((s + s // 8) % 8, rng, legal[s]) for s in range(n)])
    L = torch.from_numpy(rows).cuda().to(torch.bfloat16)
    V = torch.zeros(n, 1, dtype=torch.bfloat16, device="cuda")
    e.step_fused(L, V, record=True)
    e.raise_on_error()
    p32 = e.priors.cpu().numpy()
    cp = e.root_stats()["child_prior"].cpu().numpy()
    worst = 0.0
    for s in range(n):
        t = (np.float32(1.0 - eps) * np.where(legal[s], p32[s], np.float32(0.0))).astype(np.float64)
        v = t + eps * nz[s]
        v = np.where(legal[s], v, v * 0.0)
        S = v.sum()
        ref = v / S if S > 1e-12 else v
        ref = np.where(legal[s], ref, 0.0)
        err = np.abs(cp[s] - ref)
        assert (err <= 1e-15 * np.abs(ref)).all(), (s, cp[s] - ref)
        worst = max(worst, float((err / np.where(ref > 0, ref, 1.0)).max()))
    print(f"numerics: noised root mix: max rel err {worst:.3e}")


# ----------------------------------------------------------------------------------- B. Dirichlet root noise --
def _noise_engine(n, alpha, seed, lanes, base):
    from alphazero_othello_b200 import _lib
    from alphazero_othello_b200.engine import MctsEngine
    args = {"c_puct": 2.0, "num_simulations": 4, "dirichlet_alpha": alpha, "dirichlet_epsilon": 0.25}
    return MctsEngine(n, args, self_play=True, eval_kind=_lib.EVAL_STUB_H, lanes=lanes, seed=seed, game_id_base=base,
                      games_per_slot=1)


def _close_to_reference(got, ref):
    """Entry by entry within 1e-13 relative (CUDA's log / sqrt / cospi / pow against numpy's: a few ulp); entries
    that underflowed (alpha = 0.03) are compared at the subnormal scale."""
    err = np.abs(got - ref)
    ok = err <= 1e-13 * np.abs(ref) + 1e-300
    rel = float((err / np.where(ref > 0, ref, 1.0)).max())
    return ok, rel


@pytest.mark.parametrize("lanes", [8, 32])
@pytest.mark.parametrize("alpha", [0.03, 0.3, 1.0, 2.5, 10.0])
def test_root_noise_is_the_documented_stream(alpha, lanes):
    """e.noise of game G = game_id_base + slot at ply 0 is the restated make_noise draw for (seed, G, 0)."""
    import noise_reference as NR
    worst = 0.0
    for seed, base in ((0x5EED, 1000), (987654321, 2**32 + 7)):
        n = 96
        e = _noise_engine(n, alpha, seed, lanes, base)
        e.reset()
        got = e.noise.cpu().numpy()
        ref = NR.dirichlet_noise(seed, base + np.arange(n), alpha)
        ok, rel = _close_to_reference(got, ref)
        bad = np.argwhere(~ok)
        assert ok.all(), (seed, bad[:5], got[tuple(bad[0])], ref[tuple(bad[0])])
        worst = max(worst, rel)
    print(f"numerics: noise stream alpha={alpha} lanes={lanes}: max rel err {worst:.3e}")


@pytest.mark.parametrize("lanes", [8, 32])
def test_fresh_root_noise_at_a_later_ply_is_keyed_by_the_ply(lanes):
    """Manual mode: ``advance`` onto a child that was never expanded draws fresh noise for that root, keyed by its
    ply (counter word k | ply << 16); checked at plies 0, 1 and 2."""
    import torch
    import noise_reference as NR
    from alphazero_othello_b200 import _lib
    from alphazero_othello_b200.engine import MctsEngine
    n, seed, base, alpha = 40, 99, 500, 2.5 if lanes == 8 else 0.3
    args = {"c_puct": 2.0, "num_simulations": 1, "dirichlet_alpha": alpha, "dirichlet_epsilon": 0.25}
    e = MctsEngine(n, args, self_play=False, eval_kind=_lib.EVAL_STUB_H, lanes=lanes, seed=seed, game_id_base=base,
                   stub_salt=5, max_inline_sims=1000)
    own, opp = ROOTS["opening"]
    e.set_roots(torch.full((n,), own, dtype=torch.int64, device="cuda"), torch.full((n,), opp, dtype=torch.int64, device="cuda"),
                torch.ones(n, dtype=torch.int8, device="cuda"))
    gids = base + np.arange(n)
    for ply in range(3):
        assert (e.ctl()["ply"] == ply).all()
        ok, _ = _close_to_reference(e.noise.cpu().numpy(), NR.dirichlet_noise(seed, gids, alpha, ply))
        assert ok.all(), ply
        e.begin_search()
        for _ in range(64):
            e.step()
            if (e.ctl()["phase"] != _lib.PH_RUN).all():
                break
        e.raise_on_error()
        st = e.root_stats()
        counts, prior = st["counts"].cpu().numpy(), st["child_prior"].cpu().numpy()
        # a legal action whose child was never visited, hence never expanded
        act = np.array([int(np.nonzero((prior[s] > 0) & (counts[s] == 0))[0][s % 2 - 1]) for s in range(n)], np.int32)
        e.advance(torch.from_numpy(act).cuda())
        e.raise_on_error()
    assert (e.ctl()["ply"] == 3).all()
    ok, rel = _close_to_reference(e.noise.cpu().numpy(), NR.dirichlet_noise(seed, gids, alpha, 3))
    assert ok.all()
    assert not np.array_equal(NR.dirichlet_noise(seed, gids, alpha, 3), NR.dirichlet_noise(seed, gids, alpha, 0))


@pytest.mark.parametrize("alpha", [0.03, 0.3, 1.0, 2.5])
def test_root_noise_has_dirichlet_marginals_at_full_size(alpha):
    """16 384 slots (production C4 geometry): every column against Beta(alpha, 64 alpha) by Kolmogorov-Smirnov,
    Bonferroni-corrected over 65 columns (family-wise 1e-3).  At alpha = 0.03 entries may underflow to 0, but every
    row still sums to 1."""
    from scipy import stats
    n = 16384
    e = _noise_engine(n, alpha, 2718, None, 0)
    e.reset()
    nz = e.noise.cpu().numpy()
    assert np.isfinite(nz).all() and (nz >= 0).all()
    assert np.abs(nz.sum(1) - 1.0).max() < 1e-12
    dist = stats.beta(alpha, 64 * alpha)
    res = [stats.kstest(nz[:, c], dist.cdf) for c in range(65)]
    worst = min(res, key=lambda r: r.pvalue)
    print(f"numerics: noise law alpha={alpha}: max KS statistic {max(r.statistic for r in res):.4f}, "
          f"min p {worst.pvalue:.3e}, zeros {int((nz == 0).sum())}")
    assert worst.pvalue > 1e-3 / 65, worst


# ------------------------------------------------------------------------------ C. network-boundary kernels --
def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# grid_for caps a launch at 8 blocks of 256 threads per SM: beyond 8 x 256 x SMs threads the grid-stride loops wrap
def _wrap_threads():
    import torch
    return 8 * 256 * torch.cuda.get_device_properties(0).multi_processor_count


def _im2col_ref(planes):
    P = np.pad(planes.reshape(-1, 8, 8), ((0, 0), (1, 1), (1, 1)))
    out = np.zeros((planes.shape[0], 8, 8, 16), np.float32)
    for dy in range(3):
        for dx in range(3):
            out[..., dy * 3 + dx] = P[:, dy:dy + 8, dx:dx + 8]
    return out.reshape(-1, 64, 16)


@pytest.mark.parametrize("n", [1, 3, 255, 256, 257, 4097, "wrap"])
def test_stem_im2col_matches_numpy_bit_for_bit(n):
    """Taps in (dy, dx) order, zero padding, columns 9..15 zero; float32 -> bf16 rounded to nearest even, as torch's
    ``.to(torch.bfloat16)``.  Planes are arbitrary float32, including exact bf16 ties and values that round to inf."""
    import torch
    from alphazero_othello_b200 import _lib
    if n == "wrap":
        n = _wrap_threads() // 64 * 2 + 37
    rng = np.random.default_rng(n)
    planes = (rng.normal(0, 1, (n, 64)) * np.exp2(rng.integers(-20, 20, (n, 64)))).astype(np.float32)
    ties = np.array([1 + 2.0 ** -8, 1 + 3 * 2.0 ** -8, -(1 + 2.0 ** -8), 3.4e38, -3.4e38, -0.0, 1e-40], np.float32)
    planes.reshape(-1)[rng.choice(planes.size, min(planes.size, 64), replace=False)] = rng.choice(ties, min(planes.size, 64))
    x = torch.from_numpy(planes).cuda()
    cols = torch.full((n, 64, 16), 12345.0, dtype=torch.bfloat16, device="cuda")  # garbage: every column is written
    _lib.check(_lib.lib().oth_nn_stem_im2col_bf16(x.data_ptr(), cols.data_ptr(), n, _stream()))
    torch.cuda.synchronize()
    ref = torch.from_numpy(_im2col_ref(planes)).to(torch.bfloat16)
    assert torch.equal(cols.cpu().view(torch.int16), ref.view(torch.int16))


def test_stem_im2col_rejects_bad_arguments():
    import torch
    from alphazero_othello_b200 import _lib
    L = _lib.lib()
    x = torch.zeros(4, 64, device="cuda")
    cols = torch.zeros(4 * 64 * 16 + 8, dtype=torch.bfloat16, device="cuda")
    assert L.oth_nn_stem_im2col_bf16(x.data_ptr(), cols.data_ptr() + 2, 1, _stream()) == _lib.OTH_E_ARG
    assert L.oth_nn_stem_im2col_bf16(x.data_ptr(), cols.data_ptr() + 8, 1, _stream()) == _lib.OTH_E_ARG
    assert L.oth_nn_stem_im2col_bf16(x.data_ptr(), cols.data_ptr(), -1, _stream()) == _lib.OTH_E_ARG
    assert L.oth_nn_stem_im2col_bf16(x.data_ptr(), cols.data_ptr(), 0, _stream()) == _lib.OTH_OK
    torch.cuda.synchronize()
    assert not cols.any()


def _bias_add_relu(x, r, b):
    from alphazero_othello_b200 import _lib
    return _lib.lib().oth_nn_bias_add_relu_bf16(x.data_ptr(), r.data_ptr(), b.data_ptr(), x.numel(), x.size(-1), _stream())


def _bias_add_relu_ref(x, r, b):
    """bf16(relu((x + b) + r)) with the sum in float32, on the CPU."""
    import torch
    return torch.relu((x.float().cpu() + b.float().cpu()) + r.float().cpu()).to(torch.bfloat16)


@pytest.mark.parametrize("C", [8, 24, 64, 128, 256])
def test_bias_add_relu_matches_float32_bit_for_bit(C):
    import torch
    from alphazero_othello_b200 import _lib
    g = torch.Generator().manual_seed(C)
    for rows in (1, 7, 193, _wrap_threads() * 8 * 2 // C + 5):
        x = (torch.randn(rows, C, generator=g) * 4).to(torch.bfloat16).cuda()
        r = (torch.randn(rows, C, generator=g) * 4).to(torch.bfloat16).cuda()
        b = (torch.randn(C, generator=g) * 4).to(torch.bfloat16).cuda()
        ref = _bias_add_relu_ref(x, r, b)
        assert _bias_add_relu(x, r, b) == _lib.OTH_OK
        torch.cuda.synchronize()
        assert torch.equal(x.cpu().view(torch.int16), ref.view(torch.int16)), (C, rows)


def test_bias_add_relu_keeps_non_finite_values_like_torch_relu():
    """+inf stays +inf, -inf becomes 0 and NaN stays NaN, as torch.relu of the float32 sum: a NaN activation in the
    trunk must reach the network's outputs, where the engine's non-finite guard stops the slot."""
    import torch
    from alphazero_othello_b200 import _lib
    inf, nan = float("inf"), float("nan")
    xs = [inf, -inf, nan, 1.0, -1.0, 3e38, -3e38, inf, nan, 0.0, 2.0, -2.0, inf, -inf, 5.0, 0.5]
    rs = [0.0, 0.0, 0.0, nan, inf, 3e38, -3e38, -inf, 1.0, -inf, nan, 0.0, 1.0, 1.0, -inf, inf]
    x = torch.tensor(xs * 4, dtype=torch.float32).view(8, 8).to(torch.bfloat16)
    r = torch.tensor(rs * 4, dtype=torch.float32).view(8, 8).to(torch.bfloat16)
    b = torch.tensor([0.0, 1.0, -1.0, nan, inf, -inf, 2.0, 0.25], dtype=torch.float32).to(torch.bfloat16)
    ref = _bias_add_relu_ref(x, r, b)
    xg = x.cuda()
    assert _bias_add_relu(xg, r.cuda(), b.cuda()) == _lib.OTH_OK
    got = xg.cpu()
    isn = torch.isnan(ref)
    assert isn.any() and torch.equal(torch.isnan(got), isn)
    assert torch.equal(got.view(torch.int16)[~isn], ref.view(torch.int16)[~isn])
    assert torch.isinf(ref).any()


def test_bias_add_relu_rejects_bad_arguments():
    import torch
    from alphazero_othello_b200 import _lib
    L = _lib.lib()
    x = torch.zeros(64 + 8, dtype=torch.bfloat16, device="cuda")
    r = torch.zeros(64 + 8, dtype=torch.bfloat16, device="cuda")
    b = torch.zeros(8 + 8, dtype=torch.bfloat16, device="cuda")
    f = lambda xp, rp, bp, n, c: L.oth_nn_bias_add_relu_bf16(xp, rp, bp, n, c, _stream())
    X, R, B = x.data_ptr(), r.data_ptr(), b.data_ptr()
    assert f(X, R, B, 64, 8) == _lib.OTH_OK
    assert f(X, R, B, 60, 8) == _lib.OTH_E_ARG      # n % 8
    assert f(X, R, B, 48, 12) == _lib.OTH_E_ARG     # C % 8
    assert f(X, R, B, 64, 0) == _lib.OTH_E_ARG
    assert f(X, R, B, -8, 8) == _lib.OTH_E_ARG
    for dx, dr, db in ((2, 0, 0), (0, 8, 0), (0, 0, 4)):  # 16-byte vector loads: every pointer must be aligned
        assert f(X + dx, R + dr, B + db, 56, 8) == _lib.OTH_E_ARG
    assert f(X, R, B, 0, 8) == _lib.OTH_OK
    torch.cuda.synchronize()
