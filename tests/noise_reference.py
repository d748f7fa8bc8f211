"""float64 numpy restatement of the engine's Dirichlet root noise (``make_noise``, csrc/mcts_kernels.cu).

Entry ``e`` of the noise of game ``game_id`` at ply ``ply`` is a Marsaglia-Tsang gamma draw: attempt ``k`` (0..255) of
that entry reads the Philox4x32-10 block with key ``seed ^ 0x6e6f697365`` and counter ``(game_id, e, k | ply << 16)``
(csrc/philox.cuh); the first accepted attempt gives ``g = d v``, boosted by ``U^(1/alpha)`` when alpha < 1.  The 65
gammas are summed in index order and divided by that sum.  Every operation below is the kernel's, in its order; only
the libm calls (log, sqrt, cospi, pow) may differ from CUDA's by an ulp or two.
"""
import numpy as np

SALT_NOISE = 0x6E6F697365
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)
_LO = np.uint64(0xFFFFFFFF)


def philox4x32_10(seed, ctr_lo, h0, h1):
    """Vectorised Philox4x32-10 (csrc/philox.cuh): key ``seed`` (uint64), counter words (lo32(ctr_lo), hi32(ctr_lo),
    h0, h1).  Array arguments broadcast; returns four uint32 arrays (x, y, z, w)."""
    ctr_lo = np.asarray(ctr_lo, dtype=np.uint64)
    shape = np.broadcast_shapes(ctr_lo.shape, np.shape(h0), np.shape(h1))
    c0 = np.broadcast_to(ctr_lo & _LO, shape).astype(np.uint32)
    c1 = np.broadcast_to(ctr_lo >> np.uint64(32), shape).astype(np.uint32)
    c2 = np.broadcast_to(np.asarray(h0, dtype=np.uint32), shape).copy()
    c3 = np.broadcast_to(np.asarray(h1, dtype=np.uint32), shape).copy()
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    k0, k1 = np.uint32(seed & 0xFFFFFFFF), np.uint32(seed >> 32)
    with np.errstate(over="ignore"):
        for _ in range(10):
            p0 = _M0 * c0.astype(np.uint64)
            p1 = _M1 * c2.astype(np.uint64)
            n0 = (p1 >> np.uint64(32)).astype(np.uint32) ^ c1 ^ k0
            n2 = (p0 >> np.uint64(32)).astype(np.uint32) ^ c3 ^ k1
            c1 = (p1 & _LO).astype(np.uint32)
            c3 = (p0 & _LO).astype(np.uint32)
            c0, c2 = n0, n2
            k0 = k0 + _W0
            k1 = k1 + _W1
    return c0, c1, c2, c3


def cospi(t):
    """cos(pi t) for t in [0, 2) with exact argument reduction to [0, 1/4] (CUDA's cospi is within 2 ulp)."""
    t = np.where(t > 1.0, 2.0 - t, t)  # cos(pi (2 - t)) = cos(pi t); exact
    sign = np.where(t > 0.5, -1.0, 1.0)
    t = np.where(t > 0.5, 1.0 - t, t)  # cos(pi t) = -cos(pi (1 - t)); exact (Sterbenz)
    return sign * np.where(t > 0.25, np.sin(np.pi * (0.5 - t)), np.cos(np.pi * t))


def gammas(seed, game_ids, alpha, ply=0):
    """The unnormalised Marsaglia-Tsang draws g[len(game_ids), 65] of ``make_noise`` (float64)."""
    gid = np.asarray(game_ids, dtype=np.uint64).reshape(-1)
    alpha = float(alpha)
    a = alpha + 1.0 if alpha < 1.0 else alpha
    d = a - 1.0 / 3.0
    cc = 1.0 / np.sqrt(9.0 * d)
    key = int(seed) ^ SALT_NOISE
    G = np.repeat(gid, 65)
    E = np.tile(np.arange(65, dtype=np.uint32), len(gid))
    g = np.full(G.shape, d)  # the kernel's value if no attempt is accepted
    todo = np.arange(G.size)
    for k in range(256):
        if todo.size == 0:
            break
        x_, y_, z_, w_ = philox4x32_10(key, G[todo], E[todo], np.uint32(k | (int(ply) << 16)))
        u1 = (x_.astype(np.float64) + 1.0) * (1.0 / 4294967296.0)
        u2 = y_.astype(np.float64) * (1.0 / 4294967296.0)
        x = np.sqrt(-2.0 * np.log(u1)) * cospi(2.0 * u2)
        v = 1.0 + cc * x
        pos = v > 0.0
        v = np.where(pos, v, 1.0)
        v = v * v * v
        u = (z_.astype(np.float64) + 0.5) * (1.0 / 4294967296.0)
        acc = pos & (np.log(u) < 0.5 * x * x + d - d * v + d * np.log(v))
        gk = d * v
        if alpha < 1.0:
            gk = gk * np.power((w_.astype(np.float64) + 0.5) * (1.0 / 4294967296.0), 1.0 / alpha)
        g[todo[acc]] = gk[acc]
        todo = todo[~acc]
    return g.reshape(len(gid), 65)


def dirichlet_noise(seed, game_ids, alpha, ply=0):
    """Root noise [len(game_ids), 65] as ``make_noise`` writes it: gammas divided by their index-order sum."""
    g = gammas(seed, game_ids, alpha, ply)
    s = np.zeros(g.shape[0])
    for e in range(65):  # sequential, like the kernel's loop (numpy's sum() would be pairwise)
        s = s + g[:, e]
    return g / s[:, None]
