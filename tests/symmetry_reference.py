"""numpy restatement of the leaf-symmetry contract (include/othello_b200.h, "network boundary"; csrc/symmetry_kernels.cu).

* ``sym_ids``: s = Philox4x32-10(seed ^ OTH_SYM_SALT; counter (own, lo32(opp), hi32(opp))).x & 7 (tests/noise_reference.py
  restates the generator);
* ``transform``: T_s, np.rot90 (s & 3) times then np.fliplr if s >> 2 -- oth_symmetry's mapping -- on the 64 squares;
* ``unsymmetrise``: the inverse on the 64 square entries of a row; entries from 64 on are kept;
* ``mean``: float64 (1/8) sum_j unsym_j(softmax(logits_j)) and the mean value.
"""
import numpy as np

from noise_reference import philox4x32_10

SYM_SALT = 0x73796D6D65747279
_W = np.uint64(1) << np.arange(64, dtype=np.uint64)


def bitboards(planes):
    """(own, opp) uint64 of float planes [n,64]: the +1 and the -1 squares."""
    p = np.asarray(planes).reshape(-1, 64)
    return ((p == 1) * _W).sum(1, dtype=np.uint64), ((p == -1) * _W).sum(1, dtype=np.uint64)


def sym_ids(seed, own, opp):
    own, opp = np.asarray(own, np.uint64), np.asarray(opp, np.uint64)
    lo = (opp & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    hi = (opp >> np.uint64(32)).astype(np.uint32)
    x, _, _, _ = philox4x32_10((int(seed) & (2**64 - 1)) ^ SYM_SALT, own, lo, hi)
    return (x & np.uint32(7)).astype(np.uint8)


def plane_ids(seed, planes):
    return sym_ids(seed, *bitboards(planes))


def src_squares(s):
    """src[e]: T_s(x)[e] = x[src[e]]."""
    idx = np.arange(64).reshape(8, 8)
    return np.fliplr(np.rot90(idx, s & 3)).reshape(64) if s >> 2 else np.rot90(idx, s & 3).reshape(64)


def transform(rows, s):
    """T_s of the 64 square entries of each row of ``rows`` [n, >=64] (entries from 64 on are kept)."""
    rows = np.array(rows, copy=True)
    rows[:, :64] = rows[:, src_squares(s)]
    return rows


def unsymmetrise(rows, s):
    """u with transform(u, s) == rows."""
    out = np.array(rows, copy=True)
    out[:, src_squares(s)] = rows[:, :64]
    return out


def softmax64(x):
    x = np.asarray(x, np.float64)
    e = np.exp(x - x.max(-1, keepdims=True))
    return e / e.sum(-1, keepdims=True)


def mean(logits, values):
    """logits [8n, 65], values [8n] (rows 8i+j = image j of leaf i) -> float64 priors [n,65], values [n]."""
    n = logits.shape[0] // 8
    p = softmax64(logits[:, :65]).reshape(n, 8, 65)
    pri = sum(unsymmetrise(p[:, j], j) for j in range(8)) / 8
    return pri, np.asarray(values, np.float64).reshape(n, 8).mean(1)
