"""A fixed-depth alpha-beta Othello player on the GPU (oth_alphabeta, csrc/alphabeta_kernels.cu).

Network-vs-network matches only say which of two networks is stronger.  ``AlphaBetaPlayer`` is a fixed yardstick: the
arena (``eval.play_matches_batched``, ``eval.evaluate_vs_alphabeta``) accepts it wherever it accepts a network, and
searches every pending position of a batch in one launch.  The search semantics are documented in
include/othello_b200.h.
"""
import numpy as np
import torch

from . import _lib

NONE, WIN_SCALE, MAX_DEPTH, MAX_EXACT = _lib.AB_NONE, _lib.AB_WIN_SCALE, _lib.AB_MAX_DEPTH, _lib.AB_MAX_EXACT


def search(own, opp, depth, exact_empties=0):
    """Search n positions (``own`` to move) on their device.  own / opp: int64 or uint64 bitboard tensors [n] on a
    CUDA device.  Returns (values int32 [n,65], best int32 [n], nodes int64 [n,65]): the negamax value of every legal
    root action from the mover's side (``NONE`` elsewhere), the lowest best action (-1 at a terminal root), and the
    positions visited below each action."""
    if own.shape != opp.shape or own.dim() != 1 or own.device != opp.device or own.device.type != "cuda":
        raise ValueError("own / opp: two 1-D bitboard tensors of the same length on one CUDA device")
    if own.dtype not in (torch.int64, torch.uint64) or opp.dtype != own.dtype:
        raise ValueError("own / opp: int64 or uint64 bitboards")
    own, opp = own.contiguous(), opp.contiguous()
    n = own.numel()
    values = torch.empty((n, 65), dtype=torch.int32, device=own.device)
    best = torch.empty(n, dtype=torch.int32, device=own.device)
    nodes = torch.empty((n, 65), dtype=torch.int64, device=own.device)
    with torch.cuda.device(own.device):
        stream = torch.cuda.current_stream(own.device).cuda_stream
        _lib.check(_lib.lib().oth_alphabeta(own.data_ptr(), opp.data_ptr(), n, int(depth), int(exact_empties),
                                            values.data_ptr(), best.data_ptr(), nodes.data_ptr(), stream), "oth_alphabeta")
    return values, best, nodes


def tie_pick(cands, u):
    """The arena's pick among ``cands`` (ascending) with one logged uniform u: np.random.choice(best_actions)."""
    return cands[min(int(u * len(cands)), len(cands) - 1)]


def pick(values, margin, u):
    """The move an AlphaBetaPlayer makes from one row of root values: uniform (by u) among the root actions whose value
    is >= best - margin, in ascending action order."""
    values = np.asarray(values)
    legal = values != NONE
    if not legal.any():
        raise ValueError("no legal root action (terminal position)")
    best = values[legal].max()
    return int(tie_pick(np.nonzero(legal & (values >= best - int(margin)))[0], u))


class AlphaBetaPlayer:
    """Arena opponent: a ``depth``-ply alpha-beta search, perfect play from ``exact_empties`` empty squares on, and a
    pick among the moves within ``margin`` of the best (margin 0: exact ties only; margin > 0: varied games)."""

    def __init__(self, depth=4, exact_empties=10, margin=0):
        if not 1 <= int(depth) <= MAX_DEPTH or not 0 <= int(exact_empties) <= MAX_EXACT or int(margin) < 0:
            raise ValueError(f"depth 1..{MAX_DEPTH}, exact_empties 0..{MAX_EXACT}, margin >= 0")
        self.depth, self.exact_empties, self.margin = int(depth), int(exact_empties), int(margin)

    def __repr__(self):
        return f"AlphaBetaPlayer(depth={self.depth}, exact_empties={self.exact_empties}, margin={self.margin})"
