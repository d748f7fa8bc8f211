"""Exact win/draw/loss of endgame positions on the GPU (oth_solve_wld, csrc/endgame_kernels.cu), and the relabelling of
self-play value targets with it.

A self-play value target is a lambda-return: it mixes the network's root values with the outcome of the game as it was
played, and in the last plies that outcome is mostly the noise of sampled moves and a weak network's misplays.  A
position with few enough empty squares has a known result, and ``relabel`` replaces those targets with it.  The search
semantics are documented in include/othello_b200.h.
"""
import torch

from . import _lib

MAX_EMPTIES, UNSOLVED = _lib.SOLVE_MAX_EMPTIES, _lib.WLD_UNSOLVED


def _check_max_empties(max_empties):
    if not 0 <= int(max_empties) <= MAX_EMPTIES:
        raise ValueError(f"max_empties must be in 0..{MAX_EMPTIES}, got {max_empties}")
    return int(max_empties)


def solve_wld(own, opp, max_empties=MAX_EMPTIES):
    """Solve n positions (``own`` to move) on their device.  own / opp: int64 or uint64 bitboard tensors [n] on a CUDA
    device.  Returns (wld int8 [n], nodes int64 [n]): +1 / 0 / -1 for the side to move under perfect play, ``UNSOLVED``
    (and 0 nodes) for positions with more than ``max_empties`` empty squares, and the positions each search visited."""
    if own.shape != opp.shape or own.dim() != 1 or own.device != opp.device or own.device.type != "cuda":
        raise ValueError("own / opp: two 1-D bitboard tensors of the same length on one CUDA device")
    if own.dtype not in (torch.int64, torch.uint64) or opp.dtype != own.dtype:
        raise ValueError("own / opp: int64 or uint64 bitboards")
    max_empties = _check_max_empties(max_empties)
    own, opp = own.contiguous(), opp.contiguous()
    n = own.numel()
    wld = torch.empty(n, dtype=torch.int8, device=own.device)
    nodes = torch.empty(n, dtype=torch.int64, device=own.device)
    with torch.cuda.device(own.device):
        stream = torch.cuda.current_stream(own.device).cuda_stream
        _lib.check(_lib.lib().oth_solve_wld(own.data_ptr(), opp.data_ptr(), n, max_empties, wld.data_ptr(),
                                            nodes.data_ptr(), stream), "oth_solve_wld")
    return wld, nodes


def relabel(out, max_empties, device=None):
    """A drained self-play output (``MctsEngine.drain()`` or ``collect_self_play_games(..., return_raw=True)``) with the
    value target of every position that has at most ``max_empties`` empty squares replaced by its solved result,
    ``float(wld)`` from the mover's side, the side the lambda-return it replaces is from.

    Returns a new dict: ``values`` relabelled, ``solved`` (bool [n]) marking the replaced rows, every other entry the
    caller's tensor.  Unsolved rows keep their values bit for bit, and every tensor stays on the device it came from.
    The search runs on ``device`` (default: the device of ``out["boards"]`` when that is a CUDA device, else the
    current one).  ``max_empties = 0`` solves nothing: self-play rows are never terminal, so none has 0 empties."""
    max_empties = _check_max_empties(max_empties)
    boards, values = out["boards"], out["values"]
    res = dict(out)
    if max_empties == 0:
        res["solved"] = torch.zeros(values.shape, dtype=torch.bool, device=values.device)
        return res
    if device is None:
        device = boards.device if boards.device.type == "cuda" else torch.device("cuda", torch.cuda.current_device())
    b = boards.to(device)
    wld, _ = solve_wld(b[:, 0], b[:, 1], max_empties)
    solved = (wld != UNSOLVED).to(values.device)
    res["values"] = torch.where(solved, wld.to(device=values.device, dtype=values.dtype), values)
    res["solved"] = solved
    return res
