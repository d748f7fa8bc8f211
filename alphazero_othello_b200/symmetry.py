"""Leaf symmetry at the network boundary (csrc/symmetry_kernels.cu, include/othello_b200.h).

Othello's value and move probabilities are the same in all eight orientations of the board (D4), up to relabelling
the squares; a network only learns that approximately.  The consumers of the search can therefore show the network
each leaf differently (keyword ``leaf_symmetry``):

* ``None`` (default): the leaf as the search wrote it -- no extra launch, no extra buffer;
* ``"random"``: the leaf in one orientation T_s, s = 0..7 drawn by ``oth_nn_leaf_symmetry`` from (seed, position) alone,
  and the policy logits mapped back (``oth_nn_unsymmetrise_logits``) before the softmax;
* ``"mean"``: the leaf in all eight orientations, priors and value averaged over them (``oth_nn_symmetry_mean``).  It
  costs eight network rows per leaf, so self-play does not offer it.

Every function takes CUDA tensors, launches on the current stream of their device and never synchronises, so the
calls can be captured in CUDA graphs.
"""
import ctypes as C

import torch

from . import _lib

MODES = ("random", "mean")


def check_mode(mode, supported=MODES):
    """``mode`` if it is None or one of ``supported``; otherwise ValueError (before any device work)."""
    if mode is None:
        return None
    if not isinstance(mode, str) or mode not in MODES:
        raise ValueError(f"leaf_symmetry must be None or one of {MODES}, got {mode!r}")
    if mode not in supported:
        raise ValueError(f"leaf_symmetry={mode!r} is not supported here (supported: None, {', '.join(supported)})")
    return mode


def _stream(t):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _rows(planes):
    assert planes.dtype == torch.float32 and planes.is_contiguous() and planes.numel() % 64 == 0
    return planes.numel() // 64


def leaf_symmetry(planes, seed, out_planes, out_sym):
    """out_planes = T_s(planes) row by row and out_sym uint8 [n] = s, for float32 planes [n,1,8,8] (or [n,64])."""
    n = _rows(planes)
    assert out_planes.shape == planes.shape and out_planes.dtype == torch.float32 and out_planes.is_contiguous()
    assert out_sym.dtype == torch.uint8 and out_sym.numel() == n
    with torch.cuda.device(planes.device):
        _lib.check(_lib.lib().oth_nn_leaf_symmetry(planes.data_ptr(), n, int(seed) & (2**64 - 1), out_planes.data_ptr(),
                                                   out_sym.data_ptr(), _stream(planes)), "oth_nn_leaf_symmetry")


def unsymmetrise_logits(logits, sym):
    """In place on the 64 square entries of each row of ``logits`` [n, >=65] (float32 or bfloat16, unit column
    stride): T_sym[i] of row i afterwards is the row the network returned.  Entry 64 (pass) is left alone."""
    assert logits.dtype in (torch.float32, torch.bfloat16) and logits.dim() == 2 and logits.stride(1) == 1
    assert sym.dtype == torch.uint8 and sym.numel() == logits.size(0)
    with torch.cuda.device(logits.device):
        _lib.check(_lib.lib().oth_nn_unsymmetrise_logits(logits.data_ptr(), logits.stride(0),
                                                         1 if logits.dtype == torch.bfloat16 else 0, sym.data_ptr(),
                                                         logits.size(0), _stream(logits)), "oth_nn_unsymmetrise_logits")


def images(planes, out):
    """out [8n,1,8,8] (float32): row 8i+j = T_j(planes[i])."""
    n = _rows(planes)
    assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == 8 * 64 * n
    with torch.cuda.device(planes.device):
        _lib.check(_lib.lib().oth_nn_symmetry_images(planes.data_ptr(), n, out.data_ptr(), _stream(planes)),
                   "oth_nn_symmetry_images")


def mean(logits, values, priors_out, values_out):
    """priors_out [n,65] / values_out [n] from the network's outputs on the 8n images of ``images``: logits float32
    [8n, >=65] (unit column stride), values float32 [8n] or [8n,1] (tanh'd)."""
    n = priors_out.size(0)
    assert logits.dtype == torch.float32 and logits.dim() == 2 and logits.stride(1) == 1 and logits.size(0) == 8 * n
    assert values.dtype == torch.float32 and values.size(0) == 8 * n
    assert priors_out.dtype == values_out.dtype == torch.float32 and priors_out.is_contiguous() and values_out.numel() == n
    assert priors_out.shape == (n, 65) and values_out.is_contiguous()
    with torch.cuda.device(logits.device):
        _lib.check(_lib.lib().oth_nn_symmetry_mean(logits.data_ptr(), logits.stride(0), values.data_ptr(), values.stride(0),
                                                   n, priors_out.data_ptr(), values_out.data_ptr(), _stream(logits)),
                   "oth_nn_symmetry_mean")
