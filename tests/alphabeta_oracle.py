"""CPU reference of oth_alphabeta -- TEST INFRASTRUCTURE ONLY.

ctypes front-end of ``tests/alphabeta_oracle.c`` (plain negamax and ascending-order alpha-beta on the CPU oracle's
boards and rules).  The library is compiled once per process into a temporary directory, never into the tree.
"""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="alphabeta-oracle-")
        try:
            path = os.path.join(tmp, "libalphabeta_oracle.so")
            # the flags of oracle/Makefile
            subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off",
                                   "-fno-fast-math", "-o", path, os.path.join(_HERE, "alphabeta_oracle.c"), "-lm"])
            L = C.CDLL(path)
        finally:
            shutil.rmtree(tmp)  # the loaded library stays mapped
        for fn in (L.orc_negamax, L.orc_alphabeta):
            fn.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_long)]
            fn.restype = C.c_int
        _lib = L
    return _lib


def _search(fn, state, player, depth, exact_empties):
    s = np.ascontiguousarray(np.asarray(state, dtype=np.int8).reshape(64))
    values = np.zeros(65, np.int32)
    nodes = C.c_long(0)
    best = fn(s.ctypes.data_as(C.c_void_p), int(player), int(depth), int(exact_empties),
              values.ctypes.data_as(C.c_void_p), C.byref(nodes))
    return values, best, nodes.value


def negamax(state, player, depth, exact_empties=0):
    """oth_alphabeta's search without pruning: (values int32[65] per root action, lowest best action or -1, nodes)."""
    return _search(lib().orc_negamax, state, player, depth, exact_empties)


def alphabeta(state, player, depth, exact_empties=0):
    """The same search as ``negamax`` with fail-hard alpha-beta in ascending action order."""
    return _search(lib().orc_alphabeta, state, player, depth, exact_empties)
