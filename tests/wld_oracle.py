"""CPU reference of oth_solve_wld -- TEST INFRASTRUCTURE ONLY.

ctypes front-end of ``tests/wld_oracle.c`` (the oracle's ascending-order alpha-beta to the end of the game with the
window (-1, 1)).  The library is compiled once per process into a temporary directory, never into the tree.
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
        tmp = tempfile.mkdtemp(prefix="wld-oracle-")
        try:
            path = os.path.join(tmp, "libwld_oracle.so")
            # the flags of oracle/Makefile
            subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off",
                                   "-fno-fast-math", "-o", path, os.path.join(_HERE, "wld_oracle.c"), "-lm"])
            L = C.CDLL(path)
        finally:
            shutil.rmtree(tmp)  # the loaded library stays mapped
        L.orc_wld.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_long)]
        L.orc_wld.restype = C.c_int
        _lib = L
    return _lib


def wld(state, player):
    """(+1 / 0 / -1 for ``player`` to move under perfect play, positions visited)."""
    s = np.ascontiguousarray(np.asarray(state, dtype=np.int8).reshape(64))
    nodes = C.c_long(0)
    v = lib().orc_wld(s.ctypes.data_as(C.c_void_p), int(player), C.byref(nodes))
    return v, nodes.value
