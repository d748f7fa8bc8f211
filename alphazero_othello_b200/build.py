"""Compile libothello_b200.so in-tree with nvcc for sm_100a (B200).

    python -m alphazero_othello_b200.build        # or __graft_entry__.build()

No torch extension machinery: the library is a plain C-ABI shared object
(include/othello_b200.h) that Python binds with ctypes.
"""
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(HERE, "..", "include")
LIB = os.path.join(HERE, "libothello_b200.so")
LIB_DEBUG = os.path.join(HERE, "libothello_b200_debug.so")  # -DOTH_DEBUG: arena index assertions (OTH_B200_DEBUG=1 loads it)
SOURCES = ["env_kernels.cu", "mcts_kernels.cu", "replay_kernels.cu", "dedup_kernels.cu", "alphabeta_kernels.cu",
           "endgame_kernels.cu", "symmetry_kernels.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--fmad=false",            # numpy rounds every float op: no FMA contraction anywhere
    "-Xcompiler", "-fPIC", "-shared",
    "-Xptxas", "-v",
]
LINK_FLAGS = ["-ldl"]


def _nvcc():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found: libothello_b200 cannot be built (there is no CPU fallback)")


def _inputs_digest(debug):
    """sha256 of what the library is compiled from: the flags and every file under csrc/ and include/."""
    h = hashlib.sha256(repr((NVCC_FLAGS, LINK_FLAGS, debug)).encode())
    for d in (CSRC, INCLUDE):
        for name in sorted(os.listdir(d)):
            with open(os.path.join(d, name), "rb") as f:
                h.update(name.encode() + b"\0" + f.read())
    return h.hexdigest()


def needs_build(debug=False):
    """Whether the in-tree library is missing or was built from other sources or flags.  Judged by content, not
    timestamps, so that a copy of a built tree still loads what build() left there."""
    lib = LIB_DEBUG if debug else LIB
    try:
        with open(lib + ".inputs.sha256") as f:
            return f.read() != _inputs_digest(debug)
    except OSError:
        return True


def build(force=False, verbose=False, debug=False, out_dir=HERE):
    """Compile the library into ``out_dir`` (the package directory unless a caller must not write there) and record the
    digest of its inputs next to it.  In the package directory an up-to-date library is kept unless ``force``."""
    lib = os.path.join(out_dir, os.path.basename(LIB_DEBUG if debug else LIB))
    if not force and out_dir == HERE and not needs_build(debug):
        return lib
    digest = _inputs_digest(debug)
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    cmd = [_nvcc()] + NVCC_FLAGS + (["-DOTH_DEBUG"] if debug else []) + ["-o", lib] + srcs + LINK_FLAGS
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    log = os.path.join(out_dir, "build_debug.log" if debug else "build.log")
    with open(log, "w") as f:
        f.write(" ".join(cmd) + "\n" + p.stdout)
    if verbose or p.returncode != 0:
        sys.stderr.write(p.stdout)
    if p.returncode != 0:
        raise RuntimeError(f"nvcc failed ({p.returncode}); see {log}")
    with open(lib + ".inputs.sha256", "w") as f:
        f.write(digest)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True, debug="--debug" in sys.argv))
