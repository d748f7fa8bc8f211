"""ctypes binding of libothello_b200.so (C ABI: include/othello_b200.h).

There is NO CPU fallback: if the CUDA library cannot be loaded (or built with
nvcc), importing the compute paths raises.
"""
import ctypes as C
import os
import shutil
import tempfile

from . import build as _build

ABI_VERSION = 2
OTH_NUM_ACTIONS = 65
OTH_PASS = 64
OTH_MAX_PLIES = 128
OTH_MAX_CHILDREN = 40

OTH_OK, OTH_E_CUDA, OTH_E_ARG, OTH_E_ILLEGAL, OTH_E_NO_DEVICE = 0, -1, -2, -3, -4
F_ILLEGAL, F_TERMINAL, F_WIN, F_LOSS, F_MUST_PASS = 1, 2, 4, 8, 16
AB_NONE, AB_WIN_SCALE, AB_MAX_DEPTH, AB_MAX_EXACT = -2**31, 10000, 7, 12
SOLVE_MAX_EMPTIES, WLD_UNSOLVED = 14, -128

EVAL_EXTERNAL, EVAL_STUB_A, EVAL_STUB_B, EVAL_STUB_H, EVAL_ROLLOUT = 0, 1, 2, 3, 4
PH_RUN, PH_WAIT_EVAL, PH_IDLE, PH_DONE, PH_ERROR, PH_MOVE = 0, 1, 2, 3, 4, 5
ERR_NAMES = {1: "node arena overflow", 2: "path overflow", 4: "output ring overflow", 8: "ply overflow",
             16: "action has no child (KeyError)", 32: "non-finite prior or value from the evaluator",
             64: "debug assertion (arena index out of range)"}

(BUF_NODES, BUF_BOARDS, BUF_CTL, BUF_PATH, BUF_ROOT_PRIOR64, BUF_NOISE, BUF_U_MOVE, BUF_U_TIE, BUF_TRAJ_BOARD,
 BUF_TRAJ_PI, BUF_TRAJ_ROOTV, BUF_TRAJ_META, BUF_OUT_BOARD, BUF_OUT_PI, BUF_OUT_VALUE, BUF_OUT_META, BUF_OUT_GAMES,
 BUF_COUNTERS, BUF_SLOT_COUNTERS, BUF_HOT, BUF_MOVE_FLAGS, BUF_MOVE_LIST, BUF_COUNT) = range(23)

(CNT_SIMS, CNT_EVALS, CNT_TERMINAL, CNT_GAMES, CNT_POSITIONS, CNT_OUT_GAMES, CNT_MOVES, CNT_ERRORS, CNT_MAX_TOP,
 CNT_MAX_DEPTH, CNT_NODES, CNT_COPIED, CNT_WAITING, CNT_ACTIVE, CNT_LEVELS, CNT_CHILDREN) = range(16)
CNT_NAMES = ["sims", "evals", "terminal_sims", "games", "positions", "out_games", "moves", "errors", "max_top",
             "max_depth", "nodes", "copied", "waiting", "active", "levels", "children"]


class MctsConfig(C.Structure):
    _fields_ = [
        ("n_slots", C.c_int32), ("node_cap", C.c_int32), ("path_cap", C.c_int32), ("num_simulations", C.c_int32),
        ("num_exploratory_moves", C.c_int32), ("eval_kind", C.c_int32), ("self_play", C.c_int32),
        ("games_per_slot", C.c_int32), ("max_inline_sims", C.c_int32), ("inject_random", C.c_int32),
        ("lanes", C.c_int32), ("hot_path", C.c_int32), ("split_stub", C.c_int32), ("move_launch", C.c_int32),
        ("reserved0", C.c_int32),
        ("out_pos_cap", C.c_int64), ("out_game_cap", C.c_int64),
        ("c_puct", C.c_double), ("dirichlet_alpha", C.c_double), ("dirichlet_epsilon", C.c_double),
        ("temperature", C.c_double), ("lambda_", C.c_double),
        ("seed", C.c_uint64), ("game_id_base", C.c_uint64), ("game_id_stride", C.c_uint64), ("stub_salt", C.c_uint64),
    ]


class MctsCtl(C.Structure):
    _fields_ = [
        ("phase", C.c_int32), ("root", C.c_int32), ("top", C.c_int32), ("arena", C.c_int32), ("ply", C.c_int32),
        ("sims_done", C.c_int32), ("pending", C.c_int32), ("path_len", C.c_int32), ("flags", C.c_int32),
        ("player", C.c_int32), ("games_left", C.c_int32), ("error", C.c_int32), ("game_id", C.c_int64),
        ("reserved", C.c_int64),
    ]


assert C.sizeof(MctsCtl) == 64


class MctsBuffers(C.Structure):
    _fields_ = [("buf", C.c_void_p * BUF_COUNT), ("profile", C.c_void_p)]


class OthelloB200Error(RuntimeError):
    pass


_lib = None

_SIGS = {
    "oth_abi_version": (C.c_int, []),
    "oth_error_string": (C.c_char_p, [C.c_int]),
    "oth_last_cuda_error": (C.c_char_p, []),
    "oth_device_count": (C.c_int, []),
    "oth_legal_moves": (C.c_int, [C.c_void_p] * 3 + [C.c_int64, C.c_void_p]),
    "oth_step": (C.c_int, [C.c_void_p] * 7 + [C.c_int64, C.c_void_p]),
    "oth_rollout": (C.c_int, [C.c_uint64, C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "oth_pack_states": (C.c_int, [C.c_void_p] * 4 + [C.c_int64, C.c_void_p]),
    "oth_unpack_states": (C.c_int, [C.c_void_p] * 4 + [C.c_int64, C.c_void_p]),
    "oth_valid_moves_i8": (C.c_int, [C.c_void_p] * 3 + [C.c_int64, C.c_void_p]),
    "oth_symmetry": (C.c_int, [C.c_void_p] * 6 + [C.c_int64, C.c_void_p]),
    "oth_host_valid_moves": (C.c_int, [C.c_void_p] * 3 + [C.c_int64]),
    "oth_host_next_state": (C.c_int, [C.c_void_p] * 5 + [C.c_int64]),
    "oth_host_value_terminated": (C.c_int, [C.c_void_p] * 4 + [C.c_int64]),
    "oth_host_symmetry": (C.c_int, [C.c_void_p] * 6 + [C.c_int64]),
    "oth_host_rollout": (C.c_int, [C.c_uint64, C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "oth_host_int32_peak": (C.c_int, [C.c_void_p, C.c_void_p]),
    "oth_host_random_read_probe": (C.c_int, [C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "oth_mcts_buffer_bytes": (C.c_int, [C.c_void_p, C.c_void_p]),
    "oth_mcts_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "oth_mcts_set_roots": (C.c_int, [C.c_void_p] * 6),
    "oth_mcts_begin_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "oth_mcts_set_roots_masked": (C.c_int, [C.c_void_p] * 7),
    "oth_mcts_begin_search_masked": (C.c_int, [C.c_void_p] * 4),
    "oth_mcts_step": (C.c_int, [C.c_void_p] * 6),
    "oth_mcts_step_fused": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "oth_mcts_step_fused_mapped": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "oth_mcts_dedup_workspace_bytes": (C.c_int, [C.c_int32, C.c_void_p]),
    "oth_mcts_dedup": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p]),
    "oth_mcts_advance": (C.c_int, [C.c_void_p] * 4),
    "oth_mcts_poll": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "oth_mcts_profile_create": (C.c_int, [C.c_int32, C.c_void_p]),
    "oth_mcts_profile_read": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "oth_mcts_profile_destroy": (C.c_int, [C.c_void_p]),
    "oth_mcts_root_stats": (C.c_int, [C.c_void_p] * 9),
    "oth_unpack_canonical": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "oth_replay_aggregate_workspace_bytes": (C.c_int, [C.c_int64, C.c_void_p]),
    "oth_replay_aggregate": (C.c_int, [C.c_void_p] * 4 + [C.c_int64, C.c_void_p, C.c_int64] + [C.c_void_p] * 7),
    "oth_nn_stem_im2col_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "oth_nn_bias_add_relu_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "oth_nn_leaf_symmetry": (C.c_int, [C.c_void_p, C.c_int64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "oth_nn_unsymmetrise_logits": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "oth_nn_symmetry_images": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "oth_nn_symmetry_mean": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                       C.c_void_p]),
    "oth_alphabeta": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32] + [C.c_void_p] * 4),
    "oth_host_alphabeta": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32] + [C.c_void_p] * 3),
    "oth_solve_wld": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32] + [C.c_void_p] * 3),
    "oth_host_solve_wld": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32] + [C.c_void_p] * 2),
}

EXPORTED_SYMBOLS = tuple(_SIGS)


def lib():
    """Load (building with nvcc if needed) the CUDA library. Raises if impossible."""
    global _lib
    if _lib is None:
        debug = os.environ.get("OTH_B200_DEBUG", "") not in ("", "0")  # the -DOTH_DEBUG build (arena index assertions)
        path, tmp = (_build.LIB_DEBUG if debug else _build.LIB), None
        if _build.needs_build(debug):  # not what build() left for these sources: compile a private copy, not into the tree
            tmp = tempfile.mkdtemp(prefix="othello_b200-")
            path = _build.build(debug=debug, out_dir=tmp)
        L = C.CDLL(path)
        if tmp:
            shutil.rmtree(tmp)  # the loaded library stays mapped
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)  # AttributeError = ABI mismatch: fail loudly
            fn.restype = res
            fn.argtypes = args
        if L.oth_abi_version() != ABI_VERSION:
            raise OthelloB200Error("libothello_b200 ABI version mismatch")
        _lib = L
    return _lib


def check(rc, what=""):
    if rc == OTH_OK:
        return
    L = lib()
    msg = L.oth_error_string(rc).decode()
    if rc == OTH_E_ILLEGAL:
        raise ValueError(f"Illegal move{': ' + what if what else ''}")
    if rc in (OTH_E_CUDA, OTH_E_NO_DEVICE):
        msg += " [" + L.oth_last_cuda_error().decode() + "]"
    raise OthelloB200Error(f"{what or 'libothello_b200'}: {msg}")


def require_device():
    if lib().oth_device_count() <= 0:
        raise OthelloB200Error("no CUDA device visible: alphazero_othello_b200 has no CPU fallback")
