"""CPU oracle -- TEST INFRASTRUCTURE ONLY.

ctypes front-end of ``oracle/othello_oracle.c``, a plain-C restatement of the
reference's self-play hot path (envs/othello.py, MCTS_model.py,
self_play_worker.py).  It is the checker the CUDA engine is compared with:
only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline /
``--impl reference`` legs may import it.  The product package
``alphazero_othello_b200`` never does.

Parity is pinned by ``tests/test_oracle_golden.py`` against
``tests/golden/ref_golden.npz`` (generated from the reference itself by
``tests/golden/make_golden.py``).
"""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "liboracle.so")

EVAL_FN = C.CFUNCTYPE(None, C.c_void_p, C.POINTER(C.c_int8), C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_double))

STUB_A, STUB_B, STUB_H, STUB_TABLE, STUB_TAPE = 0, 1, 2, 3, 4


def _stale():
    return not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(os.path.join(_HERE, "othello_oracle.c"))


def build(force=False, out_dir=_HERE):
    """Compile liboracle.so with gcc (oracle/Makefile) into ``out_dir``; in this directory only when missing or stale,
    unless ``force``."""
    lib = os.path.join(out_dir, "liboracle.so")
    if force or out_dir != _HERE or _stale():
        subprocess.check_call(["make", "-s", "-C", _HERE, "-B", "OUT=" + lib, lib])
    return lib


_lib = None


def lib():
    global _lib
    if _lib is None:
        path, tmp = _LIB_PATH, None
        if _stale():  # compiled at run time into a temporary directory, never into the tree
            tmp = tempfile.mkdtemp(prefix="oracle-")
            path = build(out_dir=tmp)
        L = C.CDLL(path)
        if tmp:
            shutil.rmtree(tmp)  # the loaded library stays mapped
        vp, i32, f64 = C.c_void_p, C.c_int, C.c_double
        L.orc_initial_state.argtypes = [vp]
        L.orc_valid_moves.argtypes = [vp, i32, vp]
        L.orc_valid_moves.restype = i32
        L.orc_next_state.argtypes = [vp, i32, i32, vp]
        L.orc_next_state.restype = i32
        L.orc_score.argtypes = [vp, i32]
        L.orc_score.restype = i32
        L.orc_value_terminated.argtypes = [vp, i32, C.POINTER(i32), C.POINTER(i32)]
        L.orc_symmetry.argtypes = [vp, vp, i32, i32, vp, vp]
        L.orc_symmetries.argtypes = [vp, vp, vp, vp]
        L.orc_choice.argtypes = [vp, i32, f64]
        L.orc_choice.restype = i32
        L.orc_mcts_new.argtypes = [f64, i32, f64, vp, vp]
        L.orc_mcts_new.restype = vp
        L.orc_mcts_free.argtypes = [vp]
        L.orc_mcts_search.argtypes = [vp, vp, i32, vp]
        L.orc_mcts_search.restype = i32
        L.orc_mcts_root_stats.argtypes = [vp, vp, vp, vp, vp, vp]
        L.orc_mcts_counters.argtypes = [vp, vp]
        L.orc_mcts_policy.argtypes = [vp, f64, f64, vp]
        L.orc_philox4x32_10.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, vp]
        L.orc_mcts_set_rollout.argtypes = [vp, C.c_uint64, C.c_uint64]
        L.orc_mcts_set_ply.argtypes = [vp, i32]
        L.orc_mcts_make_move.argtypes = [vp, i32]
        L.orc_mcts_make_move.restype = i32
        L.orc_self_play.argtypes = [f64, i32, f64, f64, i32, f64, vp, vp, vp, vp, vp, i32] + [vp] * 8
        L.orc_self_play.restype = i32
        L.orc_get_stub.argtypes = [i32]
        L.orc_get_stub.restype = vp
        L.orc_table_new.argtypes = [C.c_uint64]
        L.orc_table_new.restype = vp
        L.orc_table_free.argtypes = [vp]
        L.orc_table_put.argtypes = [vp, C.c_uint64, C.c_uint64, vp, C.c_float]
        L.orc_table_put.restype = i32
        L.orc_table_put_planes.argtypes = [vp, vp, vp, vp, vp, C.c_long, vp]
        L.orc_table_put_planes.restype = i32
        L.orc_mcts_set_picks.argtypes = [vp, vp, C.c_long]
        L.orc_mcts_picks_used.argtypes = [vp]
        L.orc_mcts_picks_used.restype = C.c_long
        L.orc_tape_new.argtypes = [C.c_long, C.c_long]
        L.orc_tape_new.restype = vp
        L.orc_tape_free.argtypes = [vp]
        L.orc_tape_put_planes.argtypes = [vp, vp, vp, vp, vp, C.c_long]
        L.orc_tape_put_planes.restype = i32
        L.orc_tape_stat.argtypes = [vp, C.c_long, i32]
        L.orc_tape_stat.restype = C.c_long
        L.orc_table_misses.argtypes = [vp]
        L.orc_table_misses.restype = C.c_long
        L.orc_table_hits.argtypes = [vp]
        L.orc_table_hits.restype = C.c_long
        L.orc_random_playout.argtypes = [C.c_uint64, C.POINTER(i32), vp, i32]
        L.orc_random_playout.restype = i32
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _state(s):
    return np.ascontiguousarray(np.asarray(s, dtype=np.int8).reshape(64))


# ------------------------------------------------------------------ env ----
class OracleGame:
    """Game-API view (envs/game.py:5-57) of the C oracle env."""

    def __init__(self, n=8):
        assert n == 8
        self.n = n

    action_size = 65
    state_size = 64

    def get_initial_state(self):
        s = np.zeros(64, np.int8)
        lib().orc_initial_state(_p(s))
        return s.reshape(8, 8)

    def get_valid_moves(self, state, player):
        out = np.zeros(65, np.uint8)
        lib().orc_valid_moves(_p(_state(state)), int(player), _p(out))
        return out

    def get_next_state(self, state, action, player):
        out = np.zeros(64, np.int8)
        if lib().orc_next_state(_p(_state(state)), int(action), int(player), _p(out)) != 0:
            raise ValueError(f"Illegal move: {action}")
        return out.reshape(8, 8)

    def get_value_and_terminated(self, state, action, player):
        v, t = C.c_int(0), C.c_int(0)
        lib().orc_value_terminated(_p(_state(state)), int(player), C.byref(v), C.byref(t))
        return v.value, bool(t.value)

    def get_score(self, state, player):
        return lib().orc_score(_p(_state(state)), int(player))

    def get_opponent(self, player):
        return -player


def symmetry(state, pi, k, flip):
    """get_random_symmetry (envs/othello.py:501-526) for a given (k, flip)."""
    pi = np.ascontiguousarray(pi, dtype=np.float32)
    os_, op = np.zeros(64, np.float32), np.zeros(65, np.float32)
    lib().orc_symmetry(_p(_state(state)), _p(pi), int(k), int(bool(flip)), _p(os_), _p(op))
    return os_.reshape(1, 8, 8), op


def symmetries(state, pi):
    """OthelloGame.get_symmetries (envs/othello.py:286-298): 8 images."""
    pi = np.ascontiguousarray(pi, dtype=np.float32)
    os_, op = np.zeros((8, 64), np.float32), np.zeros((8, 65), np.float32)
    lib().orc_symmetries(_p(_state(state)), _p(pi), _p(os_), _p(op))
    return os_.reshape(8, 8, 8), op


def choice(p, u):
    p = np.ascontiguousarray(p, dtype=np.float32)
    return lib().orc_choice(_p(p), len(p), float(u))


# ----------------------------------------------------------- evaluators ----
class Evaluator:
    """Wraps either a C stub (by id) or a Python callable
    ``fn(state int8[8,8], player) -> (priors f32[65], value float)`` -- the
    signature of Models.Inference.inference (Models.py:11-31)."""

    def __init__(self, stub=None, fn=None, salt=0, table=None, tape=None, slot=0):
        self._keep = []
        self.ctx = None
        if tape is not None:  # the slot's recorded evaluation sequence, served in order
            self.fn_ptr = lib().orc_get_stub(STUB_TAPE)
            self._cursor = (C.c_void_p * 2)(tape.handle, int(slot))  # {EvalTape*, long slot}
            self.ctx = C.cast(self._cursor, C.c_void_p)
            self._keep.append(tape)
        elif fn is not None:
            def cb(_ctx, s_ptr, player, pri_ptr, val_ptr):
                s = np.ctypeslib.as_array(s_ptr, shape=(64,)).reshape(8, 8).copy()
                pri, val = fn(s, int(player))
                out = np.ctypeslib.as_array(pri_ptr, shape=(65,))
                out[:] = np.asarray(pri, dtype=np.float32)
                val_ptr[0] = float(val)
            self._cb = EVAL_FN(cb)
            self.fn_ptr = C.cast(self._cb, C.c_void_p)
        elif table is not None:
            self.fn_ptr = lib().orc_get_stub(STUB_TABLE)
            self.ctx = table.handle
            self._keep.append(table)
        else:
            self.fn_ptr = lib().orc_get_stub(int(stub))
            if stub == STUB_H:
                self._salt = C.c_uint64(salt)
                self.ctx = C.cast(C.pointer(self._salt), C.c_void_p)


class EvalTable:
    """Recorded (canonical bitboards -> priors, value) table (SURVEY 8c)."""

    def __init__(self, cap_pow2=1 << 20):
        self.handle = lib().orc_table_new(cap_pow2)
        self.stats = np.zeros(3, np.int64)  # put_planes: inserted / identical repeats / conflicts

    def put(self, own, opp, priors, value):
        priors = np.ascontiguousarray(priors, dtype=np.float32)
        return lib().orc_table_put(self.handle, int(own), int(opp), _p(priors), float(value))

    def put_planes(self, planes, mask, priors, values):
        """One leaf batch: planes f32[n,64] canonical, mask uint8/bool[n] (rows to record), priors f32[n,65],
        values f32[n].  Accumulates self.stats = [inserted, repeated identically, CONFLICTING]."""
        planes = np.ascontiguousarray(planes, dtype=np.float32).reshape(-1, 64)
        n = len(planes)
        mask = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        priors = np.ascontiguousarray(priors, dtype=np.float32).reshape(n, 65)
        values = np.ascontiguousarray(values, dtype=np.float32).reshape(n)
        if lib().orc_table_put_planes(self.handle, _p(planes), _p(mask), _p(priors), _p(values), n, _p(self.stats)) != 0:
            raise RuntimeError("EvalTable full")

    @property
    def misses(self):
        return lib().orc_table_misses(self.handle)

    @property
    def hits(self):
        return lib().orc_table_hits(self.handle)

    def __del__(self):
        try:
            lib().orc_table_free(self.handle)
        except Exception:
            pass


class EvalTape:
    """Per-slot sequence of the evaluations an engine consumed (oracle/othello_oracle.c EvalTape): the oracle
    replaying slot s is served the k-th recorded output on its k-th request and checks that the positions agree."""

    def __init__(self, n_slots, cap_per_slot):
        self.n_slots = int(n_slots)
        self.handle = lib().orc_tape_new(self.n_slots, int(cap_per_slot))
        if not self.handle:
            raise MemoryError("EvalTape")

    def put_planes(self, planes, mask, priors, values):
        planes = np.ascontiguousarray(planes, dtype=np.float32).reshape(self.n_slots, 64)
        mask = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        priors = np.ascontiguousarray(priors, dtype=np.float32).reshape(self.n_slots, 65)
        values = np.ascontiguousarray(values, dtype=np.float32).reshape(self.n_slots)
        rc = lib().orc_tape_put_planes(self.handle, _p(planes), _p(mask), _p(priors), _p(values), self.n_slots)
        if rc != 0:
            raise RuntimeError(f"EvalTape.put_planes rc={rc} (tape full?)")

    @property
    def mismatches(self):
        return lib().orc_tape_stat(self.handle, 0, 0)

    @property
    def served(self):
        return lib().orc_tape_stat(self.handle, 0, 1)

    def recorded(self, slot):
        return lib().orc_tape_stat(self.handle, slot, 2)

    def consumed(self, slot):
        return lib().orc_tape_stat(self.handle, slot, 3)

    def __del__(self):
        try:
            lib().orc_tape_free(self.handle)
        except Exception:
            pass


# ----------------------------------------------------------------- MCTS ----
class OracleMCTS:
    """MCTS surface (MCTS_model.py:172-274), num_threads=1 semantics, with
    the reference's np.random draws replaced by injected values."""

    def __init__(self, c_puct, num_simulations, evaluator, dirichlet_epsilon=0.0, rollout_seed=0, game_id=0, picks=None):
        """evaluator=None selects the reference's policy=None mode (uniform priors + random playout); ``picks`` =
        the indices np.random.choice returned in a reference run (else playouts draw from Philox)."""
        self.ev = evaluator
        if evaluator is None:
            self.h = lib().orc_mcts_new(float(c_puct), int(num_simulations), float(dirichlet_epsilon), None, None)
            lib().orc_mcts_set_rollout(self.h, int(rollout_seed), int(game_id))
            if picks is not None:
                self._picks = np.ascontiguousarray(picks, dtype=np.int32)
                lib().orc_mcts_set_picks(self.h, _p(self._picks), len(self._picks))
        else:
            self.h = lib().orc_mcts_new(float(c_puct), int(num_simulations), float(dirichlet_epsilon),
                                        evaluator.fn_ptr, evaluator.ctx)
        self.ply = 0

    def __del__(self):
        try:
            lib().orc_mcts_free(self.h)
        except Exception:
            pass

    def search(self, state, player, noise=None):
        if noise is not None:
            noise = np.ascontiguousarray(noise, dtype=np.float64)
        lib().orc_mcts_set_ply(self.h, self.ply)
        rc = lib().orc_mcts_search(self.h, _p(_state(state)), int(player), _p(noise))
        if rc != 0:
            raise AssertionError("root does not match the given state/player")

    def policy(self, temp, u_tie=0.0):
        probs = np.zeros(65, np.float32)
        lib().orc_mcts_policy(self.h, float(temp), float(u_tie), _p(probs))
        return probs

    def policy_improve_step(self, state, player, temp=1.0, noise=None, u_tie=0.0):
        self.search(state, player, noise)
        return self.policy(temp, u_tie)

    def make_move(self, action):
        if lib().orc_mcts_make_move(self.h, int(action)) != 0:
            raise KeyError(int(action))
        self.ply += 1

    @property
    def picks_used(self):
        return lib().orc_mcts_picks_used(self.h)

    def root_stats(self):
        counts = np.zeros(65, np.int32)
        cval, cpri = np.zeros(65, np.float64), np.zeros(65, np.float64)
        rv, rn = np.zeros(1, np.float64), np.zeros(1, np.int64)
        lib().orc_mcts_root_stats(self.h, _p(counts), _p(cval), _p(cpri), _p(rv), _p(rn))
        return dict(counts=counts, child_value=cval, child_prior=cpri, root_value=float(rv[0]), root_n=int(rn[0]))

    def counters(self):
        out = np.zeros(5, np.int64)
        lib().orc_mcts_counters(self.h, _p(out))
        return dict(evals=int(out[0]), sims=int(out[1]), nodes=int(out[2]), max_depth=int(out[3]),
                    max_children=int(out[4]))


def self_play(args, evaluator, noise, u_move, u_tie=None, max_plies=128):
    """one_self_play (self_play_worker.py:38-88) with injected randomness.
    Returns dict(states int8[T,8,8], pis f32[T,65], values f64[T], players,
    root_values, actions, counts int32[T,65], counters)."""
    T = max_plies
    states = np.zeros((T, 64), np.int8)
    pis = np.zeros((T, 65), np.float32)
    values = np.zeros(T, np.float64)
    players = np.zeros(T, np.int8)
    rvals = np.zeros(T, np.float64)
    actions = np.zeros(T, np.int32)
    counts = np.zeros((T, 65), np.int32)
    counters = np.zeros(5, np.int64)
    noise = None if noise is None else np.ascontiguousarray(noise, dtype=np.float64)
    u_move = np.ascontiguousarray(u_move, dtype=np.float64)
    assert len(u_move) >= T
    if u_tie is not None:
        u_tie = np.ascontiguousarray(u_tie, dtype=np.float64)
        assert len(u_tie) >= T
    n = lib().orc_self_play(float(args["c_puct"]), int(args["num_simulations"]), float(args["dirichlet_epsilon"]),
                            float(args["mcts_temperature"]), int(args["num_exploratory_moves"]),
                            float(args["lambda"]), evaluator.fn_ptr, evaluator.ctx, _p(noise), _p(u_move),
                            _p(u_tie), T, _p(states), _p(pis), _p(values), _p(players), _p(rvals), _p(actions),
                            _p(counts), _p(counters))
    if n < 0:
        raise RuntimeError(f"oracle self_play failed rc={n}")
    return dict(states=states[:n].reshape(n, 8, 8), pis=pis[:n], values=values[:n], players=players[:n],
                root_values=rvals[:n], actions=actions[:n], counts=counts[:n],
                counters=dict(evals=int(counters[0]), sims=int(counters[1]), nodes=int(counters[2]),
                              max_depth=int(counters[3]), max_children=int(counters[4])))


def philox(seed, ctr_lo, h0, h1):
    """Philox4x32-10 block (four uint32) for key ``seed`` and counter (ctr_lo, h0, h1)."""
    out = np.zeros(4, np.uint32)
    lib().orc_philox4x32_10(int(seed), int(ctr_lo), int(h0), int(h1), _p(out))
    return out


def random_playout(seed, max_plies=128):
    score = C.c_int(0)
    tr = np.zeros(max_plies, np.int32)
    n = lib().orc_random_playout(int(seed), C.byref(score), _p(tr), max_plies)
    return n, score.value, tr[:n]
