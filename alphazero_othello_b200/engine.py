"""Host driver of the batched MCTS self-play engine (CUDA kernels in csrc/mcts_kernels.cu).

PyTorch is used for device memory, streams, CUDA graphs and the policy/value
network only; every search / env / self-play step is a kernel behind the C ABI
(include/othello_b200.h).  One process drives one GPU; games are sharded over
ranks by game id (no collective on the search path).
"""
import copy
import ctypes as C
import os

import numpy as np
import torch

from . import _lib, symmetry


def default_lanes(n_slots):
    """Threads per slot.  A slot's work per launch is one dependent chain (expand, back up, descend); 32 lanes keep
    every step of it one round wide (<= 32 children) and free of intra-warp divergence between slots.  8 lanes -- four
    slots per warp -- only pay once 32 lanes would need more than one wave of the 7 x 148 resident 128-thread blocks."""
    return 32 if n_slots * 32 <= 7 * 148 * 128 else (16 if n_slots * 16 <= 7 * 148 * 128 else 8)


def default_node_cap(num_simulations):
    """Arena size per slot: kept subtree + one expansion (<= 33 children) per simulation,
    with headroom; measured high-water marks: 13.6k of 20.2k nodes at 400 simulations (16 384 complete games),
    5.5k of 10.6k at 200."""
    return int(max(2048, 48 * num_simulations + 1024))


class MctsEngine:
    """Owns the device buffers of ``n_slots`` concurrent search trees and launches the kernels.

    ``args`` carries the reference's keys (train.py:399-425): c_puct, num_simulations,
    dirichlet_alpha, dirichlet_epsilon, mcts_temperature, num_exploratory_moves, lambda.
    """

    def __init__(self, n_slots, args, *, self_play=True, eval_kind=_lib.EVAL_EXTERNAL, games_per_slot=-1,
                 device="cuda:0", node_cap=None, path_cap=128, max_inline_sims=8, inject_random=False, lanes=None,
                 seed=0, game_id_base=0, game_id_stride=None, stub_salt=0, out_pos_cap=None, out_game_cap=None,
                 hot_path=0, split_stub=False, move_launch=None):
        _lib.require_device()
        self.device = torch.device(device)
        self.n_slots = int(n_slots)
        cfg = _lib.MctsConfig()
        cfg.n_slots = self.n_slots
        cfg.num_simulations = int(args["num_simulations"])
        cfg.node_cap = int(node_cap or default_node_cap(cfg.num_simulations))
        cfg.path_cap = int(path_cap)
        cfg.num_exploratory_moves = int(args.get("num_exploratory_moves", 0))
        cfg.eval_kind = int(eval_kind)
        cfg.self_play = 1 if self_play else 0
        cfg.games_per_slot = int(games_per_slot)
        cfg.max_inline_sims = int(max_inline_sims)
        cfg.inject_random = 1 if inject_random else 0
        cfg.lanes = int(lanes or default_lanes(self.n_slots))
        cfg.hot_path = int(hot_path)
        cfg.split_stub = 1 if split_stub else 0
        if move_launch is None:
            move_launch = int(os.environ.get("OTH_MOVE_LAUNCH", "1"))
        cfg.move_launch = int(move_launch)
        if out_game_cap is None:
            out_game_cap = self.n_slots * (2 if games_per_slot < 0 else max(1, games_per_slot)) + 16
        if out_pos_cap is None:
            out_pos_cap = out_game_cap * 72
        cfg.out_pos_cap = int(out_pos_cap)
        cfg.out_game_cap = int(out_game_cap)
        cfg.c_puct = float(args["c_puct"])
        cfg.dirichlet_alpha = float(args.get("dirichlet_alpha", 0.03))
        cfg.dirichlet_epsilon = float(args.get("dirichlet_epsilon", 0.0))
        cfg.temperature = float(args.get("mcts_temperature", 1.0))
        cfg.lambda_ = float(args.get("lambda", 1.0))
        cfg.seed = int(seed)
        cfg.game_id_base = int(game_id_base)
        cfg.game_id_stride = int(game_id_stride if game_id_stride is not None else self.n_slots)
        cfg.stub_salt = int(stub_salt)
        self.cfg = cfg
        self.L = _lib.lib()
        sizes = (C.c_int64 * _lib.BUF_COUNT)()
        _lib.check(self.L.oth_mcts_buffer_bytes(C.byref(cfg), sizes), "oth_mcts_buffer_bytes")
        self.buf_bytes = list(sizes)
        self.bufs = _lib.MctsBuffers()
        self._t = []
        with torch.cuda.device(self.device):
            for i, nb in enumerate(self.buf_bytes):
                # int64 storage: every buffer is at least 8-byte aligned (torch gives 512 B)
                t = torch.zeros((max(nb, 8) + 7) // 8, dtype=torch.int64, device=self.device)
                self._t.append(t)
                self.bufs.buf[i] = t.data_ptr()
            self.nn_input = torch.zeros((self.n_slots, 1, 8, 8), dtype=torch.float32, device=self.device)
            self.priors = torch.zeros((self.n_slots, 65), dtype=torch.float32, device=self.device)
            self.values = torch.zeros((self.n_slots,), dtype=torch.float32, device=self.device)
        self.launches = 0

    # ---------------------------------------------------------------- views
    def _view(self, i, dtype, shape):
        return self._t[i].view(dtype)[: int(np.prod(shape))].view(*shape)

    @property
    def counters_t(self):
        return self._t[_lib.BUF_COUNTERS][:16]

    def counters(self, poll=True):
        """Event counters (cumulative) + gauges (waiting / active / errors / max_top, refreshed here)."""
        if poll:
            self._call(self.L.oth_mcts_poll, self._stream())
        v = self.counters_t.cpu().numpy()
        return {n: int(v[i]) for i, n in enumerate(_lib.CNT_NAMES)}

    def ctl(self):
        raw = self._t[_lib.BUF_CTL][: self.n_slots * 8].cpu().numpy().view(np.int32).reshape(self.n_slots, 16)
        names = ["phase", "root", "top", "arena", "ply", "sims_done", "pending", "path_len", "flags", "player", "games_left",
                 "error"]
        d = {n: raw[:, i].copy() for i, n in enumerate(names)}
        d["game_id"] = raw[:, 12:14].copy().view(np.int64).reshape(-1)
        return d

    @property
    def noise(self):
        return self._view(_lib.BUF_NOISE, torch.float64, (self.n_slots, 65))

    @property
    def u_move(self):
        return self._view(_lib.BUF_U_MOVE, torch.float64, (self.n_slots, _lib.OTH_MAX_PLIES))

    @property
    def u_tie(self):
        return self._view(_lib.BUF_U_TIE, torch.float64, (self.n_slots, _lib.OTH_MAX_PLIES))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _call(self, fn, *a):
        with torch.cuda.device(self.device):
            _lib.check(fn(C.byref(self.cfg), C.byref(self.bufs), *a), fn.__name__)

    # -------------------------------------------------------------- kernels
    def reset(self):
        self._call(self.L.oth_mcts_reset, self._stream())

    def set_roots(self, own, opp, players, mask=None):
        """own/opp int64 [n_slots] device tensors, players int8 [n_slots]; mask uint8 [n_slots] limits the slots."""
        self._call(self.L.oth_mcts_set_roots_masked, own.data_ptr(), opp.data_ptr(), players.data_ptr(),
                   None if mask is None else mask.data_ptr(), self._stream())

    def begin_search(self, mask=None):
        self._call(self.L.oth_mcts_begin_search_masked, None if mask is None else mask.data_ptr(), self._stream())

    def step(self):
        """One launch of the fused expand/backup/select/self-play kernel on the engine's
        priors/values/nn_input tensors."""
        self._call(self.L.oth_mcts_step, self.priors.data_ptr(), self.values.data_ptr(), self.nn_input.data_ptr(),
                   self._stream())
        self.launches += 1

    def dedup(self, bucket, compact_input, eval_map, stats, workspace):
        """oth_mcts_dedup: distinct pending leaves -> compact_input [bucket,1,8,8] + eval_map int32[n_slots]; stats int32[2]."""
        self._call(self.L.oth_mcts_dedup, int(bucket), workspace.data_ptr(), workspace.numel(),
                   None if compact_input is None else compact_input.data_ptr(), None if eval_map is None else eval_map.data_ptr(),
                   stats.data_ptr(), self._stream())

    def step_fused(self, logits, value_preact, record=False, eval_map=None):
        """``step`` with the network's softmax / tanh applied in-kernel: ``logits`` [n_slots, >=65] and
        ``value_preact`` [n_slots, >=1] are (possibly strided) float32 or bfloat16 views of the head outputs.
        ``record=True`` writes the priors / values the kernel used to ``self.priors`` / ``self.values``."""
        assert logits.dtype == value_preact.dtype and logits.dtype in (torch.float32, torch.bfloat16)
        assert logits.stride(1) == 1 and logits.size(0) == value_preact.size(0)
        assert eval_map is not None or logits.size(0) == self.n_slots  # de-duplicated batches are indexed through eval_map
        self._call(self.L.oth_mcts_step_fused_mapped, logits.data_ptr(), logits.stride(0), value_preact.data_ptr(), value_preact.stride(0),
                   1 if logits.dtype == torch.bfloat16 else 0, None if eval_map is None else eval_map.data_ptr(),
                   self.priors.data_ptr() if record else None, self.values.data_ptr() if record else None, self.nn_input.data_ptr(),
                   self._stream())
        self.launches += 1

    # per-launch timing of the step / move kernels (othello_b200_experimental.h), per engine
    def profile_begin(self, max_launches):
        h = C.c_void_p()
        _lib.check(self.L.oth_mcts_profile_create(int(max_launches), C.byref(h)), "oth_mcts_profile_create")
        self.bufs.profile = h.value
        self._prof_cap = int(max_launches)

    def profile_end(self):
        """-> (step_ms list, move_ms list) of the launches recorded since profile_begin; detaches the handle."""
        h, cap = self.bufs.profile, self._prof_cap
        self.bufs.profile = None
        a, b, n = (C.c_float * cap)(), (C.c_float * cap)(), C.c_int32(0)
        try:
            _lib.check(self.L.oth_mcts_profile_read(h, a, b, C.byref(n)), "oth_mcts_profile_read")
        finally:
            self.L.oth_mcts_profile_destroy(h)
        return list(a[: n.value]), list(b[: n.value])

    def advance(self, actions):
        self._call(self.L.oth_mcts_advance, actions.data_ptr(), self._stream())

    def root_stats(self):
        n = self.n_slots
        dev = self.device
        counts = torch.empty((n, 65), dtype=torch.int32, device=dev)
        cval = torch.empty((n, 65), dtype=torch.float64, device=dev)
        cpri = torch.empty((n, 65), dtype=torch.float64, device=dev)
        rv = torch.empty(n, dtype=torch.float64, device=dev)
        rn = torch.empty(n, dtype=torch.int32, device=dev)
        rb = torch.empty((n, 2), dtype=torch.int64, device=dev)
        self._call(self.L.oth_mcts_root_stats, counts.data_ptr(), cval.data_ptr(), cpri.data_ptr(), rv.data_ptr(),
                   rn.data_ptr(), rb.data_ptr(), self._stream())
        return dict(counts=counts, child_value=cval, child_prior=cpri, root_value=rv, root_n=rn, root_board=rb)

    def raise_on_error(self):
        c = self.ctl()
        bad = np.nonzero(c["error"])[0]
        if len(bad):
            e = int(c["error"][bad[0]])
            names = [v for k, v in _lib.ERR_NAMES.items() if e & k]
            if e == 16:
                raise KeyError("; ".join(names))
            raise _lib.OthelloB200Error(f"slot {int(bad[0])}: {'; '.join(names)} (node_cap={self.cfg.node_cap})")

    # -------------------------------------------------------------- outputs
    def drain(self, to_host=True):
        """Collect the replay tuples of games finished since the last drain and reset the
        output ring.  Returns dict(boards int64[n,2] (own,opp canonical), pis f32[n,65],
        values f64[n], meta int64[n], games int64[g,4] = (game_id, first, n, winner))."""
        torch.cuda.nvtx.range_push("oth:drain")
        cnt = self.counters_t[_lib.CNT_POSITIONS:_lib.CNT_OUT_GAMES + 1].cpu()
        n, g = int(cnt[0]), int(cnt[1])
        n, g = min(n, self.cfg.out_pos_cap), min(g, self.cfg.out_game_cap)
        out = dict(
            boards=self._view(_lib.BUF_OUT_BOARD, torch.int64, (self.cfg.out_pos_cap, 2))[:n],
            pis=self._view(_lib.BUF_OUT_PI, torch.float32, (self.cfg.out_pos_cap, 65))[:n],
            values=self._view(_lib.BUF_OUT_VALUE, torch.float64, (self.cfg.out_pos_cap,))[:n],
            meta=self._view(_lib.BUF_OUT_META, torch.int64, (self.cfg.out_pos_cap,))[:n],
            games=self._view(_lib.BUF_OUT_GAMES, torch.int64, (self.cfg.out_game_cap, 4))[:g],
        )
        states = torch.empty((n, 8, 8), dtype=torch.int8, device=self.device)
        if n:
            with torch.cuda.device(self.device):
                _lib.check(self.L.oth_unpack_canonical(out["boards"].data_ptr(), states.data_ptr(), n, self._stream()))
        out["states"] = states
        if to_host:
            out = {k: v.cpu() for k, v in out.items()}
        else:
            out = {k: v.clone() for k, v in out.items()}
        self.counters_t[_lib.CNT_POSITIONS:_lib.CNT_OUT_GAMES + 1].zero_()
        torch.cuda.nvtx.range_pop()
        return out


def private_copy(policy, device):
    """The caller's module is never moved or switched to eval mode: like the reference's workers, which rebuild the
    network from (class, config, state_dict) (self_play_worker.py:49-52), the engine works on its own copy."""
    on_dev = next((p.device for p in policy.parameters()), None) == torch.device(device)
    if on_dev and not policy.training:
        return policy  # already an inference copy on the right device (e.g. a FoldedNet the caller built)
    return copy.deepcopy(policy).to(device).eval()


class BatchedPolicy:
    """The policy/value network at the engine boundary.  It stays PyTorch
    (Models.py:93-221 architectures): ``policy(x[B,1,8,8]) -> (logits[B,65], value[B,1])``,
    softmax over actions as Models.py:24-25.  Runs in eval mode on the GPU; ``dtype``
    torch.bfloat16 uses autocast + channels_last."""

    def __init__(self, policy, device="cuda:0", dtype=torch.float32):
        self.device = torch.device(device)
        self.dtype = dtype
        self.policy = private_copy(policy, self.device)
        if dtype != torch.float32:
            self.policy = self.policy.to(memory_format=torch.channels_last)

    @property
    def has_raw(self):
        return bool(getattr(self.policy, "supports_raw", False))

    @torch.no_grad()
    def raw(self, x):
        """(logits [B,65], value pre-activation [B,1]) views of the twin's head GEMM outputs."""
        return self.policy(x, raw=True)

    @torch.no_grad()
    def __call__(self, x, priors_out, values_out, sym=None):
        """``sym`` (uint8 [B], optional): row i of ``x`` is the leaf in orientation T_sym[i] (symmetry.leaf_symmetry);
        its logits are mapped back to the leaf's orientation before the softmax."""
        if self.has_raw:
            # network twin: logits / value pre-activation straight from the head GEMMs; one softmax kernel
            # (cast fused) and one cast + one tanh for the values
            logits, v = self.policy(x, raw=True)
            if sym is not None:
                symmetry.unsymmetrise_logits(logits, sym)
            torch.softmax(logits, dim=-1, dtype=torch.float32, out=priors_out)
            values_out.copy_(v.reshape(-1))
            values_out.tanh_()
            return
        if self.dtype != torch.float32:
            with torch.autocast("cuda", dtype=self.dtype):
                logits, value = self.policy(x)
        else:
            logits, value = self.policy(x)
        logits = logits.float()
        if sym is not None:
            symmetry.unsymmetrise_logits(logits, sym)
        torch.softmax(logits, dim=-1, out=priors_out)
        values_out.copy_(value.float().reshape(-1))


class SelfPlayRunner:
    """Batched replacement of ``Trainer.collect_self_play_games`` (train.py:199-225):
    plays ``n_slots`` concurrent games with one network evaluation per simulation per game.

    ``dedup``: evaluation de-duplication (oth_mcts_dedup).  Games that start from the same position ask for the same
    leaves during their first plies; with it the network runs on the DISTINCT pending positions of a batch, padded to
    a few bucket sizes (n/8 ... 7n/8, n/16, n/32; each captured as its own CUDA graph), and the step kernel reads every
    slot's outputs through an index map.  The bucket is chosen on the host from the distinct-position count the device
    reported a few iterations earlier; positions that do not fit the bucket just wait one launch, so the choice only
    affects speed.  "auto" enables it for the fused pipeline from 8192 slots up (measured: at 4096 slots of the
    small network a half-size batch costs 2/3 of a full one and the compaction pass eats the rest).

    ``leaf_symmetry="random"``: every batch the network sees -- the whole leaf batch or a de-duplicated bucket -- is
    first rotated / reflected row by row (oth_nn_leaf_symmetry, the orientation keyed by the engine's seed and the
    position alone) and the network's logits are mapped back before the softmax (oth_nn_unsymmetrise_logits).
    ``engine.nn_input`` itself is left as the step kernel wrote it."""

    DEDUP_BLOCK = 16  # iterations per host decision (and per throttling event)

    def __init__(self, engine, evaluator=None, use_graph=True, fused=True, record=False, dedup=False, leaf_symmetry=None):
        """``record=True``: every launch also writes the priors / values it consumed to ``engine.priors`` /
        ``engine.values`` (fused path: what the kernel's own softmax / tanh produced), so a checker can replay them."""
        self.leaf_symmetry = symmetry.check_mode(leaf_symmetry, ("random",))
        if self.leaf_symmetry and engine.cfg.eval_kind != _lib.EVAL_EXTERNAL:
            raise ValueError("leaf_symmetry needs a network evaluator: the device evaluators see no leaf planes")
        self.e = engine
        self.record = record
        # diagnostic hooks, called around every EXECUTED iteration (eager ones, the warm-up iterations of the graph
        # capture, graph replays): a checker snapshots the leaf batch before and the consumed outputs after
        self.before_iteration = None
        self.after_iteration = None
        self.evaluator = evaluator
        self.external = engine.cfg.eval_kind == _lib.EVAL_EXTERNAL
        assert not self.external or evaluator is not None
        self.use_graph = use_graph
        self.graph = None
        # network twins hand the kernel raw logits: softmax / tanh are fused into oth_mcts_step_fused
        self.fused = fused and self.external and getattr(evaluator, "raw", None) is not None and evaluator.has_raw
        if dedup == "auto":  # pays where the network's time is linear in the batch: large batches of the large network
            dedup = self.fused and engine.n_slots >= 8192 and os.environ.get("OTH_DEDUP", "1") != "0"
        self.dedup = bool(dedup) and self.fused
        # iterations captured per CUDA graph: launching a graph has a fixed cost that shows when an iteration is a few tens
        # of microseconds (measured: one game, 25.6 k -> 27.2 k simulations/s with 8-32 iterations per graph; nothing at
        # 4 096 games); with hooks installed every iteration is its own launch
        self.unroll = int(os.environ.get("OTH_GRAPH_UNROLL", "16" if engine.n_slots <= 256 else "1"))
        self._graph_k = None
        self.last_map = None        # eval_map of the iteration being executed (None: every waiting slot is served)
        self.rows_evaluated = 0     # network rows computed so far (== n_slots per iteration without de-duplication)
        self.force_bucket = None    # test knob: always use this bucket, however many distinct positions there are
        if self.dedup:
            n, dev = engine.n_slots, engine.device
            # batch sizes the network is captured at: n/8 ... 7n/8 in steps of n/8, then n/16, n/32 (never below 256 rows)
            self.buckets = sorted({n * k // 8 for k in range(1, 8)} | {n // 16, n // 32}, reverse=True)
            self.buckets = [b for b in self.buckets if b >= 256 and b % 8 == 0]
            # cost model of an iteration at b rows until the graphs have been timed (_calibrate): fixed + b, in units of one
            # network row (C4: a 512-row iteration takes 340 us, a 16 384-row one 2 870 us = 175 ns per row -> ~1 400 rows)
            self.fixed_cost_rows = max(256, n // 10)
            self.iteration_ms = {}  # measured duration of one iteration per variant ("plain", 0, bucket sizes)
            self.use_measured_times = True  # False: keep the (fixed + rows) model even after the graphs have been timed
            nb = C.c_int64(0)
            _lib.check(engine.L.oth_mcts_dedup_workspace_bytes(n, C.byref(nb)), "oth_mcts_dedup_workspace_bytes")
            self._ws = torch.zeros(nb.value, dtype=torch.uint8, device=dev)
            self._map = torch.full((n,), -1, dtype=torch.int32, device=dev)
            self._stats = torch.zeros(2, dtype=torch.int32, device=dev)
            self._stats_host = torch.zeros(2, dtype=torch.int32).pin_memory()
            self._compact = {b: torch.zeros((b, 1, 8, 8), dtype=torch.float32, device=dev) for b in self.buckets}
            self._graphs = {}      # bucket (0 = whole batch + count) -> CUDA graph
            self._events = []      # throttle: the host stays at most two blocks ahead of the device
            self._recent = [n, n]  # distinct-position counts last reported by the device
            self.bucket_iterations = {0: 0, **{b: 0 for b in self.buckets}}
        if self.leaf_symmetry:
            # the planes the network sees and their symmetry ids: one persistent pair per batch size (the whole batch and
            # every bucket), so that the addresses captured in the CUDA graphs stay valid
            sizes = [engine.n_slots] + (self.buckets if self.dedup else [])
            self._sym = {b: (torch.zeros((b, 1, 8, 8), dtype=torch.float32, device=engine.device),
                             torch.zeros(b, dtype=torch.uint8, device=engine.device)) for b in sizes}

    def _symmetrised(self, x):
        """(the planes the network is shown for the leaf batch ``x``, their symmetry ids or None)."""
        if not self.leaf_symmetry:
            return x, None
        xs, sym = self._sym[x.size(0)]
        symmetry.leaf_symmetry(x, self.e.cfg.seed, xs, sym)
        return xs, sym

    def _iteration(self):
        x, sym = self._symmetrised(self.e.nn_input)
        if self.external and self.fused:
            logits, v = self.evaluator.raw(x)
            if sym is not None:
                symmetry.unsymmetrise_logits(logits, sym)
            self.e.step_fused(logits, v, record=self.record)
            return
        if self.external:
            if sym is None:
                self.evaluator(x, self.e.priors, self.e.values)
            else:
                self.evaluator(x, self.e.priors, self.e.values, sym)
        self.e.step()

    def _dedup_iteration(self, bucket):
        """bucket = 0: the whole batch as usual, plus a count of its distinct positions (the host's next decision);
        otherwise: compact the distinct positions into ``bucket`` rows, evaluate those, map the outputs back."""
        e = self.e
        if bucket == 0:
            e.dedup(0, None, None, self._stats, self._ws)
            self._stats_host.copy_(self._stats, non_blocking=True)
            self._iteration()
            return
        x = self._compact[bucket]
        e.dedup(bucket, x, self._map, self._stats, self._ws)
        self._stats_host.copy_(self._stats, non_blocking=True)
        x, sym = self._symmetrised(x)
        logits, v = self.evaluator.raw(x)
        if sym is not None:
            symmetry.unsymmetrise_logits(logits, sym)
        e.step_fused(logits, v, record=self.record, eval_map=self._map)

    def warm_start(self):
        self.e.reset()
        if self.external:
            self.e.priors.fill_(1.0 / 65.0)  # nothing is consumed by the first launch, but keep the operands finite
            self.e.values.zero_()
        self.e.step()  # emits the root leaves

    def _capture(self, fn=None):
        fn = fn or self._iteration
        dev = self.e.device
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            for _ in range(2):  # executed (they are real iterations), so lazy initialisation is done before capture
                self._hooked(fn)
        torch.cuda.current_stream(dev).wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()  # recorded, not executed
        return g

    def _hooked(self, fn):
        if self.before_iteration is not None:
            self.before_iteration()
        fn()
        if self.after_iteration is not None:
            self.after_iteration()

    def _choose_bucket(self):
        """The batch size with the lowest cost per served evaluation.  A bucket of b rows costs T(b) -- the measured
        duration of that graph (_calibrate), or (fixed + b) rows before the graphs have been timed -- and serves
        min(u, b) distinct positions (u = distinct pending positions reported lately; positions beyond b wait one launch
        and are served next time -- rows are never wasted on duplicates, so a bucket BELOW u runs at full efficiency);
        the whole batch costs T(n) and serves all u.  0 = evaluate the whole batch."""
        if self.force_bucket is not None:
            return self.force_bucket
        n = self.e.n_slots
        u = max(1, min(n, max(self._recent)))
        t = self.iteration_ms
        if t and self.use_measured_times:  # whole-batch mode = one counting iteration per block, plain ones for the rest
            k = self.DEDUP_BLOCK
            # a bucket has to beat the whole batch by 3 %: the timings are three-replay bursts, and with every position
            # distinct a bucket just below u only wins by the noise of that measurement
            best, best_cost = 0, 0.97 * (t[0] + (k - 1) * t["plain"]) / k / u
            for b in self.buckets:
                cost = t[b] / min(u, b)
                if cost < best_cost:
                    best, best_cost = b, cost
            return best
        best, best_cost = 0, n / u
        for b in self.buckets:
            cost = (self.fixed_cost_rows + b) / min(u, b)
            if cost < best_cost:
                best, best_cost = b, cost
        return best

    def _calibrate(self, reps=3):
        """Time one iteration of every captured variant (the replays are real iterations like any other)."""
        dev = self.e.device
        for key, g in self._graphs.items():
            b = None if key == "plain" else key
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                self.last_map = self._map if b else None
                self.rows_evaluated += b or self.e.n_slots
                self.e.launches += 1
                self._hooked(g.replay)
            e1.record()
            torch.cuda.synchronize(dev)
            self.iteration_ms[key] = e0.elapsed_time(e1) / reps

    def _dedup_graph(self, b):
        """The CUDA graph of one iteration variant: b = None plain, 0 whole batch + count, else compacted to b rows.
        Capturing executes two real iterations of that variant first (lazy initialisation, cuDNN plan selection)."""
        key = "plain" if b is None else b
        g = self._graphs.get(key)
        if g is None:
            self.last_map = self._map if b else None
            g = self._graphs[key] = self._capture((lambda: self._dedup_iteration(b)) if b is not None else self._iteration)
            self.rows_evaluated += 2 * (b or self.e.n_slots)
            self.e.launches += 2
        return g

    def _run_dedup(self, n):
        if self.use_graph and not self._graphs:  # every variant is captured (and timed) up front, not in the middle of a run
            for b in [None, 0] + self.buckets:
                self._dedup_graph(b)
            if self.force_bucket is None:
                self._calibrate()
        done = 0
        while done < n:
            k = min(self.DEDUP_BLOCK, n - done)
            if len(self._events) >= 2:  # wait for the block before the previous one: its counts are on the host now
                self._events.pop(0).synchronize()
            self._recent = [self._recent[1], int(self._stats_host[0])]
            bucket = self._choose_bucket()
            for i in range(k):
                b = bucket if (bucket or i == 0) else None  # whole-batch mode: count once per block, then the plain graph
                self.last_map = self._map if b else None
                self.rows_evaluated += b or self.e.n_slots
                if not self.use_graph:
                    self._hooked((lambda: self._dedup_iteration(b)) if b is not None else self._iteration)
                else:
                    self._hooked(self._dedup_graph(b).replay)
                self.e.launches += 1
                self.bucket_iterations[bucket] = self.bucket_iterations.get(bucket, 0) + 1
            ev = torch.cuda.Event()
            ev.record()
            self._events.append(ev)
            done += k

    def run_iterations(self, n):
        """n x (network forward over the leaf batch + one fused MCTS kernel launch), as CUDA-graph replays."""
        torch.cuda.nvtx.range_push(f"selfplay:{n} iterations (network + oth_mcts_step)")
        if self.dedup:
            self._run_dedup(n)
            torch.cuda.nvtx.range_pop()
            return
        if self.use_graph and self.graph is None:
            self.graph = self._capture()
        k = self.unroll if (self.graph is not None and self.before_iteration is None and self.after_iteration is None) else 1
        done = 0
        if k > 1:  # short iterations (small batches): several of them per graph launch
            if self._graph_k is None:
                def several():
                    for _ in range(k):
                        self._iteration()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    several()
                self._graph_k = g
            while n - done >= k:
                self._graph_k.replay()
                done += k
            self.e.launches += done
        for _ in range(n - done):
            if self.graph is not None:
                self._hooked(self.graph.replay)
                self.e.launches += 1
            else:
                self._hooked(self._iteration)
        self.rows_evaluated += n * self.e.n_slots
        torch.cuda.nvtx.range_pop()

    def play(self, check_every=64, max_iterations=None):
        """Run until every slot is DONE; returns the drained replay tuples."""
        self.warm_start()
        it = 0
        while True:
            self.run_iterations(check_every)
            it += check_every
            c = self.e.counters()
            if c["errors"]:
                self.e.raise_on_error()
            if c["active"] == 0:
                break
            if max_iterations is not None and it >= max_iterations:
                break
        return self.e.drain()


def split_games(out):
    """Drained output -> the reference's per-game lists of (state int8[8,8], pi f32[65], value float)
    (self_play_worker.py:31,85-86), ordered by game id."""
    games = out["games"].numpy() if hasattr(out["games"], "numpy") else np.asarray(out["games"])
    states = out["states"].numpy()
    pis = out["pis"].numpy()
    values = out["values"].numpy()
    res = []
    for gid, first, n, _w in sorted(map(tuple, games)):
        res.append([(states[first + t].copy(), pis[first + t].copy(), float(values[first + t])) for t in range(n)])
    return res
