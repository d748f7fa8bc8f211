#!/usr/bin/env python
"""bench.py -- MCTS self-play throughput of the B200 engine (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c3|c2] [--impl reference] [--dump-outputs DIR]

A "step" = `iters_per_step` (= num_simulations) engine iterations: one policy/value forward
over the leaf batch of every concurrent game + one launch of the fused MCTS kernel, i.e.
about one move of search for every game.  Games start from the initial position, play
themselves (moves sampled in-kernel, trees re-rooted, finished games emitted and restarted).

One JSON line (rank 0):
  value    whole-job simulations/s, everything resident in HBM, CUDA-graph replay
  e2e      same through the host-facing call: per step H2D of the network weights from pinned
           memory, the iterations, D2H of the step's policy targets / root values and of every
           finished game's replay tuples
  roofline the MCTS kernel against HBM: algorithmic bytes per launch (from the engine's own
           counters, formula in DESIGN.md) / CUDA-event launch duration
  cpu_baseline  the oracle port (C tree/env + the same torch net at batch 1) on the host cores
  aux      config C1: env steps/s of the random-rollout kernel and its INT32 roofline
`--impl reference` times the CPU port alone on the same config (rank 0 only).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (description, net, concurrent games per GPU, sims/move)
    "c4": ("big-model batched self-play, 16384 concurrent games, 400 sims/move", "big", 16384, 400),
    "c3": ("small-model batched self-play, 4096 concurrent games, 200 sims/move", "small", 4096, 200),
    "c2": ("small-model MCTS self-play, 100 sims/move, 1 game", "small", 1, 100),
}
TRAIN_ARGS = {"c_puct": 2.0, "dirichlet_alpha": 1.0, "dirichlet_epsilon": 0.3, "mcts_temperature": 1.0,
              "num_exploratory_moves": 35, "lambda": 0.98}  # train.py:399-423 values


def make_net(kind):
    import torch
    from alphazero_othello_b200.Models import AlphaZeroNet, FastOthelloNet
    torch.manual_seed(0)
    return (AlphaZeroNet(8, 65, 5, 128) if kind == "big" else FastOthelloNet(8, 65)).eval()


# ------------------------------------------------------------------ CPU arm --
def _cpu_worker(job):
    kind, sims, n_search, warm = job
    import numpy as np
    import torch
    torch.set_num_threads(1)
    import oracle as O
    net = make_net(kind)
    ev = O.Evaluator(fn=net.inference)
    g = O.OracleGame()
    noise = np.random.RandomState(os.getpid()).dirichlet([1.0] * 65)
    times = []
    for i in range(warm + n_search):
        m = O.OracleMCTS(TRAIN_ARGS["c_puct"], sims, ev, dirichlet_epsilon=TRAIN_ARGS["dirichlet_epsilon"])
        t0 = time.perf_counter()
        m.search(g.get_initial_state(), 1, noise)
        times.append(time.perf_counter() - t0)
    return times[warm:]


def cpu_port_rate(kind, sims, steps, warm, cores):
    """Oracle port on all host cores: every core runs `steps` searches of `sims` simulations
    (one policy_improve_step each, batch-1 torch CPU forward per simulation as the reference does)."""
    import multiprocessing as mp
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    with mp.get_context("spawn").Pool(cores) as pool:
        t0 = time.perf_counter()
        res = pool.map(_cpu_worker, [(kind, sims, steps, warm)] * cores)
        wall = time.perf_counter() - t0
    per_step = [max(r[i] for r in res) for i in range(steps)]  # slowest core per step
    total = sum(per_step)
    return cores * sims * steps / total, 1e3 * total / steps, wall


def _cpu_env_worker(job):
    seed0, seconds = job
    import oracle as O
    O.random_playout(seed0)  # load the library
    plies = games = 0
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        for k in range(64):
            plies += O.random_playout(seed0 + games + k)[0]
        games += 64
    return plies, games, time.perf_counter() - t0


def cpu_env_rate(cores, seconds=2.0):
    """Config C1 on the host: the oracle's Game-API random playout (legal mask, pick, next state,
    terminal test per ply on int8[8,8] boards) on every core for `seconds`."""
    import multiprocessing as mp
    with mp.get_context("spawn").Pool(cores) as pool:
        res = pool.map(_cpu_env_worker, [(1000003 * i, seconds) for i in range(cores)])
    return sum(r[0] for r in res) / max(r[2] for r in res), sum(r[1] for r in res)


# ------------------------------------------------- the reference itself -----
# baseline/_ref/ holds the reference's own, unmodified hot-path sources (tools/stage_reference.sh; git-ignored, ships
# to the GPU box).  The arm below drives them exactly as Trainer.collect_self_play_games does (train.py:199-225): a
# spawn Pool of one process per host core, initialised by the reference's eval._worker_init, each task one
# one_self_play((board_size, args, (policy_class, policy_config, state_dict), cache)) with the default num_threads (4)
# and OMP_NUM_THREADS=1 (MCTS_model.py:3).  A whole game at 400 simulations x ~60 plies takes minutes per core, so a
# task is stopped after a fixed number of plies: two counting wrappers are put around MCTS._simulate (simulations
# completed) and MCTS.policy_improve_step (plies searched; raises after the budget) -- the reference's code is not edited.
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
REF_PLIES_PER_STEP = {"c4": 2, "c3": 6, "c2": 12}


def reference_available():
    return os.path.exists(os.path.join(REF_DIR, "self_play_worker.py"))


class _PlyBudget(Exception):
    pass


_REF = {}


def _ref_worker_init(seed_base):
    os.environ["OMP_NUM_THREADS"] = "1"
    sys.dont_write_bytecode = True
    sys.path.insert(0, REF_DIR)
    import MCTS_model
    import self_play_worker
    import eval as ref_eval
    ref_eval._worker_init(seed_base)  # the reference's own per-process seeding (eval.py:77-84)
    st = {"sims": 0, "plies": 0, "budget": 1 << 30}
    sim, pis = MCTS_model.MCTS._simulate, MCTS_model.MCTS.policy_improve_step

    def counted_simulate(self, root):
        r = sim(self, root)
        st["sims"] += 1
        return r

    def budgeted_pis(self, init_state, init_player, temp=1):
        if st["plies"] >= st["budget"]:
            raise _PlyBudget()
        st["plies"] += 1
        return pis(self, init_state, init_player, temp=temp)

    MCTS_model.MCTS._simulate, MCTS_model.MCTS.policy_improve_step = counted_simulate, budgeted_pis
    _REF.update(st=st, one_self_play=self_play_worker.one_self_play)


def _ref_task(job):
    args_tuple, plies = job
    st = _REF["st"]
    st.update(sims=0, plies=0, budget=plies)
    t0 = time.perf_counter()
    try:
        _REF["one_self_play"](args_tuple)  # returns only if the game ended inside the budget
    except _PlyBudget:
        pass
    return st["sims"], st["plies"], time.perf_counter() - t0


def reference_rate(workload, steps, warm, cores):
    """The unmodified reference's one_self_play on all host cores.  Returns (sims/s, ms per step, description)."""
    import multiprocessing as mp
    desc, kind, G, sims = WORKLOADS[workload]
    plies = REF_PLIES_PER_STEP[workload]
    os.environ["OMP_NUM_THREADS"] = "1"
    sys.path.insert(0, REF_DIR)
    try:
        import torch
        import Models as RefModels  # baseline/_ref/Models.py
        torch.manual_seed(0)
        net = RefModels.AlphaZeroNet(8, 65, 5, 128) if kind == "big" else RefModels.FastOthelloNet(8, 65)
        policy_state = (net.__class__, net.get_config(), net.state_dict())
    finally:
        sys.path.remove(REF_DIR)
    args = dict(TRAIN_ARGS, num_simulations=sims)  # no "num_threads": the reference's default of 4 applies
    job = ((8, args, policy_state, None), plies)
    per_step = []
    with mp.get_context("spawn").Pool(cores, initializer=_ref_worker_init, initargs=(12345,)) as pool:
        for i in range(warm + steps):
            t0 = time.perf_counter()
            res = pool.map(_ref_task, [job] * cores, chunksize=1)
            per_step.append((sum(r[0] for r in res), time.perf_counter() - t0))
    timed = per_step[warm:]
    total_sims, total_s = sum(s for s, _ in timed), sum(t for _, t in timed)
    sample = (f"per step every one of {cores} spawn-Pool processes runs the unmodified reference one_self_play "
              f"(baseline/_ref, default num_threads=4, OMP_NUM_THREADS=1, f32 torch CPU network at batch 1) for the first "
              f"{plies} plies of a game ({sims} simulations each); step time = wall clock until the slowest process returns")
    return total_sims / total_s, 1e3 * total_s / len(timed), sample


def whole_game_profile(workload):
    """Whole-game throughput with / without evaluation de-duplication: NOT measured in this run (a complete C4 batch takes
    a minute each way) -- read from the committed runs of tools/full_games.py."""
    out = {}
    for dd in (1, 0):
        p = os.path.join(ROOT, "profiles", f"r02_full_games_{workload}_dedup{dd}.json")
        if os.path.exists(p):
            d = json.load(open(p))
            out["dedup_on" if dd else "dedup_off"] = {"complete_games": d["complete_games"], "seconds": d["seconds"], "sims_per_s": d["sims_per_s"],
                                                      "positions_per_s": d["positions_per_s"]}
    if out:
        out["source"] = f"committed runs profiles/r02_full_games_{workload}_dedup{{1,0}}.json (tools/full_games.py; not measured in this run)"
    return out or None


def workload_config(workload, G, sims, iters):
    """What is computed -- identical in the B200 arm and in the reference arm (the driver compares the two)."""
    node_cap = max(2048, 48 * sims + 1024)
    return {"workload": f"{workload}: {WORKLOADS[workload][0]}", "net": WORKLOADS[workload][1], "games_per_gpu": G,
            "sims_per_move": sims, "iters_per_step": iters,
            "l2": f"inputs larger than L2: tree arenas {G * 2 * node_cap * 48 >> 20} MiB per GPU vs 126 MB L2 (no flush needed)"
                  if G * 2 * node_cap * 48 > (256 << 20) else
                  "working set fits L2 by construction of this config; L2 is flushed by the network's activations between launches"}


# ---------------------------------------------------------------- utilities --
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.p = index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) > 3 + j and r[3 + j].startswith("Active") for r in self.rows)]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "", 1).isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}


DUMP_LIMIT = 64 * 10**6


def dump_outputs(path, arrays, limit=DUMP_LIMIT):
    """Write every float array of ``arrays`` as ``path/<name>.npy``.  If together they would exceed ``limit`` bytes, every
    array keeps the same fraction of its rows, a sample drawn with a fixed seed from its row count (the kept row indices
    go to ``<name>_rows.npy``), so that two runs with the same arguments write the same rows."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    limit -= 2 * 128 * len(arrays)  # .npy headers of the data and row-index files
    need = sum(v.nbytes + 8 * len(v) for v in arrays.values())
    for name, v in arrays.items():
        assert v.dtype in (np.float32, np.float64), name
        if need > limit and len(v):
            rows = np.sort(np.random.default_rng(0).choice(len(v), max(1, len(v) * limit // need), replace=False))
            np.save(os.path.join(path, f"{name}_rows.npy"), rows.astype(np.float64))
            v = v[rows]
        np.save(os.path.join(path, f"{name}.npy"), v)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


NET_FLOP_PER_EVAL = {"big": 188.99e6, "small": 15.29e6}  # forward MACs x 2 per position (SURVEY 8d)


def network_roofline(kind, evals_per_s, n_gpus=1):
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak, src = 1370.8, "fallback"
    if os.path.exists(p):
        d = json.load(open(p))
        peak, src = float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", peak))), "measured sustained (MEASURED_PEAKS.json)"
    peak *= n_gpus
    ach = evals_per_s * NET_FLOP_PER_EVAL[kind] / 1e12
    return {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "peak_source": src,
            "what": "policy/value network forward (cuDNN/cuBLAS via PyTorch, outside this repo's kernels): evaluations/s x FLOP per evaluation"}


def algorithmic_bytes(d, n_slots, launches, kernel="both"):
    """HBM bytes the MCTS kernels must move for the work the counters record (DESIGN.md 'Kernel roofline'):
    kernel = "step" (k_mcts_step), "move" (k_mcts_move: policy target, re-rooting copy) or "both"."""
    depth_nodes = d["levels"] + d["sims"]            # path entries = levels descended + the root of every simulation
    b = 0
    b += 32 * d["children"]                          # select: child records scanned (2 x 128-bit per child)
    b += 32 * d["sims"]                              # select: root record
    b += (12 + 12) * depth_nodes                     # backup: N (4 B) + W (8 B) read and written per path node
    b += (4 + 4) * depth_nodes                       # path spilled to HBM across the network call, read back
    b += d["evals"] * (16 + 16 + 32 + 8)             # leaf board (select + expand), leaf record, first_child/meta update
    b += d["evals"] * (256 + 260 + 4)                # network input plane written, priors + value read
    b += 48 * d["nodes"]                             # expansion: child record + child board written
    b += 2 * 64 * n_slots * launches                 # per-slot control block read and written every launch
    if kernel in ("both", "move"):
        mv = (48 + 48) * d["copied"]                 # re-root: kept subtree read and written
        mv += d["moves"] * (32 * 12 + 260 + 32 + 16)  # policy target: root children, trajectory row
        if kernel == "move":
            return mv + n_slots * launches           # + the move-flag byte per slot per launch
        b += mv
    return b


def measure_kernel_roofline(eng, run, ev, iters, workload, per_iteration_ms, games_overridden=False):
    """Roofline block of the MCTS kernels for the pipeline in `run`: an un-graphed pass of `iters` iterations of the same
    pipeline in which the library records CUDA events around the step kernel and around the move kernel of every launch
    (othello_b200_experimental.h, per-engine handle), algorithmic bytes from the engine's own counters, the streaming
    peak from MEASURED_PEAKS.json and the random-access rate measured live."""
    import ctypes as C
    import torch
    from alphazero_othello_b200 import _lib
    dev, G, lanes = eng.device, eng.n_slots, int(eng.cfg.lanes)
    torch.cuda.synchronize(dev)
    c0 = eng.counters()
    gap_cycles = int(float(os.environ.get("OTH_BENCH_GAP_US", "0")) * 1400)
    eng.profile_begin(iters)
    for i in range(iters):
        if run.fused:  # same launch as in the timed region: softmax / tanh fused into the step kernel
            lg, vp = ev.raw(eng.nn_input)
            if gap_cycles:  # experiment: idle gap between the network and the step kernel
                torch.cuda._sleep(gap_cycles)
            eng.step_fused(lg, vp)
        else:
            ev(eng.nn_input, eng.priors, eng.values)
            eng.step()
    kms_seq, mms_seq = eng.profile_end()
    torch.cuda.synchronize(dev)
    assert len(kms_seq) == iters
    c1 = eng.counters()
    dk = {k: c1[k] - c0[k] for k in c1}
    if os.environ.get("OTH_BENCH_DUMP_LAUNCHES"):
        json.dump({"step_ms": kms_seq, "move_ms": mms_seq}, open(os.environ["OTH_BENCH_DUMP_LAUNCHES"], "w"))
    kms = sorted(kms_seq)
    k_avg = sum(kms) / len(kms)
    alg = algorithmic_bytes(dk, G, iters, "step") / iters
    peak, peak_src = measured_peaks()
    achieved = alg / (k_avg * 1e-3) / 1e9
    mms = sorted(mms_seq)
    m_avg = sum(mms) / len(mms)
    alg_move = algorithmic_bytes(dk, G, iters, "move") / iters
    # what HBM delivers for the tree's access pattern: independent random 64-byte reads over a
    # footprint the size of the arenas (row-activation / TLB bound, far below the streaming copy peak)
    rnd_gbs, rnd_ms = C.c_double(0), C.c_float(0)
    foot = min(max(eng.buf_bytes[0] + eng.buf_bytes[1], 1 << 30), 24 << 30)
    if _lib.lib().oth_host_random_read_probe(foot, 64, C.byref(rnd_gbs), C.byref(rnd_ms)) != 0:
        rnd_gbs.value = 0.0
    # dram__bytes_read+write per launch: NOT measured in this run -- taken from the committed `ncu --set full` capture of this config
    traffic, traffic_src = None, None
    for tag in ("r02", "r01"):
        prof = os.path.join(ROOT, "profiles", f"{tag}_mcts_step_{workload}_l{lanes}.json")
        if os.path.exists(prof) and not games_overridden:
            traffic = json.load(open(prof)).get("dram_bytes_per_launch")
            traffic_src = f"committed ncu capture profiles/{os.path.basename(prof)} (not measured in this run)"
            break
    eng.drain(to_host=False)
    # what a CUDA-event pair with NOTHING between them reads on this stream: part of every per-launch figure above
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(65)]
    for e in evs:
        e.record()
    torch.cuda.synchronize(dev)
    ovh = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(64))[32]
    move_kernel = "k_mcts_move_list (due list)" if eng.cfg.move_launch else "k_mcts_move (flag scan)"
    return {"bound": "hbm", "kernel": f"k_mcts_step{'_fused' if run.fused else ''}<{lanes}>", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": alg, "launch_ms_avg": k_avg, "launch_ms_median": kms[len(kms) // 2], "launch_ms_max": kms[-1],
            "launch_ms_p90": kms[int(len(kms) * 0.9)],
            "bytes_per_sim": algorithmic_bytes(dk, G, iters) / max(dk["sims"], 1),
            "random_access": {"peak": rnd_gbs.value, "unit": "GB/s", "frac": achieved / rnd_gbs.value if rnd_gbs.value else None,
                              "how": f"measured live: independent random 64-byte reads over {foot >> 20} MiB (oth_host_random_read_probe)"},
            "move_kernel": {"kernel": move_kernel + ": policy target, move sampling, re-rooting copy, game hand-off",
                            "launch_ms_avg": m_avg, "launch_ms_median": mms[len(mms) // 2], "launch_ms_max": mms[-1],
                            "note": "runs after every step kernel; in most launches no move is due (median), the copy work sits in "
                                    "the launch per move where the in-step games all re-root (max)",
                            "algorithmic_bytes_per_launch": alg_move,
                            "achieved": alg_move / (m_avg * 1e-3) / 1e9, "frac": alg_move / (m_avg * 1e-3) / 1e9 / peak,
                            "random_access_frac": alg_move / (m_avg * 1e-3) / 1e9 / rnd_gbs.value if rnd_gbs.value else None},
            "kernel_share_of_iteration": (k_avg + m_avg) / per_iteration_ms,
            "event_pair_overhead_ms": ovh,
            "kernel_share_of_iteration_net_of_event_overhead": max(k_avg + m_avg - 2 * ovh, 0.0) / per_iteration_ms,
            "event_pair_overhead_note": "an empty CUDA-event pair on this stream reads event_pair_overhead_ms (measured live, median of "
                                        "64); every per-launch figure above includes it once, kernel_share_of_iteration twice"}


# -------------------------------------------------------------- B200 arm ----
def run_b200(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    from alphazero_othello_b200 import _lib
    from alphazero_othello_b200.Models import fold_for_inference, refold_
    from alphazero_othello_b200.engine import BatchedPolicy, MctsEngine, SelfPlayRunner

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=120))
    desc, kind, G, sims = WORKLOADS[a.workload]
    if a.games:
        G = a.games
    iters = a.iters_per_step or sims
    args = dict(TRAIN_ARGS, num_simulations=sims)

    if os.environ.get("OTH_NO_GRAPH_FUSION"):
        from alphazero_othello_b200 import Models
        Models._FusedConv.graph_fusion = False
    net = make_net(kind)
    # host copy of the weights (pinned), as Trainer.collect_self_play_games ships them (train.py:207-217)
    flat_host = torch.cat([p.detach().reshape(-1) for p in net.state_dict().values() if p.dtype.is_floating_point]).pin_memory()
    net = net.to(dev)
    flat_dev = torch.empty_like(flat_host, device=dev)

    folded = None

    def load_weights():  # H2D (+ NCCL broadcast from rank 0 when sharded) and re-fold in place
        flat_dev.copy_(flat_host, non_blocking=True)
        if world > 1 and not os.environ.get("OTH_BENCH_NO_BCAST"):
            dist.broadcast(flat_dev, 0)
        off = 0
        for p in net.state_dict().values():
            if p.dtype.is_floating_point:
                n = p.numel()
                p.copy_(flat_dev[off:off + n].view_as(p))
                off += n
        return fold_for_inference(net, torch.bfloat16) if folded is None else refold_(folded, net)

    folded = load_weights()
    ev = BatchedPolicy(folded, dev, torch.float32)
    eng = MctsEngine(G, args, self_play=True, eval_kind=_lib.EVAL_EXTERNAL, games_per_slot=-1, device=dev, seed=a.seed,
                     game_id_base=rank * G, game_id_stride=G * world, lanes=a.lanes or None, max_inline_sims=a.max_inline,
                     out_pos_cap=G * 160, out_game_cap=2 * G + 64, node_cap=a.node_cap or None,
                     move_launch=None if a.move_launch < 0 else a.move_launch)
    a.lanes = int(eng.cfg.lanes)
    run = SelfPlayRunner(eng, ev, use_graph=not a.no_graph, dedup="auto" if a.dedup else False)
    run.warm_start()

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    step_ms_log = []

    def timed(fn, steps):
        barrier()
        c0 = eng.counters()
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        e0, e1 = marks[0], marks[-1]
        e0.record()
        for i in range(steps):
            fn()
            marks[i + 1].record()
        barrier()
        ms = e0.elapsed_time(e1)
        step_ms_log.append([marks[i].elapsed_time(marks[i + 1]) for i in range(steps)])
        c1 = eng.counters()
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms, {k: c1[k] - c0[k] for k in c1}

    def total(x):
        if world == 1:
            return x
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        dist.all_reduce(t)
        return float(t)

    n_plain = [0]

    def plain_step():
        run.run_iterations(iters)
        n_plain[0] += 1
        if n_plain[0] % 32 == 0:  # long runs: finished games leave the output ring (it holds ~2 rounds of games)
            eng.drain(to_host=False)

    for _ in range(a.warmup):
        plain_step()
    eng.drain(to_host=False)

    clocks = ClockSampler(local)
    clocks.start()
    rows0 = run.rows_evaluated
    b0 = dict(run.bucket_iterations) if run.dedup else {}
    ms, d = timed(plain_step, a.steps)
    rows_timed = run.rows_evaluated - rows0
    buckets_timed = dict(run.bucket_iterations) if run.dedup else None
    # this repo's de-duplication kernels in the timed region: 4 per compacted iteration (keys, heads, emit, planes), 3 per
    # counting iteration (one per 16-iteration block in whole-batch mode); the CUB sort / scan between them are library code
    dedup_launches = sum(4 * (v - b0.get(k, 0)) for k, v in (buckets_timed or {}).items() if k) + \
        3 * (((buckets_timed or {}).get(0, 0) - b0.get(0, 0)) // 16)
    clk = clocks.stop()
    eng.raise_on_error()
    sims_total = total(d["sims"])
    moves_total = total(d["moves"])
    evals_total = total(d["evals"])
    rows_total = total(rows_timed)  # (collective: every rank)
    value = sims_total / (ms * 1e-3)
    eng.drain(to_host=False)

    # ---- e2e: weights H2D (+broadcast), iterations, D2H of targets and finished games (+gather)
    pin_counts = torch.empty((G, 65), dtype=torch.int32).pin_memory()
    pin_rootv = torch.empty((G,), dtype=torch.float64).pin_memory()
    io = {"h2d": 0, "d2h": 0}

    trace = [] if os.environ.get("OTH_BENCH_E2E_TRACE") else None  # diagnosis: synchronised stage times (perturbs e2e)

    def mark(tag):
        if trace is not None:
            torch.cuda.synchronize(dev)
            trace.append((tag, time.perf_counter()))

    def e2e_step():
        mark("start")
        load_weights()
        if os.environ.get("OTH_BENCH_SYNC_W"):
            torch.cuda.synchronize(dev)
        mark("weights")
        io["h2d"] += flat_host.numel() * 4
        run.run_iterations(iters)
        mark("iterations")
        st = eng.root_stats()
        pin_counts.copy_(st["counts"], non_blocking=True)
        pin_rootv.copy_(st["root_value"], non_blocking=True)
        out = eng.drain(to_host=True)
        io["d2h"] += pin_counts.numel() * 4 + pin_rootv.numel() * 8 + sum(v.numel() * v.element_size() for v in out.values())
        if world > 1:  # replay gather to rank 0 (sizes, then padded payload)
            n = torch.tensor([out["values"].numel()], device=dev)
            ns = [torch.zeros_like(n) for _ in range(world)]
            dist.all_gather(ns, n)
            mx = max(int(x) for x in ns)
            if mx:
                pay = torch.zeros((mx, 65 + 4), dtype=torch.float32, device=dev)
                k = out["values"].numel()
                if k:
                    pay[:k, :65] = out["pis"].to(dev)
                    pay[:k, 65] = out["values"].to(dev).float()
                    pay[:k, 66:68] = out["boards"].to(dev).view(torch.float32).view(k, 4)[:, :2]
                lst = [torch.zeros_like(pay) for _ in range(world)] if rank == 0 else None
                dist.gather(pay, lst, 0)
        torch.cuda.synchronize(dev)
        mark("outputs")

    # the e2e window is the value window: the games are started again and warmed up through the same plies, now with
    # the host-facing work of every step (weights in, targets and finished games out) inside
    run.warm_start()
    for _ in range(a.warmup):
        e2e_step()
    if world > 1:  # NCCL sets up the gather's send/recv connections on first use (~0.25 s at 2 ranks, >1 s at 8): the first
        pay = torch.zeros((1, 69), dtype=torch.float32, device=dev)  # games end at move 9, so do it before the timed region
        dist.gather(pay, [torch.zeros_like(pay) for _ in range(world)] if rank == 0 else None, 0)
        torch.cuda.synchronize(dev)
    io["h2d"] = io["d2h"] = 0
    ms2, d2 = timed(e2e_step, a.steps)
    e2e_value = total(d2["sims"]) / (ms2 * 1e-3)
    if a.dump_outputs and rank == 0:
        # what the last timed step handed to the host for every game: root visit counts (the policy targets) and root value.
        # The replay tuples of the games that finished in that step are left out: how many finish varies from run to run and
        # is zero in the opening plies the default window covers.  Two runs of one build differ by a few visits per game:
        # the de-duplication buckets and the cuDNN plans are chosen by timing, and the network's bf16 results depend on the
        # batch shape
        dump_outputs(a.dump_outputs, {"root_visit_counts": pin_counts.numpy().astype(np.float32),
                                      "root_value": pin_rootv.numpy().copy()})
    if trace:
        print(f"rank {rank} e2e stages (ms):", [(b[0], round((b[1] - a[1]) * 1e3, 1)) for a, b in zip(trace, trace[1:])], file=sys.stderr)

    roof = measure_kernel_roofline(eng, run, ev, iters, a.workload, per_iteration_ms=ms / a.steps / iters, games_overridden=bool(a.games))

    from alphazero_othello_b200 import _cudnn_fused
    fused_plans = _cudnn_fused.chosen_plans()
    out = None
    if rank == 0:
        out = {
            "metric": "MCTS simulations/s (self-play, one network evaluation per simulation)", "value": value,
            "unit": "sims/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32/f64 search (u64 boards), bf16 network",
            "data": "synthetic: self-play from the initial position, random-init weights (torch.manual_seed(0))",
            "config": workload_config(a.workload, G, sims, iters),
            "per_step_ms": step_ms_log[0],
            "engine": {"lanes": a.lanes, "cuda_graph": not a.no_graph, "move_launch": int(eng.cfg.move_launch),
                       "evaluation_dedup": {"enabled": bool(run.dedup), "buckets": getattr(run, "buckets", None),
                                            "iteration_ms_by_variant": {str(k): v for k, v in getattr(run, "iteration_ms", {}).items()} or None,
                                            "iterations_by_bucket_since_start": buckets_timed,
                                            "network_rows_per_evaluation_timed": rows_timed / max(evals_total / world, 1),
                                            "what": "the network runs on the DISTINCT pending positions of a batch (oth_mcts_dedup), bucketed "
                                                    "batch sizes; every simulation still gets the evaluation of its own leaf. Games start "
                                                    "together, so the saving sits in the first plies (per_step_ms); aux.without_dedup is the "
                                                    "same window with it off",
                                            "whole_games": whole_game_profile(a.workload)},
                       "arena_mib": eng.buf_bytes[0] + eng.buf_bytes[1] >> 20,
                       "sharding": "games by id, no collective on the search path",
                       "network_twin": {"residual_conv": "one cuDNN graph relu(bias(conv+residual)) per block" if fused_plans
                                        else "cuDNN conv + k_bias_add_relu_bf16", "cudnn_plans": fused_plans},
                       "roofline_timing": "CUDA events recorded by the library on the launching stream around k_mcts_step and around "
                                          "k_mcts_move of every launch (oth_mcts_profile_create / _read, othello_b200_experimental.h) in an un-graphed pass of "
                                          "iters_per_step iterations of the same pipeline right after the timed region "
                                          "(events cannot be recorded inside the replayed graph)"},
            "positions_per_s": moves_total / (ms * 1e-3),
            "e2e": {"value": e2e_value, "unit": "sims/s", "h2d_bytes_per_step": io["h2d"] // a.steps,
                    "d2h_bytes_per_step": io["d2h"] // a.steps, "ms_per_step": ms2 / a.steps,
                    "per_step_ms": step_ms_log[1],
                    "includes": "weights H2D from pinned host (+NCCL broadcast if sharded), BN re-fold, "
                                "D2H of policy targets/root values and finished games' replay tuples (+gather to rank 0); "
                                "same plies as `value` (games restarted, same warm-up)"},
            # this repo's kernels per iteration: k_mcts_step, k_mcts_move, k_stem_im2col_bf16 and -- only when the
            # residual convolutions do not run as one cuDNN graph -- one k_bias_add_relu_bf16 per residual block
            "gpu_launches": a.steps * iters * (3 + (0 if fused_plans else (5 if kind == "big" else 1))) + dedup_launches,
            "clocks": clk,
            "roofline": roof,
            # the step's dominant cost is the (library) network: its share of the dense bf16 peak sustained by cuBLAS on this pool
            # FLOPs the network actually executed: rows evaluated (bucket sizes when de-duplicated), not simulations
            "network_roofline": network_roofline(kind, rows_total / (ms * 1e-3), world),
            "search_counters_per_step": {k: d[k] / a.steps for k in ("sims", "evals", "terminal_sims", "moves", "games", "nodes", "copied", "levels", "children")},
        }
    if world > 1:
        if not a.no_aux:
            env_aux = aux_env_sharded(dev, rank, world)
            if rank == 0:
                out["aux"] = env_aux
        dist.barrier()
        dist.destroy_process_group()
    return out, dev


def aux_selfplay_rate(dev, workload, steps=8, warm=3, dtype=None, tf32=False, iters=None, with_roofline=False, dedup="auto"):
    """Resident self-play throughput of another BASELINE config on the same GPU (same pipeline as the
    headline: network twin + oth_mcts_step_fused replayed as a CUDA graph; a step = sims/move iterations).
    dtype torch.float32 (+ tf32) runs the float32 twin of the network: the same-precision comparator of the headline."""
    import torch
    from alphazero_othello_b200 import _lib
    from alphazero_othello_b200.Models import fold_for_inference
    from alphazero_othello_b200.engine import BatchedPolicy, MctsEngine, SelfPlayRunner
    desc, kind, G, sims = WORKLOADS[workload]
    iters = iters or sims
    args = dict(TRAIN_ARGS, num_simulations=sims)
    dtype = dtype or torch.bfloat16
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    if dtype == torch.float32:
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = bool(tf32)
    try:
        eng = MctsEngine(G, args, self_play=True, eval_kind=_lib.EVAL_EXTERNAL, games_per_slot=-1, device=dev,
                         out_pos_cap=G * 80 + 4096, out_game_cap=G + 64)
        ev = BatchedPolicy(fold_for_inference(make_net(kind).to(dev), dtype), dev, torch.float32)
        run = SelfPlayRunner(eng, ev, dedup=dedup)
        run.warm_start()
        for _ in range(warm):
            run.run_iterations(iters)
        torch.cuda.synchronize(dev)
        c0 = eng.counters()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            run.run_iterations(iters)
        e1.record()
        torch.cuda.synchronize(dev)
        c1 = eng.counters()
        eng.raise_on_error()
        ms = e0.elapsed_time(e1)
        sims_s = (c1["sims"] - c0["sims"]) / (ms * 1e-3)
        out = {"workload": f"{workload}: {desc}", "net": kind, "network_dtype": str(dtype).replace("torch.", "") + ("+tf32" if dtype == torch.float32 and tf32 else ""),
               "sims_per_s": sims_s, "positions_per_s": (c1["moves"] - c0["moves"]) / (ms * 1e-3), "steps": steps, "warmup": warm,
               "iters_per_step": iters, "ms_per_step": ms / steps, "lanes": int(eng.cfg.lanes), "evaluation_dedup": bool(run.dedup),
               "network_roofline": network_roofline(kind, (c1["evals"] - c0["evals"]) / (ms * 1e-3)) if dtype == torch.bfloat16 else None}
        if with_roofline:
            out["roofline"] = measure_kernel_roofline(eng, run, ev, min(iters, 200), workload, per_iteration_ms=ms / steps / iters)
        return out
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def aux_one_self_play(dev):
    """Config C2 through the drop-in surface: ``one_self_play((8, args, (class, config, state_dict), None))`` exactly as
    train.py:199-225 calls the reference's worker -- one whole game, 100 simulations per move, the float32 small network
    evaluated on the GPU at batch 1 by the drop-in MCTS class (one CUDA-graph replay per simulation)."""
    import numpy as np
    import torch
    from alphazero_othello_b200.Models import FastOthelloNet
    from alphazero_othello_b200.self_play_worker import one_self_play
    desc, kind, G, sims = WORKLOADS["c2"]
    args = dict(TRAIN_ARGS, num_simulations=sims)
    torch.manual_seed(0)
    net = FastOthelloNet(8, 65).eval()
    state = (FastOthelloNet, net.get_config(), net.state_dict())
    best = None
    for rep in range(2):
        np.random.seed(rep)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        traj = one_self_play((8, args, state, None))
        dt = time.perf_counter() - t0
        if best is None or dt / len(traj) < best[0] / best[1]:
            best = (dt, len(traj))
    return {"workload": f"c2: {desc} -- through the drop-in one_self_play (host loop over the GPU tree, float32 network, whole game, "
                        "engine construction and graph capture included)",
            "seconds": best[0], "plies": best[1], "sims_per_s": best[1] * sims / best[0], "positions_per_s": best[1] / best[0]}


def aux_public_api(dev, workload="c3"):
    """The call a user of the reference makes, end to end: ``collect_self_play_games(policy, args, n_games)`` with the
    policy's weights on the HOST, every game played to the end, the per-game lists of (int8[8,8], float32[65], float)
    back on the host (train.py:199-225 + 136-140).  Wall clock, everything included (engine allocation, BN folding,
    cuDNN plan selection, graph capture, ragged tail of the longest games, D2H, splitting into Python lists)."""
    import torch
    from alphazero_othello_b200.self_play_worker import collect_self_play_games
    desc, kind, G, sims = WORKLOADS[workload]
    args = dict(TRAIN_ARGS, num_simulations=sims)
    net = make_net(kind)  # CPU module, as the trainer holds it
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    games = collect_self_play_games(net, args, G, n_slots=G, device=dev, seed=1)
    dt = time.perf_counter() - t0
    npos = sum(len(g) for g in games)
    return {"workload": f"{workload}: {desc} -- {G} complete games through collect_self_play_games (host weights in, host lists out)",
            "seconds": dt, "games": len(games), "positions": npos, "positions_per_s": npos / dt, "sims_per_s": npos * sims / dt}


def aux_env_sharded(dev, rank, world):
    """Config C1 over all ranks: every rank rolls out its own 2^22 games (ids offset by rank); whole-job
    plies / max-over-ranks device time.  No collective on the path -- the all-reduce only gathers the timing."""
    import torch
    import torch.distributed as dist
    from alphazero_othello_b200.envs.othello import BatchedOthello
    env = BatchedOthello(dev)
    n = 1 << 22
    best = None
    for rep in range(4):
        torch.cuda.synchronize(dev)
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = env.rollout(n, seed=rep, game_id_base=rank * n)
        e1.record()
        torch.cuda.synchronize(dev)
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        p = torch.tensor([float(int(r["counters"][0]))], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(p)
        if rep and (best is None or float(t) < best[0]):
            best = (float(t), float(p))
    return {"workload": f"c1: Othello 8x8 random-policy rollouts, 2^22 games per GPU x {world} GPUs",
            "env_steps_per_s": best[1] / (best[0] * 1e-3), "kernel_ms_max_over_ranks": best[0], "plies": best[1]}


def aux_env(dev):
    """Config C1: random-rollout env throughput + INT32 roofline (rank 0, N=1)."""
    import ctypes as C
    import torch
    from alphazero_othello_b200 import _lib
    from alphazero_othello_b200.envs.othello import BatchedOthello
    env = BatchedOthello(dev)
    n = 1 << 22
    best = None
    for rep in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        r = env.rollout(n, seed=rep)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        if rep and (best is None or ms < best[0]):
            best = (ms, int(r["counters"][0]))
    ips, kms = C.c_double(0), C.c_float(0)
    _lib.check(_lib.lib().oth_host_int32_peak(C.byref(ips), C.byref(kms)))
    # e2e through the host-buffer C-ABI call (results copied back to host arrays)
    import numpy as np
    sc, pl = np.empty(n, np.int32), np.empty(n, np.int32)
    tot, k2 = C.c_ulonglong(0), C.c_float(0)
    t0 = time.perf_counter()
    _lib.check(_lib.lib().oth_host_rollout(9, 0, n, sc.ctypes.data, pl.ctypes.data, None, 0, None, None, C.byref(tot), C.byref(k2)))
    t1 = time.perf_counter()
    steps_s = best[1] / (best[0] * 1e-3)
    # instructions per ply and the ALU-pipe utilisation are NOT measured in this run: they come from the committed
    # `ncu --set full` capture of the same kernel and size (the survey's estimate was 600 instructions per ply)
    instr, ncu = 600.0, {"instr_per_ply_source": "SURVEY 8(d) estimate"}
    prof = os.path.join(ROOT, "profiles", "r01_rollout_c1.json")
    if os.path.exists(prof):
        pj = json.load(open(prof))
        instr = float(pj["thread_instructions_per_ply"])
        ncu = {"instr_per_ply_source": "committed ncu capture profiles/r01_rollout_c1.json (smsp__inst_executed x threads / plies)",
               "alu_pipe_frac": pj["alu_pipe_pct_of_peak"] / 100.0,
               "alu_pipe_frac_source": "committed ncu capture profiles/r01_rollout_c1.json "
                                       "(sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active; the kernel's binding pipe)"}
    return {"workload": "c1: Othello 8x8 random-policy rollouts, 2^22 games", "env_steps_per_s": steps_s, "kernel_ms": best[0],
            "plies": best[1], "e2e_env_steps_per_s": tot.value / (t1 - t0), "e2e_d2h_bytes": n * 8,
            "int32_roofline": {"bound": "int32-alu", "instr_per_ply": instr, "achieved_ginstr_s": steps_s * instr / 1e9,
                               "mixed_pipe_probe_peak_ginstr_s": ips.value / 1e9, "frac_of_mixed_pipe_probe": steps_s * instr / ips.value,
                               "mixed_pipe_probe": "measured live: LOP3+IADD3 probe kernel (oth_host_int32_peak); it issues to the ALU AND "
                                                   "FMA pipes, which k_rollout's shift/logic mix cannot -- an upper bound no shift-heavy kernel reaches",
                               **ncu}}


def aux_env_step_api(dev):
    """Stepwise env API on packed boards (oth_legal_moves / oth_step): HBM-bound, 24 / 42 bytes per position."""
    import torch
    from alphazero_othello_b200.envs.othello import BatchedOthello
    env = BatchedOthello(dev)
    n = 1 << 24
    own, opp = env.initial(n)
    gen = torch.Generator(device=dev)
    gen.manual_seed(0)
    for ply in range(16):  # mid-game positions: 16 plies, each the r-th lowest legal square (r random per game)
        lm = env.legal_moves(own, opp)
        r = torch.randint(0, 4, (n,), device=dev, generator=gen)
        pick = lm
        for _ in range(3):  # clear up to r lowest bits, keeping at least one
            nxt = pick & (pick - 1)
            pick = torch.where((r > 0) & (nxt != 0), nxt, pick)
            r = r - 1
        bit = pick & (-pick)
        act = torch.where(lm == 0, torch.full_like(bit, 64), (torch.log2(bit.double().abs()) + 0.5).long() % 64)
        act = torch.where((bit < 0) & (lm != 0), torch.full_like(act, 63), act).to(torch.uint8)
        own, opp, _, fl = env.step(own, opp, act)
        assert int((fl & 1).sum()) == 0
    peak, _ = measured_peaks()
    out = {}
    for name, fn, nbytes in (("legal_moves", lambda: env.legal_moves(own, opp), 24), ("step", lambda: env.step(own, opp, act), 42)):
        fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / 5
        out[name] = {"positions_per_s": n / (ms * 1e-3), "ms": ms, "bytes_per_position": nbytes,
                     "hbm_gbs": n * nbytes / (ms * 1e-3) / 1e9, "hbm_frac": n * nbytes / (ms * 1e-3) / 1e9 / peak}
    out["workload"] = f"{n} mid-game positions (16 plies in), packed boards resident in HBM (> L2), includes torch output allocation"
    return out


def aux_search_only(dev, G, sims):
    """Search-only variant (SURVEY 8d) through the PRODUCTION kernel pair: the step kernel with the device hash stub in
    the network's place (cfg.split_stub) + the move kernel, back to back -- exactly one evaluation per slot per launch,
    as behind the network, but with nothing in between."""
    import ctypes as C
    import torch
    from alphazero_othello_b200 import _lib
    from alphazero_othello_b200.engine import MctsEngine
    args = dict(TRAIN_ARGS, num_simulations=sims)
    eng = MctsEngine(G, args, self_play=True, eval_kind=_lib.EVAL_STUB_H, games_per_slot=-1, device=dev, split_stub=True,
                     out_pos_cap=G * 80 + 4096, out_game_cap=G + 64, stub_salt=1)
    eng.reset()
    for _ in range(sims + sims // 2):  # into the second move: trees with re-used subtrees
        eng.step()
    eng.drain(to_host=False)
    torch.cuda.synchronize(dev)
    c0 = eng.counters()
    n = min(sims, 200)
    eng.profile_begin(n)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        eng.step()
    e1.record()
    torch.cuda.synchronize(dev)
    kms, mms = eng.profile_end()
    c1 = eng.counters()
    ms = e0.elapsed_time(e1)
    d = {k: c1[k] - c0[k] for k in c1}
    eng.raise_on_error()
    peak, _ = measured_peaks()
    rnd_gbs, rnd_ms = C.c_double(0), C.c_float(0)
    foot = min(max(eng.buf_bytes[0] + eng.buf_bytes[1], 1 << 30), 24 << 30)
    if _lib.lib().oth_host_random_read_probe(foot, 64, C.byref(rnd_gbs), C.byref(rnd_ms)) != 0:
        rnd_gbs.value = 0.0
    k_avg = sum(kms) / len(kms)
    alg_step = algorithmic_bytes(dict(d, evals=0), G, n, "step") + d["evals"] * (16 + 16 + 32 + 8)  # no network I/O in this variant
    gbs = alg_step / n / (k_avg * 1e-3) / 1e9
    return {"workload": f"search-only: {G} games, {sims} sims/move, k_mcts_step_devstub<{int(eng.cfg.lanes)}> + move kernel, "
                        "one evaluation per slot per launch",
            "sims_per_s": d["sims"] / (ms * 1e-3), "sims_per_s_step_kernel_alone": d["sims"] / n / (k_avg * 1e-3),
            "launch_ms_step_avg": k_avg, "launch_ms_move_avg": sum(mms) / len(mms), "launch_ms_move_max": max(mms),
            "hbm_gbs": gbs, "hbm_frac": gbs / peak, "random_access_gbs": rnd_gbs.value,
            "random_access_frac": gbs / rnd_gbs.value if rnd_gbs.value else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    # defaults = the window the round-1 driver used: plies 5..24 of games that start together.  (A shorter window close to the
    # start would sit in the plies where almost every leaf of a batch is a duplicate -- see per_step_ms / aux.without_dedup.)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--games", type=int, default=0, help="override concurrent games per GPU")
    ap.add_argument("--iters-per-step", type=int, default=0)
    ap.add_argument("--lanes", type=int, default=0, help="threads per game slot: 8 / 16 / 32 (0 = engine default for the slot count)")
    ap.add_argument("--move-launch", type=int, default=-1, help="move kernel: 0 host-launched flag scan, 1 device tail launch (-1 = engine default)")
    ap.add_argument("--max-inline", type=int, default=8)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--node-cap", type=int, default=0, help="experiment: arena size per slot (default 48*sims+1024)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--dedup", type=int, default=1, help="evaluation de-duplication (oth_mcts_dedup): 1 on (default), 0 off")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aux", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write every game's root visit counts and root value from the "
                    "last timed e2e step as DIR/<name>.npy (float32 / float64, at most 64 MB, rank 0)")
    a = ap.parse_args()
    # stdout carries exactly ONE JSON line: everything else this process, its libraries (NCCL prints its
    # version banner to stdout when NCCL_DEBUG is set) and its children write goes to stderr
    result_out = os.fdopen(os.dup(1), "w")
    sys.stdout.flush()
    os.dup2(2, 1)
    a.warmup = max(a.warmup, 3) if a.impl == "b200" else a.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    desc, kind, G, sims = WORKLOADS[a.workload]
    cores = len(os.sched_getaffinity(0))

    if a.impl == "reference":
        if rank != 0:
            return
        iters = a.iters_per_step or sims
        G_ref = a.games or G
        if reference_available() and not os.environ.get("OTH_BENCH_FORCE_PORT"):
            rate, ms_step, sample = reference_rate(a.workload, a.steps, a.warmup, cores)
            ref_kind = "reference"
        else:  # no staged reference on this box: the oracle port (C tree/env + the same torch net at batch 1)
            import oracle
            oracle.lib()
            rate, ms_step, wall = cpu_port_rate(kind, sims, a.steps, a.warmup, cores)
            sample = f"per step every core runs one policy_improve_step of {sims} simulations from the initial position " \
                     f"(batch-1 torch CPU forward per simulation), {cores} processes"
            ref_kind = "port"
        print(json.dumps({
            "impl": "reference", "metric": "MCTS simulations/s (self-play, one network evaluation per simulation)",
            "value": rate, "unit": "sims/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32/f64 search, f32 network (CPU)",
            "data": "synthetic: random-init weights (torch.manual_seed(0))",
            "config": workload_config(a.workload, G_ref, sims, iters),
            "cpu_baseline": {"value": rate, "unit": "sims/s", "cores": cores, "kind": ref_kind, "sample": sample},
            "e2e": {"value": rate, "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}), file=result_out, flush=True)
        return

    out, dev = run_b200(a)
    if rank == 0:
        if world == 1 and not a.no_aux:
            out["aux"] = aux_env(dev)
            import torch
            out["aux"]["search_only"] = aux_search_only(dev, out["config"]["games_per_gpu"], sims)
            out["aux"]["env_step_api"] = aux_env_step_api(dev)
            other = "c3" if a.workload != "c3" else "c4"  # north_star: both architectures, every BASELINE config
            out["aux"]["other_architecture"] = aux_selfplay_rate(dev, other, with_roofline=True)
            out["aux"]["other_architecture_without_dedup"] = aux_selfplay_rate(dev, other, dedup=False)
            if a.workload != "c2":
                out["aux"]["c2_one_game"] = aux_selfplay_rate(dev, "c2", steps=12, warm=3, with_roofline=True)
            out["aux"]["c2_one_self_play_dropin"] = aux_one_self_play(dev)
            # same-precision comparator of the headline: the float32 twin of the same network (TF32 tensor cores, and plain FP32)
            out["aux"]["network_precision"] = {
                "tf32": aux_selfplay_rate(dev, a.workload, steps=2, warm=1, dtype=torch.float32, tf32=True, iters=40, dedup=False),
                "note": "float32 twin of the same network on TF32 tensor cores, every leaf evaluated in its own row (compare with "
                        "aux.without_dedup).  Plain FP32 without tensor cores lands on cuDNN's SIMT kernels: 63 k simulations/s, "
                        "measured once (profiles/r02_bench_c4_1gpu_first.json), not repeated in every run"}
            out["aux"]["public_api_whole_games"] = aux_public_api(dev, "c3")
            if out["engine"]["evaluation_dedup"]["enabled"]:  # the same plies with every leaf evaluated in its own row
                out["aux"]["without_dedup"] = aux_selfplay_rate(dev, a.workload, steps=a.steps, warm=a.warmup, dedup=False)
            import oracle
            oracle.lib()
            rate, games = cpu_env_rate(cores)
            out["aux"]["cpu_env_baseline"] = {"value": rate, "unit": "env steps/s", "cores": cores, "kind": "port",
                                              "sample": f"{games} random playouts (oracle Game-API loop on int8[8,8] boards), {cores} processes x 2 s"}
        if world == 1 and not a.no_cpu_baseline:
            import oracle
            oracle.lib()
            rate, ms_step, wall = cpu_port_rate(kind, sims, 2, 1, cores)
            port = {"value": rate, "unit": "sims/s", "cores": cores, "kind": "port",
                    "sample": f"{cores} processes x 2 searches of {sims} simulations from the initial position "
                              f"(oracle C tree/env + batch-1 torch CPU forward of the {kind} net), {wall:.1f} s wall"}
            if reference_available():
                rate, ms_step, sample = reference_rate(a.workload, 2, 1, cores)
                out["cpu_baseline"] = {"value": rate, "unit": "sims/s", "cores": cores, "kind": "reference", "sample": sample,
                                       "port": port}
            else:
                out["cpu_baseline"] = port
        else:
            out["cpu_baseline"] = None
        print(json.dumps(out), file=result_out, flush=True)


def stop_resource_tracker():
    """The spawn pools of the CPU arms start multiprocessing's resource tracker, which would outlive this process (and
    be left to whatever adopts orphans); stop it and reap it here, so the benchmark leaves no process behind."""
    from multiprocessing import resource_tracker
    resource_tracker._resource_tracker._stop()


if __name__ == "__main__":
    try:
        main()
    finally:
        stop_resource_tracker()
