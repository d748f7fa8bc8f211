"""Throughput of oth_alphabeta on one GPU, and arena wall time of a network against the alpha-beta player.

    python tools/alphabeta_bench.py --out profiles/alphabeta_bench.json

- positions/s and nodes/s at depths 2/4/6/7 (mid-game and late-game roots; 7 = OTH_AB_MAX_DEPTH) and exactly solved
  endgames with 10/11/12 empties (12 = OTH_AB_MAX_EXACT), over 4 096 and 16 384 roots, and over 512 roots (the batch
  an arena ply searches) at depth 7 and 11 and 12 exact empties: CUDA events around whole launches, after one warm-up
  launch of the same shape;
- lane balance, for the roots k_alphabeta searches (all but exact ones with 12+ empties) = sum of nodes / (32 x the
  largest per-lane node count), summed over warps (one warp per root, lane l searches the root actions of rank l and
  l + 32): the share of lane-time that does work.  The split search's lanes share (root action, reply) tasks
  dynamically, so no formula gives their lanes; its cases report launch time, nodes/s and nodes per position;
- wall time of 1 024 arena matches of a FastOthelloNet (100 simulations per move) against depth 4 and depth 6 (exact
  from 10 empties) and depth 7 (exact from 12 empties).
Roots come from uniform-random games played by the library's own rollout kernel (seeded).  The GPU's name and power
limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from alphazero_othello_b200 import _lib  # noqa: E402
from alphazero_othello_b200.alphabeta import AlphaBetaPlayer, search  # noqa: E402


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = out
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"not read: {e}"
    return info


def roots(n, empties, seed):
    """n non-terminal roots with exactly `empties` empty squares, from seeded random games (oth_host_rollout traces)."""
    from alphazero_othello_b200.envs.othello import OthelloGameNew
    env = OthelloGameNew(8)
    L = _lib.lib()
    m = 2 * n + 64
    trace = np.zeros((m, 128), np.uint8)
    _lib.check(L.oth_host_rollout(seed, 0, m, None, None, None, m, trace.ctypes.data_as(C.c_void_p), None, None, None))
    states = np.repeat(env.get_initial_state().reshape(1, 64), m, 0).astype(np.int8)
    players = np.ones(m, np.int8)
    own, opp = [], []
    w = np.uint64(1) << np.arange(64, dtype=np.uint64)
    taken = np.zeros(m, bool)
    for ply in range(128):
        e = (states == 0).sum(1)
        live = trace[:, ply] != 0xFF
        pick = live & ~taken & (e == empties)
        for i in np.nonzero(pick)[0]:
            own.append(((states[i] == players[i]) * w).sum(dtype=np.uint64))
            opp.append(((states[i] == -players[i]) * w).sum(dtype=np.uint64))
        taken |= pick
        if not live.any() or len(own) >= n:
            break
        idx = np.nonzero(live)[0]
        states[idx] = env.next_state_batch(states[idx], trace[idx, ply].astype(np.int32), players[idx]).reshape(-1, 64)
        players[idx] = -players[idx]
    assert len(own) >= n, (len(own), n, empties)
    to = lambda a: torch.from_numpy(np.array(a[:n], np.uint64).view(np.int64)).cuda()
    return to(own), to(opp)


def lane_balance(values, nodes):
    legal = values != _lib.AB_NONE
    rank = np.cumsum(legal, 1) - 1
    lane = np.where(legal, rank % 32, 32)
    per_lane = np.zeros((len(values), 33), np.int64)
    np.add.at(per_lane, (np.repeat(np.arange(len(values)), 65), lane.reshape(-1)), nodes.reshape(-1))
    per_lane = per_lane[:, :32]
    return float(per_lane.sum() / (32 * per_lane.max(1)).sum())


def time_search(own, opp, depth, exact, reps, split):
    search(own, opp, depth, exact)  # warm-up: same shape
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(reps):
        e0.record()
        v, b, nodes = search(own, opp, depth, exact)
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    v, nodes = v.cpu().numpy(), nodes.cpu().numpy()
    n = len(v)
    total = int(nodes.sum())
    t = min(ms) / 1e3
    r = {"positions": n, "depth": depth, "exact_empties": exact, "launch_ms": [round(x, 3) for x in ms],
         "positions_per_s": n / t, "nodes": total, "nodes_per_s": total / t, "nodes_per_position": total / n,
         "mean_root_actions": float((v != _lib.AB_NONE).sum(1).mean())}
    if not split:
        r["lane_balance"] = lane_balance(v, nodes)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/alphabeta_bench.json")
    ap.add_argument("--sizes", default="4096,16384")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--arena-matches", type=int, default=1024)
    ap.add_argument("--arena-sims", type=int, default=100)
    ap.add_argument("--arena-levels", default="4:10,6:10,7:12", help="depth:exact_empties of each arena run")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    res = {"gpu": gpu_info(), "search": [], "arena": []}
    sizes = [int(x) for x in a.sizes.split(",")]
    cases = [("mid-game", 40, d, 0) for d in (2, 4, 6, 7)] + [("late-game", 24, d, 0) for d in (2, 4, 6, 7)] + \
            [("endgame", e, 1, e) for e in (10, 11, 12)]
    arena_batch = [("mid-game", 40, 7, 0)] + [("endgame", e, 1, e) for e in (11, 12)]
    for n, case in [(n, c) for n in sizes for c in cases] + [(512, c) for c in arena_batch]:
        phase, empties, depth, exact = case
        split = 11 < empties <= exact  # every root of a case has `empties` empty squares: one path searches them all
        own, opp = roots(n, empties, seed=1000 + empties)
        r = time_search(own, opp, depth, exact, a.reps, split)
        r.update(phase=phase, root_empties=empties, path="split" if split else "per-action")
        print(json.dumps(r), flush=True)
        res["search"].append(r)
    from alphazero_othello_b200.Models import FastOthelloNet
    from alphazero_othello_b200.eval import evaluate_vs_alphabeta
    torch.manual_seed(0)
    net = FastOthelloNet(8, 65).eval()
    args = {"c_puct": 2.0, "num_simulations": a.arena_sims}
    for level in [x for x in a.arena_levels.split(",") if x]:
        d, x = (int(v) for v in level.split(":"))
        np.random.seed(0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rates, log = evaluate_vs_alphabeta(net, args, a.arena_matches, player=AlphaBetaPlayer(depth=d, exact_empties=x))
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        r = {"matches": a.arena_matches, "simulations": a.arena_sims, "depth": d, "exact_empties": x, "wall_s": dt,
             "plies": int(log["plies"].sum()), "rates": rates}
        print(json.dumps(r), flush=True)
        res["arena"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
