"""Throughput of the endgame solver oth_solve_wld on one GPU, against the alpha-beta player's exact path, and the cost of
relabelling a self-play batch with it.

    python tools/endgame_bench.py --out profiles/endgame_bench.json

- positions/s, nodes/s and nodes per position over 512, 4 096 and 16 384 roots with exactly 10, 12, 14 and 16 empty
  squares and OTH_SOLVE_MAX_EMPTIES (cases above the cap are skipped): CUDA events around whole launches, best of
  --reps after one warm-up launch of the same shape;
- the same roots at 10-12 empties solved with oth_alphabeta(depth 1, exact_empties 12), taking the maximum of each row:
  the way a win/draw/loss could be had without the solver.  Its signs are checked against the solver's;
- 4 096 self-play games of BASELINE config C3 (small network, 200 simulations per move) played to the end with
  collect_self_play_games(return_raw=True), then relabelled at 12, 14 and OTH_SOLVE_MAX_EMPTIES empties: rows solved,
  seconds (host clock around the call, which ends in a device synchronise), and that time as a share of the self-play.
Roots come from uniform-random games played by the library's own rollout kernel (seeded), as in alphabeta_bench.py.
The GPU's name, power limit and maximum SM clock are read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from alphabeta_bench import gpu_info, roots  # noqa: E402
from alphazero_othello_b200 import endgame  # noqa: E402
from alphazero_othello_b200.alphabeta import NONE, search  # noqa: E402


def best_ms(fn, reps):
    fn()  # warm-up: same shape
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(reps):
        e0.record()
        res = fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/endgame_bench.json")
    ap.add_argument("--sizes", default="512,4096,16384")
    ap.add_argument("--empties", default="10,12,14,16")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--games", type=int, default=4096)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    cap = endgame.MAX_EMPTIES
    res = {"gpu": gpu_info(), "solve_max_empties": cap, "solve": [], "alphabeta_max_of_row": [], "relabel": {}}
    empties = sorted({int(x) for x in a.empties.split(",")} | {cap})
    for n in [int(x) for x in a.sizes.split(",")]:
        for e in empties:
            if e > cap:
                res["solve"].append({"positions": n, "root_empties": e, "skipped": f"above OTH_SOLVE_MAX_EMPTIES = {cap}"})
                continue
            own, opp = roots(n, e, seed=2000 + e)
            ms, (w, nodes) = best_ms(lambda: endgame.solve_wld(own, opp, e), a.reps)
            w, nodes = w.cpu().numpy(), nodes.cpu().numpy()
            t = min(ms) / 1e3
            r = {"positions": n, "root_empties": e, "launch_ms": [round(x, 3) for x in ms], "positions_per_s": n / t,
                 "nodes": int(nodes.sum()), "nodes_per_s": float(nodes.sum()) / t, "nodes_per_position": float(nodes.mean()),
                 "max_nodes_of_a_position": int(nodes.max()), "wins_draws_losses": [int((w == v).sum()) for v in (1, 0, -1)]}
            print(json.dumps(r), flush=True)
            res["solve"].append(r)
            if e <= 12:
                ms_ab, (v, _, ab_nodes) = best_ms(lambda: search(own, opp, 1, 12), a.reps)
                v = v.cpu().numpy().astype(np.int64)
                sign = np.sign(np.where(v != NONE, v, -2**40).max(1))
                t_ab = min(ms_ab) / 1e3
                c = {"positions": n, "root_empties": e, "launch_ms": [round(x, 3) for x in ms_ab], "positions_per_s": n / t_ab,
                     "nodes": int(ab_nodes.sum().item()), "solver_speedup": t_ab / t, "signs_agree": bool((sign == w).all())}
                print(json.dumps(c), flush=True)
                res["alphabeta_max_of_row"].append(c)
    from bench import TRAIN_ARGS, WORKLOADS, make_net
    from alphazero_othello_b200.self_play_worker import collect_self_play_games
    _, kind, _, sims = WORKLOADS["c3"]
    net = make_net(kind)
    args = dict(TRAIN_ARGS, num_simulations=sims)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = collect_self_play_games(net, args, a.games, seed=1, return_raw=True)
    torch.cuda.synchronize()
    t_play = time.perf_counter() - t0
    out = {k: v.cuda() for k, v in out.items()}
    rel = {"games": a.games, "config": "c3", "simulations": sims, "positions": int(out["values"].numel()),
           "self_play_s": t_play, "levels": []}
    endgame.relabel(out, 12)  # warm-up
    for e in sorted({12, 14, cap}):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = endgame.relabel(out, e)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        lv = {"max_empties": e, "rows_solved": int(r["solved"].sum()), "seconds": dt, "share_of_self_play": dt / t_play}
        print(json.dumps(lv), flush=True)
        rel["levels"].append(lv)
    res["relabel"] = rel
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
