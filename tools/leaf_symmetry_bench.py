"""What leaf symmetry (keyword ``leaf_symmetry``, csrc/symmetry_kernels.cu) costs on one GPU.

    python tools/leaf_symmetry_bench.py --out profiles/r06_leaf_symmetry.json

- the four kernels at 16 384 rows (a C4 leaf batch; its planes, 4 MiB, stay in L2 between launches) and 131 072 rows:
  CUDA events around 200 back-to-back launches after 20 warm-up launches, and the bytes each launch must move;
- seconds per self-play iteration (network + step kernels, CUDA-graph replays) of C4 (big net, 16 384 slots,
  400 simulations, de-duplication "auto"), C3 (small net, 4 096 slots, 200 simulations) and the one-slot runner (small
  net, 100 simulations) with leaf_symmetry off and "random": two runners of the same configuration, warmed up past the
  opening (about ply 16) and timed in alternating windows;
- wall time and win / draw / loss rates of 1 024 arena matches of a FastOthelloNet (100 simulations) against
  AlphaBetaPlayer(4, 10), with leaf_symmetry off, "random" and "mean".
The GPU's name and power limit are read in the same run, once per section.
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from alphabeta_bench import gpu_info  # noqa: E402
from alphazero_othello_b200 import _lib, symmetry  # noqa: E402


def _events_ms(fn, reps=200, warm=20):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernels():
    out = {"gpu": gpu_info(), "timing": "CUDA events around 200 launches after 20 warm-up launches", "cases": []}
    for n in (16384, 131072):
        g = torch.Generator(device="cuda").manual_seed(n)
        planes = torch.randint(-1, 2, (n, 1, 8, 8), device="cuda", generator=g).float()
        xs, sym = torch.empty_like(planes), torch.empty(n, dtype=torch.uint8, device="cuda")
        symmetry.leaf_symmetry(planes, 0, xs, sym)
        logits_f32 = torch.randn(n, 72, device="cuda", generator=g)[:, :65]   # FoldedNet-like strided head views
        logits_bf16 = torch.randn(n, 72, device="cuda", generator=g).to(torch.bfloat16)[:, :65]
        images = torch.empty((8 * n, 1, 8, 8), device="cuda")
        ml = torch.randn(8 * n, 72, device="cuda", generator=g)[:, :65]
        mv = torch.randn(8 * n, device="cuda", generator=g).tanh()
        pri, val = torch.empty((n, 65), device="cuda"), torch.empty(n, device="cuda")
        moved = 7 / 8  # rows with s = 0 are skipped by the unsymmetrise kernel
        cases = [("oth_nn_leaf_symmetry", lambda: symmetry.leaf_symmetry(planes, 0, xs, sym), n * (256 + 256 + 1)),
                 ("oth_nn_unsymmetrise_logits f32", lambda: symmetry.unsymmetrise_logits(logits_f32, sym),
                  n * 1 + n * moved * 2 * 256),
                 ("oth_nn_unsymmetrise_logits bf16", lambda: symmetry.unsymmetrise_logits(logits_bf16, sym),
                  n * 1 + n * moved * 2 * 128),
                 ("oth_nn_symmetry_images", lambda: symmetry.images(planes, images), n * (256 + 8 * 256)),
                 ("oth_nn_symmetry_mean", lambda: symmetry.mean(ml, mv, pri, val), n * (8 * (260 + 4) + 260 + 4))]
        for name, fn, nbytes in cases:
            ms = _events_ms(fn)
            out["cases"].append({"kernel": name, "rows": n, "us_per_launch": ms * 1e3, "bytes": int(nbytes),
                                 "GB_per_s": nbytes / (ms * 1e-3) / 1e9})
    return out


def runners(windows, plan):
    from bench import TRAIN_ARGS, WORKLOADS, make_net
    from alphazero_othello_b200.Models import fold_for_inference
    from alphazero_othello_b200.engine import BatchedPolicy, MctsEngine, SelfPlayRunner
    out = {"gpu": gpu_info(), "method": f"{windows} alternating timed windows per mode (CUDA events), after the same "
                                        "warm-up iterations per runner; runners share the network", "cases": []}
    for w, (warm, iters) in plan.items():
        desc, kind, G, sims = WORKLOADS[w] if w != "one-slot" else ("one slot, small net, 100 sims/move", "small", 1, 100)
        args = dict(TRAIN_ARGS, num_simulations=sims)
        net = fold_for_inference(make_net(kind).cuda(), torch.bfloat16)
        runs = {}
        for mode in (None, "random"):
            eng = MctsEngine(G, args, self_play=True, eval_kind=_lib.EVAL_EXTERNAL, games_per_slot=-1, seed=1,
                             out_pos_cap=G * 80 + 4096, out_game_cap=G + 64)
            runs[mode] = SelfPlayRunner(eng, BatchedPolicy(net, "cuda:0", torch.float32), dedup="auto", leaf_symmetry=mode)
            runs[mode].warm_start()
            runs[mode].run_iterations(warm)  # past the opening: the timed windows see whole batches
        torch.cuda.synchronize()
        ms = {None: [], "random": []}
        for _ in range(windows):
            for mode, run in runs.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run.run_iterations(iters)
                e1.record()
                torch.cuda.synchronize()
                ms[mode].append(e0.elapsed_time(e1) / iters)
                run.e.raise_on_error()
        off, on = sorted(ms[None]), sorted(ms["random"])
        med = lambda v: v[len(v) // 2]
        out["cases"].append({"workload": w, "desc": desc, "warmup_iterations": warm, "iterations_per_window": iters,
                             "dedup": runs[None].dedup,
                             "ms_per_iteration_off": ms[None], "ms_per_iteration_random": ms["random"],
                             "median_off_ms": med(off), "median_random_ms": med(on),
                             "overhead_pct_of_medians": 100.0 * (med(on) / med(off) - 1.0)})
        del runs
        torch.cuda.empty_cache()
    return out


def arena(n_matches):
    from bench import make_net
    from alphazero_othello_b200.alphabeta import AlphaBetaPlayer
    from alphazero_othello_b200.eval import evaluate_vs_alphabeta
    out = {"gpu": gpu_info(), "net": "FastOthelloNet (seeded random init), bf16 folded twin", "matches": n_matches,
           "simulations": 100, "opponent": "AlphaBetaPlayer(4, 10)", "cases": []}
    net = make_net("small").cuda()
    args = {"c_puct": 2.0, "num_simulations": 100}
    evaluate_vs_alphabeta(net, args, 64, AlphaBetaPlayer(4, 10))  # warm-up: module loads, cuDNN plans
    for mode in (None, "random", "mean"):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rates, log = evaluate_vs_alphabeta(net, args, n_matches, AlphaBetaPlayer(4, 10), leaf_symmetry=mode, seed=0)
        torch.cuda.synchronize()
        out["cases"].append({"leaf_symmetry": mode, "wall_s": time.perf_counter() - t0, "plies": int(log["plies"].sum()),
                             "rates": rates})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_leaf_symmetry.json"))
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--matches", type=int, default=1024)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing here is measured without one")
    res = {"kernels": kernels()}
    print(json.dumps(res["kernels"], indent=1), flush=True)
    # warm-up to about ply 16 (C4, C3): the de-duplicated opening is over and every iteration evaluates a whole batch
    res["runners"] = runners(a.windows, {"c4": (6400, 100), "c3": (3200, 200), "one-slot": (1600, 1600)})
    print(json.dumps(res["runners"], indent=1), flush=True)
    res["arena"] = arena(a.matches)
    print(json.dumps(res["arena"], indent=1), flush=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
