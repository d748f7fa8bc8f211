"""Leaf symmetry at the network boundary (csrc/symmetry_kernels.cu; keyword ``leaf_symmetry``) on the GPU.

1. the four kernels against the numpy restatement (tests/symmetry_reference.py), bit for bit or against float64;
2. an exactly D4-equivariant network (small integer weights, elementwise ops: exact float32 outputs): every consumer
   plays bit for bit the same games with ``"random"`` as without, and ``"mean"`` gives the same priors within 1e-6;
3. real, non-equivariant networks: self-play with ``"random"`` replays through the CPU oracle from its tape, and the
   consumed priors / values are unsym(softmax(net(T_s(plane)))) with s the documented id;
4. the arena with ``"random"`` / ``"mean"`` against a network and against the alpha-beta player;
5. off by default: no extra kernel in the iteration.
"""
import ctypes as C

import numpy as np
import pytest

import symmetry_reference as R

pytestmark = pytest.mark.gpu

TRAIN_ARGS = {"c_puct": 2.0, "dirichlet_alpha": 1.0, "dirichlet_epsilon": 0.3, "mcts_temperature": 1.0,
              "num_exploratory_moves": 35, "lambda": 0.98}


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _planes(n, seed):
    """n random canonical planes, row 0 the initial position (invariant under four of the eight symmetries)."""
    rng = np.random.default_rng(seed)
    p = rng.integers(-1, 2, (n, 64)).astype(np.float32)
    p[0] = 0
    p[0, [27, 36]], p[0, [28, 35]] = -1, 1
    return p


# ------------------------------------------------------------------------------------------------------ 1. kernels --
@pytest.mark.parametrize("n", [1, 4097, 20011])
def test_leaf_symmetry_ids_and_images_match_numpy(n):
    import torch
    from alphazero_othello_b200 import symmetry
    planes = _planes(n, n)
    x = torch.from_numpy(planes).cuda().view(n, 1, 8, 8)
    for seed in (0, 2**64 - 1, 987654321):
        out = torch.full_like(x, 5.0)
        sym = torch.full((n,), 99, dtype=torch.uint8, device="cuda")
        symmetry.leaf_symmetry(x, seed, out, sym)
        ids = R.plane_ids(seed, planes)
        assert np.array_equal(sym.cpu().numpy(), ids)
        got = out.view(n, 64).cpu().numpy()
        for s in range(8):
            rows = ids == s
            assert np.array_equal(got[rows], R.transform(planes[rows], s)), s
    assert np.array_equal(x.view(n, 64).cpu().numpy(), planes)  # the input is untouched
    img = torch.full((8 * n, 1, 8, 8), 5.0, device="cuda")
    symmetry.images(x, img)
    got = img.view(n, 8, 64).cpu().numpy()
    for j in range(8):
        assert np.array_equal(got[:, j], R.transform(planes, j)), j
    # the initial position is its own image under the identity, the half turn and the two diagonal reflections
    same = [j for j in range(8) if np.array_equal(got[0, j], planes[0])]
    assert same == [0, 2, 5, 7], same


@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
def test_unsymmetrise_strided_rows_bit_for_bit(dtype):
    import torch
    from alphazero_othello_b200 import symmetry
    n, width = 20011, 80
    g = torch.Generator().manual_seed(5)
    full = (torch.randn(n, width, generator=g) * 8).to(getattr(torch, dtype))
    sym = torch.randint(0, 8, (n,), generator=g, dtype=torch.uint8)
    dev = full.cuda()
    symmetry.unsymmetrise_logits(dev[:, :65], sym.cuda())
    got = dev.cpu()
    bits = torch.int16 if dtype == "bfloat16" else torch.int32
    ref_bits = full.view(bits).numpy()
    got_bits = got.view(bits).numpy()
    assert np.array_equal(got_bits[:, 64:], ref_bits[:, 64:])  # pass entry and padding columns untouched
    for s in range(8):
        rows = sym.numpy() == s
        assert np.array_equal(got_bits[rows], R.unsymmetrise(ref_bits[rows], s)), s


def test_symmetry_mean_matches_float64():
    import torch
    from alphazero_othello_b200 import symmetry
    n = 5003
    g = torch.Generator().manual_seed(11)
    logits = torch.randn(8 * n, 72, generator=g) * 4
    logits[::7, 64] += 30.0  # some rows dominated by the pass, some by one square
    logits[::5, 3] += 40.0
    vals = torch.tanh(torch.randn(8 * n, 3, generator=g))
    pri = torch.full((n, 65), 7.0, device="cuda")
    val = torch.full((n,), 7.0, device="cuda")
    lg, vg = logits.cuda(), vals.cuda()
    symmetry.mean(lg[:, :65], vg[:, 1], pri, val)
    ref_p, ref_v = R.mean(logits[:, :65].numpy(), vals[:, 1].numpy())
    assert np.abs(pri.cpu().numpy() - ref_p).max() < 1e-6
    assert np.abs(val.cpu().numpy() - ref_v).max() < 1e-6


def test_argument_errors_return_before_any_launch():
    import torch
    from alphazero_othello_b200 import _lib
    L = _lib.lib()
    E = _lib.OTH_E_ARG
    x = torch.zeros(4, 64, device="cuda")
    o = torch.full((8 * 4 + 1, 64), 3.0, device="cuda")
    s = torch.full((8,), 9, dtype=torch.uint8, device="cuda")
    lg = torch.full((32, 72), 3.0, device="cuda")
    v = torch.full((32,), 3.0, device="cuda")
    X, O, S, LG, V = x.data_ptr(), o.data_ptr(), s.data_ptr(), lg.data_ptr(), v.data_ptr()
    st = _stream()
    assert L.oth_nn_leaf_symmetry(X, -1, 0, O, S, st) == E
    assert L.oth_nn_leaf_symmetry(None, 4, 0, O, S, st) == E
    assert L.oth_nn_leaf_symmetry(X, 4, 0, None, S, st) == E
    assert L.oth_nn_leaf_symmetry(X, 4, 0, O, None, st) == E
    assert L.oth_nn_leaf_symmetry(X, 4, 0, X, S, st) == E       # out of place only
    assert L.oth_nn_leaf_symmetry(X + 2, 4, 0, O, S, st) == E   # float alignment
    assert L.oth_nn_unsymmetrise_logits(LG, 64, 0, S, 4, st) == E   # stride < 65
    assert L.oth_nn_unsymmetrise_logits(LG, 72, 2, S, 4, st) == E   # is_bf16 not 0 / 1
    assert L.oth_nn_unsymmetrise_logits(LG, 72, 0, S, -1, st) == E
    assert L.oth_nn_unsymmetrise_logits(None, 72, 0, S, 4, st) == E
    assert L.oth_nn_unsymmetrise_logits(LG, 72, 0, None, 4, st) == E
    assert L.oth_nn_unsymmetrise_logits(LG + 2, 72, 0, S, 4, st) == E
    assert L.oth_nn_unsymmetrise_logits(LG + 1, 72, 1, S, 4, st) == E
    assert L.oth_nn_symmetry_images(X, -1, O, st) == E
    assert L.oth_nn_symmetry_images(None, 4, O, st) == E
    assert L.oth_nn_symmetry_images(X, 4, None, st) == E
    assert L.oth_nn_symmetry_mean(LG, 64, V, 1, 4, O, V, st) == E
    assert L.oth_nn_symmetry_mean(LG, 72, V, 0, 4, O, V, st) == E
    assert L.oth_nn_symmetry_mean(LG, 72, V, 1, -1, O, V, st) == E
    assert L.oth_nn_symmetry_mean(LG, 72, None, 1, 4, O, V, st) == E
    assert L.oth_nn_symmetry_mean(LG, 72, V, 1, 4, None, V, st) == E
    assert L.oth_nn_symmetry_mean(LG, 72, V, 1, 4, O, None, st) == E
    for f in (lambda: L.oth_nn_leaf_symmetry(X, 0, 0, O, S, st), lambda: L.oth_nn_unsymmetrise_logits(LG, 72, 0, S, 0, st),
              lambda: L.oth_nn_symmetry_images(X, 0, O, st), lambda: L.oth_nn_symmetry_mean(LG, 72, V, 1, 0, O, V, st)):
        assert f() == _lib.OTH_OK
    torch.cuda.synchronize()
    assert bool((o == 3.0).all()) and bool((s == 9).all()) and bool((lg == 3.0).all()) and bool((v == 3.0).all())


# ---------------------------------------------------------------------------------- 2. an equivariant network --
def _equivariant_net(supports_raw=True):
    """logits of square e = f(x_e, sum of e's eight neighbours), pass and value = functions of disc counts: small integers
    times powers of two, so every output is exact in float32 and T_s(net(x)) == net(T_s(x)) bit for bit."""
    import torch
    import torch.nn.functional as F

    class Equivariant(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.register_buffer("one", torch.ones(1))
            self.supports_raw = supports_raw

        def forward(self, x, raw=False):
            x = x.reshape(-1, 1, 8, 8).float()
            B = x.size(0)
            p = F.pad(x, (1, 1, 1, 1))
            nb = None
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    if dy or dx:
                        t = p[:, :, 1 + dy:9 + dy, 1 + dx:9 + dx]
                        nb = t if nb is None else nb + t
            sq = (2 * x - nb + x * nb + (x == 0).float() * nb * nb) * 0.25
            own, opp = (x == 1).float().sum((1, 2, 3)), (x == -1).float().sum((1, 2, 3))
            y = torch.cat([sq.reshape(B, 64), ((own - opp) * 0.125)[:, None], ((own - 2 * opp) * 0.0625)[:, None],
                           torch.zeros(B, 6, device=x.device)], 1)  # [B, 72]: strided head views like FoldedNet's
            if raw:
                return y[:, :65], y[:, 65:66]
            return y[:, :65], torch.tanh(y[:, 65:66])
    return Equivariant().cuda().eval()


def _self_play(net, mode, n_slots, sims, fused, graph, dedup, seed=21):
    import torch
    from alphazero_othello_b200 import _lib
    from alphazero_othello_b200.engine import BatchedPolicy, MctsEngine, SelfPlayRunner
    args = dict(TRAIN_ARGS, num_simulations=sims)
    e = MctsEngine(n_slots, args, self_play=True, eval_kind=_lib.EVAL_EXTERNAL, games_per_slot=1, seed=seed)
    run = SelfPlayRunner(e, BatchedPolicy(net, "cuda:0", torch.float32), use_graph=graph, fused=fused, dedup=dedup,
                         leaf_symmetry=mode)
    assert run.fused == fused and run.dedup == dedup
    if dedup:
        run.force_bucket = 256
    out = run.play(check_every=32)
    e.raise_on_error()
    return out, e, run


@pytest.mark.parametrize("fused,graph,dedup,raw", [(False, True, False, True), (False, False, False, False),
                                                   (True, True, False, True), (True, False, False, True),
                                                   (True, True, True, True), (True, False, True, True)])
def test_equivariant_network_self_play_is_identical_with_random_symmetry(fused, graph, dedup, raw):
    """Boards, policy targets, value targets, game descriptors and the number of launches: bit for bit."""
    net = _equivariant_net(supports_raw=raw)
    n_slots, sims = (512, 16) if dedup else (64, 24)
    off, e0, _ = _self_play(net, None, n_slots, sims, fused, graph, dedup)
    on, e1, run = _self_play(net, "random", n_slots, sims, fused, graph, dedup)
    assert len(off["games"]) == n_slots
    # finished games enter the output ring in the order their slots reach it: compare position by position keyed by
    # (game id, ply), and the game descriptors by game id
    for k in ("boards", "pis", "values", "meta", "states"):
        x0 = off[k].numpy()[np.argsort(off["meta"].numpy(), kind="stable")]
        x1 = on[k].numpy()[np.argsort(on["meta"].numpy(), kind="stable")]
        assert np.array_equal(x0, x1), k
    g0, g1 = off["games"].numpy(), on["games"].numpy()
    assert np.array_equal(g0[np.argsort(g0[:, 0])][:, [0, 2, 3]], g1[np.argsort(g1[:, 0])][:, [0, 2, 3]])
    assert e0.launches == e1.launches and e0.counters() == e1.counters()
    if not dedup:  # the network really was shown other orientations (the last whole batch)
        assert len(set(run._sym[n_slots][1].cpu().numpy().tolist())) > 1


def test_equivariant_network_arena_and_mcts_are_identical_with_random_and_close_with_mean():
    import torch
    from alphazero_othello_b200.MCTS_model import MCTS
    from alphazero_othello_b200.envs.othello import OthelloGameNew
    from alphazero_othello_b200.eval import play_matches_batched
    net = _equivariant_net(supports_raw=False)
    args = {"c_puct": 2.0, "num_simulations": 24}
    n = 16
    u = np.random.default_rng(3).random((n, 128))
    worst = [0.0]

    def check_mean(side):  # the mean of the eight images == the leaf's own outputs (within float32 rounding)
        e = side.eng
        logits, value = side.net(e.nn_input)
        p = torch.softmax(logits.float(), -1)
        worst[0] = max(worst[0], float((p - e.priors).abs().max()), float((value.reshape(-1) - e.values).abs().max()))

    ref = play_matches_batched(net, net, args, n, dtype=None, u_tie=u)
    rnd = play_matches_batched(net, net, args, n, dtype=None, u_tie=u, leaf_symmetry="random", seed=9)
    mean = play_matches_batched(net, net, args, n, dtype=None, u_tie=u, leaf_symmetry="mean", record=check_mean)
    assert ref[0] == rnd[0] and np.array_equal(ref[1]["actions"], rnd[1]["actions"])
    assert all(r in ("A", "B", "Draw") for r in mean[0]) and worst[0] < 1e-6

    env = OthelloGameNew(8)
    margs = dict(TRAIN_ARGS, num_simulations=32)
    res = {}
    for mode in (None, "random", "mean"):
        np.random.seed(4)
        m = MCTS(env, margs, net, dirichlet_alpha=1.0, dirichlet_epsilon=0.25, leaf_symmetry=mode, seed=17)
        s, pl, trace = env.get_initial_state(), 1, []
        for _ in range(6):
            pi = m.policy_improve_step(s, pl, temp=1.0)
            pri = np.array([m.root.children[a].prior for a in sorted(m.root.children)])
            a = int(np.argmax(pi))
            trace.append((pi, m.root.value, pri, a))
            m.make_move(a)
            s, pl = env.get_next_state(s, a, pl), -pl
        assert m._graph is not None  # the captured (network + step) graph ran
        res[mode] = trace
    same_root = True  # "mean" searches the same positions as long as its moves agree with the plain search's
    for (p0, v0, q0, a0), (p1, v1, q1, a1), (_, _, q2, a2) in zip(res[None], res["random"], res["mean"]):
        assert np.array_equal(p0, p1) and v0 == v1 and np.array_equal(q0, q1) and a0 == a1
        if same_root:
            assert np.abs(q0 - q2).max() < 1e-6
        same_root = same_root and a0 == a2


# ------------------------------------------------------------------------------------ 3. a real network, recorded --
class _SampleTape:
    """Forwards to an oracle EvalTape and keeps a sample of the leaf batches with what the step kernel consumed."""

    def __init__(self, tape, every=7):
        self.tape, self.every, self.calls, self.samples = tape, every, 0, []

    def put_planes(self, planes, mask, priors, values):
        self.tape.put_planes(planes, mask, priors, values)
        if self.calls % self.every == 0 and mask.any():
            self.samples.append((planes.copy(), mask.copy(), priors.copy(), values.copy()))
        self.calls += 1


@pytest.fixture
def no_tf32():
    """Full float32 convolutions and matmuls: the host recomputation below evaluates the leaves in other batches than
    the engine did, and TF32's rounding would differ between them by more than the tolerance."""
    import torch
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@pytest.mark.parametrize("kind,dedup", [("small", False), ("big", False), ("small", True)])
def test_real_network_random_symmetry_replays_through_the_oracle(kind, dedup, no_tf32):
    import torch
    import oracle as O
    from oracle.record_replay import record_self_play, replay_and_compare
    from alphazero_othello_b200 import _lib
    from alphazero_othello_b200.Models import AlphaZeroNet, FastOthelloNet, fold_for_inference
    from alphazero_othello_b200.engine import BatchedPolicy, MctsEngine, SelfPlayRunner
    seed = 31
    torch.manual_seed(seed)
    net = fold_for_inference((AlphaZeroNet(8, 65, 2, 32) if kind == "big" else FastOthelloNet(8, 65)).cuda().eval(),
                             torch.float32)
    n_slots, sims = (512, 16) if dedup else (96, 48)
    args = dict(TRAIN_ARGS, num_simulations=sims)
    e = MctsEngine(n_slots, args, self_play=True, eval_kind=_lib.EVAL_EXTERNAL, games_per_slot=1, seed=seed)
    run = SelfPlayRunner(e, BatchedPolicy(net, "cuda:0", torch.float32), use_graph=True, record=True, dedup=dedup,
                         leaf_symmetry="random")
    assert run.fused
    if dedup:
        run.force_bucket = 256
    tape = O.EvalTape(n_slots, sims * 70 + 128)
    sampler = _SampleTape(tape)
    record_self_play(run, sampler, poll_every=64)
    e.raise_on_error()
    c = e.counters()
    assert c["games"] == n_slots and c["errors"] == 0
    checked, oracle_sims = replay_and_compare(e, args, tape)
    assert checked == n_slots and oracle_sims == c["sims"] and tape.served == c["evals"]
    # the consumed priors / values are the network's on the leaf's documented image, mapped back
    planes = np.concatenate([p[m] for p, m, _, _ in sampler.samples])
    pri = np.concatenate([q[m] for _, m, q, _ in sampler.samples])
    val = np.concatenate([v[m] for _, m, _, v in sampler.samples])
    ids = R.plane_ids(seed, planes)
    assert len(planes) > 1000 and len(set(ids.tolist())) == 8
    xs = np.empty_like(planes)
    for s in range(8):
        xs[ids == s] = R.transform(planes[ids == s], s)
    with torch.no_grad():
        logits, value = net(torch.from_numpy(xs).cuda().view(-1, 1, 8, 8))
    ref = R.softmax64(logits.double().cpu().numpy())
    for s in range(8):
        ref[ids == s] = R.unsymmetrise(ref[ids == s], s)
    assert np.abs(pri - ref).max() < 1e-5
    assert np.abs(val - value.double().cpu().numpy().reshape(-1)).max() < 1e-6


# --------------------------------------------------------------------------------------------------- 4. arena --
def _linear_net(seed):
    from test_arena_gpu import _net
    return _net(seed).cuda().eval()


@pytest.mark.parametrize("mode", ["random", "mean"])
def test_arena_with_leaf_symmetry_replays_through_the_oracle(mode):
    import torch
    import oracle as O
    from alphazero_othello_b200 import _lib, symmetry
    from alphazero_othello_b200.eval import play_matches_batched
    args = {"c_puct": 3.0, "num_simulations": 20}
    tables = {}
    worst = [0.0]
    key = (1 << (63 - np.arange(64, dtype=np.uint64)))  # the oracle's table key: square 0 is the top bit

    def record(side):
        t = tables.setdefault(id(side), O.EvalTable(1 << 18))
        e = side.eng
        ph = e.ctl()["phase"]
        x = e.nn_input.view(-1, 64).cpu().numpy()
        pr, va = e.priors.cpu().numpy(), e.values.cpu().numpy()
        for s in np.nonzero(ph == _lib.PH_WAIT_EVAL)[0]:  # a position gets one answer, in any row
            assert t.put(int((key * (x[s] == 1)).sum()), int((key * (x[s] == -1)).sum()), pr[s], va[s]) in (0, 1)
        side._table = t
        if mode == "mean":  # every image of a leaf, averaged the same way, gives the leaf's priors permuted
            leaves = np.nonzero(ph == _lib.PH_WAIT_EVAL)[0][:4]
            if len(leaves):
                imgs = torch.zeros((8 * len(leaves), 1, 8, 8), device="cuda")
                symmetry.images(e.nn_input[torch.from_numpy(leaves).cuda()].contiguous(), imgs)
                im8 = torch.zeros((64 * len(leaves), 1, 8, 8), device="cuda")
                symmetry.images(imgs, im8)
                logits, value = side.net(im8)
                p8, v8 = torch.zeros((8 * len(leaves), 65), device="cuda"), torch.zeros(8 * len(leaves), device="cuda")
                symmetry.mean(logits.float(), value.float().reshape(-1), p8, v8)
                p8 = p8.cpu().numpy().reshape(len(leaves), 8, 65)
                for k, slot in enumerate(leaves):
                    for j in range(8):
                        worst[0] = max(worst[0], np.abs(p8[k, j] - R.transform(pr[slot:slot + 1], j)[0]).max())

    np.random.seed(6)
    n = 10
    results, log = play_matches_batched(_linear_net(1), _linear_net(2), args, n, dtype=None, record=record,
                                        leaf_symmetry=mode, seed=3)
    assert all(r in ("A", "B", "Draw") for r in results) and len(results) == n
    assert worst[0] < 1e-6
    ta, tb = list(tables.values())
    g = O.OracleGame()
    for i in range(n):
        first_t, second_t = (ta, tb) if i % 2 == 0 else (tb, ta)
        trees = {1: O.OracleMCTS(3.0, 20, O.Evaluator(table=first_t)), -1: O.OracleMCTS(3.0, 20, O.Evaluator(table=second_t))}
        searched = {1: False, -1: False}
        s, pl = g.get_initial_state(), 1
        res = None
        for ply in range(200):
            probs = trees[pl].policy_improve_step(s, pl, 0.0, None, log["u_tie"][i, ply])
            searched[pl] = True
            a = int(np.argmax(probs))
            assert a == log["actions"][i, ply], (i, ply)
            s = g.get_next_state(s, a, pl)
            rew, done = g.get_value_and_terminated(s, a, pl)
            if done:
                res = "Draw" if rew == 0 else ("A" if (rew == 1) == (pl == 1) else "B")
                break
            for p2 in (1, -1):
                if searched[p2]:
                    trees[p2].make_move(a)
            pl = -pl
        if i % 2 == 1 and res != "Draw":
            res = "B" if res == "A" else "A"
        assert res == results[i] and log["plies"][i] == ply + 1
    assert ta.misses == 0 and tb.misses == 0


@pytest.mark.parametrize("mode", ["random", "mean"])
def test_arena_against_alphabeta_and_folded_network_runs_to_completion(mode):
    import torch
    from alphazero_othello_b200.Models import FastOthelloNet
    from alphazero_othello_b200.alphabeta import AlphaBetaPlayer
    from alphazero_othello_b200.eval import evaluate_vs_alphabeta, play_matches_batched
    torch.manual_seed(0)
    net = FastOthelloNet(8, 65).cuda().eval()
    args = {"c_puct": 2.0, "num_simulations": 16}
    rates, log = evaluate_vs_alphabeta(net, args, 8, AlphaBetaPlayer(2, 6), leaf_symmetry=mode, seed=1)
    assert abs(sum(rates.values()) - 1.0) < 1e-9 and (log["plies"] > 0).all()
    torch.manual_seed(1)
    results, _ = play_matches_batched(net, FastOthelloNet(8, 65).cuda().eval(), args, 8, leaf_symmetry=mode)  # bf16 twins
    assert len(results) == 8 and all(r in ("A", "B", "Draw") for r in results)


# ------------------------------------------------------------------------------------------- 5. off by default --
def test_off_by_default_adds_no_kernel():
    """The graph of 16 iterations runs exactly two more kernels per iteration with "random" and none of them without."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    net = _equivariant_net()

    def kernels(mode):
        from alphazero_othello_b200 import _lib
        from alphazero_othello_b200.engine import BatchedPolicy, MctsEngine, SelfPlayRunner
        e = MctsEngine(64, dict(TRAIN_ARGS, num_simulations=16), self_play=True, eval_kind=_lib.EVAL_EXTERNAL,
                       games_per_slot=1, seed=2)
        run = SelfPlayRunner(e, BatchedPolicy(net, "cuda:0", torch.float32), leaf_symmetry=mode)
        run.warm_start()
        run.run_iterations(32)  # captures the graphs
        torch.cuda.synchronize()
        launches = e.launches
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run.run_iterations(32)
            torch.cuda.synchronize()
        assert e.launches - launches == 32
        names = [ev.name for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]
        return [k for k in names if "k_nn_" in k], len(names)

    sym0, n0 = kernels(None)
    sym1, n1 = kernels("random")
    assert sym0 == [] and n0 > 0
    assert len(sym1) == 64 and n1 - n0 == 64, (len(sym1), n0, n1)
