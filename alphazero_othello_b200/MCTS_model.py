"""Drop-in for the reference's ``MCTS_model.MCTS`` (MCTS_model.py:172-274) on the B200 engine.

Same constructor, ``policy_improve_step`` / ``make_move`` and ``root`` surface; the tree
lives on the GPU (csrc/mcts_kernels.cu, manual mode, one slot).  Semantics are the
reference's sequential ones (``num_threads=1``): with the same ``np.random`` state and the
same policy outputs the visit counts, root values and policy targets are bit-identical,
because the host side makes the same numpy calls in the same order:
``np.random.dirichlet`` when the root is expanded with noise (:340-343) and
``np.random.choice`` for the temp~0 tie pick (:249-255); the policy target is formed with
the reference's own numpy expressions (:244-274).

``policy`` is either a torch module ``policy(x[B,1,8,8]) -> (logits, value)`` (evaluated on
the GPU straight from the engine's leaf batch) or any object with
``inference(state, player) -> (priors f32[65], value)`` (called on the host per leaf).
``policy=None`` selects the reference's rollout mode (uniform priors + one random playout per
leaf, MCTS_model.py:276-303, 332-335) evaluated in-kernel; its playouts draw from the engine's
Philox streams (keyed by ``seed``), not from ``np.random``.

``leaf_symmetry`` (torch-module policies only): ``"random"`` evaluates every leaf in one of its eight orientations,
drawn from (``seed``, position), and maps the policy back; ``"mean"`` evaluates all eight and averages priors and
values (symmetry.py).  ``apply_symmetry``, the reference's dead switch for the same idea, stays accepted and ignored.

Restrictions (stated, not silent): ``args["num_threads"]`` is accepted and ignored -- searches
run with the reference's ``num_threads=1`` semantics, the only deterministic mode (its default
of 4 races virtual losses between Python threads); the caller's ``policy`` module is neither
moved nor switched to eval mode, the search works on a private copy made at construction
(later weight updates need a new ``MCTS`` object, as in the reference's workers).
"""
import numpy as np
import torch

from . import _lib, symmetry
from .engine import MctsEngine, private_copy


class _Child:
    __slots__ = ("action", "visit_count", "value", "prior")

    def __init__(self, action, n, v, p):
        self.action, self.visit_count, self.value, self.prior = action, n, v, p


class _Root:
    """Read-only view of the device root with the attributes callers use (SURVEY 8b)."""

    def __init__(self, state, player, stats, valid_actions):
        self.state, self.player = state, player
        self.visit_count = int(stats["root_n"])
        self.value = float(stats["root_value"])
        self.valid_actions = valid_actions
        self.children = {int(a): _Child(int(a), int(stats["counts"][a]), float(stats["child_value"][a]),
                                        stats["child_prior"][a]) for a in valid_actions} if stats["expanded"] else {}

    def is_leaf(self):
        return not self.children


class MCTS:
    def __init__(self, env, args, policy, apply_symmetry=False, dirichlet_alpha=0.03, dirichlet_epsilon=0.0,
                 inference_cache=None, device="cuda:0", seed=0, leaf_symmetry=None):
        self.leaf_symmetry = symmetry.check_mode(leaf_symmetry)
        if self.leaf_symmetry and not isinstance(policy, torch.nn.Module):
            raise ValueError("leaf_symmetry needs a torch module policy (the network is evaluated on the device)")
        self.env, self.args, self.policy = env, args, policy
        self.use_rollout = policy is None
        self.num_actions = env.action_size
        # apply_symmetry / inference_cache are accepted and ignored: dead code in every reference caller
        self.apply_symmetry, self.inference_cache = apply_symmetry, inference_cache
        self.dirichlet_alpha, self.dirichlet_epsilon = dirichlet_alpha, dirichlet_epsilon
        self.num_threads = 1
        self.device = torch.device(device)
        eargs = dict(args)
        eargs.update(dirichlet_alpha=dirichlet_alpha, dirichlet_epsilon=dirichlet_epsilon)
        self._e = MctsEngine(1, eargs, self_play=False, eval_kind=_lib.EVAL_ROLLOUT if self.use_rollout else _lib.EVAL_EXTERNAL,
                             inject_random=True, device=device, max_inline_sims=64, seed=seed)
        self._module = isinstance(policy, torch.nn.Module)
        if self._module:
            self.policy = private_copy(policy, self.device)
        self._seed = int(seed)
        if self.leaf_symmetry == "random":
            self._xs = torch.zeros_like(self._e.nn_input)
            self._sym = torch.zeros(1, dtype=torch.uint8, device=self.device)
        elif self.leaf_symmetry == "mean":
            self._images = torch.zeros((8, 1, 8, 8), dtype=torch.float32, device=self.device)
        self._graph = None        # CUDA graph of (network forward + oth_mcts_step) for module policies
        self._graph_failed = False
        self._state = None  # host copy of the root position
        self._player = None
        self.root = None

    # -- helpers ---------------------------------------------------------------
    def _root_record(self):
        c = self._e.ctl()
        idx = (int(c["arena"][0]) * self._e.cfg.node_cap + int(c["root"][0])) * 4
        rec = self._e._t[_lib.BUF_NODES][idx:idx + 4].cpu().numpy().view(np.int32)
        return int(rec[4]), int(rec[5])  # first_child, meta

    def _refresh_root(self):
        st = {k: v.cpu().numpy()[0] for k, v in self._e.root_stats().items()}
        fc, _meta = self._root_record()
        st["expanded"] = fc >= 0
        valid = np.nonzero(self.env.get_valid_moves(self._state, self._player))[0]
        self.root = _Root(self._state, self._player, st, valid)

    @torch.no_grad()
    def _evaluate(self):
        e = self._e
        if self._module:
            if self.leaf_symmetry == "mean":
                symmetry.images(e.nn_input, self._images)
                logits, value = self.policy(self._images)
                symmetry.mean(logits.float(), value.float().reshape(-1), e.priors, e.values)
                return
            x = e.nn_input
            if self.leaf_symmetry == "random":
                symmetry.leaf_symmetry(x, self._seed, self._xs, self._sym)
                x = self._xs
            logits, value = self.policy(x)
            logits = logits.float()
            if self.leaf_symmetry == "random":
                symmetry.unsymmetrise_logits(logits, self._sym)
            e.priors.copy_(torch.softmax(logits, -1))
            e.values.copy_(value.float().reshape(-1))
            return
        canon = e.nn_input.view(8, 8).cpu().numpy().astype(np.int8)
        pri, val = self.policy.inference(canon, 1)  # canonical plane == player*state (Models.py:16)
        e.priors.copy_(torch.from_numpy(np.asarray(pri, np.float32)).view(1, 65))
        e.values.fill_(float(val))

    def _eval_and_step(self):
        self._evaluate()
        self._e.step()

    def _run_search(self):
        """num_simulations simulations on the device tree.  Every launch after the first consumes one evaluation
        and completes at least one simulation (the root initialisation excepted), so ``num_simulations + 1``
        evaluate+launch pairs always suffice: a module policy is driven without reading anything back per
        simulation (one CUDA-graph replay each), a host ``inference`` policy needs the leaf on the host anyway."""
        e = self._e
        sims = int(self.args["num_simulations"])
        e.step()
        if self._module:
            if self._graph is None and not self._graph_failed:
                self._capture()
            for _ in range(sims + 1):
                if self._graph is not None:
                    self._graph.replay()
                else:
                    self._eval_and_step()
        for _ in range(sims + 2):  # host policies; for module policies this loop only confirms the search is over
            ph = int(e.ctl()["phase"][0])
            if ph == _lib.PH_WAIT_EVAL:
                self._evaluate()
            elif ph != _lib.PH_RUN:
                break
            e.step()

    def _capture(self):
        """Capture (network forward, softmax, oth_mcts_step) once; fall back to eager launches if the module cannot
        be captured.  The two warm-up iterations are real ones (an evaluation of a slot that is not waiting is ignored)."""
        dev = self.device
        try:
            s = torch.cuda.Stream(device=dev)
            s.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(s):
                self._evaluate()  # warm-up of lazy initialisation only: outputs are rewritten by the first replay
            torch.cuda.current_stream(dev).wait_stream(s)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._eval_and_step()
            self._graph = g
        except Exception:
            self._graph, self._graph_failed = None, True
            torch.cuda.synchronize(dev)

    # -- the reference's surface -------------------------------------------------
    def make_move(self, action):
        action = int(action)
        if self.root is None:  # "in case we play 2nd and it is the 1st move" (:209-211)
            return
        if action not in self.root.children:
            raise KeyError(action)
        self._e.advance(torch.tensor([action], dtype=torch.int32, device=self.device))
        self._e.raise_on_error()
        self._state = self.env.get_next_state(self._state, action, self._player)
        self._player = self.env.get_opponent(self._player)
        self._refresh_root()

    def policy_improve_step(self, init_state, init_player, temp=1):
        e = self._e
        if self.root is None:
            st = np.asarray(init_state)
            canon = (st.astype(np.int64) * int(init_player)).ravel()
            own = int(sum(1 << i for i in np.nonzero(canon == 1)[0]))
            opp = int(sum(1 << i for i in np.nonzero(canon == -1)[0]))
            as_i64 = lambda x: torch.from_numpy(np.array([x], np.uint64).view(np.int64)).to(self.device)
            e.set_roots(as_i64(own), as_i64(opp), torch.tensor([int(init_player)], dtype=torch.int8, device=self.device))
            self._state, self._player = st.copy(), int(init_player)
            self._refresh_root()
        else:
            assert np.all(self.root.state == init_state)
            assert self.root.player == init_player
        if self.root.is_leaf() and self.dirichlet_epsilon > 0:
            # the draw the reference makes inside _expand_and_evaluate(root) (:340-343)
            noise = np.random.dirichlet([self.dirichlet_alpha] * self.num_actions)
            e.noise[0] = torch.from_numpy(noise).to(self.device)
        e.begin_search()
        self._run_search()
        e.raise_on_error()
        self._refresh_root()
        counts = np.zeros(self.num_actions, dtype=np.float32)
        for a, ch in self.root.children.items():
            counts[a] = ch.visit_count
        if abs(temp) < 1e-1:
            best_actions = np.where(counts == counts.max())[0]
            best_action = np.random.choice(best_actions)
            probs = np.zeros_like(counts)
            if len(self.root.valid_actions) != 0:
                probs[best_action] = 1.0
            return probs
        counts_exp = counts ** (1.0 / temp)
        norm = np.sum(counts_exp)
        if norm < 1e-12:
            probs = np.zeros(self.num_actions, dtype=np.float32)
            for a in self.root.valid_actions:
                probs[a] = 1.0 / len(self.root.valid_actions)
            return probs
        return counts_exp / norm
