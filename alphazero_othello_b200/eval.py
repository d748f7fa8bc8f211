"""Batched arena on the B200 engine (SURVEY 8f rank 2): the second consumer of the MCTS surface.

Restates ``eval.py:12-178`` of the reference -- ``play_match`` (mover searches with temp=0, arg-max
move, BOTH trees advance), ``_run_one_match`` (even matches: candidate plays +1, odd: the incumbent)
and ``evaluate_models_parallel`` (win rates) -- for ``n_matches`` concurrent matches: two engines
(one per network) hold one tree per match; in every ply only the trees of the side to move search.

Tie-breaks among equally visited moves (``np.random.choice(best_actions)``, MCTS_model.py:249-255)
use one logged uniform per match and ply (``np.random.random_sample``), so a match can be replayed.
"""
import numpy as np
import torch

from . import _lib, alphabeta
from .alphabeta import AlphaBetaPlayer
from .engine import MctsEngine, private_copy
from .envs.othello import OthelloGameNew


def _pack(states, players):
    canon = states.reshape(len(states), 64).astype(np.int64) * players.astype(np.int64)[:, None]
    w = np.uint64(1) << np.arange(64, dtype=np.uint64)
    own = ((canon == 1) * w).sum(1, dtype=np.uint64)
    opp = ((canon == -1) * w).sum(1, dtype=np.uint64)
    return own.view(np.int64), opp.view(np.int64)


class DeviceStubPolicy:
    """A deterministic evaluator that lives in the kernels (OTH_EVAL_STUB_A / _B / _H of the C ABI) in the place of a
    network: parity tests replay matches of the reference played with the same stub, benches search without a network."""

    KINDS = {"A": _lib.EVAL_STUB_A, "B": _lib.EVAL_STUB_B, "H": _lib.EVAL_STUB_H}

    def __init__(self, kind="H", salt=0):
        self.eval_kind, self.salt = self.KINDS[kind], int(salt)


class _Side:
    """One network + one manual-mode engine holding a tree per match."""

    def __init__(self, policy, args, n, device, lanes, dtype):
        from .Models import fold_for_inference
        self.stub = isinstance(policy, DeviceStubPolicy)
        self.eng = MctsEngine(n, args, self_play=False, eval_kind=policy.eval_kind if self.stub else _lib.EVAL_EXTERNAL,
                              stub_salt=policy.salt if self.stub else 0, device=device, lanes=lanes, max_inline_sims=16)
        if not self.stub:
            net = private_copy(policy, device)
            self.net = fold_for_inference(net, dtype) if dtype is not None else net
        self.has_tree = np.zeros(n, bool)  # "self.root is None" of the reference until the first own search
        self.record = None

    @torch.no_grad()
    def evaluate(self):
        e = self.eng
        logits, value = self.net(e.nn_input)
        torch.softmax(logits.float(), dim=-1, out=e.priors)
        e.values.copy_(value.float().reshape(-1))

    def search(self, mask_np, states, players, sims):
        e = self.eng
        dev = e.device
        mask = torch.from_numpy(mask_np.astype(np.uint8)).to(dev)
        fresh = mask_np & ~self.has_tree
        if fresh.any():  # first own search: root created from the current position (MCTS_model.py:223-228)
            own, opp = _pack(states, players)
            e.set_roots(torch.from_numpy(own).to(dev), torch.from_numpy(opp).to(dev),
                        torch.from_numpy(players.astype(np.int8)).to(dev), torch.from_numpy(fresh.astype(np.uint8)).to(dev))
            self.has_tree |= fresh
        e.begin_search(mask)
        e.step()
        for _ in range(sims + 1):
            if not self.stub:
                self.evaluate()
                if self.record is not None:
                    self.record(self)  # test hook: sees (nn_input, priors, values, phases) of this evaluation
            e.step()
        assert e.counters()["active"] == 0, "search did not finish"
        self.counts = e.root_stats()["counts"].cpu().numpy()

    def pick(self, i, u):
        counts = self.counts[i].astype(np.float32)
        return alphabeta.tie_pick(np.where(counts == counts.max())[0], u)  # MCTS_model.py:249-255, then np.argmax (eval.py:161)


class _AlphaBetaSide:
    """An AlphaBetaPlayer in the arena: one oth_alphabeta launch over the matches it moves in; it keeps no tree."""

    def __init__(self, player, n, device):
        self.player, self.device = player, device
        self.has_tree = np.zeros(n, bool)  # never advanced
        self.values = np.full((n, 65), alphabeta.NONE, np.int32)

    def search(self, mask_np, states, players, sims):
        idx = np.nonzero(mask_np)[0]
        own, opp = _pack(states[idx], players[idx])
        p = self.player
        values, _, _ = alphabeta.search(torch.from_numpy(own).to(self.device), torch.from_numpy(opp).to(self.device),
                                        p.depth, p.exact_empties)
        self.values[idx] = values.cpu().numpy()

    def pick(self, i, u):
        return alphabeta.pick(self.values[i], self.player.margin, u)


def _side(policy, args, n, device, lanes, dtype):
    return _AlphaBetaSide(policy, n, device) if isinstance(policy, AlphaBetaPlayer) else _Side(policy, args, n, device, lanes, dtype)


def play_matches_batched(policy_a, policy_b, args, n_matches, *, device="cuda:0", lanes=None, dtype=torch.bfloat16, record=None,
                         max_plies=128, u_tie=None):
    """n_matches concurrent games; match i: policy_a plays +1 if i is even, policy_b otherwise
    (eval.py:115-126).  Either policy, or both, may be a network, a ``DeviceStubPolicy`` or an ``AlphaBetaPlayer``.
    Returns (results, log): results[i] in {"A", "B", "Draw"} from policy_a's
    point of view as evaluate_models_parallel counts them; log holds per-match actions and tie uniforms.
    ``u_tie`` float64 [n_matches, max_plies]: the tie-pick uniforms to use instead of drawing them (replay of a
    logged match, or of a match of the reference whose np.random.choice(best_actions) picks were tapped)."""
    env = OthelloGameNew(8)
    n = int(n_matches)
    sims = int(args["num_simulations"])
    A = _side(policy_a, args, n, device, lanes, dtype)
    B = _side(policy_b, args, n, device, lanes, dtype)
    A.record = B.record = record
    a_first = (np.arange(n) % 2 == 0)
    states = np.repeat(env.get_initial_state()[None], n, 0)
    players = np.ones(n, np.int8)
    active = np.ones(n, bool)
    results = [None] * n
    log = dict(actions=np.full((n, max_plies), -1, np.int32), u_tie=np.zeros((n, max_plies)), plies=np.zeros(n, np.int32))
    for ply in range(max_plies):
        if not active.any():
            break
        a_moves = active & (a_first == (players == 1))  # first tree moves for +1 (eval.py:153-160)
        b_moves = active & ~a_moves
        if a_moves.any():
            A.search(a_moves, states, players, sims)
        if b_moves.any():
            B.search(b_moves, states, players, sims)
        actions = np.full(n, -1, np.int32)
        for i in np.nonzero(active)[0]:
            u = np.random.random_sample() if u_tie is None else float(u_tie[i, ply])
            actions[i] = (A if a_moves[i] else B).pick(i, u)
            log["u_tie"][i, ply] = u
            log["actions"][i, ply] = actions[i]
        idx = np.nonzero(active)[0]
        nxt = env.next_state_batch(states[idx], actions[idx], players[idx])
        rew, done = env.value_and_terminated_batch(nxt, players[idx])
        states[idx] = nxt
        log["plies"][idx] = ply + 1
        for j, i in enumerate(idx):
            if done[j]:
                first_won = (rew[j] == 1) == (players[i] == 1)
                res = "Draw" if rew[j] == 0 else ("A" if first_won else "B")  # A/B = first/second tree (eval.py:165-173)
                if not a_first[i] and res != "Draw":  # _run_one_match inverts odd matches (eval.py:127-131)
                    res = "B" if res == "A" else "A"
                results[i] = res
                active[i] = False
        # both trees follow the move (eval.py:175-176); a tree that was never searched stays None
        for side in (A, B):
            act = np.where(active & side.has_tree, actions, -1).astype(np.int32)
            if (act >= 0).any():
                side.eng.advance(torch.from_numpy(act).to(side.eng.device))
                side.eng.raise_on_error()
        players[active] = -players[active]
    return results, log


@torch.no_grad()
def evaluate_models_parallel(board_size, args, policy_state, best_policy_state, n_matches=20, **kw):
    """Drop-in for eval.py:40-74: returns (win rate of the candidate, win rate of the incumbent)."""
    assert board_size == 8
    nets = []
    for cls, cfg, sd in (policy_state, best_policy_state):
        net = cls(**cfg)
        net.load_state_dict(sd)
        nets.append(net.eval())
    results, _ = play_matches_batched(nets[0], nets[1], args, n_matches, **kw)
    return results.count("A") / n_matches, results.count("B") / n_matches


def evaluate_vs_alphabeta(policy, args, n_matches, player=AlphaBetaPlayer(), **kw):
    """A network's strength on a fixed scale: ``n_matches`` arena matches of ``policy`` (MCTS with ``args``) against
    an ``AlphaBetaPlayer``, colours alternating.  Returns ({"win", "draw", "loss"} rates of the network, the match
    log of ``play_matches_batched``)."""
    results, log = play_matches_batched(policy, player, args, n_matches, **kw)
    n = int(n_matches)
    return {"win": results.count("A") / n, "draw": results.count("Draw") / n, "loss": results.count("B") / n}, log
