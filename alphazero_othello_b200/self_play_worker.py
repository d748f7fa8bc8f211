"""Self-play on the B200 engine behind the reference's worker surface.

* ``one_self_play(args_tuple)`` -- same signature, RNG call order and return value as
  ``self_play_worker.py:38-88`` (one game, host loop over the GPU-resident tree).
* ``collect_self_play_games(policy, args, n_games, ...)`` -- the batched replacement of
  ``Trainer.collect_self_play_games`` (train.py:199-225): thousands of concurrent games,
  one network evaluation per simulation per game, moves sampled / trees re-rooted /
  lambda-returns formed in-kernel; returns the same per-game lists of
  ``(state int8[8,8], pi float32[65], value float)`` that ``Trainer._extend_buffer``
  (train.py:136-140) consumes.
"""
import numpy as np
import torch

from . import _lib, endgame, symmetry
from .MCTS_model import MCTS
from .engine import BatchedPolicy, MctsEngine, SelfPlayRunner, private_copy, split_games
from .envs.othello import OthelloGameNew as OthelloGame


def get_training_data(trajectory, winning_player, lambd=1.0):
    """Value targets for one finished game: the backward lambda-return of self_play_worker.py:8-35.
    ``trajectory`` rows are ``(state, pi, player, root_value)``; returns ``(state, pi, G_t)`` rows.
    The batched engine evaluates the same recurrence in-kernel (emit_game, csrc/mcts_kernels.cu)."""
    def outcome(p):
        return 0.0 if winning_player == 0 else (1.0 if p == winning_player else -1.0)

    rows = [None] * len(trajectory)
    later = None  # (G_{t+1}, player_{t+1})
    for t in reversed(range(len(trajectory))):
        state, pi, player, v_root = trajectory[t]
        if later is None:
            g = outcome(player)
        else:
            g_next, p_next = later
            sign = 1.0 if player == p_next else -1.0
            g = (1.0 - lambd) * v_root + lambd * sign * g_next
        rows[t] = (state, pi, g)
        later = (g, player)
    return rows


def _rebuild_policy(policy_state):
    cls, cfg, weights = policy_state
    net = cls(**cfg)
    net.load_state_dict(weights)
    net.eval()
    return net


@torch.no_grad()
def one_self_play(args_tuple):
    """One complete game on the GPU-resident tree, behind the reference's worker signature
    (self_play_worker.py:38-88): ``(board_size, args, (policy_class, policy_config, state_dict),
    inference_cache) -> [(state int8[8,8], pi float32[65], value float), ...]``.  np.random is
    consumed in the reference's order (root noise, tie picks, one ``choice(65, p)`` per ply)."""
    board_size, args, policy_state, inference_cache = args_tuple
    env = OthelloGame(board_size)
    search = MCTS(env, args, _rebuild_policy(policy_state), dirichlet_alpha=args["dirichlet_alpha"],
                  dirichlet_epsilon=args["dirichlet_epsilon"], inference_cache=inference_cache)
    history = []
    board, mover = env.get_initial_state(), 1
    while True:
        exploring = len(history) < args["num_exploratory_moves"]
        pi = search.policy_improve_step(board, mover, temp=args["mcts_temperature"] if exploring else 0.0)
        history.append((board.copy() * mover, pi.copy(), mover, search.root.value))
        move = np.random.choice(env.action_size, p=pi)
        search.make_move(move)
        board = env.get_next_state(board, move, mover)
        reward, over = env.get_value_and_terminated(board, move, mover)
        if over:
            winner = 0 if reward == 0 else (mover if reward > 0 else env.get_opponent(mover))
            return get_training_data(history, winner, args["lambda"])
        mover = env.get_opponent(mover)


def collect_self_play_games(policy, args, n_games, *, n_slots=None, device="cuda:0", dtype=torch.bfloat16, seed=0,
                            game_id_base=0, fold=True, use_graph=True, return_raw=False, dedup="auto", solve_empties=0,
                            leaf_symmetry=None):
    """Play ``n_games`` self-play games with ``policy`` (a torch module) on one GPU.  With ``solve_empties`` > 0 the
    value target of every position with at most that many empty squares is its solved win / draw / loss
    (``endgame.relabel``) instead of its lambda-return.  ``leaf_symmetry="random"``: the network sees every leaf in
    one of its eight orientations, drawn from (``seed``, position) (``engine.SelfPlayRunner``)."""
    from .Models import fold_for_inference
    symmetry.check_mode(leaf_symmetry, ("random",))
    if not 0 <= int(solve_empties) <= endgame.MAX_EMPTIES:
        raise ValueError(f"solve_empties must be in 0..{endgame.MAX_EMPTIES}, got {solve_empties}")
    n_slots = int(n_slots or min(n_games, 4096))
    gps = -(-n_games // n_slots)
    eng = MctsEngine(n_slots, args, self_play=True, eval_kind=_lib.EVAL_EXTERNAL, games_per_slot=gps, device=device,
                     seed=seed, game_id_base=game_id_base)
    net = private_copy(policy, device)  # the trainer's module stays where it is, in the mode it is in
    if fold:
        net = fold_for_inference(net, dtype)
        ev = BatchedPolicy(net, device, torch.float32)
    else:
        ev = BatchedPolicy(net, device, dtype)
    out = SelfPlayRunner(eng, ev, use_graph=use_graph, dedup=dedup, leaf_symmetry=leaf_symmetry).play()
    eng.raise_on_error()
    if solve_empties:
        out = endgame.relabel(out, solve_empties, device=device)
    return out if return_raw else split_games(out)[:n_games]


def collect_self_play_games_distributed(policy, args, n_games_per_rank, *, n_slots=None, dtype=torch.bfloat16, seed=0, version=0,
                                        leaf_symmetry=None):
    """Sharded ``collect_self_play_games`` (launch with torchrun, one process per GPU, NCCL initialised):
    rank 0's weights are broadcast, every rank plays its own game ids with no collective on the
    search path, and the replay tuples are gathered to rank 0, which gets the per-game lists
    (other ranks get None).  BASELINE config C5 is this with 16 384 slots per rank on 8 GPUs."""
    symmetry.check_mode(leaf_symmetry, ("random",))
    import torch.distributed as dist
    from . import parallel
    from .Models import fold_for_inference
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", torch.cuda.current_device())
    net = private_copy(policy, dev)
    parallel.broadcast_weights(net, src=0, version=version)
    n_slots = int(n_slots or min(n_games_per_rank, 4096))
    gps = -(-n_games_per_rank // n_slots)
    base, stride = parallel.shard_game_ids(rank, world, n_slots)
    eng = MctsEngine(n_slots, args, self_play=True, eval_kind=_lib.EVAL_EXTERNAL, games_per_slot=gps, device=dev, seed=seed,
                     game_id_base=base, game_id_stride=stride)
    out = SelfPlayRunner(eng, BatchedPolicy(fold_for_inference(net, dtype), dev, torch.float32), dedup="auto",
                         leaf_symmetry=leaf_symmetry).play()
    eng.raise_on_error()
    merged = parallel.gather_replay({k: v.to(dev) for k, v in out.items() if k != "states"}, dst=0, device=dev)
    if merged is None:
        return None
    n = merged["values"].numel()
    states = torch.empty((n, 8, 8), dtype=torch.int8, device=dev)
    if n:
        import ctypes as C
        _lib.check(_lib.lib().oth_unpack_canonical(merged["boards"].contiguous().data_ptr(), states.data_ptr(), n,
                                                   C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    merged["states"] = states
    return split_games({k: v.cpu() for k, v in merged.items()})
