/*
 * othello_b200.h -- C ABI of libothello_b200.so, the B200 (sm_100a) self-play
 * hot path behind the call surface of AfoninAndrei/alphaZero-Othello.
 *
 * The reference is pure Python and has no FFI; its boundary is duck typing on
 * three surfaces (envs/game.py:5-57 as implemented by envs/othello.py:309-460,
 * MCTS_model.py:172-274, self_play_worker.py:38-88).  Each entry point below
 * names the reference code it replaces.  INTEGRATION.md shows the ctypes
 * binding a maintainer adds.
 *
 * Conventions
 *  - plain pointers and sizes only; `stream` is a cudaStream_t passed as void*
 *    (NULL = the legacy default stream);
 *  - oth_* functions without "_host" take DEVICE pointers, never allocate and
 *    never synchronise: the caller owns every buffer (oth_mcts_buffer_bytes
 *    tells it how large each must be);
 *  - oth_host_* functions take HOST pointers and do H2D copy, kernel, D2H copy
 *    and a stream synchronise inside the call;
 *  - return value 0 = OK, < 0 = an OTH_E_* code (oth_error_string decodes);
 *  - bitboards: bit i = square index i = row*8+col = the Game API's action
 *    index; `own` = discs of the side to move, `opp` = the other side.
 */
#ifndef OTHELLO_B200_H
#define OTHELLO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OTH_ABI_VERSION 2
#define OTH_NUM_ACTIONS 65 /* envs/othello.py:325 action_size: 64 squares + pass */
#define OTH_PASS 64
#define OTH_MAX_PLIES 128 /* trace / trajectory rows per game */
#define OTH_MAX_CHILDREN 40 /* >= 33, the largest legal-move count on 8x8 */

enum {
    OTH_OK = 0,
    OTH_E_CUDA = -1,     /* a CUDA runtime call failed (see oth_last_cuda_error) */
    OTH_E_ARG = -2,      /* bad argument */
    OTH_E_ILLEGAL = -3,  /* illegal move: the reference's ValueError, envs/othello.py:419-421 */
    OTH_E_NO_DEVICE = -4 /* no CUDA device: there is no CPU fallback */
};

/* step flags (oth_step / oth_host_next_state out_flags) */
#define OTH_F_ILLEGAL 1u  /* action not legal: outputs hold the unchanged position */
#define OTH_F_TERMINAL 2u /* neither side can move after the action */
#define OTH_F_WIN 4u      /* terminal and the mover has more discs */
#define OTH_F_LOSS 8u     /* terminal and the mover has fewer discs */
#define OTH_F_MUST_PASS 16u /* next side to move has no board move (and game not over) */

int oth_abi_version(void);
const char* oth_error_string(int code);
const char* oth_last_cuda_error(void);
int oth_device_count(void);

/* ------------------------------------------------------------------ env -- */

/* _BitBoard.valid_mask / _legal_moves, envs/othello.py:157-169, batched. */
int oth_legal_moves(const uint64_t* own, const uint64_t* opp, uint64_t* out_moves, int64_t n, void* stream);

/* _BitBoard.make_move (envs/othello.py:171-200) + the terminal test of
 * get_value_and_terminated (:435-454), batched.  action 0..63 or 64 = pass.
 * Outputs are from the NEXT mover's perspective (sides swapped), plus that
 * mover's legal set and OTH_F_* flags (value is from the MOVER's side, as
 * self_play_worker.py:78-82 reads it). */
int oth_step(const uint64_t* own, const uint64_t* opp, const uint8_t* action, uint64_t* out_own, uint64_t* out_opp,
             uint64_t* out_moves, uint8_t* out_flags, int64_t n, void* stream);

/* Config C1: n_games uniform-random playouts from the start position, one
 * thread per game, whole game in registers (the loop of
 * envs/test_equivalence_game.py:158-190 / MCTS._rollout MCTS_model.py:276-303).
 * Game g draws from Philox4x32-10 keyed (seed; game_id_base+g, ply).
 * out_score[g]  = final disc difference for +1 (get_score(state, 1)),
 * out_plies[g]  = plies played (passes count), out_final[2g..] = (+1 discs,
 * -1 discs).  The first n_trace games also write their action per ply to
 * trace_actions[g][OTH_MAX_PLIES] (0xFF padded) and the mover's legal set to
 * trace_moves[g][OTH_MAX_PLIES].  counters[0] += total plies. Any output
 * pointer may be NULL. */
int oth_rollout(uint64_t seed, uint64_t game_id_base, int64_t n_games, int32_t* out_score, int32_t* out_plies,
                uint64_t* out_final, int64_t n_trace, uint8_t* trace_actions, uint64_t* trace_moves,
                unsigned long long* counters, void* stream);

/* OthelloGameNew._np_to_bitboards / _bitboards_to_np, envs/othello.py:358-388:
 * int8[n,64] boards (+ the player whose discs become `own`) <-> bitboards. */
int oth_pack_states(const int8_t* states, const int8_t* players, uint64_t* own, uint64_t* opp, int64_t n, void* stream);
int oth_unpack_states(const uint64_t* own, const uint64_t* opp, const int8_t* players, int8_t* states, int64_t n,
                      void* stream);

/* get_valid_moves on int8 boards, envs/othello.py:394-411: uint8[n,65]. */
int oth_valid_moves_i8(const int8_t* states, const int8_t* players, uint8_t* out_masks, int64_t n, void* stream);

/* get_random_symmetry (envs/othello.py:501-526) / get_symmetries (:286-298)
 * for given per-sample k (quarter turns, np.rot90) and flip (np.fliplr):
 * float32 boards [n,64] and policies [n,65]. */
int oth_symmetry(const int8_t* states, const float* pis, const int32_t* ks, const uint8_t* flips, float* out_states,
                 float* out_pis, int64_t n, void* stream);

/* Host-buffer forms of the Game API (what envs.othello.OthelloGameNew calls). */
int oth_host_valid_moves(const int8_t* states, const int8_t* players, uint8_t* out_masks, int64_t n);
int oth_host_next_state(const int8_t* states, const int32_t* actions, const int8_t* players, int8_t* out_states,
                        uint8_t* out_flags, int64_t n);
int oth_host_value_terminated(const int8_t* states, const int8_t* players, int8_t* out_values, uint8_t* out_terms,
                              int64_t n);
int oth_host_symmetry(const int8_t* states, const float* pis, const int32_t* ks, const uint8_t* flips,
                      float* out_states, float* out_pis, int64_t n);
int oth_host_rollout(uint64_t seed, uint64_t game_id_base, int64_t n_games, int32_t* out_score, int32_t* out_plies,
                     uint64_t* out_final, int64_t n_trace, uint8_t* trace_actions, uint64_t* trace_moves,
                     unsigned long long* total_plies, float* kernel_ms);

/* ------------------------------------------------------- alpha-beta player -- */

/* A fixed-depth alpha-beta player: an absolute yardstick for the arena (eval.evaluate_vs_alphabeta).
 *
 * For each position (own, opp; own to move) and each legal root action a (board moves, or the pass when the
 * mover has none), out_values[i][a] = the negamax value of the position after a, from the root mover's side;
 * every other entry is OTH_AB_NONE.  out_best[i] = the LOWEST action whose value is the maximum, -1 when the
 * root is terminal.  out_nodes[i][a] (may be NULL) = positions visited below action a, the position after a
 * included: > 0 exactly for the legal actions.  It depends on how the root is searched (below), not on the launch.
 *
 * Search semantics (the values are unique: any correct negamax gives them, in any order, with any pruning):
 *  - every ply costs one depth level; a forced pass is a ply;
 *  - a position where neither side can move is terminal: OTH_AB_WIN_SCALE * (own discs - opp discs), empty
 *    squares not awarded (get_score);
 *  - at depth 0 a non-terminal position scores, from the side to move,
 *      h = sum_sq W[sq] * (own_sq - opp_sq) + 10 * (#legal(own, opp) - #legal(opp, own)),
 *    W the D4-symmetric square table, rows 0-3 (rows 4-7 mirror them):
 *      100 -20  10   5   5  10 -20 100
 *      -20 -50  -2  -2  -2  -2 -50 -20
 *       10  -2  -1  -1  -1  -1  -2  10
 *        5  -2  -1  -1  -1  -1  -2   5
 *    |h| < 1 300, below one disc of a decided game; all arithmetic is int32;
 *  - a root with <= exact_empties empty squares is searched to the end of the game (no depth limit).
 * depth 1..OTH_AB_MAX_DEPTH, exact_empties 0..OTH_AB_MAX_EXACT, else OTH_E_ARG (checked before any device
 * call).
 *
 * The search, one warp per position: a depth-limited root, or an exact one with <= 11 empties, gives each root
 * action to one lane, which runs a full-window alpha-beta below it.  An exact root with 12..exact_empties empties is
 * split one level further (Young Brothers Wait): below root action a, the first reply in the search's move order is
 * searched with a full window, which bounds the value of the position after a; every other reply is then its own
 * task, searched with the window that bound leaves (fail-hard), and the warp's lanes share these tasks.  On that
 * path out_nodes counts the positions of all these searches.  The caps bound every launch: 4 096 mid-game positions
 * at depth 7 take 1.9 s on a B200 (1 000 W), 4 096 exact endgames with 12 empties 2.0 s.  Depth 8 (11.7 s) and
 * 13 empties (10.7 s) miss a 4 s budget even on the split search (DESIGN.md 4). */
#define OTH_AB_NONE INT32_MIN
#define OTH_AB_WIN_SCALE 10000
#define OTH_AB_MAX_DEPTH 7
#define OTH_AB_MAX_EXACT 12
int oth_alphabeta(const uint64_t* own, const uint64_t* opp, int64_t n, int32_t depth, int32_t exact_empties,
                  int32_t* out_values /* [n][65] */, int32_t* out_best /* [n] */, uint64_t* out_nodes /* [n][65] */,
                  void* stream);
int oth_host_alphabeta(const uint64_t* own, const uint64_t* opp, int64_t n, int32_t depth, int32_t exact_empties,
                       int32_t* out_values, int32_t* out_best, uint64_t* out_nodes);

/* ------------------------------------------------------- endgame solver -- */

/* The game-theoretic result of endgame positions: the truth a self-play value target can be replaced with
 * (endgame.relabel).
 *
 * For each position (own, opp; own to move) with at most max_empties empty squares, out_wld[i] = +1, 0 or -1: the
 * result for own under perfect play by both sides to the end of the game, forced passes included.  The result is the
 * sign of the final disc difference, empty squares not awarded (get_value_and_terminated; the sign of oth_alphabeta's
 * exact values).  A terminal position gets its own result.  A position with more empty squares gets
 * OTH_WLD_UNSOLVED and 0 nodes.  out_nodes[i] (may be NULL) = positions the search visited, the root included; it
 * depends on the position alone, not on the launch.  max_empties 0..OTH_SOLVE_MAX_EMPTIES, else OTH_E_ARG (checked
 * before any device call).
 *
 * The search, one thread per position: a sequential alpha-beta with the window (-1, +1) on that sign, which stops at
 * the first winning move; children are searched fastest-first (fewest replies for the opponent) from 7 empty squares
 * up, in the alpha-beta player's static order below.  The cap bounds a launch: 4 096 positions with 14 empties took
 * 1.53 s on a B200 (1 000 W), with 15 empties 7.7 s and with 16 empties 54 s (DESIGN.md 4). */
#define OTH_SOLVE_MAX_EMPTIES 14
#define OTH_WLD_UNSOLVED (-128)
int oth_solve_wld(const uint64_t* own, const uint64_t* opp, int64_t n, int32_t max_empties, int8_t* out_wld /* [n] */,
                  uint64_t* out_nodes /* [n] */, void* stream);
int oth_host_solve_wld(const uint64_t* own, const uint64_t* opp, int64_t n, int32_t max_empties, int8_t* out_wld,
                       uint64_t* out_nodes);

/* INT32-ALU roofline probe:dependent-free LOP3/IADD3/SHF mix; returns the
 * measured thread-instructions per second in *out_ips (BASELINE.md 3). */
int oth_host_int32_peak(double* out_ips, float* kernel_ms);

/* Random-access HBM probe: independent pseudo-random reads of chunk_bytes (32, 64 or 128) from a
 * buffer_bytes buffer (>> L2), the access pattern of tree records; GB/s in *out_gbs. */
int oth_host_random_read_probe(int64_t buffer_bytes, int32_t chunk_bytes, double* out_gbs, float* kernel_ms);

/* ----------------------------------------------------------------- MCTS -- */

/* evaluator kinds */
#define OTH_EVAL_EXTERNAL 0 /* policy/value net outside the library (PyTorch) */
#define OTH_EVAL_STUB_A 1   /* uniform priors, value 0 (SURVEY Appendix A) */
#define OTH_EVAL_STUB_B 2   /* weighted-sum stub (SURVEY Appendix A) */
#define OTH_EVAL_STUB_H 3   /* hash stub (oracle/othello_oracle.c orc_stub_h) */
#define OTH_EVAL_ROLLOUT 4  /* policy=None: uniform priors + one random playout (MCTS_model.py:276-303, 332-335) */

/* per-slot phases (oth_mcts_ctl.phase) */
#define OTH_PH_RUN 0       /* searching, nothing pending */
#define OTH_PH_WAIT_EVAL 1 /* a leaf sits in nn_input[slot]; needs priors/values[slot] */
#define OTH_PH_IDLE 2      /* manual mode: num_simulations done, waiting for oth_mcts_advance */
#define OTH_PH_DONE 3      /* self-play mode: this slot has played all its games */
#define OTH_PH_ERROR 4     /* see ctl.error */
#define OTH_PH_MOVE 5      /* transient inside oth_mcts_step: simulations done, the move kernel takes over */

/* ctl.error bits */
#define OTH_ERR_NODE_OVERFLOW 1
#define OTH_ERR_PATH_OVERFLOW 2
#define OTH_ERR_OUT_OVERFLOW 4
#define OTH_ERR_PLY_OVERFLOW 8
#define OTH_ERR_BAD_ACTION 16 /* MCTS.make_move KeyError, MCTS_model.py:214 */
#define OTH_ERR_NONFINITE 32  /* the evaluator handed a NaN / infinite prior or value to this slot: the slot stops
                                 (nothing non-finite ever enters a tree; the reference would carry on with NaN scores) */
#define OTH_ERR_DEBUG 64      /* an index / ownership assertion of the -DOTH_DEBUG build failed */

typedef struct oth_mcts_config {
    int32_t n_slots;          /* concurrent games on this GPU */
    int32_t node_cap;         /* nodes per arena per slot (two arenas per slot) */
    int32_t path_cap;         /* max search depth (<= 128) */
    int32_t num_simulations;  /* args["num_simulations"], MCTS_model.py:237 */
    int32_t num_exploratory_moves; /* self_play_worker.py:66-67 */
    int32_t eval_kind;        /* OTH_EVAL_* */
    int32_t self_play;        /* 1: moves are sampled and games restarted in-kernel (one_self_play);
                                 0: manual -- the host calls oth_mcts_advance (MCTS.make_move) */
    int32_t games_per_slot;   /* self-play: games each slot plays (<0 = endless) */
    int32_t max_inline_sims;  /* simulations a slot may finish inside one launch without an
                                 external evaluation (terminal hits; all of them with a stub) */
    int32_t inject_random;    /* 1: read noise / u_move / u_tie from the buffers instead of Philox */
    int32_t lanes;            /* threads cooperating on one slot: 8, 16 or 32 */
    int32_t hot_path;         /* path entries carried in the 256-byte hot record (1..52, 0 = 52); deeper entries
                                 live in OTH_BUF_PATH.  A tuning / test knob: small values force the HBM path tail */
    int32_t split_stub;       /* device evaluators (OTH_EVAL_STUB_*) only.  0: one monolithic kernel runs whole
                                 simulations back to back; 1: the production kernel pair -- the 64-register step
                                 kernel expands with the stub's output, descends and parks the next leaf (one
                                 evaluation per slot per launch), the move kernel plays the moves */
    int32_t move_launch;      /* form of the move kernel that follows every step kernel.  0: it scans the move flags;
                                 1: the step kernel lists the due slots, the move kernel exits at once when the list
                                 is empty and otherwise gives one warp to each listed slot */
    int32_t reserved0;
    int64_t out_pos_cap;      /* replay tuples the output ring can hold */
    int64_t out_game_cap;     /* finished-game descriptors it can hold */
    double c_puct;            /* args["c_puct"], MCTS_model.py:131,136 */
    double dirichlet_alpha;   /* MCTS_model.py:341 */
    double dirichlet_epsilon; /* MCTS_model.py:340-343 */
    double temperature;       /* args["mcts_temperature"] */
    double lambda;            /* args["lambda"], self_play_worker.py:8-35 */
    uint64_t seed;            /* Philox key */
    uint64_t game_id_base;    /* slot s plays games base + s + k*stride, k = 0.. */
    uint64_t game_id_stride;
    uint64_t stub_salt;       /* OTH_EVAL_STUB_H salt */
} oth_mcts_config;

/* 64-byte per-slot control block (device memory; readable by the host). */
typedef struct oth_mcts_ctl {
    int32_t phase;
    int32_t root;      /* node index of the root in the current arena */
    int32_t top;       /* bump pointer of the current arena */
    int32_t arena;     /* 0/1 */
    int32_t ply;
    int32_t sims_done; /* simulations finished for the current move */
    int32_t pending;   /* leaf awaiting evaluation */
    int32_t path_len;
    int32_t flags;     /* bit0 pending is a root initialisation (not a simulation); bit1 root priors are float64 */
    int32_t player;    /* colour to move at the root: +1 / -1 */
    int32_t games_left;
    int32_t error;
    int64_t game_id;
    int64_t reserved;
} oth_mcts_ctl;

/* Device buffers the engine works on; sizes from oth_mcts_buffer_bytes(). */
enum {
    OTH_BUF_NODES = 0,   /* 32 B/node  [slot][2][node_cap] */
    OTH_BUF_BOARDS,      /* 16 B/node  [slot][2][node_cap] */
    OTH_BUF_CTL,         /* oth_mcts_ctl [slot] */
    OTH_BUF_PATH,        /* int32 [slot][path_cap] */
    OTH_BUF_ROOT_PRIOR64,/* double [slot][OTH_MAX_CHILDREN] */
    OTH_BUF_NOISE,       /* double [slot][65]  Dirichlet draw used at ply 0 (recorded, or injected) */
    OTH_BUF_U_MOVE,      /* double [slot][OTH_MAX_PLIES] np.random.choice(65,p) uniform per ply */
    OTH_BUF_U_TIE,       /* double [slot][OTH_MAX_PLIES] temp~0 tie-pick uniform per ply */
    OTH_BUF_TRAJ_BOARD,  /* 16 B [slot][OTH_MAX_PLIES] canonical position per ply */
    OTH_BUF_TRAJ_PI,     /* float [slot][OTH_MAX_PLIES][65] */
    OTH_BUF_TRAJ_ROOTV,  /* double [slot][OTH_MAX_PLIES] mcts.root.value after the search */
    OTH_BUF_TRAJ_META,   /* int32 [slot][OTH_MAX_PLIES]: player (low byte, signed) | action << 8 */
    OTH_BUF_OUT_BOARD,   /* 16 B [out_pos_cap] */
    OTH_BUF_OUT_PI,      /* float [out_pos_cap][65] */
    OTH_BUF_OUT_VALUE,   /* double [out_pos_cap]  value target G_t */
    OTH_BUF_OUT_META,    /* int64 [out_pos_cap]: game_id << 16 | ply << 8 | (player & 0xff) */
    OTH_BUF_OUT_GAMES,   /* int64 [out_game_cap][4]: game_id, first position, n positions, winner */
    OTH_BUF_COUNTERS,    /* uint64 [16], see OTH_CNT_*: refreshed by oth_mcts_poll */
    OTH_BUF_SLOT_COUNTERS, /* uint32 [slot][16] cumulative per-slot event counters */
    OTH_BUF_HOT,         /* 256 B [slot]: pending leaf (board, legal set, meta), root header mirror, path[0..52) */
    OTH_BUF_MOVE_FLAGS,  /* uint8 [slot rounded up to 64]: slots whose move is due (step kernel -> move kernel) */
    OTH_BUF_MOVE_LIST,   /* int32 [4 + n_slots]: [0] slots due, [1] move-kernel block tickets, [4..] the due slots
                            (move_launch = 1: step kernel -> move kernel) */
    OTH_BUF_COUNT
};

enum {
    OTH_CNT_SIMS = 0,     /* simulations completed */
    OTH_CNT_EVALS,        /* leaves evaluated (network slots used) */
    OTH_CNT_TERMINAL,     /* simulations that ended on a terminal node */
    OTH_CNT_GAMES,        /* games finished */
    OTH_CNT_POSITIONS,    /* replay tuples emitted since the last drain */
    OTH_CNT_OUT_GAMES,    /* finished-game descriptors since the last drain */
    OTH_CNT_MOVES,        /* moves played */
    OTH_CNT_ERRORS,       /* slots in error (gauge, oth_mcts_poll) */
    OTH_CNT_MAX_TOP,      /* arena high-water mark over all slots */
    OTH_CNT_MAX_DEPTH,    /* deepest path seen */
    OTH_CNT_NODES,        /* nodes created */
    OTH_CNT_COPIED,       /* nodes copied by re-rooting */
    OTH_CNT_WAITING,      /* slots in OTH_PH_WAIT_EVAL (gauge, oth_mcts_poll) */
    OTH_CNT_ACTIVE,       /* slots not DONE/IDLE/ERROR (gauge, oth_mcts_poll) */
    OTH_CNT_LEVELS,       /* tree levels descended (select steps) */
    OTH_CNT_CHILDREN      /* child records scanned by select */
};

typedef struct oth_mcts_buffers {
    void* buf[OTH_BUF_COUNT];
    void* profile; /* NULL, or an oth_mcts_profile handle (othello_b200_experimental.h): per-engine launch timing */
} oth_mcts_buffers;

/* Sizes (bytes) of the OTH_BUF_* buffers for a configuration.  The caller allocates them in device
 * memory (16-byte aligned; cudaMalloc / torch give far more) and ZERO-FILLS them once before the first
 * oth_mcts_reset / oth_mcts_set_roots: a zeroed control block means "slot has no tree yet" and is
 * skipped by every kernel. */
int oth_mcts_buffer_bytes(const oth_mcts_config* cfg, int64_t* out_bytes /* [OTH_BUF_COUNT] */);

/* Start every slot on a fresh game from the initial position (one_self_play's
 * setup, self_play_worker.py:60-62) and zero the counters.  The first
 * oth_mcts_step after it consumes nothing and emits the root leaves. */
int oth_mcts_reset(const oth_mcts_config* cfg, const oth_mcts_buffers* b, void* stream);

/* Manual mode: give every slot a new tree rooted at (own, opp) with `player`
 * to move (MCTS.policy_improve_step's root creation, MCTS_model.py:223-228). */
int oth_mcts_set_roots(const oth_mcts_config* cfg, const oth_mcts_buffers* b, const uint64_t* own, const uint64_t* opp,
                       const int8_t* players, void* stream);

/* As oth_mcts_set_roots / oth_mcts_begin_search, restricted to slots with mask[slot] != 0
 * (device uint8 [n_slots]; NULL = all).  The batched arena (eval.py:134-178) uses them: in every
 * ply only the trees of the side to move search. */
int oth_mcts_set_roots_masked(const oth_mcts_config* cfg, const oth_mcts_buffers* b, const uint64_t* own, const uint64_t* opp,
                              const int8_t* players, const uint8_t* mask, void* stream);
int oth_mcts_begin_search_masked(const oth_mcts_config* cfg, const oth_mcts_buffers* b, const uint8_t* mask, void* stream);

/* Manual mode: begin a search of num_simulations on every idle slot
 * (MCTS.policy_improve_step, MCTS_model.py:234-242). */
int oth_mcts_begin_search(const oth_mcts_config* cfg, const oth_mcts_buffers* b, void* stream);

/* THE hot kernel. For each slot: consume priors[slot][65] / values[slot] for
 * its pending leaf (expand + backup: MCTS_model.py:325-360, 146-169), then run
 * PUCT descents (:362-395, 129-139) until a leaf needs the network -- its
 * canonical plane goes to nn_input[slot] -- or the move's simulations are done,
 * in which case (self-play mode) the policy target is formed (:244-274), the
 * move sampled (self_play_worker.py:64-88), the tree re-rooted (:200-215) and
 * finished games are emitted with their lambda-returns (:8-35). */
int oth_mcts_step(const oth_mcts_config* cfg, const oth_mcts_buffers* b, const float* priors, const float* values,
                  float* nn_input, void* stream);

/* oth_mcts_step with the network's tail fused in: `logits` [n_slots] rows of >= 65 raw policy logits
 * (row stride in elements) and `value_preact` [n_slots] pre-tanh values (stride in elements), both
 * float32 (is_bf16 = 0) or bfloat16 (1) -- typically views into the head GEMM outputs.  The kernel
 * applies softmax over the 65 logits (Models.py:24-25) and tanh itself.  priors_out / values_out
 * (both or neither): float32 [n_slots][65] / [n_slots] receive what it applied, for record & replay. */
int oth_mcts_step_fused(const oth_mcts_config* cfg, const oth_mcts_buffers* b, const void* logits, int64_t logits_stride,
                        const void* value_preact, int64_t value_stride, int32_t is_bf16, float* priors_out, float* values_out,
                        float* nn_input, void* stream);

/* Evaluation de-duplication.  Concurrent games that start from the same position ask, for their first plies, for
 * the same leaf positions over and over (the reference evaluates each of them: one Inference.inference call per
 * simulation per game, MCTS_model.py:325-336 / Models.py:11-31).  oth_mcts_dedup finds the DISTINCT positions among
 * the slots in OTH_PH_WAIT_EVAL, writes their canonical planes to compact_input [bucket][64] (row u = the u-th
 * distinct position) and eval_map[slot] = the row that holds the slot's position, or -1 if the slot is not waiting or
 * its position did not fit into `bucket` rows.  The caller runs the network on the `bucket` rows and hands the
 * outputs to oth_mcts_step_fused_mapped, which reads logits[eval_map[slot]]; slots mapped to -1 stay as they are and
 * are served by a later launch.  A slot's sequence of evaluated positions is unchanged, so results depend on this
 * only through the network's outputs.  stats (device int32[2]) receives {distinct pending positions, waiting slots}
 * of this batch; bucket = 0 only counts (compact_input / eval_map may be NULL).  workspace: device scratch of
 * oth_mcts_dedup_workspace_bytes(n_slots) bytes, zero-filled once by the caller. */
int oth_mcts_dedup_workspace_bytes(int32_t n_slots, int64_t* bytes);
int oth_mcts_dedup(const oth_mcts_config* cfg, const oth_mcts_buffers* b, int32_t bucket, void* workspace, int64_t workspace_bytes,
                   float* compact_input, int32_t* eval_map, int32_t* stats, void* stream);
int oth_mcts_step_fused_mapped(const oth_mcts_config* cfg, const oth_mcts_buffers* b, const void* logits, int64_t logits_stride,
                               const void* value_preact, int64_t value_stride, int32_t is_bf16, const int32_t* eval_map,
                               float* priors_out, float* values_out, float* nn_input, void* stream);

/* Refresh OTH_BUF_COUNTERS: sums the per-slot event counters and derives the gauges (WAITING /
 * ACTIVE / ERRORS / MAX_TOP) from the control blocks.  Kept out of the hot kernel; hosts call
 * it when they want totals or need to know whether to stop. */
int oth_mcts_poll(const oth_mcts_config* cfg, const oth_mcts_buffers* b, void* stream);

/* Manual mode: MCTS.make_move (MCTS_model.py:200-215) on every slot;
 * actions[slot] < 0 leaves that slot alone.  Root noise: the reference draws a fresh
 * np.random.dirichlet whenever a search starts on an unexpanded root (MCTS_model.py:234-235, 339-343).
 * When the new root is such a leaf and dirichlet_epsilon > 0, this call therefore replaces the slot's
 * OTH_BUF_NOISE row with a fresh Philox draw keyed (seed; game id, ply) -- unless inject_random is set,
 * in which case the HOST must write the row before the next oth_mcts_begin_search (the MCTS class does). */
int oth_mcts_advance(const oth_mcts_config* cfg, const oth_mcts_buffers* b, const int32_t* actions, void* stream);

/* mcts.root.* as the reference exposes it: child visit counts / values /
 * priors by action, root value and visit count, root position. NULL = skip. */
int oth_mcts_root_stats(const oth_mcts_config* cfg, const oth_mcts_buffers* b, int32_t* counts, double* child_value,
                        double* child_prior, double* root_value, int32_t* root_n, uint64_t* root_board, void* stream);

/* Replay tuples -> the reference's array form: int8 [n,64] canonical states
 * (state*player, self_play_worker.py:72) from packed boards. */
int oth_unpack_canonical(const uint64_t* boards /* [n][2] own,opp */, int8_t* states, int64_t n, void* stream);

/* ------------------------------------------------------- replay ingest -- */

/* Trainer._aggregate_duplicates (train.py:142-173) on the GPU: collapse replay tuples with the
 * same (canonical board, model version) into one sample -- mean policy re-normalised, mean value
 * -- in order of first occurrence.  Inputs: boards uint64[n][2] (own, opp), pis float32[n][65],
 * values float64[n], versions int32[n] (n < 2^31).  Outputs are sized n; *out_m (device int64)
 * receives the number of unique samples; out_counts their multiplicities.  workspace: device
 * scratch of oth_replay_aggregate_workspace_bytes(n) bytes. */
int oth_replay_aggregate_workspace_bytes(int64_t n, int64_t* bytes);
int oth_replay_aggregate(const uint64_t* boards, const float* pis, const double* values, const int32_t* versions, int64_t n,
                         void* workspace, int64_t workspace_bytes, uint64_t* out_boards, float* out_pis, float* out_values,
                         int32_t* out_versions, int32_t* out_counts, int64_t* out_m, void* stream);

/* Network boundary helper (the policy/value network itself stays PyTorch, Models.py):
 * in-place x = relu(x + bias[channel] + res) on channels-last bf16 activations -- the residual
 * epilogue of ResidualBlock.forward (Models.py:81-89) after BatchNorm folding.
 * n = element count (multiple of 8), channels multiple of 8, 16-byte aligned pointers. */
int oth_nn_bias_add_relu_bf16(void* x, const void* res, const void* bias, int64_t n, int32_t channels, void* stream);

/* Network boundary helper: im2col of the leaf planes for the 1-input-channel 3x3 stem convolution
 * (Models.py:105-107 / :179): float32 [n,64] -> bf16 [n,64,16] (9 taps + 7 zero columns), so the
 * stem runs as one GEMM with a fused bias+ReLU epilogue and writes channels-last output. */
int oth_nn_stem_im2col_bf16(const float* planes, void* cols, int64_t n, void* stream);

/* Network boundary: leaf symmetry.  Othello's value and move probabilities are invariant under the eight symmetries
 * of the square; a network only approximates that.  These kernels show it a leaf in another orientation and map
 * its outputs back.  T_s, s = 0..7, is oth_symmetry's mapping with k = s & 3 quarter turns (np.rot90) and
 * flip = s >> 2 (np.fliplr): image[e] = plane[src_s(e)] for the 64 squares.
 *
 * The symmetry id of a canonical plane (+1 = side to move, -1 = opponent, as oth_mcts_step writes nn_input) is
 *   s = philox4x32_10(seed ^ OTH_SYM_SALT; counter (own, lo32(opp), hi32(opp))).x & 7
 * with own / opp the bitboards of the +1 / -1 squares: it depends on (seed, position) only, not on the batch row,
 * the launch or a de-duplicated bucket, so a search's results do not depend on how its leaves were batched.
 *
 * oth_nn_leaf_symmetry: out_planes[i] = T_{s_i}(planes[i]) (float32 [n,64], out of place) and out_sym[i] = s_i.
 * oth_nn_unsymmetrise_logits: in place, for the 64 square entries of each of n rows (row stride in elements, >= 65;
 *   float32, or bfloat16 when is_bf16): row[src_s(e)] = row[e], so T_s of the result is the row the network gave.
 *   Entry 64 (pass) and padding columns are untouched.  Softmax commutes with it: unsymmetrising the logits gives
 *   the priors of unsymmetrising after the softmax.
 * oth_nn_symmetry_images: out[i][j] = T_j(planes[i]), float32 [n,8,64].
 * oth_nn_symmetry_mean: rows 8i+j (j = 0..7) of logits (float32, row stride >= 65) and values (float32, stride >= 1)
 *   are the network's logits and tanh'd value for image j of leaf i; priors[i] (float32 [n,65]) =
 *   (1/8) sum_j unsym_j(softmax(logits[8i+j])) and out_values[i] = (1/8) sum_j values[8i+j], summed in the
 *   order j = 0..7.
 * Bad sizes, strides, NULL or misaligned pointers return OTH_E_ARG before any device call; n = 0 is a no-op. */
#define OTH_SYM_SALT 0x73796D6D65747279ull /* "symmetry" */
int oth_nn_leaf_symmetry(const float* planes, int64_t n, uint64_t seed, float* out_planes, uint8_t* out_sym, void* stream);
int oth_nn_unsymmetrise_logits(void* logits, int64_t stride, int32_t is_bf16, const uint8_t* sym, int64_t n, void* stream);
int oth_nn_symmetry_images(const float* planes, int64_t n, float* out, void* stream);
int oth_nn_symmetry_mean(const float* logits, int64_t stride, const float* values, int64_t value_stride, int64_t n,
                         float* priors, float* out_values, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OTHELLO_B200_H */
