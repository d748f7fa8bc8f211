// Batched fixed-depth alpha-beta player (oth_alphabeta): a fixed yardstick opponent for the arena.
//
// One warp per position, two kernels that split the roots of a launch between them:
//  - k_alphabeta (depth-limited roots, and exact ones with <= 11 empties): lane l searches the root actions of rank l,
//    l+32 (ascending action order) with a full-window alpha-beta below each of them;
//  - k_alphabeta_split (exact roots with 12 or more empties): the Young Brothers Wait split one level below each root
//    action, so the warp's lanes share (root action, reply) tasks instead of idling beside the longest root action.
// Either way every root value is the exact negamax value whatever the move ordering inside a subtree.  The search
// semantics (ply = one depth level, forced pass included, terminal = 10 000 x disc difference, depth-0 heuristic) are
// defined once, in ab_leaf() / ab_subtree() below, and documented in include/othello_b200.h;
// tests/alphabeta_oracle.c restates them on the CPU oracle's mailbox boards.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/othello_b200.h"
#include "bitboard.cuh"
#include "common.cuh"

using namespace oth;

namespace {

// Explicit per-lane stack: the ancestors of the current node.  An exact search from <= OTH_AB_MAX_EXACT empties
// visits at most 2*empties plies below the root action (a forced pass may precede every move), a depth-limited one
// at most OTH_AB_MAX_DEPTH - 1.
constexpr int AB_STACK = 2 * OTH_AB_MAX_EXACT + 2;
static_assert(AB_STACK >= OTH_AB_MAX_DEPTH, "stack shorter than the depth cap");
// The most empties k_alphabeta solves exactly.  Its roots keep their values and node counts whatever the cap above.
constexpr int AB_SEQ_MAX_EXACT = 11;
constexpr int AB_INF = 1 << 30;   // > every value: |terminal| <= 640 000, |heuristic| < 1 300
constexpr u64 PASS_ONLY = ~0ULL;  // "remaining moves" of a node whose only action is the pass (no real move set is full)

// Square-weight classes of the D4-symmetric table W (header): mask of the squares with each weight.
constexpr u64 W_100 = 0x8100000000000081ULL, W_M20 = 0x4281000000008142ULL, W_M50 = 0x0042000000004200ULL,
              W_10 = 0x2400810000810024ULL, W_5 = 0x1800008181000018ULL, W_M2 = 0x003C424242423C00ULL,
              W_M1 = 0x00003C3C3C3C0000ULL;
// Move ordering inside a subtree (any order gives the same values): corners, then squares not next to a corner,
// then the X- and C-squares.
constexpr u64 ORDER_NEAR_CORNER = W_M20 | W_M50;

__device__ __forceinline__ int wdiff(u64 own, u64 opp, u64 m) { return __popcll(own & m) - __popcll(opp & m); }

// Depth-0 score of a non-terminal position, from the side to move (OTH_AB_* in the header).
__device__ __forceinline__ int ab_heuristic(u64 own, u64 opp, int own_mob, int opp_mob)
{
    return 100 * wdiff(own, opp, W_100) - 20 * wdiff(own, opp, W_M20) - 50 * wdiff(own, opp, W_M50) +
           10 * wdiff(own, opp, W_10) + 5 * wdiff(own, opp, W_5) - 2 * wdiff(own, opp, W_M2) - wdiff(own, opp, W_M1) +
           10 * (own_mob - opp_mob);
}

// Classifies a node: returns true with *value set when it is a leaf (terminal, or depth 0), else false with
// *rem = its actions (PASS_ONLY for a forced pass).
__device__ __forceinline__ bool ab_leaf(u64 own, u64 opp, int depth, int* value, u64* rem)
{
    const u64 m = legal_moves(own, opp);
    if (m) {
        if (depth > 0) {
            *rem = m;
            return false;
        }
        *value = ab_heuristic(own, opp, __popcll(m), __popcll(legal_moves(opp, own)));
        return true;
    }
    const u64 m2 = legal_moves(opp, own);
    if (!m2) {
        *value = OTH_AB_WIN_SCALE * (__popcll(own) - __popcll(opp));
        return true;
    }
    if (depth > 0) {
        *rem = PASS_ONLY;
        return false;
    }
    *value = ab_heuristic(own, opp, 0, __popcll(m2));
    return true;
}

// Takes the next action out of *rem (ordered as above) and returns the child position.
__device__ __forceinline__ Board ab_next_child(u64 own, u64 opp, u64* rem)
{
    if (*rem == PASS_ONLY) {
        *rem = 0;
        return apply_move(own, opp, OTH_PASS, 0);
    }
    const u64 r = *rem;
    const u64 corner = r & W_100, plain = r & ~(W_100 | ORDER_NEAR_CORNER);
    const u64 pick = corner ? corner : (plain ? plain : r);
    const int sq = __ffsll((long long)pick) - 1;
    *rem = r & ~(1ULL << sq);
    return apply_move(own, opp, sq, flips(own, opp, 1ULL << sq));
}

struct Frame {
    u64 own, opp, rem;
    int alpha, beta;
};

// Negamax value of (own, opp) searched `depth` plies deep: iterative fail-hard alpha-beta with the window
// (alpha, beta) at the top, exact when it lies inside the window, beta when it is >= beta.  *nodes += positions visited.
__device__ int ab_subtree(u64 own, u64 opp, int depth, int alpha, int beta, unsigned long long* nodes)
{
    Frame st[AB_STACK];
    int sp = 0, v;
    u64 rem;
    unsigned long long cnt = 0;
    for (;;) {
        // enter (own, opp) at level sp with window (alpha, beta)
        cnt++;
        if (!ab_leaf(own, opp, depth - sp, &v, &rem)) {
            const Board c = ab_next_child(own, opp, &rem);
            st[sp++] = Frame{own, opp, rem, alpha, beta};
            own = c.own;
            opp = c.opp;
            const int a = alpha;
            alpha = -beta;
            beta = -a;
            continue;
        }
        // v = value of the node just finished; hand it to its ancestors until one has a child left to search
        for (;;) {
            if (sp == 0) {
                *nodes += cnt;
                return v;
            }
            Frame& f = st[--sp];
            const int s = -v;
            if (s >= f.beta) {
                v = f.beta;
                continue;
            }
            if (s > f.alpha) f.alpha = s;
            if (f.rem == 0) {
                v = f.alpha;
                continue;
            }
            const Board c = ab_next_child(f.own, f.opp, &f.rem);
            alpha = -f.beta;
            beta = -f.alpha;
            sp++;  // the frame stays where it is, updated
            own = c.own;
            opp = c.opp;
            break;
        }
    }
}

// Whether a root is searched by k_alphabeta_split: only the exact searches beyond k_alphabeta's.
__device__ __forceinline__ bool ab_split_root(int empties, int exact_empties)
{
    return empties <= exact_empties && empties > AB_SEQ_MAX_EXACT;
}

__global__ void __launch_bounds__(128) k_alphabeta(const u64* __restrict__ own_in, const u64* __restrict__ opp_in, int64_t n,
                                                   int depth, int exact_empties, int32_t* __restrict__ out_values,
                                                   int32_t* __restrict__ out_best, unsigned long long* __restrict__ out_nodes)
{
    const int lane = threadIdx.x & 31;
    const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += nw) {
        const u64 own = own_in[i], opp = opp_in[i];
        const u64 m = legal_moves(own, opp);
        const bool pass = !m && legal_moves(opp, own);
        const int k = m ? __popcll(m) : (pass ? 1 : 0);  // root actions; 0 = terminal root
        const int empties = 64 - __popcll(own | opp);
        if (ab_split_root(empties, exact_empties)) continue;  // k_alphabeta_split's root
        // below a root action: depth - 1 plies, or (exact) deeper than any game from here can last
        const int sub_depth = empties <= exact_empties ? AB_STACK : depth - 1;
        int val[2] = {OTH_AB_NONE, OTH_AB_NONE};
        unsigned long long cnt[2] = {0, 0};
        int best_v = OTH_AB_NONE, best_a = 65;
#pragma unroll
        for (int s = 0; s < 2; s++) {
            const int r = lane + 32 * s;
            if (r < k) {
                const int a = pass ? OTH_PASS : nth_set_bit(m, r);
                const Board c = apply_move(own, opp, a, pass ? 0ULL : flips(own, opp, 1ULL << a));
                val[s] = -ab_subtree(c.own, c.opp, sub_depth, -AB_INF, AB_INF, &cnt[s]);
                if (val[s] > best_v) {  // ranks ascend with the action index: the first maximum is the lowest action
                    best_v = val[s];
                    best_a = a;
                }
            }
        }
        // lowest action among the maxima over the warp
        for (int o = 16; o; o >>= 1) {
            const int ov = __shfl_xor_sync(0xffffffffu, best_v, o), oa = __shfl_xor_sync(0xffffffffu, best_a, o);
            if (ov > best_v || (ov == best_v && oa < best_a)) {
                best_v = ov;
                best_a = oa;
            }
        }
        if (lane == 0) out_best[i] = k ? best_a : -1;
        // entry e of the output row comes from the lane that owns its rank
#pragma unroll
        for (int s = 0; s < 3; s++) {
            const int e = lane + 32 * s;
            const bool legal = e < 64 ? ((m >> (e & 63)) & 1) : pass;
            const int r = e < 64 ? __popcll(m & ((1ULL << (e & 63)) - 1)) : 0;
            const int v0 = __shfl_sync(0xffffffffu, val[0], r & 31), v1 = __shfl_sync(0xffffffffu, val[1], r & 31);
            const unsigned long long c0 = __shfl_sync(0xffffffffu, cnt[0], r & 31), c1 = __shfl_sync(0xffffffffu, cnt[1], r & 31);
            if (e < OTH_NUM_ACTIONS) {
                out_values[i * OTH_NUM_ACTIONS + e] = legal ? (r < 32 ? v0 : v1) : OTH_AB_NONE;
                if (out_nodes) out_nodes[i * OTH_NUM_ACTIONS + e] = legal ? (r < 32 ? c0 : c1) : 0ULL;
            }
        }
    }
}

// Per-warp state of one root in k_alphabeta_split, indexed by root-action rank (a position has < 64 actions).
struct SplitRoot {
    int next;              // next task to claim
    int ntasks;
    int young_begin[65];   // younger-brother tasks of rank r: ntasks' indices k + young_begin[r] .. k + young_begin[r+1]-1
    u64 young[64];         // their reply squares (the child's actions minus the eldest)
    int beta[64];          // window top of those tasks = the eldest's value; AB_INF until it is known
    int val[64];           // min over the rank's task results = its root value
    unsigned long long nodes[64];
};

// Exact roots beyond k_alphabeta's (ab_split_root), one warp each, split one level below the root actions
// (Young Brothers Wait).  For root action a with child c and replies g_1 .. g_m (ab_next_child's order):
//  - eldest task: g_1 with a full window, so L = -V(g_1) is a lower bound on V(c);
//  - younger tasks: every other g_j with the window (-AB_INF, -L), fail-hard, so -result = max(L, -V(g_j)) exactly;
// and the root value -V(c) = min(V(g_1), min_j result_j).  A child that is terminal, a forced pass or has one
// reply is one task (its whole subtree).  The lanes claim tasks from a counter, eldest tasks first; a younger
// task waits for its eldest.  Every task's window is fixed by the position alone and results are combined with min
// and sum, so values and node counts do not depend on which lane ran which task.
__global__ void __launch_bounds__(128) k_alphabeta_split(const u64* __restrict__ own_in, const u64* __restrict__ opp_in,
                                                         int64_t n, int exact_empties,
                                                         int32_t* __restrict__ out_values, int32_t* __restrict__ out_best,
                                                         unsigned long long* __restrict__ out_nodes)
{
    __shared__ SplitRoot sh_roots[4];
    SplitRoot& R = sh_roots[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += nw) {
        const u64 own = own_in[i], opp = opp_in[i];
        if (!ab_split_root(64 - __popcll(own | opp), exact_empties)) continue;
        const u64 m = legal_moves(own, opp);
        const bool pass = !m && legal_moves(opp, own);
        const int k = m ? __popcll(m) : (pass ? 1 : 0);
        // the tasks of every root action
        for (int r = lane; r < k; r += 32) {
            const int a = pass ? OTH_PASS : nth_set_bit(m, r);
            const Board c = apply_move(own, opp, a, pass ? 0ULL : flips(own, opp, 1ULL << a));
            int v;
            u64 rem = 0;
            if (!ab_leaf(c.own, c.opp, AB_STACK, &v, &rem) && rem != PASS_ONLY)
                ab_next_child(c.own, c.opp, &rem);  // rem = the younger brothers
            else
                rem = 0;
            R.young[r] = rem;
            R.young_begin[r + 1] = __popcll(rem);
            R.beta[r] = AB_INF;
            R.val[r] = AB_INF;
            R.nodes[r] = 0;
        }
        __syncwarp();
        if (lane == 0) {
            R.young_begin[0] = 0;
            for (int r = 0; r < k; r++) R.young_begin[r + 1] += R.young_begin[r];
            R.ntasks = k + R.young_begin[k];
            R.next = 0;
        }
        __syncwarp();
        for (int t = atomicAdd(&R.next, 1); t < R.ntasks; t = atomicAdd(&R.next, 1)) {
            int r = t;
            if (t >= k)
                for (r = 0; t - k >= R.young_begin[r + 1]; r++) {}
            const int a = pass ? OTH_PASS : nth_set_bit(m, r);
            const Board c = apply_move(own, opp, a, pass ? 0ULL : flips(own, opp, 1ULL << a));
            unsigned long long cnt = 0;
            int v;
            if (t >= k) {  // younger brother: wait for the eldest's value
                volatile int* vb = &R.beta[r];
                int beta;
                while ((beta = *vb) == AB_INF) __nanosleep(256);
                const int sq = nth_set_bit(R.young[r], t - k - R.young_begin[r]);
                const Board g = apply_move(c.own, c.opp, sq, flips(c.own, c.opp, 1ULL << sq));
                v = ab_subtree(g.own, g.opp, AB_STACK - 1, -AB_INF, beta, &cnt);
            } else if (R.young[r]) {  // eldest brother
                u64 rem = legal_moves(c.own, c.opp);
                const Board g = ab_next_child(c.own, c.opp, &rem);
                v = ab_subtree(g.own, g.opp, AB_STACK - 1, -AB_INF, AB_INF, &cnt);
                cnt++;  // c
                *(volatile int*)&R.beta[r] = v;
            } else {  // c unsplit
                v = -ab_subtree(c.own, c.opp, AB_STACK, -AB_INF, AB_INF, &cnt);
            }
            atomicMin(&R.val[r], v);
            atomicAdd(&R.nodes[r], cnt);
        }
        __syncwarp();
        // lowest action among the maxima, as in k_alphabeta
        int best_v = OTH_AB_NONE, best_a = 65;
        for (int r = lane; r < k; r += 32) {
            const int a = pass ? OTH_PASS : nth_set_bit(m, r);
            if (R.val[r] > best_v || (R.val[r] == best_v && a < best_a)) {
                best_v = R.val[r];
                best_a = a;
            }
        }
        for (int o = 16; o; o >>= 1) {
            const int ov = __shfl_xor_sync(0xffffffffu, best_v, o), oa = __shfl_xor_sync(0xffffffffu, best_a, o);
            if (ov > best_v || (ov == best_v && oa < best_a)) {
                best_v = ov;
                best_a = oa;
            }
        }
        if (lane == 0) out_best[i] = k ? best_a : -1;
        for (int e = lane; e < OTH_NUM_ACTIONS; e += 32) {
            const bool legal = e < 64 ? ((m >> e) & 1) : pass;
            const int r = e < 64 ? __popcll(m & ((1ULL << e) - 1)) : 0;
            out_values[i * OTH_NUM_ACTIONS + e] = legal ? R.val[r] : OTH_AB_NONE;
            if (out_nodes) out_nodes[i * OTH_NUM_ACTIONS + e] = legal ? R.nodes[r] : 0ULL;
        }
        __syncwarp();  // R is reused by the warp's next root
    }
}

}  // namespace

extern "C" int oth_alphabeta(const uint64_t* own, const uint64_t* opp, int64_t n, int32_t depth, int32_t exact_empties,
                             int32_t* out_values, int32_t* out_best, uint64_t* out_nodes, void* stream)
{
    if (n < 0 || depth < 1 || depth > OTH_AB_MAX_DEPTH || exact_empties < 0 || exact_empties > OTH_AB_MAX_EXACT) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    if (!own || !opp || !out_values || !out_best) return OTH_E_ARG;
    k_alphabeta<<<grid_for(n * 32, 128), 128, 0, (cudaStream_t)stream>>>((const u64*)own, (const u64*)opp, n, depth, exact_empties,
                                                                         out_values, out_best, (unsigned long long*)out_nodes);
    int rc = cuda_status(cudaGetLastError());
    if (rc == OTH_OK && exact_empties > AB_SEQ_MAX_EXACT) {
        k_alphabeta_split<<<grid_for(n * 32, 128), 128, 0, (cudaStream_t)stream>>>(
            (const u64*)own, (const u64*)opp, n, exact_empties, out_values, out_best, (unsigned long long*)out_nodes);
        rc = cuda_status(cudaGetLastError());
    }
    return rc;
}

extern "C" int oth_host_alphabeta(const uint64_t* own, const uint64_t* opp, int64_t n, int32_t depth, int32_t exact_empties,
                                  int32_t* out_values, int32_t* out_best, uint64_t* out_nodes)
{
    if (n < 0 || depth < 1 || depth > OTH_AB_MAX_DEPTH || exact_empties < 0 || exact_empties > OTH_AB_MAX_EXACT) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    if (!own || !opp || !out_values || !out_best) return OTH_E_ARG;
    const size_t nb = (size_t)n * 8, vb = (size_t)n * OTH_NUM_ACTIONS * 4, bb = (size_t)n * 4,
                 cb = out_nodes ? (size_t)n * OTH_NUM_ACTIONS * 8 : 0;
    char* d = nullptr;
    int rc = cuda_status(cudaMalloc((void**)&d, 2 * nb + vb + bb + cb));
    if (rc != OTH_OK) return rc;
    uint64_t *down = (uint64_t*)d, *dopp = (uint64_t*)(d + nb), *dnodes = out_nodes ? (uint64_t*)(d + 2 * nb + vb + bb) : nullptr;
    int32_t *dval = (int32_t*)(d + 2 * nb), *dbest = (int32_t*)(d + 2 * nb + vb);
    if (rc == OTH_OK) rc = cuda_status(cudaMemcpyAsync(down, own, nb, cudaMemcpyHostToDevice, 0));
    if (rc == OTH_OK) rc = cuda_status(cudaMemcpyAsync(dopp, opp, nb, cudaMemcpyHostToDevice, 0));
    if (rc == OTH_OK) rc = oth_alphabeta(down, dopp, n, depth, exact_empties, dval, dbest, dnodes, 0);
    if (rc == OTH_OK) rc = cuda_status(cudaMemcpyAsync(out_values, dval, vb, cudaMemcpyDeviceToHost, 0));
    if (rc == OTH_OK) rc = cuda_status(cudaMemcpyAsync(out_best, dbest, bb, cudaMemcpyDeviceToHost, 0));
    if (rc == OTH_OK && out_nodes) rc = cuda_status(cudaMemcpyAsync(out_nodes, dnodes, cb, cudaMemcpyDeviceToHost, 0));
    if (rc == OTH_OK) rc = cuda_status(cudaStreamSynchronize(0));
    cudaFree(d);
    return rc;
}
