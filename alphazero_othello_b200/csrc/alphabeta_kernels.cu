// Batched fixed-depth alpha-beta player (oth_alphabeta): a fixed yardstick opponent for the arena.
//
// One warp per position; lane l searches the root actions of rank l, l+32 (ascending action order) with a
// full-window alpha-beta below each of them, so every root value is the exact negamax value whatever the
// move ordering inside a subtree.  The search semantics (ply = one depth level, forced pass included,
// terminal = 10 000 x disc difference, depth-0 heuristic) are defined once, in ab_leaf() / ab_subtree() below,
// and documented in include/othello_b200.h; tests/alphabeta_oracle.c restates them on the CPU oracle's mailbox boards.
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

// Exact negamax value of (own, opp) searched `depth` plies deep: iterative fail-hard alpha-beta with a full
// window at the top.  *nodes += positions visited.
__device__ int ab_subtree(u64 own, u64 opp, int depth, unsigned long long* nodes)
{
    Frame st[AB_STACK];
    int sp = 0, alpha = -AB_INF, beta = AB_INF, v;
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
        // below a root action: depth - 1 plies, or (exact) deeper than any game from here can last
        const int sub_depth = (64 - __popcll(own | opp) <= exact_empties) ? AB_STACK : depth - 1;
        int val[2] = {OTH_AB_NONE, OTH_AB_NONE};
        unsigned long long cnt[2] = {0, 0};
        int best_v = OTH_AB_NONE, best_a = 65;
#pragma unroll
        for (int s = 0; s < 2; s++) {
            const int r = lane + 32 * s;
            if (r < k) {
                const int a = pass ? OTH_PASS : nth_set_bit(m, r);
                const Board c = apply_move(own, opp, a, pass ? 0ULL : flips(own, opp, 1ULL << a));
                val[s] = -ab_subtree(c.own, c.opp, sub_depth, &cnt[s]);
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

}  // namespace

extern "C" int oth_alphabeta(const uint64_t* own, const uint64_t* opp, int64_t n, int32_t depth, int32_t exact_empties,
                             int32_t* out_values, int32_t* out_best, uint64_t* out_nodes, void* stream)
{
    if (n < 0 || depth < 1 || depth > OTH_AB_MAX_DEPTH || exact_empties < 0 || exact_empties > OTH_AB_MAX_EXACT) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    if (!own || !opp || !out_values || !out_best) return OTH_E_ARG;
    k_alphabeta<<<grid_for(n * 32, 128), 128, 0, (cudaStream_t)stream>>>((const u64*)own, (const u64*)opp, n, depth, exact_empties,
                                                                         out_values, out_best, (unsigned long long*)out_nodes);
    return cuda_status(cudaGetLastError());
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
