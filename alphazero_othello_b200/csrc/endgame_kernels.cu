// Batched exact win/draw/loss endgame solver (oth_solve_wld): the game-theoretic result of every root with few enough
// empty squares, for labelling self-play positions with the truth instead of a lambda-return.
//
// One thread per root runs a sequential null-window alpha-beta, window (-1, +1) on the sign of the final disc
// difference, with an explicit per-thread stack.  A root's value only needs its first winning move, and a sequential
// search keeps every cutoff: splitting a root into independent tasks would give most of them back (DESIGN.md 4).
// Children of nodes with FF_MIN_EMPTIES or more empty squares are searched fastest-first (fewest replies for the
// opponent first); nearer the leaves, where generating the children's move sets costs more than it saves, the
// static corner-first order of the alpha-beta player.  Roots are independent and nothing is shared between threads,
// so values and node counts depend on the position alone.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/othello_b200.h"
#include "bitboard.cuh"
#include "common.cuh"

using namespace oth;

namespace {

// The ancestors of a node: at most one move per empty square and a forced pass before each.
constexpr int WLD_STACK = 2 * OTH_SOLVE_MAX_EMPTIES + 1;
// Nodes with at least this many empty squares order their children fastest-first.
constexpr int FF_MIN_EMPTIES = 7;
// Fastest-first packs the node's children as 6-bit squares into one 64-bit word; nodes with more moves (rare this
// late in a game) keep the static order.
constexpr int FF_MAX_MOVES = 10;
constexpr u64 PASS_ONLY = ~0ULL;  // "remaining moves" of a node whose only action is the pass (no real move set is full)

// Square classes of the static order and of the fastest-first key.
constexpr u64 CORNERS = 0x8100000000000081ULL, X_SQUARES = 0x0042000000004200ULL,
              NEAR_CORNER = 0x4281000000008142ULL | X_SQUARES;

struct WldFrame {
    u64 own, opp;
    u64 moves;  // actions not yet searched (PASS_ONLY: the forced pass)
    u64 order;  // fastest-first: the squares still to search, 6 bits each, next in the low bits
    int8_t alpha, beta;
    bool ordered;
};

// The children of (own, opp) with legal set m (2..FF_MAX_MOVES moves) sorted by the opponent's mobility after the move,
// corners a step earlier and X-squares a step later, ties in ascending square order.  Returns the packed squares.
__device__ __forceinline__ u64 ff_order(u64 own, u64 opp, u64 m)
{
    u64 order = 0, keys = 0;
    int cnt = 0;
    for (u64 r = m; r; r &= r - 1, cnt++) {
        const int sq = __ffsll((long long)r) - 1;
        const u64 x = 1ULL << sq;
        const u64 f = flips(own, opp, x);
        int k = 4 * __popcll(legal_moves(opp ^ f, own | x | f)) + 4 - ((x & CORNERS) ? 4 : 0) + ((x & X_SQUARES) ? 4 : 0);
        k = k > 63 ? 63 : k;
        int p = 0;  // insert after every key <= k: stable
        for (int i = 0; i < cnt; i++) p += (int)((keys >> (6 * i)) & 63) <= k;
        const u64 low = (1ULL << (6 * p)) - 1;
        order = (order & low) | ((u64)sq << (6 * p)) | ((order & ~low) << 6);
        keys = (keys & low) | ((u64)k << (6 * p)) | ((keys & ~low) << 6);
    }
    return order;
}

// Takes the next action out of f and returns the child position.
__device__ __forceinline__ Board wld_next_child(WldFrame& f)
{
    if (f.moves == PASS_ONLY) {
        f.moves = 0;
        return apply_move(f.own, f.opp, OTH_PASS, 0);
    }
    int sq;
    if (f.ordered) {
        sq = (int)(f.order & 63);
        f.order >>= 6;
    } else {
        const u64 r = f.moves;
        const u64 corner = r & CORNERS, plain = r & ~(CORNERS | NEAR_CORNER);
        sq = __ffsll((long long)(corner ? corner : (plain ? plain : r))) - 1;
    }
    f.moves &= ~(1ULL << sq);
    return apply_move(f.own, f.opp, sq, flips(f.own, f.opp, 1ULL << sq));
}

// Win (+1), draw (0) or loss (-1) of (own, opp) for own under perfect play: fail-hard alpha-beta with the window
// (-1, +1) on the sign of the final disc difference, which it returns exactly.  *nodes = positions visited.
__device__ int wld_solve(u64 own, u64 opp, unsigned long long* nodes)
{
    WldFrame st[WLD_STACK];
    int sp = 0, v, alpha = -1, beta = 1;
    unsigned long long cnt = 0;
    for (;;) {
        // enter (own, opp) at level sp with window (alpha, beta)
        cnt++;
        const u64 m = legal_moves(own, opp);
        if (m || legal_moves(opp, own)) {
            WldFrame& f = st[sp++];
            f.own = own;
            f.opp = opp;
            f.alpha = (int8_t)alpha;
            f.beta = (int8_t)beta;
            f.moves = m ? m : PASS_ONLY;
            const int k = __popcll(m);
            f.ordered = 64 - __popcll(own | opp) >= FF_MIN_EMPTIES && k > 1 && k <= FF_MAX_MOVES;
            if (f.ordered) f.order = ff_order(own, opp, m);
            const Board c = wld_next_child(f);
            own = c.own;
            opp = c.opp;
            const int a = alpha;
            alpha = -beta;
            beta = -a;
            continue;
        }
        const int d = __popcll(own) - __popcll(opp);  // terminal: the sign lies in every window
        v = (d > 0) - (d < 0);
        // hand v to the ancestors until one has a child left to search
        for (;;) {
            if (sp == 0) {
                *nodes = cnt;
                return v;
            }
            WldFrame& f = st[--sp];
            const int s = -v;
            if (s >= f.beta) {
                v = f.beta;
                continue;
            }
            if (s > f.alpha) f.alpha = (int8_t)s;
            if (f.moves == 0) {
                v = f.alpha;
                continue;
            }
            const Board c = wld_next_child(f);
            alpha = -f.beta;
            beta = -f.alpha;
            sp++;  // the frame stays where it is, updated
            own = c.own;
            opp = c.opp;
            break;
        }
    }
}

// One block = one warp, whose first `per_warp` lanes each take a root at a time.  The launch picks per_warp so that
// every SM sub-partition gets warps to interleave even when a launch has only a few thousand roots.
__global__ void __launch_bounds__(32) k_solve_wld(const u64* __restrict__ own_in, const u64* __restrict__ opp_in, int64_t n,
                                                  int max_empties, int per_warp, int8_t* __restrict__ out_wld,
                                                  unsigned long long* __restrict__ out_nodes)
{
    if ((int)threadIdx.x >= per_warp) return;
    const int64_t stride = (int64_t)gridDim.x * per_warp;
    for (int64_t i = (int64_t)blockIdx.x * per_warp + threadIdx.x; i < n; i += stride) {
        const u64 own = own_in[i], opp = opp_in[i];
        int8_t w = OTH_WLD_UNSOLVED;
        unsigned long long cnt = 0;
        if (64 - __popcll(own | opp) <= max_empties) w = (int8_t)wld_solve(own, opp, &cnt);
        out_wld[i] = w;
        if (out_nodes) out_nodes[i] = cnt;
    }
}

// Warps per SM the launch aims for: two per sub-partition, so that one hides the other's latencies.
constexpr int WLD_WARPS_PER_SM = 8;

}  // namespace

extern "C" int oth_solve_wld(const uint64_t* own, const uint64_t* opp, int64_t n, int32_t max_empties, int8_t* out_wld,
                             uint64_t* out_nodes, void* stream)
{
    if (n < 0 || max_empties < 0 || max_empties > OTH_SOLVE_MAX_EMPTIES) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    if (!own || !opp || !out_wld) return OTH_E_ARG;
    const int64_t warps = (int64_t)sm_count() * WLD_WARPS_PER_SM;
    int64_t per_warp = (n + warps - 1) / warps;
    per_warp = per_warp < 1 ? 1 : (per_warp > 32 ? 32 : per_warp);
    k_solve_wld<<<grid_for(((n + per_warp - 1) / per_warp) * 32, 32), 32, 0, (cudaStream_t)stream>>>(
        (const u64*)own, (const u64*)opp, n, max_empties, (int)per_warp, out_wld, (unsigned long long*)out_nodes);
    return cuda_status(cudaGetLastError());
}

extern "C" int oth_host_solve_wld(const uint64_t* own, const uint64_t* opp, int64_t n, int32_t max_empties, int8_t* out_wld,
                                  uint64_t* out_nodes)
{
    if (n < 0 || max_empties < 0 || max_empties > OTH_SOLVE_MAX_EMPTIES) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    if (!own || !opp || !out_wld) return OTH_E_ARG;
    const size_t nb = (size_t)n * 8, wb = ((size_t)n + 7) & ~(size_t)7, cb = out_nodes ? (size_t)n * 8 : 0;
    char* d = nullptr;
    int rc = cuda_status(cudaMalloc((void**)&d, 2 * nb + cb + wb));
    if (rc != OTH_OK) return rc;
    uint64_t *down = (uint64_t*)d, *dopp = (uint64_t*)(d + nb), *dnodes = out_nodes ? (uint64_t*)(d + 2 * nb) : nullptr;
    int8_t* dwld = (int8_t*)(d + 2 * nb + cb);
    if (rc == OTH_OK) rc = cuda_status(cudaMemcpyAsync(down, own, nb, cudaMemcpyHostToDevice, 0));
    if (rc == OTH_OK) rc = cuda_status(cudaMemcpyAsync(dopp, opp, nb, cudaMemcpyHostToDevice, 0));
    if (rc == OTH_OK) rc = oth_solve_wld(down, dopp, n, max_empties, dwld, dnodes, 0);
    if (rc == OTH_OK) rc = cuda_status(cudaMemcpyAsync(out_wld, dwld, (size_t)n, cudaMemcpyDeviceToHost, 0));
    if (rc == OTH_OK && out_nodes) rc = cuda_status(cudaMemcpyAsync(out_nodes, dnodes, cb, cudaMemcpyDeviceToHost, 0));
    if (rc == OTH_OK) rc = cuda_status(cudaStreamSynchronize(0));
    cudaFree(d);
    return rc;
}
