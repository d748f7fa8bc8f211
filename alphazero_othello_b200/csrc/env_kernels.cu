// Othello environment kernels for B200 (sm_100a) and their C ABI.
// Reference behaviour: envs/othello.py (OthelloGameNew / _BitBoard); see
// include/othello_b200.h for the per-entry citations.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/othello_b200.h"
#include "bitboard.cuh"
#include "common.cuh"
#include "philox.cuh"

using namespace oth;

// ------------------------------------------------------------- kernels ----

// Two positions per thread: 128-bit loads/stores of packed uint64 boards.
__global__ void __launch_bounds__(256) k_legal_moves(const u64* __restrict__ own, const u64* __restrict__ opp,
                                                     u64* __restrict__ out, int64_t n)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t npair = n >> 1;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < npair; i += stride) {
        const ulonglong2 a = reinterpret_cast<const ulonglong2*>(own)[i];
        const ulonglong2 b = reinterpret_cast<const ulonglong2*>(opp)[i];
        ulonglong2 m;
        m.x = legal_moves(a.x, b.x);
        m.y = legal_moves(a.y, b.y);
        reinterpret_cast<ulonglong2*>(out)[i] = m;
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) out[n - 1] = legal_moves(own[n - 1], opp[n - 1]);
}

// scalar form for buffers that are not 16-byte aligned
__global__ void __launch_bounds__(256) k_legal_moves_scalar(const u64* __restrict__ own, const u64* __restrict__ opp,
                                                            u64* __restrict__ out, int64_t n)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = legal_moves(own[i], opp[i]);
}

__device__ __forceinline__ void step_one(u64 o, u64 p, int a, u64& no, u64& np, u64& nm, unsigned& fl)
{
    fl = 0;
    u64 f = 0;
    if (a != OTH_PASS) {
        const u64 x = (a >= 0 && a < 64) ? (1ULL << a) : 0ULL;
        f = (x & ~(o | p)) ? flips(o, p, x) : 0ULL;
        if (f == 0) {  // envs/othello.py:419-421 -> ValueError
            no = o;
            np = p;
            nm = legal_moves(o, p);
            fl = OTH_F_ILLEGAL;
            return;
        }
    }
    const Board b = apply_move(o, p, a, f);
    no = b.own;
    np = b.opp;
    nm = legal_moves(no, np);
    int v;
    const int st = position_status(no, np, nm, &v);
    if (st == 1) fl |= OTH_F_MUST_PASS;
    if (st == 2) {
        // v is from the next mover's side; the mover who just played sees -v
        fl |= OTH_F_TERMINAL;
        if (v < 0) fl |= OTH_F_WIN;
        if (v > 0) fl |= OTH_F_LOSS;
    }
}

__global__ void __launch_bounds__(256) k_step(const u64* __restrict__ own, const u64* __restrict__ opp,
                                              const uint8_t* __restrict__ action, u64* __restrict__ out_own,
                                              u64* __restrict__ out_opp, u64* __restrict__ out_moves,
                                              uint8_t* __restrict__ out_flags, int64_t n)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        u64 no, np, nm;
        unsigned fl;
        step_one(own[i], opp[i], action[i], no, np, nm, fl);
        out_own[i] = no;
        out_opp[i] = np;
        if (out_moves) out_moves[i] = nm;
        if (out_flags) out_flags[i] = (uint8_t)fl;
    }
}

// One thread per game, whole game in registers.
__global__ void __launch_bounds__(256) k_rollout(uint64_t seed, uint64_t base, int64_t n_games, int32_t* __restrict__ out_score,
                                                 int32_t* __restrict__ out_plies, u64* __restrict__ out_final, int64_t n_trace,
                                                 uint8_t* __restrict__ trace_actions, u64* __restrict__ trace_moves,
                                                 unsigned long long* __restrict__ counters)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned long long my_plies = 0;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_games; g += stride) {
        const uint64_t gid = base + (uint64_t)g;
        const bool tr = g < n_trace;
        u64 own = INIT_BLACK, opp = INIT_WHITE;
        int side = 0;  // 0: +1 (black) to move
        int plies = 0;
        u64 m = legal_moves(own, opp);
        Philox4 r = {0, 0, 0, 0};
        int block = -1;  // Philox block (ply >> 2) currently held in r; a forced pass can skip a block boundary
        while (plies < OTH_MAX_PLIES) {
            if ((plies >> 2) != block) {
                block = plies >> 2;
                r = philox4x32_10(seed, gid, (uint32_t)block, 0u);
            }
            const int w = plies & 3;
            const uint32_t rnd = w == 0 ? r.x : (w == 1 ? r.y : (w == 2 ? r.z : r.w));
            const int nm = __popcll(m);
            const int k = (int)__umulhi(rnd, (uint32_t)nm);
            const int sq = nth_set_bit(m, k);
            if (tr) {
                if (trace_actions) trace_actions[g * OTH_MAX_PLIES + plies] = (uint8_t)sq;
                if (trace_moves) trace_moves[g * OTH_MAX_PLIES + plies] = m;
            }
            const u64 f = flips(own, opp, 1ULL << sq);
            const Board b = apply_move(own, opp, sq, f);
            own = b.own;
            opp = b.opp;
            side ^= 1;
            plies++;
            m = legal_moves(own, opp);
            if (m == 0) {
                const u64 m2 = legal_moves(opp, own);
                if (m2 == 0) break;  // neither side can move: terminal (envs/othello.py:440-454)
                if (plies >= OTH_MAX_PLIES) break;
                if (tr) {  // forced pass is a ply of its own (self_play_worker.py:88)
                    if (trace_actions) trace_actions[g * OTH_MAX_PLIES + plies] = OTH_PASS;
                    if (trace_moves) trace_moves[g * OTH_MAX_PLIES + plies] = 0;
                }
                const u64 t = own;
                own = opp;
                opp = t;
                side ^= 1;
                plies++;
                m = m2;
            }
        }
        if (tr && trace_actions)
            for (int p = plies; p < OTH_MAX_PLIES; p++) trace_actions[g * OTH_MAX_PLIES + p] = 0xFF;
        const u64 black = side == 0 ? own : opp, white = side == 0 ? opp : own;
        if (out_score) out_score[g] = __popcll(black) - __popcll(white);
        if (out_plies) out_plies[g] = plies;
        if (out_final) {
            out_final[2 * g] = black;
            out_final[2 * g + 1] = white;
        }
        my_plies += plies;
    }
    if (counters) {
        for (int o = 16; o; o >>= 1) my_plies += __shfl_xor_sync(0xffffffffu, my_plies, o);
        if ((threadIdx.x & 31) == 0) atomicAdd(counters, my_plies);
    }
}

// One warp per board: cells -> bitboards by ballot (envs/othello.py:358-371).
__device__ __forceinline__ void warp_pack(const int8_t* __restrict__ s, int player, int lane, u64& own, u64& opp)
{
    const int c0 = s[lane], c1 = s[lane + 32];
    const unsigned o_lo = __ballot_sync(0xffffffffu, c0 == player), o_hi = __ballot_sync(0xffffffffu, c1 == player);
    const unsigned p_lo = __ballot_sync(0xffffffffu, c0 == -player), p_hi = __ballot_sync(0xffffffffu, c1 == -player);
    own = ((u64)o_hi << 32) | o_lo;
    opp = ((u64)p_hi << 32) | p_lo;
}

__global__ void __launch_bounds__(256) k_pack(const int8_t* __restrict__ states, const int8_t* __restrict__ players,
                                              u64* __restrict__ own, u64* __restrict__ opp, int64_t n)
{
    const int lane = threadIdx.x & 31;
    const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += nw) {
        u64 o, p;
        warp_pack(states + i * 64, players ? players[i] : 1, lane, o, p);
        if (lane == 0) {
            own[i] = o;
            opp[i] = p;
        }
    }
}

// bitboards -> int8 cells; own discs get the value `player` (envs/othello.py:374-388, 430-433).
__global__ void __launch_bounds__(256) k_unpack(const u64* __restrict__ own, const u64* __restrict__ opp,
                                                const int8_t* __restrict__ players, int own_stride, int8_t* __restrict__ states,
                                                int64_t n)
{
    const int lane = threadIdx.x & 31;
    const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += nw) {
        const u64 o = own[i * own_stride], p = opp[i * own_stride];
        const int pl = players ? players[i] : 1;
        // two cells per lane, written as one 16-bit store
        const int a = 2 * lane;
        const int v0 = ((o >> a) & 1) ? pl : (((p >> a) & 1) ? -pl : 0);
        const int v1 = ((o >> (a + 1)) & 1) ? pl : (((p >> (a + 1)) & 1) ? -pl : 0);
        reinterpret_cast<uint16_t*>(states + i * 64)[lane] = (uint16_t)((v0 & 0xff) | ((v1 & 0xff) << 8));
    }
}

__global__ void __launch_bounds__(256) k_valid_moves_i8(const int8_t* __restrict__ states, const int8_t* __restrict__ players,
                                                       uint8_t* __restrict__ out, int64_t n)
{
    const int lane = threadIdx.x & 31;
    const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += nw) {
        u64 o, p;
        warp_pack(states + i * 64, players[i], lane, o, p);
        const u64 m = legal_moves(o, p);
        uint8_t* dst = out + i * OTH_NUM_ACTIONS;
        dst[lane] = (uint8_t)((m >> lane) & 1);
        dst[lane + 32] = (uint8_t)((m >> (lane + 32)) & 1);
        if (lane == 0) dst[64] = (uint8_t)(m == 0);  // pass iff no board move (envs/othello.py:401-403)
    }
}

__global__ void __launch_bounds__(256) k_next_state_i8(const int8_t* __restrict__ states, const int32_t* __restrict__ actions,
                                                       const int8_t* __restrict__ players, int8_t* __restrict__ out,
                                                       uint8_t* __restrict__ out_flags, int64_t n)
{
    const int lane = threadIdx.x & 31;
    const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += nw) {
        u64 o, p;
        const int pl = players[i];
        warp_pack(states + i * 64, pl, lane, o, p);
        const int a = actions[i];
        unsigned fl = 0;
        u64 f = 0;
        if (a != OTH_PASS) {  // pass copies the board unchecked (envs/othello.py:415-416)
            const u64 x = (a >= 0 && a < 64) ? (1ULL << a) : 0ULL;
            f = (x & ~(o | p)) ? flips(o, p, x) : 0ULL;
            if (f == 0) fl = OTH_F_ILLEGAL;
            else {
                o |= x | f;
                p &= ~f;
            }
        }
        const int c = 2 * lane;  // absolute colours: player's discs stay = player
        const int v0 = ((o >> c) & 1) ? pl : (((p >> c) & 1) ? -pl : 0);
        const int v1 = ((o >> (c + 1)) & 1) ? pl : (((p >> (c + 1)) & 1) ? -pl : 0);
        reinterpret_cast<uint16_t*>(out + i * 64)[lane] = (uint16_t)((v0 & 0xff) | ((v1 & 0xff) << 8));
        if (lane == 0 && out_flags) out_flags[i] = (uint8_t)fl;
    }
}

__global__ void __launch_bounds__(256) k_value_terminated_i8(const int8_t* __restrict__ states, const int8_t* __restrict__ players,
                                                             int8_t* __restrict__ values, uint8_t* __restrict__ terms, int64_t n)
{
    const int lane = threadIdx.x & 31;
    const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += nw) {
        u64 o, p;
        warp_pack(states + i * 64, players[i], lane, o, p);
        int v;
        const int st = position_status(o, p, legal_moves(o, p), &v);
        if (lane == 0) {
            values[i] = (int8_t)v;
            terms[i] = (uint8_t)(st == 2);
        }
    }
}

// Dihedral image: out[r][c] = in[src(r,c)], np.rot90 k times then np.fliplr.
__global__ void __launch_bounds__(256) k_symmetry(const int8_t* __restrict__ states, const float* __restrict__ pis,
                                                  const int32_t* __restrict__ ks, const uint8_t* __restrict__ flips_,
                                                  float* __restrict__ out_s, float* __restrict__ out_pi, int64_t n)
{
    const int64_t total = n * 65;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
        const int64_t i = t / 65;
        const int e = (int)(t - i * 65);
        if (e == 64) {
            if (out_pi) out_pi[i * 65 + 64] = pis[i * 65 + 64];
            continue;
        }
        int r = e >> 3, c = e & 7;
        if (flips_[i]) c = 7 - c;
        const int k = ks[i] & 3;
        for (int q = 0; q < k; q++) {
            const int nr = c, nc = 7 - r;
            r = nr;
            c = nc;
        }
        const int src = r * 8 + c;
        if (out_s) out_s[i * 64 + e] = (float)states[i * 64 + src];
        if (out_pi) out_pi[i * 65 + e] = pis[i * 65 + src];
    }
}

// Network-boundary epilogue (the network itself stays PyTorch/cuDNN): x = relu(x + bias[c] + res)
// on channels-last bf16 activations, 8 elements (128 bits) per thread.
#include <cuda_bf16.h>
// relu that keeps a NaN, as torch.relu does: fmaxf(NaN, 0) would return 0 and hide it from the non-finite guard;
// every other input takes the same fmaxf as before, bit for bit
__device__ __forceinline__ float relu_keep_nan(float v) { return v != v ? v : fmaxf(v, 0.0f); }

__global__ void __launch_bounds__(256) k_bias_add_relu_bf16(uint4* __restrict__ x, const uint4* __restrict__ res,
                                                            const __nv_bfloat16* __restrict__ bias, int64_t n8, int C)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
        uint4 a = x[i];
        const uint4 r = res[i];
        const int c0 = (int)((i * 8) % C);
        const uint4 bv = *reinterpret_cast<const uint4*>(bias + c0);
        __nv_bfloat162* pa = reinterpret_cast<__nv_bfloat162*>(&a);
        const __nv_bfloat162* pr = reinterpret_cast<const __nv_bfloat162*>(&r);
        const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(&bv);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const float2 fa = __bfloat1622float2(pa[k]), fr = __bfloat1622float2(pr[k]), fb = __bfloat1622float2(pb[k]);
            pa[k] = __floats2bfloat162_rn(relu_keep_nan(fa.x + fb.x + fr.x), relu_keep_nan(fa.y + fb.y + fr.y));
        }
        x[i] = a;
    }
}

// Network-boundary im2col for the 1-channel 3x3 stem: float32 planes [n,64] -> bf16 [n,64,16]
// (9 taps in (dy,dx) order, zero padding at the border, columns 9..15 zero), one thread per square.
__global__ void __launch_bounds__(256) k_stem_im2col_bf16(const float* __restrict__ planes, uint4* __restrict__ cols, int64_t n64)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n64; t += stride) {
        const int sq = (int)(t & 63), r = sq >> 3, c = sq & 7;
        const float* p = planes + (t - sq);
        float v[9];
#pragma unroll
        for (int dy = -1; dy <= 1; dy++)
#pragma unroll
            for (int dx = -1; dx <= 1; dx++) {
                const int rr = r + dy, cc = c + dx;
                v[(dy + 1) * 3 + dx + 1] = (rr >= 0 && rr < 8 && cc >= 0 && cc < 8) ? p[rr * 8 + cc] : 0.0f;
            }
        uint4 a, b;
        __nv_bfloat162* pa = reinterpret_cast<__nv_bfloat162*>(&a);
        __nv_bfloat162* pb = reinterpret_cast<__nv_bfloat162*>(&b);
        pa[0] = __floats2bfloat162_rn(v[0], v[1]);
        pa[1] = __floats2bfloat162_rn(v[2], v[3]);
        pa[2] = __floats2bfloat162_rn(v[4], v[5]);
        pa[3] = __floats2bfloat162_rn(v[6], v[7]);
        pb[0] = __floats2bfloat162_rn(v[8], 0.0f);
        pb[1] = pb[2] = pb[3] = __floats2bfloat162_rn(0.0f, 0.0f);
        cols[2 * t] = a;
        cols[2 * t + 1] = b;
    }
}

extern "C" int oth_nn_stem_im2col_bf16(const float* planes, void* cols, int64_t n, void* stream)
{
    if (n < 0 || (n > 0 && (!planes || !cols)) || ((uintptr_t)cols & 15)) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    k_stem_im2col_bf16<<<grid_for(n * 64, 256), 256, 0, (cudaStream_t)stream>>>(planes, (uint4*)cols, n * 64);
    return cuda_status(cudaGetLastError());
}

extern "C" int oth_nn_bias_add_relu_bf16(void* x, const void* res, const void* bias, int64_t n, int32_t channels, void* stream)
{
    if (n < 0 || channels <= 0 || (channels % 8) || (n % 8) || !x || !res || !bias) return OTH_E_ARG;
    if ((((uintptr_t)x | (uintptr_t)res | (uintptr_t)bias) & 15) != 0) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    k_bias_add_relu_bf16<<<grid_for(n / 8, 256), 256, 0, (cudaStream_t)stream>>>((uint4*)x, (const uint4*)res,
                                                                                (const __nv_bfloat16*)bias, n / 8, channels);
    return cuda_status(cudaGetLastError());
}

// canonical packed boards [n][2] -> int8 [n,64] (+1 own / -1 opp)
extern "C" int oth_unpack_canonical(const uint64_t* boards, int8_t* states, int64_t n, void* stream)
{
    if (n <= 0) return OTH_OK;
    k_unpack<<<grid_for(n * 32, 256), 256, 0, (cudaStream_t)stream>>>((const u64*)boards, (const u64*)boards + 1, nullptr, 2,
                                                                      states, n);
    return cuda_status(cudaGetLastError());
}

// INT32 ALU probe: 8 independent chains of LOP3 + IADD3 per thread.
__global__ void __launch_bounds__(256) k_int32_probe(unsigned* __restrict__ out, int iters, unsigned b, unsigned c)
{
    unsigned a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
#define STEP(x)                                                                               \
    asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x) : "r"(b), "r"(c));                 \
    asm volatile("add.u32 %0, %0, %1;" : "+r"(x) : "r"(c));
            STEP(a0) STEP(a1) STEP(a2) STEP(a3) STEP(a4) STEP(a5) STEP(a6) STEP(a7)
#undef STEP
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
}

// Random-access HBM probe: every thread reads `per_thread` pseudo-random, independent chunks of
// `chunk` bytes (32/64/128) from a buffer much larger than L2 -- the access pattern of tree
// records -- so the MCTS kernel can be judged against what HBM delivers for that pattern.
__global__ void __launch_bounds__(256) k_random_read_probe(const uint4* __restrict__ buf, uint64_t n_chunks, int chunk16, int per_thread,
                                                           unsigned* __restrict__ sink)
{
    uint64_t x = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 0x9E3779B97F4A7C15ULL + 0x1234567ULL;
    unsigned acc = 0;
    for (int k = 0; k < per_thread; k += 4) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {  // 4 independent requests in flight per thread
            x ^= x >> 29;
            x *= 0xBF58476D1CE4E5B9ULL;
            x ^= x >> 32;
            const uint64_t c = x % n_chunks;
            v[u] = buf[c * chunk16];
            for (int q = 1; q < chunk16; q++) {
                const uint4 w = buf[c * chunk16 + q];
                v[u].x ^= w.x ^ w.y ^ w.z ^ w.w;
            }
        }
#pragma unroll
        for (int u = 0; u < 4; u++) acc ^= v[u].x ^ v[u].y ^ v[u].z ^ v[u].w;
    }
    if (acc == 0x7fffffff) sink[0] = acc;
}

extern "C" int oth_host_random_read_probe(int64_t buffer_bytes, int32_t chunk_bytes, double* out_gbs, float* kernel_ms)
{
    if (buffer_bytes < (1 << 20) || (chunk_bytes != 32 && chunk_bytes != 64 && chunk_bytes != 128)) return OTH_E_ARG;
    void *buf = nullptr, *sink = nullptr;
    int rc = cuda_status(cudaMalloc(&buf, (size_t)buffer_bytes));
    if (rc != OTH_OK) return rc;
    cudaMalloc(&sink, 64);
    cudaMemset(buf, 1, (size_t)buffer_bytes);
    const int blocks = sm_count() * 8, threads = 256, per_thread = 64;
    const uint64_t n_chunks = (uint64_t)buffer_bytes / chunk_bytes;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        cudaEventRecord(e0, 0);
        k_random_read_probe<<<blocks, threads>>>((const uint4*)buf, n_chunks, chunk_bytes / 16, per_thread, (unsigned*)sink);
        cudaEventRecord(e1, 0);
        cudaStreamSynchronize(0);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep > 0 && ms < best) best = ms;
    }
    rc = cuda_status(cudaGetLastError());
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(buf);
    cudaFree(sink);
    if (rc != OTH_OK) return rc;
    if (out_gbs) *out_gbs = (double)blocks * threads * per_thread * chunk_bytes / (best * 1e-3) / 1e9;
    if (kernel_ms) *kernel_ms = best;
    return OTH_OK;
}

// ----------------------------------------------------------------- C ABI --

static char g_cuda_err[256] = "";

namespace oth {
int cuda_status(cudaError_t e)
{
    if (e == cudaSuccess) return OTH_OK;
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", cudaGetErrorName(e), cudaGetErrorString(e));
    return e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? OTH_E_NO_DEVICE : OTH_E_CUDA;
}

int sm_count()
{
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = 148;
    }
    return n;
}

// grid sized in multiples of the SM count (148 on B200), capped by the work
int grid_for(int64_t threads, int block)
{
    const int64_t need = (threads + block - 1) / block;
    const int64_t full = (int64_t)sm_count() * 8;
    if (need <= 0) return 1;
    if (need >= full) return (int)full;
    const int64_t sms = sm_count();
    return (int)(need <= sms ? need : ((need + sms - 1) / sms) * sms);
}
}  // namespace oth

extern "C" int oth_abi_version(void) { return OTH_ABI_VERSION; }

extern "C" const char* oth_error_string(int code)
{
    switch (code) {
    case OTH_OK: return "ok";
    case OTH_E_CUDA: return "CUDA runtime error";
    case OTH_E_ARG: return "bad argument";
    case OTH_E_ILLEGAL: return "Illegal move";
    case OTH_E_NO_DEVICE: return "no CUDA device (libothello_b200 has no CPU fallback)";
    default: return "unknown error";
    }
}

extern "C" const char* oth_last_cuda_error(void) { return g_cuda_err; }

extern "C" int oth_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int oth_legal_moves(const uint64_t* own, const uint64_t* opp, uint64_t* out, int64_t n, void* stream)
{
    if (n < 0 || (n > 0 && (!own || !opp || !out))) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    if ((((uintptr_t)own | (uintptr_t)opp | (uintptr_t)out) & 15) != 0)  // no 128-bit access possible
        k_legal_moves_scalar<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const u64*)own, (const u64*)opp, (u64*)out, n);
    else
        k_legal_moves<<<grid_for((n + 1) / 2, 256), 256, 0, (cudaStream_t)stream>>>((const u64*)own, (const u64*)opp, (u64*)out, n);
    return cuda_status(cudaGetLastError());
}

extern "C" int oth_step(const uint64_t* own, const uint64_t* opp, const uint8_t* action, uint64_t* out_own, uint64_t* out_opp,
                        uint64_t* out_moves, uint8_t* out_flags, int64_t n, void* stream)
{
    if (n < 0 || (n > 0 && (!own || !opp || !action || !out_own || !out_opp))) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    k_step<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const u64*)own, (const u64*)opp, action, (u64*)out_own,
                                                               (u64*)out_opp, (u64*)out_moves, out_flags, n);
    return cuda_status(cudaGetLastError());
}

extern "C" int oth_rollout(uint64_t seed, uint64_t game_id_base, int64_t n_games, int32_t* out_score, int32_t* out_plies,
                           uint64_t* out_final, int64_t n_trace, uint8_t* trace_actions, uint64_t* trace_moves,
                           unsigned long long* counters, void* stream)
{
    if (n_games < 0 || n_trace < 0 || n_trace > n_games) return OTH_E_ARG;
    if (n_games == 0) return OTH_OK;
    k_rollout<<<grid_for(n_games, 256), 256, 0, (cudaStream_t)stream>>>(seed, game_id_base, n_games, out_score, out_plies,
                                                                       (u64*)out_final, n_trace, trace_actions, (u64*)trace_moves,
                                                                       counters);
    return cuda_status(cudaGetLastError());
}

extern "C" int oth_pack_states(const int8_t* states, const int8_t* players, uint64_t* own, uint64_t* opp, int64_t n, void* stream)
{
    if (n < 0 || (n > 0 && (!states || !own || !opp))) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    k_pack<<<grid_for(n * 32, 256), 256, 0, (cudaStream_t)stream>>>(states, players, (u64*)own, (u64*)opp, n);
    return cuda_status(cudaGetLastError());
}

extern "C" int oth_unpack_states(const uint64_t* own, const uint64_t* opp, const int8_t* players, int8_t* states, int64_t n,
                                 void* stream)
{
    if (n < 0 || (n > 0 && (!states || !own || !opp))) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    k_unpack<<<grid_for(n * 32, 256), 256, 0, (cudaStream_t)stream>>>((const u64*)own, (const u64*)opp, players, 1, states, n);
    return cuda_status(cudaGetLastError());
}

extern "C" int oth_valid_moves_i8(const int8_t* states, const int8_t* players, uint8_t* out_masks, int64_t n, void* stream)
{
    if (n < 0 || (n > 0 && (!states || !players || !out_masks))) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    k_valid_moves_i8<<<grid_for(n * 32, 256), 256, 0, (cudaStream_t)stream>>>(states, players, out_masks, n);
    return cuda_status(cudaGetLastError());
}

extern "C" int oth_symmetry(const int8_t* states, const float* pis, const int32_t* ks, const uint8_t* flips_, float* out_states,
                            float* out_pis, int64_t n, void* stream)
{
    if (n < 0 || (n > 0 && (!states || !pis || !ks || !flips_))) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    k_symmetry<<<grid_for(n * 65, 256), 256, 0, (cudaStream_t)stream>>>(states, pis, ks, flips_, out_states, out_pis, n);
    return cuda_status(cudaGetLastError());
}

// ------------------------------------------------------ host-buffer forms --

namespace {
struct Scratch {  // grow-only device staging for the oth_host_* calls: one per host thread and device
    void* p[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    size_t cap[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    ~Scratch()
    {
        for (int i = 0; i < 8; i++)
            if (p[i]) cudaFree(p[i]);  // may run after context teardown: the error is irrelevant
    }
    int get(int i, size_t bytes, void** out)
    {
        if (bytes > cap[i]) {
            if (p[i]) cudaFree(p[i]);
            p[i] = nullptr;
            cap[i] = 0;
            size_t want = bytes < 4096 ? 4096 : bytes + bytes / 2;
            cudaError_t e = cudaMalloc(&p[i], want);
            if (e != cudaSuccess) return cuda_status(e);
            cap[i] = want;
        }
        *out = p[i];
        return OTH_OK;
    }
};
// The reference's Game object is stateless and shared across the MCTS worker threads (MCTS_model.py:196-198,
// ThreadPoolExecutor); ctypes releases the GIL during a call.  Staging buffers are therefore per calling thread and
// per current device, so concurrent oth_host_* calls never share device memory.
constexpr int kMaxDevices = 16;
Scratch& scr()
{
    thread_local Scratch per_device[kMaxDevices];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
    return per_device[dev];
}

#define CK(x)                          \
    do {                               \
        int _rc = (x);                 \
        if (_rc != OTH_OK) return _rc; \
    } while (0)
#define CU(x) CK(cuda_status(x))
}  // namespace

extern "C" int oth_host_valid_moves(const int8_t* states, const int8_t* players, uint8_t* out_masks, int64_t n)
{
    if (n < 0 || (n > 0 && (!states || !players || !out_masks))) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    void *ds, *dp, *dm;
    CK(scr().get(0, n * 64, &ds));
    CK(scr().get(1, n, &dp));
    CK(scr().get(2, n * 65, &dm));
    CU(cudaMemcpyAsync(ds, states, n * 64, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(dp, players, n, cudaMemcpyHostToDevice, 0));
    CK(oth_valid_moves_i8((const int8_t*)ds, (const int8_t*)dp, (uint8_t*)dm, n, 0));
    CU(cudaMemcpyAsync(out_masks, dm, n * 65, cudaMemcpyDeviceToHost, 0));
    CU(cudaStreamSynchronize(0));
    return OTH_OK;
}

extern "C" int oth_host_next_state(const int8_t* states, const int32_t* actions, const int8_t* players, int8_t* out_states,
                                   uint8_t* out_flags, int64_t n)
{
    if (n < 0 || (n > 0 && (!states || !players || !actions || !out_states || !out_flags))) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    void *ds, *dp, *da, *dout, *df;
    CK(scr().get(0, n * 64, &ds));
    CK(scr().get(1, n, &dp));
    CK(scr().get(2, n * 4, &da));
    CK(scr().get(3, n * 64, &dout));
    CK(scr().get(4, n, &df));
    CU(cudaMemcpyAsync(ds, states, n * 64, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(dp, players, n, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(da, actions, n * 4, cudaMemcpyHostToDevice, 0));
    k_next_state_i8<<<grid_for(n * 32, 256), 256>>>((const int8_t*)ds, (const int32_t*)da, (const int8_t*)dp, (int8_t*)dout,
                                                    (uint8_t*)df, n);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out_states, dout, n * 64, cudaMemcpyDeviceToHost, 0));
    CU(cudaMemcpyAsync(out_flags, df, n, cudaMemcpyDeviceToHost, 0));
    CU(cudaStreamSynchronize(0));
    for (int64_t i = 0; i < n; i++)
        if (out_flags[i] & OTH_F_ILLEGAL) return OTH_E_ILLEGAL;
    return OTH_OK;
}

extern "C" int oth_host_value_terminated(const int8_t* states, const int8_t* players, int8_t* out_values, uint8_t* out_terms,
                                         int64_t n)
{
    if (n < 0 || (n > 0 && (!states || !players || !out_values || !out_terms))) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    void *ds, *dp, *dv, *dt;
    CK(scr().get(0, n * 64, &ds));
    CK(scr().get(1, n, &dp));
    CK(scr().get(2, n, &dv));
    CK(scr().get(3, n, &dt));
    CU(cudaMemcpyAsync(ds, states, n * 64, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(dp, players, n, cudaMemcpyHostToDevice, 0));
    k_value_terminated_i8<<<grid_for(n * 32, 256), 256>>>((const int8_t*)ds, (const int8_t*)dp, (int8_t*)dv, (uint8_t*)dt, n);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out_values, dv, n, cudaMemcpyDeviceToHost, 0));
    CU(cudaMemcpyAsync(out_terms, dt, n, cudaMemcpyDeviceToHost, 0));
    CU(cudaStreamSynchronize(0));
    return OTH_OK;
}

extern "C" int oth_host_symmetry(const int8_t* states, const float* pis, const int32_t* ks, const uint8_t* flips_, float* out_states,
                                 float* out_pis, int64_t n)
{
    if (n < 0 || (n > 0 && (!states || !pis || !ks || !flips_ || !out_states || !out_pis))) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    void *ds, *dpi, *dk, *df, *dos, *dop;
    CK(scr().get(0, n * 64, &ds));
    CK(scr().get(1, n * 65 * 4, &dpi));
    CK(scr().get(2, n * 4, &dk));
    CK(scr().get(3, n, &df));
    CK(scr().get(4, n * 64 * 4, &dos));
    CK(scr().get(5, n * 65 * 4, &dop));
    CU(cudaMemcpyAsync(ds, states, n * 64, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(dpi, pis, n * 65 * 4, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(dk, ks, n * 4, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(df, flips_, n, cudaMemcpyHostToDevice, 0));
    CK(oth_symmetry((const int8_t*)ds, (const float*)dpi, (const int32_t*)dk, (const uint8_t*)df, (float*)dos, (float*)dop, n, 0));
    CU(cudaMemcpyAsync(out_states, dos, n * 64 * 4, cudaMemcpyDeviceToHost, 0));
    CU(cudaMemcpyAsync(out_pis, dop, n * 65 * 4, cudaMemcpyDeviceToHost, 0));
    CU(cudaStreamSynchronize(0));
    return OTH_OK;
}

extern "C" int oth_host_rollout(uint64_t seed, uint64_t game_id_base, int64_t n_games, int32_t* out_score, int32_t* out_plies,
                                uint64_t* out_final, int64_t n_trace, uint8_t* trace_actions, uint64_t* trace_moves,
                                unsigned long long* total_plies, float* kernel_ms)
{
    if (n_games <= 0 || n_trace < 0 || n_trace > n_games) return OTH_E_ARG;
    void *dsc, *dpl, *dfin, *dta = nullptr, *dtm = nullptr, *dcnt;
    CK(scr().get(0, n_games * 4, &dsc));
    CK(scr().get(1, n_games * 4, &dpl));
    CK(scr().get(2, n_games * 16, &dfin));
    if (n_trace) {
        CK(scr().get(3, n_trace * OTH_MAX_PLIES, &dta));
        CK(scr().get(4, n_trace * OTH_MAX_PLIES * 8, &dtm));
    }
    CK(scr().get(5, 64, &dcnt));
    CU(cudaMemsetAsync(dcnt, 0, 64, 0));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    CU(cudaEventRecord(e0, 0));
    int rc = oth_rollout(seed, game_id_base, n_games, (int32_t*)dsc, (int32_t*)dpl, (uint64_t*)dfin, n_trace, (uint8_t*)dta,
                         (uint64_t*)dtm, (unsigned long long*)dcnt, 0);
    CU(cudaEventRecord(e1, 0));
    if (rc != OTH_OK) return rc;
    if (out_score) CU(cudaMemcpyAsync(out_score, dsc, n_games * 4, cudaMemcpyDeviceToHost, 0));
    if (out_plies) CU(cudaMemcpyAsync(out_plies, dpl, n_games * 4, cudaMemcpyDeviceToHost, 0));
    if (out_final) CU(cudaMemcpyAsync(out_final, dfin, n_games * 16, cudaMemcpyDeviceToHost, 0));
    if (n_trace && trace_actions) CU(cudaMemcpyAsync(trace_actions, dta, n_trace * OTH_MAX_PLIES, cudaMemcpyDeviceToHost, 0));
    if (n_trace && trace_moves) CU(cudaMemcpyAsync(trace_moves, dtm, n_trace * OTH_MAX_PLIES * 8, cudaMemcpyDeviceToHost, 0));
    if (total_plies) CU(cudaMemcpyAsync(total_plies, dcnt, 8, cudaMemcpyDeviceToHost, 0));
    CU(cudaStreamSynchronize(0));
    if (kernel_ms) CU(cudaEventElapsedTime(kernel_ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return OTH_OK;
}

extern "C" int oth_host_int32_peak(double* out_ips, float* kernel_ms)
{
    const int blocks = sm_count() * 8, threads = 256, iters = 2048;
    void* d;
    CK(scr().get(6, (size_t)blocks * threads * 4, &d));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        CU(cudaEventRecord(e0, 0));
        k_int32_probe<<<blocks, threads>>>((unsigned*)d, iters, 0x12345u + rep, 0x9e3779b9u);
        CU(cudaEventRecord(e1, 0));
        CU(cudaStreamSynchronize(0));
        CU(cudaGetLastError());
        float ms;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    const double instr = (double)blocks * threads * (double)iters * 8.0 * 8.0 * 2.0;
    if (out_ips) *out_ips = instr / (best * 1e-3);
    if (kernel_ms) *kernel_ms = best;
    return OTH_OK;
}
