// Leaf symmetry at the network boundary (include/othello_b200.h, "network boundary"): the leaf planes the search
// hands to the network are shown to it in one of the eight D4 orientations, or in all eight, and its policy rows are
// mapped back to the leaf's own orientation.  One warp per 64-square row: lane l holds squares l and l + 32, so a row
// is two coalesced 128-byte loads and every permutation is a pair of warp shuffles.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/othello_b200.h"
#include "common.cuh"
#include "philox.cuh"

using namespace oth;

namespace {

constexpr unsigned FULL = 0xffffffffu;

// T_s of oth_symmetry / k_symmetry: image[e] = plane[src(e, s)], np.rot90 (s & 3) times, then np.fliplr if s >> 2.
__device__ __forceinline__ int src_square(int e, int s)
{
    int r = e >> 3, c = e & 7;
    if (s >> 2) c = 7 - c;
    for (int q = 0; q < (s & 3); q++) {
        const int nr = c, nc = 7 - r;
        r = nr;
        c = nc;
    }
    return r * 8 + c;
}

// The inverse permutation: src_square(dst_square(d, s), s) == d.
__device__ __forceinline__ int dst_square(int d, int s)
{
    int r = d >> 3, c = d & 7;
    for (int q = 0; q < ((4 - (s & 3)) & 3); q++) {
        const int nr = c, nc = 7 - r;
        r = nr;
        c = nc;
    }
    if (s >> 2) c = 7 - c;
    return r * 8 + c;
}

// Square e of the row whose squares l and l + 32 are this lane's (a, b).
__device__ __forceinline__ float row_at(float a, float b, int e)
{
    const float va = __shfl_sync(FULL, a, e & 31), vb = __shfl_sync(FULL, b, e & 31);
    return e < 32 ? va : vb;
}

__device__ __forceinline__ int64_t warp_id() { return ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; }
__device__ __forceinline__ int64_t warp_count() { return ((int64_t)gridDim.x * blockDim.x) >> 5; }

__device__ __forceinline__ float warp_max(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(FULL, v, o));
    return v;
}

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

bool misaligned(const void* p, uintptr_t a) { return ((uintptr_t)p & (a - 1)) != 0; }

}  // namespace

__global__ void __launch_bounds__(256) k_nn_leaf_symmetry(const float* __restrict__ planes, int64_t n, uint64_t key,
                                                          float* __restrict__ out, uint8_t* __restrict__ out_sym)
{
    const int lane = threadIdx.x & 31;
    for (int64_t i = warp_id(); i < n; i += warp_count()) {
        const float a = planes[i * 64 + lane], b = planes[i * 64 + 32 + lane];
        const uint64_t own = (uint64_t)__ballot_sync(FULL, a == 1.0f) | (uint64_t)__ballot_sync(FULL, b == 1.0f) << 32;
        const uint32_t opp_lo = __ballot_sync(FULL, a == -1.0f), opp_hi = __ballot_sync(FULL, b == -1.0f);
        const int s = (int)(philox4x32_10(key, own, opp_lo, opp_hi).x & 7u);
        const float va = row_at(a, b, src_square(lane, s)), vb = row_at(a, b, src_square(lane + 32, s));
        out[i * 64 + lane] = va;
        out[i * 64 + 32 + lane] = vb;
        if (lane == 0) out_sym[i] = (uint8_t)s;
    }
}

// In place: row[src(e)] = row'[e], so that T_s(row) is the network's row' again.  Entry 64 (pass) and any padding
// columns are not touched; rows with s = 0 are left as they are.
template <typename T>
__global__ void __launch_bounds__(256) k_nn_unsymmetrise(T* __restrict__ logits, int64_t stride, const uint8_t* __restrict__ sym,
                                                         int64_t n)
{
    const int lane = threadIdx.x & 31;
    for (int64_t i = warp_id(); i < n; i += warp_count()) {
        const int s = sym[i] & 7;
        if (s == 0) continue;
        T* row = logits + i * stride;
        const T a = row[lane], b = row[lane + 32];
        __syncwarp();  // every lane has read its two entries before any lane writes
        row[src_square(lane, s)] = a;
        row[src_square(lane + 32, s)] = b;
    }
}

__global__ void __launch_bounds__(256) k_nn_symmetry_images(const float* __restrict__ planes, int64_t n, float* __restrict__ out)
{
    const int lane = threadIdx.x & 31;
    for (int64_t i = warp_id(); i < n; i += warp_count()) {
        const float a = planes[i * 64 + lane], b = planes[i * 64 + 32 + lane];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const float va = row_at(a, b, src_square(lane, j)), vb = row_at(a, b, src_square(lane + 32, j));
            float* o = out + (i * 8 + j) * 64;
            o[lane] = va;
            o[32 + lane] = vb;
        }
    }
}

// Leaf i: priors = (1/8) sum_j unsym_j(softmax(logits[8i + j])), values = (1/8) sum_j values[8i + j], j = 0..7 in order.
__global__ void __launch_bounds__(256) k_nn_symmetry_mean(const float* __restrict__ logits, int64_t stride,
                                                          const float* __restrict__ values, int64_t value_stride, int64_t n,
                                                          float* __restrict__ priors, float* __restrict__ out_values)
{
    const int lane = threadIdx.x & 31;
    for (int64_t i = warp_id(); i < n; i += warp_count()) {
        float acc0 = 0.0f, acc1 = 0.0f, acc_pass = 0.0f;
#pragma unroll 1
        for (int j = 0; j < 8; j++) {
            const float* row = logits + (i * 8 + j) * stride;
            const float a = row[lane], b = row[lane + 32], p = row[64];
            const float m = fmaxf(warp_max(fmaxf(a, b)), p);
            const float ea = expf(a - m), eb = expf(b - m), ep = expf(p - m);
            const float inv = 1.0f / (warp_sum(ea + eb) + ep);
            // the prior of square d in the leaf's orientation is the image's prior at dst(d)
            acc0 += row_at(ea, eb, dst_square(lane, j)) * inv;
            acc1 += row_at(ea, eb, dst_square(lane + 32, j)) * inv;
            acc_pass += ep * inv;
        }
        priors[i * 65 + lane] = acc0 * 0.125f;
        priors[i * 65 + 32 + lane] = acc1 * 0.125f;
        if (lane == 0) {
            priors[i * 65 + 64] = acc_pass * 0.125f;
            float v = 0.0f;
            for (int j = 0; j < 8; j++) v += values[(i * 8 + j) * value_stride];
            out_values[i] = v * 0.125f;
        }
    }
}

extern "C" int oth_nn_leaf_symmetry(const float* planes, int64_t n, uint64_t seed, float* out_planes, uint8_t* out_sym,
                                    void* stream)
{
    if (n < 0) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    if (!planes || !out_planes || !out_sym || planes == out_planes || misaligned(planes, 4) || misaligned(out_planes, 4))
        return OTH_E_ARG;
    k_nn_leaf_symmetry<<<grid_for(n * 32, 256), 256, 0, (cudaStream_t)stream>>>(planes, n, seed ^ OTH_SYM_SALT, out_planes,
                                                                                out_sym);
    return cuda_status(cudaGetLastError());
}

extern "C" int oth_nn_unsymmetrise_logits(void* logits, int64_t stride, int32_t is_bf16, const uint8_t* sym, int64_t n,
                                          void* stream)
{
    if (n < 0 || stride < OTH_NUM_ACTIONS || (is_bf16 != 0 && is_bf16 != 1)) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    if (!logits || !sym || misaligned(logits, is_bf16 ? 2 : 4)) return OTH_E_ARG;
    const int grid = grid_for(n * 32, 256);
    if (is_bf16)
        k_nn_unsymmetrise<<<grid, 256, 0, (cudaStream_t)stream>>>((__nv_bfloat16*)logits, stride, sym, n);
    else
        k_nn_unsymmetrise<<<grid, 256, 0, (cudaStream_t)stream>>>((float*)logits, stride, sym, n);
    return cuda_status(cudaGetLastError());
}

extern "C" int oth_nn_symmetry_images(const float* planes, int64_t n, float* out, void* stream)
{
    if (n < 0) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    if (!planes || !out || misaligned(planes, 4) || misaligned(out, 4)) return OTH_E_ARG;
    k_nn_symmetry_images<<<grid_for(n * 32, 256), 256, 0, (cudaStream_t)stream>>>(planes, n, out);
    return cuda_status(cudaGetLastError());
}

extern "C" int oth_nn_symmetry_mean(const float* logits, int64_t stride, const float* values, int64_t value_stride, int64_t n,
                                    float* priors, float* out_values, void* stream)
{
    if (n < 0 || stride < OTH_NUM_ACTIONS || value_stride < 1) return OTH_E_ARG;
    if (n == 0) return OTH_OK;
    if (!logits || !values || !priors || !out_values || misaligned(logits, 4) || misaligned(values, 4) ||
        misaligned(priors, 4) || misaligned(out_values, 4))
        return OTH_E_ARG;
    k_nn_symmetry_mean<<<grid_for(n * 32, 256), 256, 0, (cudaStream_t)stream>>>(logits, stride, values, value_stride, n, priors,
                                                                                out_values);
    return cuda_status(cudaGetLastError());
}
