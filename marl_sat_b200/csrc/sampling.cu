// Categorical action draw from the rollout's act_key (learner:397-403: `rng, act_key = split(rng);
// action = pi.sample(seed=act_key)`): the Gumbel-max draw of jax.random.categorical over distrax-normalised logits.
// Contract in include/marl_sat_b200.h (msat_sample_actions); oracle/sampling.py restates it.
#include <float.h>

#include "internal.h"

namespace msat {

namespace {

constexpr int kSampleThreads = 256;

// max of the logits with NaN / +inf mapped to +inf: +inf flags an invalid row, -inf an all -inf row
__device__ __forceinline__ float screened(float l) { return (l != l || l == INFINITY) ? INFINITY : l; }

// jax.random.gumbel from the 32 random bits of one element: uniform(minval=tiny, maxval=1) then -log(-log(u))
__device__ __forceinline__ float gumbel_from_bits(uint32_t bits) {
    const float f = __uint_as_float((bits >> 9) | 0x3F800000u) - 1.0f;
    const float u = fmaxf(FLT_MIN, f * (1.0f - FLT_MIN) + FLT_MIN);
    return -logf(-logf(u));
}

// best (score, class) so far: the larger score wins, ties go to the smaller class (jnp.argmax)
__device__ __forceinline__ void take_best(float s, int c, float z, float& bs, int& bc, float& bz) {
    if (s > bs || (s == bs && c < bc)) { bs = s; bc = c; bz = z; }
}

// One warp handles R = 32 / C rows of C <= 32 classes (kLoop = false: one class per lane, lanes >= R * C idle) or one
// row of C > 32 classes (kLoop = true: lane j owns classes j, j + 32, ...).  W = min(C, 32) lanes form a row's segment;
// reductions run over the segment with shuffles down by 1, 2, 4, ... < W, so the segment's first lane holds the
// result, which it broadcasts.  Consecutive lanes read consecutive floats of the row-major table.
template <bool kLoop>
__global__ void __launch_bounds__(kSampleThreads) sample_actions_kernel(
        const float* __restrict__ logits, uint32_t N, uint32_t row_offset, int num_rows, int C,
        const uint32_t* __restrict__ rng_in, int32_t* __restrict__ actions, float* __restrict__ log_prob) {
    __shared__ uint32_t act_key[2];
    const int lane = threadIdx.x & 31;
    const int W = kLoop ? 32 : C;
    const int R = kLoop ? 1 : 32 / C;
    const int seg = lane / W;                                   // row of this lane inside the warp's R rows
    const int j = lane - seg * W;                               // first class of this lane
    const int head = seg * W;
    const long long row = ((long long)blockIdx.x * (kSampleThreads / 32) + (threadIdx.x >> 5)) * R + seg;
    const bool active = seg < R && row < num_rows;
    const float* lrow = logits + row * C;
    float first = -INFINITY;
    if (active && j < C) first = __ldg(lrow + j);               // issued before the key is ready

    // act_key = split(rng_in)[1] = {x1 of block (0, 2), x1 of block (1, 3)}, once per CTA
    if (threadIdx.x < 2) {
        uint32_t x0 = threadIdx.x, x1 = 2u + threadIdx.x;
        threefry2x32(rng_in[0], rng_in[1], x0, x1);
        act_key[threadIdx.x] = x1;
    }
    __syncthreads();
    const uint32_t k0 = act_key[0], k1 = act_key[1];

    // 1. M = max over the row, +inf when the row holds a NaN or +inf
    float m = screened(first);
    if constexpr (kLoop)
        for (int c = j + 32; c < C; c += 32) m = fmaxf(m, active ? screened(__ldg(lrow + c)) : -INFINITY);
    for (int o = 1; o < W; o <<= 1) {
        const float v = __shfl_down_sync(0xffffffffu, m, o);
        if (j + o < W) m = fmaxf(m, v);
    }
    m = __shfl_sync(0xffffffffu, m, head);
    const bool valid = m != INFINITY && m != -INFINITY;

    // 2. S = sum of exp(l - M)
    float s = (j < C) ? expf(first - m) : 0.0f;
    if constexpr (kLoop)
        for (int c = j + 32; c < C; c += 32) s += expf((active ? __ldg(lrow + c) : -INFINITY) - m);
    for (int o = 1; o < W; o <<= 1) {
        const float v = __shfl_down_sync(0xffffffffu, s, o);
        if (j + o < W) s += v;
    }
    const float lse = logf(__shfl_sync(0xffffffffu, s, head));

    // 3. z = (l - M) - log S; action = the first class maximising gumbel + z
    const uint32_t e0 = (row_offset + (uint32_t)row) * (uint32_t)C;
    float bs = -INFINITY, bz = -INFINITY;
    int bc = 0x7fffffff;
    if (active && j < C) {
        const float z = (first - m) - lse;
        take_best(gumbel_from_bits(bits32_at(k0, k1, N, e0 + (uint32_t)j)) + z, j, z, bs, bc, bz);
    }
    if constexpr (kLoop)
        for (int c = j + 32; c < C; c += 32) {
            if (!active) break;
            const float z = (__ldg(lrow + c) - m) - lse;
            take_best(gumbel_from_bits(bits32_at(k0, k1, N, e0 + (uint32_t)c)) + z, c, z, bs, bc, bz);
        }
    for (int o = 1; o < W; o <<= 1) {
        const float vs = __shfl_down_sync(0xffffffffu, bs, o);
        const int vc = __shfl_down_sync(0xffffffffu, bc, o);
        const float vz = __shfl_down_sync(0xffffffffu, bz, o);
        if (j + o < W) take_best(vs, vc, vz, bs, bc, bz);
    }
    if (active && j == 0) {
        actions[row] = valid ? bc : -1;
        if (log_prob) log_prob[row] = valid ? bz : -INFINITY;
    }
}

}  // namespace

cudaError_t launch_sample_actions(const float* logits, uint32_t N, uint32_t row_offset, int num_rows, int C,
                                  const uint32_t* rng_in, int32_t* actions, float* log_prob, cudaStream_t s) {
    const int rows_per_warp = C <= 32 ? 32 / C : 1;
    const long long warps = ((long long)num_rows + rows_per_warp - 1) / rows_per_warp;
    const unsigned grid = (unsigned)((warps + kSampleThreads / 32 - 1) / (kSampleThreads / 32));
    if (C <= 32)
        sample_actions_kernel<false><<<grid, kSampleThreads, 0, s>>>(logits, N, row_offset, num_rows, C, rng_in,
                                                                     actions, log_prob);
    else
        sample_actions_kernel<true><<<grid, kSampleThreads, 0, s>>>(logits, N, row_offset, num_rows, C, rng_in,
                                                                    actions, log_prob);
    return cudaGetLastError();
}

}  // namespace msat
