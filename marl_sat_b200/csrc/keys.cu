// Rollout RNG chain on device: JAX 0.4.29 Threefry-2x32 split / randint as used by
// src/learners/mappo_gnn_sat_learner.py:397,416-417,426-434 and src/runners/mappo_runner.py:289-295.
#include "internal.h"

namespace msat {

// rng,act = split(rng); rng,step = split(rng); rng,prob,reset = split(rng,3)   (learner:397,416,426)
__global__ void rng_chain_kernel(const uint32_t* rng_in, uint32_t* out) {   // may alias (read first)
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    uint32_t out10[10];
    rng_chain_compute(rng_in[0], rng_in[1], out10);
    for (int i = 0; i < 10; ++i) out[i] = out10[i];
}

__global__ void rng_split2_kernel(const uint32_t* __restrict__ key_in, uint32_t* __restrict__ out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    uint32_t a[2], b[2];
    split2(key_in[0], key_in[1], a, b);
    out[0] = a[0]; out[1] = a[1]; out[2] = b[0]; out[3] = b[1];
}

// Weighted problem draw (msat_env_keys_weighted): u = hi * 2^32 + lo, W = cum[P-1]; W <= 0 falls back to randint;
// otherwise r = floor(u * W / 2^64) and the index is the smallest p with cum[p] > r.  The binary search runs over
// [0, P-1] whatever the table holds, so the index stays in range for a non-monotone table.
__device__ __forceinline__ uint32_t weighted_problem(uint32_t hi, uint32_t lo, const long long* __restrict__ cum,
                                                     uint32_t P) {
    const long long W = cum[P - 1];
    if (W <= 0) return randint_from_bits(hi, lo, P);
    const unsigned long long u = ((unsigned long long)hi << 32) | lo;
    const long long r = (long long)__umul64hi(u, (unsigned long long)W);   // < W <= 2^63 - 1
    uint32_t a = 0u, b = P - 1u;
    while (a < b) {
        const uint32_t mid = (a + b) >> 1;
        if (cum[mid] > r) b = mid;
        else a = mid + 1u;
    }
    return a;
}

// problem_idx = randint(prob_key, (Bg,), 0, P)[off + b]; reset_keys = split(reset_key, Bg)[off + b]
// (jax._src.random._randint: two 32-bit draws combined with multiplier (2^16 % span)^2 % span).
// kWeighted: the problem index is drawn from the inclusive prefix sums `cum` instead (weighted_problem).  `cum` is the
// last parameter so that the uniform instantiation, which ignores it, keeps the parameter layout of the plain kernel.
template <bool kWeighted>
__global__ void __launch_bounds__(256) env_keys_kernel(const uint32_t* __restrict__ prob_key,
                                                       const uint32_t* __restrict__ reset_key, uint32_t Bg,
                                                       uint32_t off, uint32_t Bl, uint32_t P,
                                                       int32_t* __restrict__ idx, uint32_t* __restrict__ keys,
                                                       const long long* __restrict__ cum) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= Bl) return;
    const uint32_t g = off + b;
    if (idx) {
        if constexpr (kWeighted) {
            uint32_t hi, lo;
            env_problem_bits(prob_key[0], prob_key[1], Bg, g, hi, lo);
            idx[b] = (int32_t)weighted_problem(hi, lo, cum, P);
        } else {
            idx[b] = (int32_t)env_problem_index(prob_key[0], prob_key[1], Bg, g, P);
        }
    }
    if (keys) {
        uint32_t k[2];
        env_reset_key(reset_key[0], reset_key[1], Bg, g, k);
        keys[2 * b + 0] = k[0];
        keys[2 * b + 1] = k[1];
    }
}

cudaError_t launch_rng_chain(const uint32_t* rng_in, uint32_t* chain_out, cudaStream_t s) {
    rng_chain_kernel<<<1, 32, 0, s>>>(rng_in, chain_out);
    return cudaGetLastError();
}
cudaError_t launch_rng_split2(const uint32_t* key_in, uint32_t* out, cudaStream_t s) {
    rng_split2_kernel<<<1, 32, 0, s>>>(key_in, out);
    return cudaGetLastError();
}
cudaError_t launch_env_keys(const uint32_t* prob_key, const uint32_t* reset_key, int Bg, int off, int Bl, int P,
                            int32_t* idx, uint32_t* keys, const long long* cum_weights, cudaStream_t s) {
    if (Bl == 0) return cudaSuccess;
    const int grid = (Bl + 255) / 256;
    if (cum_weights)
        env_keys_kernel<true><<<grid, 256, 0, s>>>(prob_key, reset_key, (uint32_t)Bg, (uint32_t)off, (uint32_t)Bl,
                                                   (uint32_t)P, idx, keys, cum_weights);
    else
        env_keys_kernel<false><<<grid, 256, 0, s>>>(prob_key, reset_key, (uint32_t)Bg, (uint32_t)off, (uint32_t)Bl,
                                                    (uint32_t)P, idx, keys, nullptr);
    return cudaGetLastError();
}

}  // namespace msat
