// Shared device helpers for the SATEnv kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace msat {

// Device-side view of a plan; passed by value to every kernel.
struct Dims {
    int n, m, k, A, V, D, AD;
    int ms;               // literal-column stride inside a bank record: m rounded up to even (32-bit paired loads)
    int action_mode, max_steps;
    int base, rem;        // contiguous balanced grouping: size_a = base + (a < rem)
    int aw, sw, xw, fw;   // words: assignment, clause status, obs value vector (+1 pad), flat mask stream
    int lits_bytes;       // padded byte size of the literal-code block inside a bank record
    int rec_bytes;        // bank record size = stride between records (multiple of 128)
    int rec_copy_bytes;   // leading part staged by observation-writing launches: literals + agent-mask stream
    int csr_off;          // byte offset of the var -> clause occurrence lists inside a record (0 = not built)
    int csr_bytes;        // their size, padded to 16 bytes (one TMA bulk copy into the group's record slot)
    int cnt_words;        // incremental clause update: words of per-clause true-literal counts (4 bits each) in the
                          // state record after the 4 scalar fields; 0 = full recompute (default)
    int state_words;      // env-state record words (multiple of 4)
    int agw;              // words of an agent bit-set = ceil(A/32)
    uint32_t inv_D;       // ceil(2^32 / D): j / D = umulhi(j, inv_D) (minus 1 when that overshoots)
};

// State record word offsets (after the aw assignment words).
enum { ST_STEP = 0, ST_PIDX = 1, ST_NUNSAT = 2, ST_FLAGS = 3 };

// Literal code of a 0-padding literal (never true): one past the last real code (var << 1 | negated), so that
// the per-env literal truth table tt[code] (2n + 1 bytes, tt[2n] = 0) answers it without a special case.
__host__ __device__ __forceinline__ uint32_t lit_pad(const Dims& d) { return 2u * (uint32_t)d.n; }

// Literal codes are stored literal-major ([k][ms], ms = m rounded up to even, the spare column holds padding
// codes) inside a bank record: consecutive lanes = consecutive clauses read consecutive u16 (conflict-free
// shared-memory loads), and one aligned 32-bit load fetches the codes of two adjacent clauses.
__host__ __device__ __forceinline__ int lit_index(int ms, int c, int j) { return j * ms + c; }

// Problem index of an env as every kernel reads it: clamped into [0, P), so an index from outside (reset_from_bank,
// import_state(validate=False)) or a corrupted state record never addresses past the bank.
__device__ __forceinline__ int clamp_problem(int pidx, int P) { return pidx < 0 ? 0 : (pidx >= P ? P - 1 : pidx); }

// ---- agent grouping (env:294-338; contiguous balanced split) --------------
__host__ __device__ __forceinline__ int group_size(const Dims& d, int a) { return d.base + (a < d.rem ? 1 : 0); }
__host__ __device__ __forceinline__ int group_start(const Dims& d, int a) { return a * d.base + (a < d.rem ? a : d.rem); }
__host__ __device__ __forceinline__ int var_to_agent(const Dims& d, int v) {
    const int big = d.rem * (d.base + 1);
    return v < big ? v / (d.base + 1) : d.rem + (v - big) / d.base;
}

// ---- Threefry-2x32 (JAX 0.4.29 default PRNG; oracle/threefry.py) ---------
__host__ __device__ __forceinline__ uint32_t rotl32(uint32_t x, int r) { return (x << r) | (x >> (32 - r)); }

__host__ __device__ __forceinline__ void threefry2x32(uint32_t k0, uint32_t k1, uint32_t& x0, uint32_t& x1) {
    const uint32_t ks[3] = {k0, k1, k0 ^ k1 ^ 0x1BD11BDAu};
    x0 += ks[0];
    x1 += ks[1];
#define MSAT_TF_ROUND(r) x0 += x1; x1 = rotl32(x1, r); x1 ^= x0;
#define MSAT_TF_A MSAT_TF_ROUND(13) MSAT_TF_ROUND(15) MSAT_TF_ROUND(26) MSAT_TF_ROUND(6)
#define MSAT_TF_B MSAT_TF_ROUND(17) MSAT_TF_ROUND(29) MSAT_TF_ROUND(16) MSAT_TF_ROUND(24)
    MSAT_TF_A x0 += ks[1]; x1 += ks[2] + 1u;
    MSAT_TF_B x0 += ks[2]; x1 += ks[0] + 2u;
    MSAT_TF_A x0 += ks[0]; x1 += ks[1] + 3u;
    MSAT_TF_B x0 += ks[1]; x1 += ks[2] + 4u;
    MSAT_TF_A x0 += ks[2]; x1 += ks[0] + 5u;
#undef MSAT_TF_A
#undef MSAT_TF_B
#undef MSAT_TF_ROUND
}

// Element i of threefry_2x32(key, arange(N)) (jax._src.prng.threefry_2x32 with
// the odd-length zero pad): first half of the counters feeds word 0, second half word 1.
__host__ __device__ __forceinline__ uint32_t bits32_at(uint32_t k0, uint32_t k1, uint32_t N, uint32_t i) {
    const uint32_t half = (N + 1u) >> 1;
    const bool lo = i < half;
    const uint32_t blk = lo ? i : i - half;
    uint32_t x0 = blk;
    uint32_t x1 = (half + blk < N) ? half + blk : 0u;   // the pad counter is 0
    threefry2x32(k0, k1, x0, x1);
    return lo ? x0 : x1;
}

// a, b = jax.random.split(key): counters [0,1,2,3] -> blocks (0,2),(1,3); a = {x0(0), x0(1)}, b = {x1(0), x1(1)}.
__host__ __device__ __forceinline__ void split2(uint32_t k0, uint32_t k1, uint32_t a[2], uint32_t b[2]) {
    uint32_t p0 = 0u, p1 = 2u, q0 = 1u, q1 = 3u;
    threefry2x32(k0, k1, p0, p1);
    threefry2x32(k0, k1, q0, q1);
    a[0] = p0; a[1] = q0; b[0] = p1; b[1] = q1;
}

// One rollout step of the key chain (learner:397,416,426):
//   rng,act = split(rng); rng,step = split(rng); rng,prob,reset = split(rng,3)
// out[10] = {rng', act_key, step_key, prob_key, reset_key}.
__host__ __device__ __forceinline__ void rng_chain_compute(uint32_t r0, uint32_t r1, uint32_t out[10]) {
    uint32_t a[2], b[2];
    split2(r0, r1, a, b);                       // rng <- a, act_key <- b
    out[2] = b[0]; out[3] = b[1];
    r0 = a[0]; r1 = a[1];
    split2(r0, r1, a, b);                       // rng <- a, step_key <- b
    out[4] = b[0]; out[5] = b[1];
    r0 = a[0]; r1 = a[1];
    // split(rng, 3) = threefry_2x32(rng, arange(6)).reshape(3, 2): blocks (0,3),(1,4),(2,5)
    uint32_t x0 = 0u, x1 = 3u, y0 = 1u, y1 = 4u, z0 = 2u, z1 = 5u;
    threefry2x32(r0, r1, x0, x1);
    threefry2x32(r0, r1, y0, y1);
    threefry2x32(r0, r1, z0, z1);
    out[0] = x0; out[1] = y0;                   // rng'
    out[6] = z0; out[7] = x1;                   // prob_key
    out[8] = y1; out[9] = z1;                   // reset_key
}

// The two 32-bit draws of randint(prob_key, (Bg,), 0, P)[g] (learner:430): (k1, k2) = split(prob_key),
// hi = bits32_at(k1, Bg, g), lo = bits32_at(k2, Bg, g).  The weighted draw (msat_env_keys_weighted) uses the same words.
__host__ __device__ __forceinline__ void env_problem_bits(uint32_t pk0, uint32_t pk1, uint32_t Bg, uint32_t g,
                                                          uint32_t& hi, uint32_t& lo) {
    uint32_t k1[2], k2[2];
    split2(pk0, pk1, k1, k2);
    hi = bits32_at(k1[0], k1[1], Bg, g);
    lo = bits32_at(k2[0], k2[1], Bg, g);
}

// jax._src.random._randint's combination of the two draws into [0, P)
__host__ __device__ __forceinline__ uint32_t randint_from_bits(uint32_t hi, uint32_t lo, uint32_t P) {
    const uint32_t span = P > 0u ? P : 1u;
    uint32_t mult = 65536u % span;
    mult = (mult * mult) % span;
    return ((hi % span) * mult + (lo % span)) % span;
}

// problem index and reset key of global env g out of Bg (learner:430,434):
//   randint(prob_key, (Bg,), 0, P)[g]  and  split(reset_key, Bg)[g]
__host__ __device__ __forceinline__ uint32_t env_problem_index(uint32_t pk0, uint32_t pk1, uint32_t Bg, uint32_t g,
                                                               uint32_t P) {
    uint32_t hi, lo;
    env_problem_bits(pk0, pk1, Bg, g, hi, lo);
    return randint_from_bits(hi, lo, P);
}
__host__ __device__ __forceinline__ void env_reset_key(uint32_t rk0, uint32_t rk1, uint32_t Bg, uint32_t g,
                                                       uint32_t key[2]) {
    key[0] = bits32_at(rk0, rk1, 2u * Bg, 2u * g);
    key[1] = bits32_at(rk0, rk1, 2u * Bg, 2u * g + 1u);
}

#ifdef __CUDACC__
// The same derivation for ONE env spread over four consecutive lanes (`lane4` = 0..3 within `mask`): the thirteen
// Threefry blocks of  chain -> (prob_key, reset_key) -> (problem index, reset key)  form five dependent levels, and
// the blocks of a level run on different lanes (branch-free: a diverging warp would run them one after the other).
//   level 1-2: split(rng), split(rng)            two blocks each (lanes 0,1)
//   level 3:   split(rng, 3)                     three blocks (lanes 0,1,2)
//   level 4:   split(prob_key) (lanes 0,1)  +  the two words of split(reset_key, Bg)[g] (lanes 2,3)
//   level 5:   the high / low draws of randint(prob_key, (Bg,), 0, P)[g] (lanes 0,1)
// have_chain: prob_key / reset_key are already known (c6..c9), levels 1-3 are skipped.  Every lane of `mask` must
// call; all of them return the same results.
__device__ __forceinline__ void env_reset_inputs_4lanes(uint32_t mask, int lane4, int base_lane, bool have_chain,
                                                        uint32_t r0, uint32_t r1, uint32_t c6, uint32_t c7, uint32_t c8,
                                                        uint32_t c9, uint32_t Bg, uint32_t g, uint32_t P,
                                                        uint32_t& pidx, uint32_t& key0, uint32_t& key1) {
    uint32_t x0, x1;
    if (!have_chain) {
        for (int lvl = 0; lvl < 2; ++lvl) {                      // rng <- split(rng)[0]: blocks (0,2), (1,3)
            x0 = (uint32_t)(lane4 & 1);
            x1 = 2u + (uint32_t)(lane4 & 1);
            threefry2x32(r0, r1, x0, x1);
            r0 = __shfl_sync(mask, x0, base_lane);
            r1 = __shfl_sync(mask, x0, base_lane + 1);
        }
        const uint32_t i = lane4 < 3 ? (uint32_t)lane4 : 0u;     // split(rng, 3): blocks (0,3), (1,4), (2,5)
        x0 = i;
        x1 = 3u + i;
        threefry2x32(r0, r1, x0, x1);
        c7 = __shfl_sync(mask, x1, base_lane);                   // prob_key = {z0, x1(block 0)}
        c8 = __shfl_sync(mask, x1, base_lane + 1);               // reset_key = {y1, z1}
        c6 = __shfl_sync(mask, x0, base_lane + 2);
        c9 = __shfl_sync(mask, x1, base_lane + 2);
    }
    // level 4: lanes 0,1 -> block lane of split(prob_key); lanes 2,3 -> word (lane - 2) of split(reset_key, Bg)[g]
    const bool upper = lane4 >= 2;
    const uint32_t N2 = 2u * Bg, half2 = (N2 + 1u) >> 1;
    const uint32_t i2 = 2u * g + (uint32_t)(lane4 & 1);
    const bool lo2 = i2 < half2;
    const uint32_t blk2 = lo2 ? i2 : i2 - half2;
    x0 = upper ? blk2 : (uint32_t)(lane4 & 1);
    x1 = upper ? ((half2 + blk2 < N2) ? half2 + blk2 : 0u) : 2u + (uint32_t)(lane4 & 1);
    threefry2x32(upper ? c8 : c6, upper ? c9 : c7, x0, x1);
    const uint32_t word = lo2 ? x0 : x1;
    key0 = __shfl_sync(mask, word, base_lane + 2);
    key1 = __shfl_sync(mask, word, base_lane + 3);
    const uint32_t k10 = __shfl_sync(mask, x0, base_lane), k11 = __shfl_sync(mask, x0, base_lane + 1);   // k1 = a
    const uint32_t k20 = __shfl_sync(mask, x1, base_lane), k21 = __shfl_sync(mask, x1, base_lane + 1);   // k2 = b
    // level 5: lane 0 (and 2) draws the high word from k1, lane 1 (and 3) the low word from k2
    const bool odd = (lane4 & 1) != 0;
    const uint32_t v = bits32_at(odd ? k20 : k10, odd ? k21 : k11, Bg, g);
    const uint32_t hi = __shfl_sync(mask, v, base_lane), lo = __shfl_sync(mask, v, base_lane + 1);
    const uint32_t span = P > 0u ? P : 1u;
    uint32_t mult = 65536u % span;
    mult = (mult * mult) % span;
    pidx = ((hi % span) * mult + (lo % span)) % span;
}
#endif

// ---- bit-stream helpers ------------------------------------------------------
// 32 bits starting at bit `pos` of a clean little-endian bit array of `nwords` words
// (bits past the logical end are zero; reads outside the array return zero).  pos may be negative.
__device__ __forceinline__ uint32_t ldw(const uint32_t* a, int i, int nwords) {
    return (i >= 0 && i < nwords) ? a[i] : 0u;
}
__device__ __forceinline__ uint32_t extract32(const uint32_t* a, int nwords, int pos) {
    const int w = pos >> 5;             // arithmetic shift: floor for negatives
    const int sh = pos & 31;
    const uint32_t lo = ldw(a, w, nwords);
    const uint32_t hi = ldw(a, w + 1, nwords);
    return __funnelshift_r(lo, hi, sh);
}

// ---- mbarrier + TMA bulk copy (global -> shared) --------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    // make the initialised barrier visible to the async (TMA) proxy; CTA scope is enough without clusters
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!ok);
}
// 1-D bulk copy through the TMA engine; bytes % 16 == 0, both addresses 16-byte aligned.
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Barrier over the GS threads that cooperate on one env (GS = 8 / 16: four / two envs share a warp and synchronise with
// sub-warp lane masks; their control flow may diverge, e.g. when only one of them auto-resets).  The named-barrier index must be an
// immediate: with a register index ptxas reserves all 16 hardware barriers for the CTA, which caps
// the number of resident CTAs per SM.
// GS < 32: lane mask of the sub-warp group (GS consecutive lanes) this thread belongs to, and its first lane
template <int GS>
__device__ __forceinline__ uint32_t subwarp_shift() { return threadIdx.x & (32u - GS) & 31u; }
template <int GS>
__device__ __forceinline__ uint32_t subwarp_mask() { return ((1u << GS) - 1u) << subwarp_shift<GS>(); }

template <int GS>
__device__ __forceinline__ void group_sync(int gid) {
    if constexpr (GS < 32) {
        __syncwarp(subwarp_mask<GS>());                 // the lanes of this warp that own this env
    } else if constexpr (GS == 32) {
        __syncwarp();
    } else if constexpr (GS == 256) {
        asm volatile("bar.sync 1, 256;" ::: "memory");
    } else if constexpr (GS == 128) {
        if (gid == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
        else asm volatile("bar.sync 2, 128;" ::: "memory");
    } else {
        switch (gid) {
            case 0: asm volatile("bar.sync 1, 64;" ::: "memory"); break;
            case 1: asm volatile("bar.sync 2, 64;" ::: "memory"); break;
            case 2: asm volatile("bar.sync 3, 64;" ::: "memory"); break;
            default: asm volatile("bar.sync 4, 64;" ::: "memory"); break;
        }
    }
}

}  // namespace msat
