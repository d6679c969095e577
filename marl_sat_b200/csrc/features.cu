// Next-tier rows of the hot path (SURVEY.md section 8f): the GNN-input emitter that the reference's
// SATDataWrapper builds from the env state (src/learners/mappo_gnn_sat_learner.py:149-195,
// src/utils/graph_constructor.py:93-114), the rollout-metric reductions (learner:661-686) and the
// first-solve tracking of the greedy evaluation loop (src/runners/mappo_runner.py:57-70).
#include "internal.h"

namespace msat {

// ---- static graph, once per formula (graph_constructor.py:93-114; learner:150-164) -------------------
// static_var_features f32[P,n,3] = [pos_degree/m, neg_degree/m, 0]; optional dense A_pos / A_neg f32[P,n,m]
// (occurrence counts: duplicates accumulate like `.at[].add`).
__global__ void __launch_bounds__(256) gnn_static_kernel(const Dims d, const uint8_t* __restrict__ bank,
                                                         float* __restrict__ svf, float* __restrict__ a_pos,
                                                         float* __restrict__ a_neg) {
    extern __shared__ int deg[];                     // [2][n] positive / negative degrees
    const int p = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const uint16_t* lits = reinterpret_cast<const uint16_t*>(bank + (size_t)p * d.rec_bytes);
    for (int i = tid; i < 2 * d.n; i += nt) deg[i] = 0;
    if (a_pos)
        for (size_t i = tid; i < (size_t)d.n * d.m; i += nt) a_pos[(size_t)p * d.n * d.m + i] = 0.0f;
    if (a_neg)
        for (size_t i = tid; i < (size_t)d.n * d.m; i += nt) a_neg[(size_t)p * d.n * d.m + i] = 0.0f;
    __syncthreads();
    for (int c = tid; c < d.m; c += nt) {            // one thread owns column c of A_pos / A_neg
        for (int j = 0; j < d.k; ++j) {
            const uint32_t code = lits[lit_index(d.ms, c, j)];
            if (code == lit_pad(d)) continue;
            const int v = (int)(code >> 1), neg = (int)(code & 1u);
            atomicAdd(&deg[neg * d.n + v], 1);
            float* A = neg ? a_neg : a_pos;
            if (A) A[(size_t)p * d.n * d.m + (size_t)v * d.m + c] += 1.0f;
        }
    }
    __syncthreads();
    if (svf)
        for (int v = tid; v < d.n; v += nt) {
            float* o = svf + ((size_t)p * d.n + v) * 3;
            o[0] = __fdiv_rn((float)deg[v], (float)d.m);            // learner:157
            o[1] = __fdiv_rn((float)deg[d.n + v], (float)d.m);      // learner:158
            o[2] = 0.0f;                                            // learner:160
        }
}

// ---- dynamic features, per env (learner:165-195) -------------------------------------------------------
// assignment i32[B,n]; clause_features f32[B,m,3] = [is_sat, n_true_literals / 3.0, 1]
// (the divisor is the literal 3.0 of learner:185 for every clause width).
__global__ void __launch_bounds__(128) gnn_dynamic_kernel(const Dims d, const uint8_t* __restrict__ bank, int P,
                                                          const uint32_t* __restrict__ state, int32_t* __restrict__ assign,
                                                          float* __restrict__ cf) {
    const int e = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const uint32_t* st = state + (size_t)e * d.state_words;
    const int pidx = clamp_problem((int)st[d.aw + ST_PIDX], P);
    const uint16_t* lits = reinterpret_cast<const uint16_t*>(bank + (size_t)pidx * d.rec_bytes);
    if (assign)
        for (int v = tid; v < d.n; v += nt) assign[(size_t)e * d.n + v] = (int)((st[v >> 5] >> (v & 31)) & 1u);
    if (cf)
        for (int c = tid; c < d.m; c += nt) {
            int ntrue = 0;
            for (int j = 0; j < d.k; ++j) {
                const uint32_t code = lits[lit_index(d.ms, c, j)];
                if (code != lit_pad(d)) {
                    const uint32_t v = code >> 1;
                    ntrue += (int)(((st[v >> 5] >> (v & 31)) ^ code) & 1u);
                }
            }
            float* o = cf + ((size_t)e * d.m + c) * 3;
            o[0] = ntrue > 0 ? 1.0f : 0.0f;
            o[1] = __fdiv_rn((float)ntrue, 3.0f);
            o[2] = 1.0f;
        }
}

// ---- rollout metrics (learner:661-686) ----------------------------------------------------------------
// sums[5] += { sum reward(agent 0), #finished, #solved at finish, sum num_unsatisfied at finish,
//              sum episode_step of solved-at-finish } over all T*B transitions.
__global__ void __launch_bounds__(256) rollout_metrics_kernel(const float* __restrict__ reward, long long rs_t,
                                                              long long rs_b, const uint8_t* __restrict__ done,
                                                              const uint8_t* __restrict__ solved,
                                                              const int32_t* __restrict__ num_unsat,
                                                              const int32_t* __restrict__ episode_step, int T, int B,
                                                              double* __restrict__ sums) {
    double acc[5] = {0, 0, 0, 0, 0};
    const long long N = (long long)T * B, stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
        const long long t = i / B, b = i - t * B;
        acc[0] += (double)reward[t * rs_t + b * rs_b];
        if (done[i]) {
            acc[1] += 1.0;
            acc[3] += (double)num_unsat[i];
            if (solved[i]) {
                acc[2] += 1.0;
                acc[4] += (double)episode_step[i];
            }
        }
    }
    __shared__ double sh[5][8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        double x = acc[k];
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) sh[k][warp] = x;
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        double x = 0.0;
        for (int w = 0; w < 8; ++w) x += sh[threadIdx.x][w];
        if (x != 0.0) atomicAdd(&sums[threadIdx.x], x);
    }
}

// ---- per-problem statistics (msat_problem_stats) ------------------------------------------------------------
// stats[p][0..3] += {#finished, #solved at finish, sum num_unsatisfied at finish, sum episode_step of solved-at-finish}
// over the rows (t, b) with done != 0, p = the clamped problem index of the row.  A warp takes 32 consecutive rows; the
// lanes whose rows end an episode of the same problem form one group (__match_any_sync) and its lowest lane adds the
// group's sums, so a hot problem costs one update per warp instead of one per row.  kSmem: the CTA accumulates into
// P * 4 shared counters and flushes each non-zero one with one global atomic.
constexpr int kStatsSmemProblems = 1024;   // 32 KB of counters: six 256-thread CTAs still fit an SM's shared memory

// exact sum of the int32 values of a lane group: the low 16 bits (unsigned) and the high 16 bits (signed) are reduced
// separately, so neither 32-bit reduction can overflow
__device__ __forceinline__ long long group_sum(unsigned grp, int v) {
    return (long long)__reduce_add_sync(grp, v >> 16) * 65536LL + (long long)__reduce_add_sync(grp, (unsigned)v & 0xFFFFu);
}

template <bool kSmem>
__global__ void __launch_bounds__(256) problem_stats_kernel(const int32_t* __restrict__ pidx, long long ps_t,
                                                            long long ps_b, const uint8_t* __restrict__ done,
                                                            const uint8_t* __restrict__ solved,
                                                            const int32_t* __restrict__ num_unsat,
                                                            const int32_t* __restrict__ episode_step, int T, int B,
                                                            int P, unsigned long long* __restrict__ stats) {
    extern __shared__ unsigned long long sacc[];          // [P][4] (kSmem)
    if constexpr (kSmem) {
        for (int i = threadIdx.x; i < 4 * P; i += blockDim.x) sacc[i] = 0ull;
        __syncthreads();
    }
    unsigned long long* acc = kSmem ? sacc : stats;
    const int lane = threadIdx.x & 31;
    const long long N = (long long)T * B, stride = (long long)gridDim.x * blockDim.x;
    // the warp's lanes share the trip count (the base is warp-aligned), so the full-warp votes below are legal
    for (long long base = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < N; base += stride) {
        const long long i = base + lane;
        int p = -1, nu = 0, es = 0;
        bool sol = false;
        if (i < N && done[i]) {
            const long long t = i / B, b = i - t * B;
            p = clamp_problem(pidx[t * ps_t + b * ps_b], P);
            sol = solved[i] != 0;
            nu = num_unsat[i];
            es = sol ? episode_step[i] : 0;
        }
        if (!__any_sync(0xffffffffu, p >= 0)) continue;
        const unsigned sol_lanes = __ballot_sync(0xffffffffu, sol);
        const unsigned grp = __match_any_sync(0xffffffffu, p);
        if (p < 0) continue;
        const unsigned nsol = __popc(grp & sol_lanes);
        const long long snu = group_sum(grp, nu), ses = group_sum(grp, es);
        if (lane != __ffs(grp) - 1) continue;
        unsigned long long* row = acc + 4 * p;
        atomicAdd(row + 0, (unsigned long long)__popc(grp));
        if (nsol) atomicAdd(row + 1, (unsigned long long)nsol);
        if (snu) atomicAdd(row + 2, (unsigned long long)snu);
        if (ses) atomicAdd(row + 3, (unsigned long long)ses);
    }
    if constexpr (kSmem) {
        __syncthreads();
        for (int i = threadIdx.x; i < 4 * P; i += blockDim.x)
            if (sacc[i]) atomicAdd(stats + i, sacc[i]);
    }
}

// ---- greedy evaluation bookkeeping (runner:57-70) --------------------------------------------------------
// After evaluation step t (0-based): envs that are solved for the first time record steps_to_solve = t+1
// and a copy of their packed assignment.
__global__ void __launch_bounds__(256) eval_track_kernel(const Dims d, const uint32_t* __restrict__ state,
                                                         const uint8_t* __restrict__ solved, int t, int B,
                                                         uint8_t* __restrict__ ever, int32_t* __restrict__ steps,
                                                         int32_t* __restrict__ solution) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B || !solved[e] || ever[e]) return;
    ever[e] = 1;
    steps[e] = t + 1;
    const uint32_t* st = state + (size_t)e * d.state_words;
    for (int v = 0; v < d.n; ++v) solution[(size_t)e * d.n + v] = (int)((st[v >> 5] >> (v & 31)) & 1u);
}

// ---- per-variable flip gains and the greedy expert labels (behavioral_cloning.py:54-100) -----------------
// delta_unsat[v] = (#unsatisfied after flipping v alone) - (#unsatisfied now) = break[v] - make[v]:
//   an unsatisfied clause becomes satisfied by flipping any variable it mentions (make, once per clause);
//   a satisfied clause breaks iff all its true literals are on v and it has no false literal on v.
// greedy label of agent a: the owned variable with the most negative delta (first wins ties), kept only
// if that delta < tau, else the no-op action V.
__global__ void __launch_bounds__(128) flip_gain_kernel(const Dims d, const uint8_t* __restrict__ bank, int P,
                                                        const uint32_t* __restrict__ state, float tau,
                                                        int32_t* __restrict__ delta_out, int32_t* __restrict__ labels) {
    extern __shared__ int gain[];                     // [n] break - make
    const int e = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    const uint32_t* st = state + (size_t)e * d.state_words;
    const int pidx = clamp_problem((int)st[d.aw + ST_PIDX], P);
    const uint16_t* lits = reinterpret_cast<const uint16_t*>(bank + (size_t)pidx * d.rec_bytes);
    for (int v = tid; v < d.n; v += nt) gain[v] = 0;
    __syncthreads();
    for (int c = tid; c < d.m; c += nt) {
        int ntrue = 0;
        for (int j = 0; j < d.k; ++j) {
            const uint32_t code = lits[lit_index(d.ms, c, j)];
            if (code != lit_pad(d)) ntrue += (int)(((st[(code >> 1) >> 5] >> ((code >> 1) & 31)) ^ code) & 1u);
        }
        for (int j = 0; j < d.k; ++j) {
            const uint32_t code = lits[lit_index(d.ms, c, j)];
            if (code == lit_pad(d)) continue;
            const uint32_t v = code >> 1;
            bool first = true;              // handle each distinct variable of the clause once
            int true_on_v = 0, false_on_v = 0;
            for (int i = 0; i < d.k; ++i) {
                const uint32_t ci = lits[lit_index(d.ms, c, i)];
                if (ci == lit_pad(d) || (ci >> 1) != v) continue;
                if (i < j) first = false;
                const int t = (int)(((st[v >> 5] >> (v & 31)) ^ ci) & 1u);
                true_on_v += t;
                false_on_v += 1 - t;
            }
            if (!first) continue;
            if (ntrue == 0) atomicSub(&gain[v], 1);                                   // make
            else if (true_on_v == ntrue && false_on_v == 0) atomicAdd(&gain[v], 1);   // break
        }
    }
    __syncthreads();
    if (delta_out)
        for (int v = tid; v < d.n; v += nt) delta_out[(size_t)e * d.n + v] = gain[v];
    if (labels)
        for (int a = tid; a < d.A; a += nt) {
            const int start = group_start(d, a), size = group_size(d, a);
            float best_delta = 0.0f;
            int best = d.V;
            for (int j = 0; j < size; ++j) {
                const float dl = (float)gain[start + j];
                if (dl < best_delta) { best_delta = dl; best = j; }
            }
            labels[(size_t)e * d.A + a] = (best_delta < tau) ? best : d.V;
        }
}

cudaError_t launch_flip_gains(const msat_plan* plan, const uint8_t* bank, int P, const uint32_t* state, int B, float tau,
                              int32_t* delta, int32_t* labels, cudaStream_t s) {
    if (B == 0) return cudaSuccess;
    flip_gain_kernel<<<B, 128, plan->d.n * sizeof(int), s>>>(plan->d, bank, P, state, tau, delta, labels);
    return cudaGetLastError();
}

cudaError_t launch_gnn_static(const msat_plan* plan, const uint8_t* bank, int P, float* svf, float* a_pos,
                              float* a_neg, cudaStream_t s) {
    if (P == 0) return cudaSuccess;
    gnn_static_kernel<<<P, 256, 2 * plan->d.n * sizeof(int), s>>>(plan->d, bank, svf, a_pos, a_neg);
    return cudaGetLastError();
}
cudaError_t launch_gnn_dynamic(const msat_plan* plan, const uint8_t* bank, int P, const uint32_t* state, int B,
                               int32_t* assign, float* cf, cudaStream_t s) {
    if (B == 0) return cudaSuccess;
    gnn_dynamic_kernel<<<B, 128, 0, s>>>(plan->d, bank, P, state, assign, cf);
    return cudaGetLastError();
}
cudaError_t launch_rollout_metrics(const float* reward, long long rs_t, long long rs_b, const uint8_t* done,
                                   const uint8_t* solved, const int32_t* num_unsat, const int32_t* episode_step, int T,
                                   int B, double* sums, cudaStream_t s) {
    const long long N = (long long)T * B;
    if (N == 0) return cudaSuccess;
    long long blocks = (N + 256 * 8 - 1) / (256 * 8);
    blocks = blocks > 148 * 8 ? 148 * 8 : (blocks < 1 ? 1 : blocks);
    rollout_metrics_kernel<<<(int)blocks, 256, 0, s>>>(reward, rs_t, rs_b, done, solved, num_unsat, episode_step, T, B,
                                                       sums);
    return cudaGetLastError();
}
cudaError_t launch_problem_stats(const int32_t* pidx, long long ps_t, long long ps_b, const uint8_t* done,
                                 const uint8_t* solved, const int32_t* num_unsat, const int32_t* episode_step, int T,
                                 int B, int P, long long* stats, cudaStream_t s) {
    const long long N = (long long)T * B;
    if (N == 0) return cudaSuccess;
    unsigned long long* out = reinterpret_cast<unsigned long long*>(stats);
    long long blocks = (N + 256 * 8 - 1) / (256 * 8);
    if (P <= kStatsSmemProblems) {
        // every CTA flushes up to 4P counters: fewer, longer-lived CTAs (four per SM) keep that cost small
        blocks = blocks > 148 * 4 ? 148 * 4 : blocks;
        problem_stats_kernel<true><<<(int)blocks, 256, 4 * P * sizeof(unsigned long long), s>>>(
            pidx, ps_t, ps_b, done, solved, num_unsat, episode_step, T, B, P, out);
    } else {
        blocks = blocks > 148 * 8 ? 148 * 8 : blocks;
        problem_stats_kernel<false><<<(int)blocks, 256, 0, s>>>(pidx, ps_t, ps_b, done, solved, num_unsat,
                                                                episode_step, T, B, P, out);
    }
    return cudaGetLastError();
}
cudaError_t launch_eval_track(const msat_plan* plan, const uint32_t* state, const uint8_t* solved, int t, int B,
                              uint8_t* ever, int32_t* steps, int32_t* solution, cudaStream_t s) {
    if (B == 0) return cudaSuccess;
    eval_track_kernel<<<(B + 255) / 256, 256, 0, s>>>(plan->d, state, solved, t, B, ever, steps, solution);
    return cudaGetLastError();
}

}  // namespace msat
