// Private declarations shared by the translation units of libmarlsat_b200.so.
#pragma once
#include <atomic>

#include "common.cuh"

namespace msat {

constexpr int kCtaThreads = 256;
constexpr int kMaxSmemOptin = 227 * 1024;

// Shared-memory carve-up of one env group (byte offsets from the group base).  Launches that write
// observations stage the whole bank record (literals + agent-mask stream) and need the value / mask
// re-basing buffers; launches without observations stage only the literal block and keep the per-clause
// true-literal counts for the GNN features, so eight one-warp groups fit in ~26 KB per CTA.
struct GroupLayout {
    int rec, st, satw, satw_old, x, smx, tt, stage, bar, misc, total;
};
constexpr int kCfStageClauses = 256;               // clauses per staging pass of the GNN clause features
constexpr int kCfStageBytes = 12 * kCfStageClauses + 16;
inline GroupLayout group_layout(const Dims& d, bool obs) {
    GroupLayout L;
    int o = 0;
    // TMA destination, 128-byte aligned: whole record (observations), literal block, or -- in the step launches of
    // an incremental plan -- the occurrence lists, whichever is larger
    const int noobs_rec = d.lits_bytes > d.csr_bytes ? d.lits_bytes : d.csr_bytes;
    L.rec = o;  o += ((obs ? d.rec_copy_bytes : noobs_rec) + 127) & ~127;
    L.st = o;   o += 4 * d.state_words;           // state record (multiple of 16 bytes)
    L.stage = o; o += obs ? 0 : kCfStageBytes;    // 16-byte aligned (rec and state sizes are multiples of 16)
    L.satw = o; o += 4 * d.sw;
    L.satw_old = o; o += 4 * d.sw;                // clause status before the flips (shaped-reward mode only)
    L.x = o;    o += obs ? 4 * d.xw : 0;
    L.tt = o;   o += ((2 * d.n + 4) & ~3) + 4;    // literal truth table: 2n + 1 bytes, written as 32-bit words
    o = (o + 7) & ~7;
    L.smx = o;  o += obs ? 8 * (d.fw + 2) : 0;    // {mask word, value word} per 32 observation ints
    L.bar = o;  o += 8;                           // mbarrier
    L.misc = o; o += 16 + 128;                    // [0] #unsatisfied accumulator, [1] new problem idx, [2..3] reset key,
                                                  // then float2[16]: {t > 0, t / 3.0} table of the GNN clause features
    L.total = (o + 127) & ~127;
    return L;
}

}  // namespace msat

struct msat_plan {
    msat::Dims d;
    int group_threads;     // GS: threads cooperating on one env (16 = two envs per warp, 32/64/128/256)
    int group_smem_bytes;  // shared memory per env group (multiple of 128)
    int smem_bytes;        // dynamic shared memory per 256-thread CTA
    int group_threads_noobs;   // GS used when a launch writes no observations (little per-env work: small groups)
    int smem_bytes_noobs;
    msat::GroupLayout layout_obs, layout_noobs;   // shared-memory carve-up of one env group, computed once
    int compile_smem_bytes;
    int requested_group_threads = 0;
    int reward_mode = 0;       // MSAT_REWARD_SPARSE / MSAT_REWARD_SHAPED (msat_plan_set_reward)
    float r_gamma = 0.99f, r_clause = 0.02f, r_sat = 1.0f;
    unsigned long long* reset_counter = nullptr;   // device counter of auto-resets (diagnostics), or null
    int obs_i8 = 0;            // MSAT_OBS_INT8: observations are written as int8 instead of int32
    // devices on which the > 48 KB dynamic shared memory opt-in of the env kernels has been made (bit = device
    // ordinal); set once per (plan, device) instead of once per launch
    mutable std::atomic<unsigned long long> prepared_devices{0};
    mutable std::atomic<unsigned long long> prepared_walksat{0};   // the same opt-in for walksat_kernel
};

namespace msat {

constexpr int kMaxFusedSteps = 64;                // K of msat_rollout_steps

struct EnvArgs {
    GroupLayout L;              // filled in by launch_env from the plan
    const uint8_t* bank;
    int P;
    const uint32_t* state_in;
    uint32_t* state_out;
    const int32_t* actions;
    const int32_t* prob_idx;
    const uint32_t* keys;
    const uint32_t* rng_in;     // fused key derivation (msat_rollout_step): rollout rng before this step
    uint32_t* chain_out;        // ... and the advanced chain {rng', act, step, prob, reset}
    uint32_t Bg, env_off;       // global batch size and this shard's first global env index
    int auto_reset;
    int32_t* obs;
    int32_t* gnn_assign;        // optional GNN-input outputs of the state the caller continues from
    float* gnn_cf;              // (learner:165-195): assignment int32[B,n], clause_features float[B,m,3]
    float* reward;
    int reward_cols;
    uint8_t* done;
    int done_cols;
    uint8_t* solved;
    int32_t* num_unsat;
    int32_t* episode_step;
    int B;
    // multi-step launches (msat_rollout_steps): K steps per env in one launch; step j reads
    // actions + j * act_step_stride and writes row j of every [K, B, ...] output; observations / GNN
    // inputs are written for every step (emit_every_step) or for the last one only
    int num_steps;
    long long act_step_stride;
    int emit_every_step;
    // reward: 0 = sparse solved reward (env:183-198); 1 = shaped reward of env:201-223
    //   gamma * (-unsat') + unsat + r_clause * #newly satisfied + [solved] * r_sat
    int reward_mode;
    float r_gamma, r_clause, r_sat;
    int32_t* newly_sat;         // optional int32[(K,) B]: clauses satisfied now that were not before the step
    unsigned long long* reset_count;   // optional device counter: += 1 for every auto-reset (msat_plan_set_reset_counter)
    int obs_i8;                 // `obs` points to int8 elements (msat_plan_set_obs_dtype)
    // state import (msat_import_state): reference-shaped leaves in place of the reset's Threefry draw;
    // assignment int32[B, n] (nonzero = 1), step int32[B] and done uint8[B] (NULL = 0)
    const int32_t* assign_in;
    const int32_t* step_in;
    const uint8_t* done_in;
    // start states (msat_apply_start_states): per-problem packed start assignments uint32[P, aw], flip thresholds
    // uint32[P] and flags uint8[P] (NULL = every problem has a start); the envs' reset key is derived from
    // reset_key with the global env index (Bg, env_off)
    const uint32_t* start_words;
    const uint32_t* flip_thr;
    const uint8_t* has_start;
    const uint32_t* reset_key;
};

// MODE_IMPORT: the reset path with the assignment, step and done flag read from memory
// MODE_START: the reset path for the envs that just restarted (step == 0) on a problem with a start state, with the
// assignment taken from that start and flipped by bits drawn from the env's reset key; every other env is left alone
enum EnvMode { MODE_RESET = 0, MODE_STEP = 1, MODE_OBS = 2, MODE_IMPORT = 3, MODE_START = 4 };

extern int g_gae_force_plain;   // gae.cu; msat_tune("gae_plain", 1)
extern int g_gae_variant;       // gae.cu; msat_tune("gae_variant", v)
extern int g_gae_pipe_min_cols; // gae.cu; msat_tune("gae_pipe_min_cols", B)
extern int g_gae_warps_per_sm;  // gae.cu; msat_tune("gae_warps_per_sm", w)

struct ExportArgs {
    const uint8_t* bank;
    int P;
    const uint32_t* state;
    int B;
    int32_t* assign;
    uint8_t* sat;
    int32_t* num_unsat;
    int32_t* step;
    uint8_t* done;
    int32_t* clauses;
    int32_t* acm;
    int32_t* anm;
    int32_t* l2a;
    int32_t* pidx;
};

// ---- WalkSAT (local_search.cu) ----------------------------------------------------------------------------
// Shared-memory carve-up of one warp's env (byte offsets from the warp base): the staged literal block, the
// var -> clause occurrence lists built from it, u8 true-literal counts, unsatisfied / repeated-variable clause bits,
// the assignment and the per-candidate break counters.
constexpr int kWalksatMaxK = 32;                   // one lane per literal column of the picked clause
constexpr int kWalksatMaxWarps = 8;
struct WalksatLayout {
    int lits, occ, row, cnt, unsat, dup, assign, brk, bar, total;
};
inline WalksatLayout walksat_layout(const Dims& d) {
    WalksatLayout L;
    int o = 0;
    L.lits = o;   o += (d.lits_bytes + 127) & ~127;          // TMA destination
    L.occ = o;    o += (2 * d.m * d.k + 15) & ~15;           // u16 (clause << 1) | negated, grouped by variable
    L.row = o;    o += (4 * d.n + 15) & ~15;                 // int: end of variable v's list (start = row[v - 1])
    L.cnt = o;    o += (d.m + 15) & ~15;                     // u8 true-literal count per clause
    L.unsat = o;  o += 4 * d.sw;
    L.dup = o;    o += 4 * d.sw;                             // clause mentions a variable more than once
    L.assign = o; o += 4 * d.aw;
    L.brk = o;    o += 4 * kWalksatMaxK;
    o = (o + 7) & ~7;
    L.bar = o;    o += 8;
    L.total = (o + 127) & ~127;
    return L;
}
// warps (envs) per CTA; 0 = one env's working set does not fit in shared memory
inline int walksat_warps(const Dims& d) {
    if (d.k > kWalksatMaxK) return 0;
    const int w = kMaxSmemOptin / walksat_layout(d).total;
    return w < kWalksatMaxWarps ? w : kWalksatMaxWarps;
}
struct WalksatArgs {
    const uint8_t* bank;
    int P;
    uint32_t* state;
    const uint32_t* keys;
    int max_flips, flip_offset;
    uint32_t thr;               // random walk iff (x1 >> 8) < thr; llrint(noise * 2^24)
    uint8_t* solved;
    int32_t* flips;
    int B;
};
cudaError_t launch_walksat(const msat_plan* plan, const WalksatArgs& a, cudaStream_t s);

cudaError_t launch_compile_bank(const msat_plan* plan, const int32_t* clauses, int P, uint8_t* bank, cudaStream_t s);
cudaError_t launch_env(const msat_plan* plan, EnvMode mode, const EnvArgs& a, cudaStream_t s);
cudaError_t launch_export(const msat_plan* plan, const ExportArgs& a, cudaStream_t s);
cudaError_t launch_rng_chain(const uint32_t* rng_in, uint32_t* chain_out, cudaStream_t s);
cudaError_t launch_rng_split2(const uint32_t* key_in, uint32_t* out, cudaStream_t s);
// cum_weights == NULL: the uniform randint draw; else the weighted draw of msat_env_keys_weighted
cudaError_t launch_env_keys(const uint32_t* prob_key, const uint32_t* reset_key, int Bg, int off, int Bl, int P,
                            int32_t* idx, uint32_t* keys, const long long* cum_weights, cudaStream_t s);
// N = global element count (< 2^32 - 1), C >= 1, num_rows > 0
cudaError_t launch_sample_actions(const float* logits, uint32_t N, uint32_t row_offset, int num_rows, int C,
                                  const uint32_t* rng_in, int32_t* actions, float* log_prob, cudaStream_t s);
cudaError_t launch_problem_stats(const int32_t* pidx, long long ps_t, long long ps_b, const uint8_t* done,
                                 const uint8_t* solved, const int32_t* num_unsat, const int32_t* episode_step, int T,
                                 int B, int P, long long* stats, cudaStream_t s);
cudaError_t launch_gae(const float* reward, long long rs_t, long long rs_b, const uint8_t* done, const float* value,
                       const float* last_val, float gamma, float gamma_lambda, float* adv, float* targets, int T, int B,
                       double* stats, cudaStream_t s);
cudaError_t launch_adv_stats(const float* adv, long long count, double* stats, cudaStream_t s);
cudaError_t launch_adv_normalize(float* adv, long long count, const double* stats, cudaStream_t s);
cudaError_t launch_gnn_static(const msat_plan* plan, const uint8_t* bank, int P, float* svf, float* a_pos, float* a_neg,
                              cudaStream_t s);
cudaError_t launch_gnn_dynamic(const msat_plan* plan, const uint8_t* bank, int P, const uint32_t* state, int B,
                               int32_t* assign, float* cf, cudaStream_t s);
cudaError_t launch_rollout_metrics(const float* reward, long long rs_t, long long rs_b, const uint8_t* done,
                                   const uint8_t* solved, const int32_t* num_unsat, const int32_t* episode_step, int T,
                                   int B, double* sums, cudaStream_t s);
cudaError_t launch_flip_gains(const msat_plan* plan, const uint8_t* bank, int P, const uint32_t* state, int B, float tau,
                              int32_t* delta, int32_t* labels, cudaStream_t s);
cudaError_t launch_eval_track(const msat_plan* plan, const uint32_t* state, const uint8_t* solved, int t, int B,
                              uint8_t* ever, int32_t* steps, int32_t* solution, cudaStream_t s);

}  // namespace msat
