// extern "C" boundary of libmarlsat_b200.so (include/marl_sat_b200.h): plan construction, argument
// validation and kernel enqueue.  No allocation, no synchronisation (except msat_step_host, which is
// documented to synchronise), no torch types.
#include <math.h>
#include <string.h>
#include <map>
#include <mutex>
#include <new>

#include "../../include/marl_sat_b200.h"
#include "internal.h"

using namespace msat;

namespace {

inline bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }
inline int cuda_rc(cudaError_t e) { return e == cudaSuccess ? MSAT_OK : (int)e; }
inline size_t actions_per_env(const Dims& d) { return (size_t)d.A * (d.action_mode == 0 ? 1 : d.V); }
// GNN clause features come from a 16-entry table indexed by the true-literal count: k <= 15.
inline bool clause_features_unsupported(const msat_plan* plan, const float* cf) { return cf && plan->d.k > 15; }
constexpr int kMaxSmem = 227 * 1024;
constexpr int kMaxPipeDepth = 4;

// Internal streams + fork/join events used by msat_rollout_step_host to overlap PCIe copies with the kernel:
// one set per device, created on first use, released by msat_shutdown().
struct SyncPipe {
    cudaStream_t ws[2] = {nullptr, nullptr};
    cudaEvent_t fork = nullptr, join[2] = {nullptr, nullptr};
    cudaError_t create() {
        cudaError_t e = cudaSuccess;
        for (int w = 0; w < 2 && e == cudaSuccess; ++w) {
            e = cudaStreamCreateWithFlags(&ws[w], cudaStreamNonBlocking);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&join[w], cudaEventDisableTiming);
        }
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&fork, cudaEventDisableTiming);
        return e;
    }
    void destroy() {
        for (int w = 0; w < 2; ++w) {
            if (ws[w]) cudaStreamDestroy(ws[w]);
            if (join[w]) cudaEventDestroy(join[w]);
            ws[w] = nullptr; join[w] = nullptr;
        }
        if (fork) cudaEventDestroy(fork);
        fork = nullptr;
    }
};
std::mutex g_pipe_mu;
std::map<int, SyncPipe> g_pipes;      // device ordinal -> pipe

// must be called with g_pipe_mu held; leaves the current device unchanged
cudaError_t sync_pipe_for_current_device(SyncPipe** out) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    auto it = g_pipes.find(dev);
    if (it == g_pipes.end()) {
        SyncPipe sp;
        e = sp.create();
        if (e != cudaSuccess) { sp.destroy(); return e; }
        it = g_pipes.emplace(dev, sp).first;
    }
    *out = &it->second;
    return cudaSuccess;
}

// Every env entry point: a plan, B >= 0, P > 0 and, when B > 0, the bank and the caller's own required pointers.
inline bool bad_env_call(const msat_plan* plan, const void* bank, int32_t P, int32_t B, bool missing) {
    return !plan || B < 0 || P <= 0 || (B > 0 && (!bank || missing));
}

// bad_env_call, then bank (128 bytes), state and observation (16 bytes) alignment; fills the base of `a`.
int env_args(EnvArgs& a, const msat_plan* plan, const void* bank, int32_t P, const uint32_t* state_in,
             uint32_t* state_out, int32_t* obs, int32_t B, bool missing) {
    if (bad_env_call(plan, bank, P, B, missing)) return MSAT_EINVAL;
    if (!aligned(bank, 128) || !aligned(state_in, 16) || !aligned(state_out, 16) || !aligned(obs, 16))
        return MSAT_EALIGN;
    a = EnvArgs{};
    a.bank = static_cast<const uint8_t*>(bank); a.P = P;
    a.state_in = state_in; a.state_out = state_out; a.obs = obs; a.B = B;
    return MSAT_OK;
}

// Per-step outputs of msat_step and the fused rollout steps, added to `a` with the plan's reward: reward
// [B, reward_cols] and done [B, done_cols] need a positive column count, newly_satisfied the shaped reward.
int step_outputs(EnvArgs& a, const msat_plan* plan, float* reward, int32_t reward_cols, uint8_t* done,
                 int32_t done_cols, uint8_t* solved, int32_t* num_unsat, int32_t* episode_step, int32_t* newly_sat) {
    if ((done && done_cols <= 0) || (reward && reward_cols <= 0)) return MSAT_EINVAL;
    if (newly_sat && plan->reward_mode != MSAT_REWARD_SHAPED) return MSAT_EINVAL;
    a.reward = reward; a.reward_cols = reward_cols; a.done = done; a.done_cols = done_cols;
    a.solved = solved; a.num_unsat = num_unsat; a.episode_step = episode_step; a.newly_sat = newly_sat;
    a.reward_mode = plan->reward_mode; a.r_gamma = plan->r_gamma; a.r_clause = plan->r_clause; a.r_sat = plan->r_sat;
    a.reset_count = plan->reset_counter;
    return MSAT_OK;
}

// A shard [off, off + B) inside a global batch of Bg envs, Bg at most 2^30.
int shard_rule(int32_t Bg, int32_t off, int32_t B) {
    if (Bg < 0 || off < 0 || B < 0 || (long long)off + B > Bg) return MSAT_EINVAL;
    return Bg > (1 << 30) ? MSAT_EUNSUPPORTED : MSAT_OK;
}

// Checks of the fused rollout steps; on success `a` is the launch for the whole batch.
int rollout_args(EnvArgs& a, const msat_plan* plan, const void* bank, int32_t P, const uint32_t* state_in,
                 uint32_t* state_out, const int32_t* actions, int32_t K, const uint32_t* rng_in, uint32_t* chain_out,
                 int32_t Bg, int32_t env_offset, int32_t* obs, int32_t* gnn_assign, float* gnn_cf,
                 int32_t emit_every_step, float* reward, int32_t reward_cols, uint8_t* done, int32_t done_cols,
                 uint8_t* solved, int32_t* num_unsat, int32_t* episode_step, int32_t* newly_sat, int32_t B) {
    if (K < 1 || K > kMaxFusedSteps || !rng_in || !chain_out || Bg <= 0) return MSAT_EINVAL;
    // the advanced chain is written while other CTAs still read rng_in: the buffers must not overlap
    const uintptr_t r = reinterpret_cast<uintptr_t>(rng_in), c = reinterpret_cast<uintptr_t>(chain_out);
    if (r + 8 > c && c + 40 > r) return MSAT_EINVAL;
    int rc = env_args(a, plan, bank, P, state_in, state_out, obs, B, !state_in || !state_out || !actions);
    if (rc == MSAT_OK) rc = step_outputs(a, plan, reward, reward_cols, done, done_cols, solved, num_unsat, episode_step,
                                         newly_sat);
    if (rc == MSAT_OK) rc = shard_rule(Bg, env_offset, B);
    if (rc != MSAT_OK) return rc;
    if (clause_features_unsupported(plan, gnn_cf)) return MSAT_EUNSUPPORTED;
    a.actions = actions; a.num_steps = K; a.act_step_stride = (long long)B * actions_per_env(plan->d);
    a.auto_reset = 1; a.rng_in = rng_in; a.chain_out = chain_out; a.Bg = (uint32_t)Bg; a.env_off = (uint32_t)env_offset;
    a.gnn_assign = gnn_assign; a.gnn_cf = gnn_cf; a.emit_every_step = emit_every_step ? 1 : 0;
    return MSAT_OK;
}

cudaError_t rollout_enqueue(const msat_plan* plan, const EnvArgs& a, cudaStream_t s) {
    if (a.B > 0) return launch_env(plan, MODE_STEP, a, s);
    cudaError_t e = cudaSuccess;   // an empty shard still advances the chain K times
    for (int j = 0; j < a.num_steps && e == cudaSuccess; ++j)
        e = launch_rng_chain(j == 0 ? a.rng_in : a.chain_out, a.chain_out, s);
    return e;
}

// A rollout step with actions and results in host memory.  check() validates the whole batch before anything is
// enqueued; after it, each stage of a slice [b0, b0 + bc) can fail only with a CUDA error.
struct HostStep {
    const msat_plan* plan;
    const int32_t* actions_host; int32_t* actions_dev;
    float* reward_host; uint8_t* done_host; uint8_t* solved_host; int32_t* nunsat_host; int32_t* estep_host;
    EnvArgs a{};                // the fused step of the whole batch
    size_t act_per_env = 0, obs_env_bytes = 0;
    int check(const void* bank, int32_t P, uint32_t* state, const uint32_t* rng_in, uint32_t* chain_out, int32_t Bg,
              int32_t env_offset, int32_t* obs_dev, float* reward_dev, int32_t reward_cols, uint8_t* done_dev,
              int32_t done_cols, uint8_t* solved_dev, int32_t* nunsat_dev, int32_t* estep_dev, int32_t B) {
        if (!plan || !actions_host || !actions_dev || B < 0) return MSAT_EINVAL;
        act_per_env = actions_per_env(plan->d);
        obs_env_bytes = (size_t)plan->d.A * plan->d.D * (plan->obs_i8 ? 1 : 4);   // int8 plans: one byte per element
        return rollout_args(a, plan, bank, P, state, state, actions_dev, 1, rng_in, chain_out, Bg, env_offset, obs_dev,
                            nullptr, nullptr, 0, reward_dev, reward_cols, done_dev, done_cols, solved_dev, nunsat_dev,
                            estep_dev, nullptr, B);
    }
    cudaError_t upload(int b0, int bc, cudaStream_t w) const {
        const size_t off = b0 * act_per_env, bytes = bc * act_per_env * sizeof(int32_t);
        if (bytes == 0) return cudaSuccess;
        return cudaMemcpyAsync(actions_dev + off, actions_host + off, bytes, cudaMemcpyHostToDevice, w);
    }
    cudaError_t step(int b0, int bc, cudaStream_t w) const {
        EnvArgs s = a;
        s.B = bc; s.env_off += b0; s.actions += b0 * act_per_env; s.act_step_stride = (long long)bc * act_per_env;
        s.state_in += (size_t)b0 * plan->d.state_words; s.state_out += (size_t)b0 * plan->d.state_words;
        if (s.obs) s.obs = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(s.obs) + b0 * obs_env_bytes);
        auto at = [b0](auto* p, size_t per_env) { return p ? p + b0 * per_env : p; };
        s.reward = at(s.reward, s.reward_cols); s.done = at(s.done, s.done_cols);
        s.solved = at(s.solved, 1); s.num_unsat = at(s.num_unsat, 1); s.episode_step = at(s.episode_step, 1);
        return rollout_enqueue(plan, s, w);
    }
    cudaError_t download(int b0, int bc, cudaStream_t w) const;
};

// Outputs that are adjacent in both address spaces (the Python layer carves them out of one device block and
// one pinned block) travel as ONE copy.
cudaError_t HostStep::download(int b0, int bc, cudaStream_t w) const {
    struct Seg { const char* dev; char* host; size_t bytes; };
    Seg seg[5];
    int ns = 0;
    auto add = [&](const void* dv, void* hs, size_t off, size_t bytes) {
        if (dv && hs && bytes) seg[ns++] = Seg{static_cast<const char*>(dv) + off, static_cast<char*>(hs) + off, bytes};
    };
    add(a.reward, reward_host, (size_t)b0 * a.reward_cols * sizeof(float), (size_t)bc * a.reward_cols * sizeof(float));
    add(a.num_unsat, nunsat_host, (size_t)b0 * 4, (size_t)bc * 4);
    add(a.episode_step, estep_host, (size_t)b0 * 4, (size_t)bc * 4);
    add(a.done, done_host, (size_t)b0 * a.done_cols, (size_t)bc * a.done_cols);
    add(a.solved, solved_host, (size_t)b0, (size_t)bc);
    for (int i = 1; i < ns; ++i)          // insertion sort by device address
        for (int j = i; j > 0 && seg[j].dev < seg[j - 1].dev; --j) { Seg t = seg[j]; seg[j] = seg[j - 1]; seg[j - 1] = t; }
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < ns && e == cudaSuccess;) {
        Seg cur = seg[i++];
        while (i < ns && seg[i].dev == cur.dev + cur.bytes && seg[i].host == cur.host + cur.bytes) cur.bytes += seg[i++].bytes;
        e = cudaMemcpyAsync(cur.host, cur.dev, cur.bytes, cudaMemcpyDeviceToHost, w);
    }
    return e;
}

// Smallest group size from gs up to 256 whose CTA (plus the K key chains of a multi-step launch) fits; 0 if none.
int fit_group_threads(int gs, const GroupLayout& L) {
    for (; gs <= 256; gs *= 2)
        if ((long long)L.total * (kCtaThreads / gs) + 40 * kMaxFusedSteps <= kMaxSmem) return gs;
    return 0;
}

// Sizes that depend on the clause-update mode (d.cnt_words), group sizes and shared-memory layouts.
int finish_plan(msat_plan* p) {
    Dims& d = p->d;
    const int n = d.n, m = d.m, k = d.k;
    d.rec_copy_bytes = (d.lits_bytes + 4 * (d.fw + 1) + 15) & ~15;
    if (d.cnt_words) {
        // incremental clause update: var -> clause occurrence lists (CSR) behind the mask stream --
        // u16 row_off[n + 1] (padded to 8 entries), u16 occ[m * k] = (clause << 1) | negated
        d.csr_off = d.rec_copy_bytes;
        d.csr_bytes = (2 * ((n + 1 + 7) & ~7) + 2 * m * k + 15) & ~15;
        d.rec_bytes = (d.csr_off + d.csr_bytes + 127) & ~127;
    } else {
        d.csr_off = 0;
        d.csr_bytes = 0;
        d.rec_bytes = (d.rec_copy_bytes + 127) & ~127;
    }
    d.state_words = (d.aw + 4 + d.cnt_words + 3) & ~3;

    const int chunks = (d.AD + 3) / 4;
    int gs = p->requested_group_threads;
    // measured on B200 (profiles/r1_group_size_sweep.md): about 16-24 store iterations per thread is the sweet
    // spot -- larger groups idle most lanes in the short per-env phases, smaller ones serialise the stores
    // -- and below ~450 chunks (uf20-91: 164, uf35-149: 384) two envs share a warp (half-warp groups): the fixed
    // per-env instruction count, not the stores, bounds those shapes (profiles/r2_group_size_sweep.md)
    if (gs == 0) gs = chunks <= 448 ? 16 : (chunks <= 768 ? 32 : (chunks <= 1536 ? 64 : (chunks <= 2048 ? 128 : 256)));
    if (p->requested_group_threads == 0 && p->obs_i8) {
        // int8 observations: a quarter of the store trips for the same per-env set-up, so smaller groups win
        // (uf100-430 x 65,536: 0.266 / 0.271 / 0.299 / 0.365 ms with 32 / 64 / 128 / 256 threads per env)
        // rule from the sweep in profiles/r2_group_size_sweep.md: store chunks plus a quarter of the literal count
        const int w8 = (d.AD + 15) / 16 + (m * k) / 4;
        gs = w8 <= 300 ? 16 : (w8 <= 1320 ? 32 : (w8 <= 1800 ? 64 : (w8 <= 4096 ? 128 : 256)));
    }
    if (gs != 16 && gs != 32 && gs != 64 && gs != 128 && gs != 256) return MSAT_EINVAL;
    const GroupLayout L = group_layout(d, true);
    gs = fit_group_threads(gs, L);
    if (gs == 0) return MSAT_EUNSUPPORTED;
    p->group_threads = gs;
    p->layout_obs = L;
    p->layout_noobs = group_layout(d, false);
    p->group_smem_bytes = L.total;
    p->smem_bytes = L.total * (kCtaThreads / gs);
    // launches that write no observations (emit_obs off, GNN-input mode) have ~m clause evaluations of work per
    // env and stage only the literal block: one warp per env unless the caller pinned the group size or eight
    // groups do not fit in shared memory (half-warp groups only with observations)
    const GroupLayout Ln = p->layout_noobs;
    const int gn = fit_group_threads(p->requested_group_threads ? (gs < 32 ? 32 : gs) : 32, Ln);
    if (gn == 0) return MSAT_EUNSUPPORTED;
    p->group_threads_noobs = gn;
    p->smem_bytes_noobs = Ln.total * (kCtaThreads / gn);
    p->compile_smem_bytes = 4 * (m + n) * d.agw + (d.cnt_words ? 4 * (n + 1) : 0);
    if (p->compile_smem_bytes > kMaxSmem) return MSAT_EUNSUPPORTED;
    return MSAT_OK;
}

// Sets an option finish_plan sizes the plan from; when the plan cannot take the value, nothing changes.
int set_and_finish(msat_plan* p, int& option, int value) {
    const int old = option;
    option = value;
    const int rc = finish_plan(p);
    if (rc != MSAT_OK) { option = old; finish_plan(p); }
    return rc;
}

}  // namespace

extern "C" {

const char* msat_version(void) { return "marl_sat_b200 0.1 (sm_100a)"; }

int32_t msat_num_agents_for(int32_t n, int32_t vars_per_agent) {
    if (n <= 0) return MSAT_EINVAL;
    if (vars_per_agent > 0) return (n + vars_per_agent - 1) / vars_per_agent;   // env:299
    if (n % 4 == 0) return n / 4;                                               // env:315-323
    int r = (int)floor(sqrt((double)n));
    while ((long long)r * r > n) --r;
    while ((long long)(r + 1) * (r + 1) <= n) ++r;
    return r > 2 ? r : 2;                                                       // env:326
}

int msat_plan_create(msat_plan** out, int32_t n, int32_t m, int32_t k, int32_t A, int32_t action_mode,
                     int32_t max_steps, int32_t group_threads) {
    if (!out) return MSAT_EINVAL;
    *out = nullptr;
    if (n <= 0 || m <= 0 || k <= 0 || A <= 0 || A > n || n > 32767 || m > 32767) return MSAT_EINVAL;
    if (action_mode != 0 && action_mode != 1) return MSAT_EINVAL;
    if ((long long)A * (2LL * n + m) > (1LL << 26)) return MSAT_EUNSUPPORTED;
    msat_plan* p = new (std::nothrow) msat_plan();
    if (!p) return MSAT_EINVAL;
    Dims& d = p->d;
    d.n = n; d.m = m; d.k = k; d.A = A;
    d.base = n / A; d.rem = n % A;
    d.V = d.base + (d.rem > 0 ? 1 : 0);
    d.D = 2 * n + m;
    d.AD = A * d.D;
    d.action_mode = action_mode;
    d.max_steps = max_steps;
    d.aw = (n + 31) / 32;
    d.sw = (m + 31) / 32;
    d.xw = (d.D + 31) / 32 + 1;
    d.fw = (d.AD + 31) / 32;
    d.agw = (A + 31) / 32;
    d.inv_D = (uint32_t)(((1ULL << 32) + (uint64_t)d.D - 1) / (uint64_t)d.D);
    d.ms = (m + 1) & ~1;
    d.lits_bytes = (d.ms * k * 2 + 15) & ~15;
    p->requested_group_threads = group_threads;
    const int rc = finish_plan(p);
    if (rc != MSAT_OK) { delete p; return rc; }
    *out = p;
    return MSAT_OK;
}

void msat_plan_destroy(msat_plan* plan) { delete plan; }

int msat_plan_set_reward(msat_plan* plan, int32_t mode, double gamma, double r_clause, double r_sat) {
    if (!plan || (mode != MSAT_REWARD_SPARSE && mode != MSAT_REWARD_SHAPED)) return MSAT_EINVAL;
    plan->reward_mode = mode;
    plan->r_gamma = (float)gamma;
    plan->r_clause = (float)r_clause;
    plan->r_sat = (float)r_sat;
    return MSAT_OK;
}

int msat_plan_set_obs_dtype(msat_plan* plan, int32_t dtype) {
    if (!plan || (dtype != MSAT_OBS_INT32 && dtype != MSAT_OBS_INT8)) return MSAT_EINVAL;
    return set_and_finish(plan, plan->obs_i8, dtype == MSAT_OBS_INT8);   // the group size follows the store width
}

int msat_plan_set_clause_update(msat_plan* plan, int32_t mode) {
    if (!plan || (mode != MSAT_CLAUSES_FULL && mode != MSAT_CLAUSES_INCREMENTAL)) return MSAT_EINVAL;
    if (mode == MSAT_CLAUSES_INCREMENTAL && plan->d.k > 15) return MSAT_EUNSUPPORTED;     // 4-bit counts
    return set_and_finish(plan, plan->d.cnt_words, mode == MSAT_CLAUSES_INCREMENTAL ? (plan->d.m + 7) / 8 : 0);
}

int msat_plan_set_reset_counter(msat_plan* plan, uint64_t* counter_dev) {
    if (!plan || (reinterpret_cast<uintptr_t>(counter_dev) & 7)) return MSAT_EINVAL;
    plan->reset_counter = reinterpret_cast<unsigned long long*>(counter_dev);
    return MSAT_OK;
}

int msat_tune(const char* key, int32_t value) {
    if (!key) return MSAT_EINVAL;
    if (!strcmp(key, "gae_plain")) { g_gae_force_plain = value; return MSAT_OK; }
    if (!strcmp(key, "gae_variant")) { g_gae_variant = value; return MSAT_OK; }
    if (!strcmp(key, "gae_pipe_min_cols")) { g_gae_pipe_min_cols = value; return MSAT_OK; }
    if (!strcmp(key, "gae_warps_per_sm")) { g_gae_warps_per_sm = value > 0 ? value : 0; return MSAT_OK; }
    return MSAT_EINVAL;
}

int msat_plan_dims(const msat_plan* plan, msat_dims* o) {
    if (!plan || !o) return MSAT_EINVAL;
    const Dims& d = plan->d;
    o->n = d.n; o->m = d.m; o->k = d.k; o->A = d.A; o->V = d.V; o->D = d.D;
    o->action_mode = d.action_mode; o->max_steps = d.max_steps;
    o->rec_bytes = d.rec_bytes; o->state_words = d.state_words;
    o->group_threads = plan->group_threads; o->smem_bytes = plan->smem_bytes;
    return MSAT_OK;
}

int msat_compile_bank(const msat_plan* plan, const int32_t* clauses, int32_t P, void* bank, void* stream) {
    if (!plan || P < 0 || (P > 0 && (!clauses || !bank))) return MSAT_EINVAL;
    if (!aligned(bank, 128) || !aligned(clauses, 4)) return MSAT_EALIGN;
    return cuda_rc(launch_compile_bank(plan, clauses, P, static_cast<uint8_t*>(bank), (cudaStream_t)stream));
}

int msat_reset(const msat_plan* plan, const void* bank, int32_t P, const int32_t* problem_idx, const uint32_t* keys,
               uint32_t* state, int32_t* obs, int32_t B, void* stream) {
    EnvArgs a;
    if (const int rc = env_args(a, plan, bank, P, nullptr, state, obs, B, !problem_idx || !keys || !state)) return rc;
    a.prob_idx = problem_idx; a.keys = keys;
    return cuda_rc(launch_env(plan, MODE_RESET, a, (cudaStream_t)stream));
}

int msat_import_state(const msat_plan* plan, const void* bank, int32_t P, const int32_t* problem_idx,
                      const int32_t* variable_assignments, const int32_t* step, const uint8_t* done, uint32_t* state_out,
                      int32_t* obs, int32_t B, void* stream) {
    EnvArgs a;
    if (const int rc = env_args(a, plan, bank, P, nullptr, state_out, obs, B,
                                !problem_idx || !variable_assignments || !state_out))
        return rc;
    a.prob_idx = problem_idx; a.assign_in = variable_assignments; a.step_in = step; a.done_in = done;
    return cuda_rc(launch_env(plan, MODE_IMPORT, a, (cudaStream_t)stream));
}

int msat_apply_start_states(const msat_plan* plan, const void* bank, int32_t P, uint32_t* state,
                            const uint32_t* reset_key, int32_t Bg, int32_t env_offset, const uint32_t* start_words,
                            const uint32_t* flip_thr, const uint8_t* has_start, int32_t* obs, int32_t* gnn_assignment,
                            float* gnn_clause_features, int32_t B, void* stream) {
    EnvArgs a;
    int rc = env_args(a, plan, bank, P, state, state, obs, B, !state || !reset_key || !start_words || !flip_thr);
    if (rc == MSAT_OK) rc = shard_rule(Bg, env_offset, B);
    if (rc != MSAT_OK) return rc;
    if (!aligned(start_words, 4) || !aligned(flip_thr, 4) || !aligned(gnn_assignment, 4) ||
        !aligned(gnn_clause_features, 4))
        return MSAT_EALIGN;
    if (clause_features_unsupported(plan, gnn_clause_features)) return MSAT_EUNSUPPORTED;
    if (B == 0) return MSAT_OK;
    a.Bg = (uint32_t)Bg; a.env_off = (uint32_t)env_offset; a.reset_key = reset_key;
    a.start_words = start_words; a.flip_thr = flip_thr; a.has_start = has_start;
    // observations and GNN inputs come from differently shaped launches; the rewrite depends only on the key and
    // the tables, so the second launch selects the same envs and writes the same states again
    cudaError_t e = cudaSuccess;
    if (obs || !(gnn_assignment || gnn_clause_features)) e = launch_env(plan, MODE_START, a, (cudaStream_t)stream);
    if (e == cudaSuccess && (gnn_assignment || gnn_clause_features)) {
        a.obs = nullptr; a.gnn_assign = gnn_assignment; a.gnn_cf = gnn_clause_features;
        e = launch_env(plan, MODE_START, a, (cudaStream_t)stream);
    }
    return cuda_rc(e);
}

int msat_walksat(const msat_plan* plan, const void* bank, int32_t P, uint32_t* state, const uint32_t* keys,
                 int32_t max_flips, int32_t flip_offset, double noise, uint8_t* solved, int32_t* flips, int32_t B,
                 void* stream) {
    if (bad_env_call(plan, bank, P, B, !state || !keys)) return MSAT_EINVAL;
    if (!(noise >= 0.0 && noise <= 1.0)) return MSAT_EINVAL;          // also NaN
    if (max_flips < 0 || flip_offset < 0 || (long long)flip_offset + max_flips > 2147483647LL) return MSAT_EINVAL;
    if (!aligned(bank, 128) || !aligned(state, 16)) return MSAT_EALIGN;
    if (walksat_warps(plan->d) == 0) return MSAT_EUNSUPPORTED;
    WalksatArgs a{};
    a.bank = static_cast<const uint8_t*>(bank); a.P = P; a.state = state; a.keys = keys;
    a.max_flips = max_flips; a.flip_offset = flip_offset;
    a.thr = (uint32_t)llrint(noise * 16777216.0);
    a.solved = solved; a.flips = flips; a.B = B;
    return cuda_rc(launch_walksat(plan, a, (cudaStream_t)stream));
}

int msat_step(const msat_plan* plan, const void* bank, int32_t P, const uint32_t* state_in, uint32_t* state_out,
              const int32_t* actions, int32_t auto_reset, const int32_t* new_problem_idx, const uint32_t* reset_keys,
              int32_t* obs, float* reward, int32_t reward_cols, uint8_t* done, int32_t done_cols, uint8_t* solved,
              int32_t* num_unsatisfied, int32_t* episode_step, int32_t* newly_satisfied, int32_t B, void* stream) {
    EnvArgs a;
    int rc = env_args(a, plan, bank, P, state_in, state_out, obs, B,
                      !state_in || !state_out || !actions || (auto_reset && (!new_problem_idx || !reset_keys)));
    if (rc == MSAT_OK) rc = step_outputs(a, plan, reward, reward_cols, done, done_cols, solved, num_unsatisfied,
                                         episode_step, newly_satisfied);
    if (rc != MSAT_OK) return rc;
    a.actions = actions; a.auto_reset = auto_reset ? 1 : 0; a.prob_idx = new_problem_idx; a.keys = reset_keys;
    return cuda_rc(launch_env(plan, MODE_STEP, a, (cudaStream_t)stream));
}

int msat_rollout_step(const msat_plan* plan, const void* bank, int32_t P, const uint32_t* state_in,
                      uint32_t* state_out, const int32_t* actions, const uint32_t* rng_in, uint32_t* chain_out,
                      int32_t Bg, int32_t env_offset, int32_t* obs, float* reward, int32_t reward_cols, uint8_t* done,
                      int32_t done_cols, uint8_t* solved, int32_t* num_unsatisfied, int32_t* episode_step, int32_t B,
                      void* stream) {
    return msat_rollout_steps(plan, bank, P, state_in, state_out, actions, 1, rng_in, chain_out, Bg, env_offset, obs,
                              nullptr, nullptr, 0, reward, reward_cols, done, done_cols, solved, num_unsatisfied,
                              episode_step, nullptr, B, stream);
}

int msat_rollout_step_gnn(const msat_plan* plan, const void* bank, int32_t P, const uint32_t* state_in,
                          uint32_t* state_out, const int32_t* actions, const uint32_t* rng_in, uint32_t* chain_out,
                          int32_t Bg, int32_t env_offset, int32_t* assignment, float* clause_features, float* reward,
                          int32_t reward_cols, uint8_t* done, int32_t done_cols, uint8_t* solved,
                          int32_t* num_unsatisfied, int32_t* episode_step, int32_t B, void* stream) {
    return msat_rollout_steps(plan, bank, P, state_in, state_out, actions, 1, rng_in, chain_out, Bg, env_offset,
                              nullptr, assignment, clause_features, 0, reward, reward_cols, done, done_cols, solved,
                              num_unsatisfied, episode_step, nullptr, B, stream);
}

int msat_rollout_steps(const msat_plan* plan, const void* bank, int32_t P, const uint32_t* state_in,
                       uint32_t* state_out, const int32_t* actions, int32_t num_steps, const uint32_t* rng_in,
                       uint32_t* chain_out, int32_t Bg, int32_t env_offset, int32_t* obs, int32_t* gnn_assignment,
                       float* gnn_clause_features, int32_t emit_every_step, float* reward, int32_t reward_cols,
                       uint8_t* done, int32_t done_cols, uint8_t* solved, int32_t* num_unsatisfied,
                       int32_t* episode_step, int32_t* newly_satisfied, int32_t B, void* stream) {
    if (obs && (gnn_assignment || gnn_clause_features)) return MSAT_EINVAL;   // one kind of policy input per launch
    EnvArgs a;
    const int rc = rollout_args(a, plan, bank, P, state_in, state_out, actions, num_steps, rng_in, chain_out, Bg,
                                env_offset, obs, gnn_assignment, gnn_clause_features, emit_every_step, reward,
                                reward_cols, done, done_cols, solved, num_unsatisfied, episode_step, newly_satisfied, B);
    return rc != MSAT_OK ? rc : cuda_rc(rollout_enqueue(plan, a, (cudaStream_t)stream));
}

int msat_get_obs(const msat_plan* plan, const void* bank, int32_t P, const uint32_t* state, int32_t* obs, int32_t B,
                 void* stream) {
    EnvArgs a;
    const int rc = env_args(a, plan, bank, P, state, nullptr, obs, B, !state || !obs);
    return rc != MSAT_OK ? rc : cuda_rc(launch_env(plan, MODE_OBS, a, (cudaStream_t)stream));
}

int msat_export_state(const msat_plan* plan, const void* bank, int32_t P, const uint32_t* state, int32_t B,
                      int32_t* variable_assignments, uint8_t* clauses_satisfied_status, int32_t* num_unsatisfied,
                      int32_t* step, uint8_t* done, int32_t* clauses, int32_t* agent_clause_masks,
                      int32_t* agent_neighbor_masks, int32_t* literal_to_agent_idx, int32_t* problem_idx,
                      void* stream) {
    if (bad_env_call(plan, bank, P, B, !state)) return MSAT_EINVAL;
    ExportArgs a{};
    a.bank = static_cast<const uint8_t*>(bank); a.P = P; a.state = state; a.B = B;
    a.assign = variable_assignments; a.sat = clauses_satisfied_status; a.num_unsat = num_unsatisfied;
    a.step = step; a.done = done; a.clauses = clauses; a.acm = agent_clause_masks; a.anm = agent_neighbor_masks;
    a.l2a = literal_to_agent_idx; a.pidx = problem_idx;
    return cuda_rc(launch_export(plan, a, (cudaStream_t)stream));
}

int msat_rollout_step_host(const msat_plan* plan, const void* bank, int32_t P, uint32_t* state,
                           const int32_t* actions_host, int32_t* actions_dev, const uint32_t* rng_in,
                           uint32_t* chain_out, int32_t Bg, int32_t env_offset, int32_t* obs_dev, float* reward_dev,
                           int32_t reward_cols, uint8_t* done_dev, int32_t done_cols, uint8_t* solved_dev,
                           int32_t* num_unsatisfied_dev, int32_t* episode_step_dev, float* reward_host,
                           uint8_t* done_host, uint8_t* solved_host, int32_t* num_unsatisfied_host,
                           int32_t* episode_step_host, int32_t B, void* stream) {
    HostStep h{plan, actions_host, actions_dev, reward_host, done_host, solved_host, num_unsatisfied_host,
               episode_step_host};
    if (const int rc = h.check(bank, P, state, rng_in, chain_out, Bg, env_offset, obs_dev, reward_dev, reward_cols,
                               done_dev, done_cols, solved_dev, num_unsatisfied_dev, episode_step_dev, B))
        return rc;
    cudaStream_t s = (cudaStream_t)stream;
    auto run_slice = [&](int b0, int bc, cudaStream_t w) {
        cudaError_t e = h.upload(b0, bc, w);
        if (e == cudaSuccess) e = h.step(b0, bc, w);
        if (e == cudaSuccess) e = h.download(b0, bc, w);
        return e;
    };
    constexpr int kSlices = 4;
    if (B < 32768) {   // one slice on the caller's stream (slicing only pays when the kernel is long)
        const cudaError_t e = run_slice(0, B, s);
        return cuda_rc(e != cudaSuccess ? e : cudaStreamSynchronize(s));
    }
    // Large batch: slices alternate between two internal streams so that the action upload of slice
    // i+1 and the result download of slice i-1 overlap the kernel of slice i (separate copy engines).
    cudaError_t e = cudaSuccess;
    {
        std::lock_guard<std::mutex> lock(g_pipe_mu);
        SyncPipe* pipe = nullptr;
        e = sync_pipe_for_current_device(&pipe);
        if (e == cudaSuccess) e = cudaEventRecord(pipe->fork, s);
        for (int w = 0; w < 2 && e == cudaSuccess; ++w) e = cudaStreamWaitEvent(pipe->ws[w], pipe->fork, 0);
        if (e != cudaSuccess) return (int)e;
        const int per = (((B + kSlices - 1) / kSlices) + 63) & ~63;   // multiple of 64 envs keeps every slice aligned
        for (int c = 0, b0 = 0; b0 < B && e == cudaSuccess; ++c, b0 += per) {
            const int bc = B - b0 < per ? B - b0 : per;
            e = run_slice(b0, bc, pipe->ws[c & 1]);
        }
        // always join the internal streams back into the caller's stream -- also after a failed slice, so that
        // nothing enqueued so far is still running when the caller sees the error
        for (int w = 0; w < 2; ++w) {
            cudaError_t j = cudaEventRecord(pipe->join[w], pipe->ws[w]);
            if (j == cudaSuccess) j = cudaStreamWaitEvent(s, pipe->join[w], 0);
            if (j != cudaSuccess && e == cudaSuccess) e = j;
        }
    }
    const cudaError_t se = cudaStreamSynchronize(s);
    return cuda_rc(e != cudaSuccess ? e : se);
}

// ---- asynchronous host pipeline (double-buffered host I/O) -------------------------------------------------
struct msat_host_pipe {
    int dev = 0, depth = 0;
    cudaStream_t s_in = nullptr, s_out = nullptr;
    cudaEvent_t ev_h2d[kMaxPipeDepth] = {}, ev_kernel[kMaxPipeDepth] = {}, ev_d2h[kMaxPipeDepth] = {};
    bool kernel_valid[kMaxPipeDepth] = {}, d2h_valid[kMaxPipeDepth] = {};
};

int msat_host_pipe_create(msat_host_pipe** out, int32_t depth) {
    if (!out || depth < 1 || depth > kMaxPipeDepth) return MSAT_EINVAL;
    *out = nullptr;
    msat_host_pipe* p = new (std::nothrow) msat_host_pipe();
    if (!p) return MSAT_EINVAL;
    p->depth = depth;
    cudaError_t e = cudaGetDevice(&p->dev);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&p->s_in, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&p->s_out, cudaStreamNonBlocking);
    for (int i = 0; i < depth && e == cudaSuccess; ++i) {
        e = cudaEventCreateWithFlags(&p->ev_h2d[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_kernel[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_d2h[i], cudaEventDisableTiming);
    }
    if (e != cudaSuccess) { msat_host_pipe_destroy(p); return (int)e; }
    *out = p;
    return MSAT_OK;
}

void msat_host_pipe_destroy(msat_host_pipe* p) {
    if (!p) return;
    if (p->s_in) cudaStreamSynchronize(p->s_in);
    if (p->s_out) cudaStreamSynchronize(p->s_out);
    for (int i = 0; i < kMaxPipeDepth; ++i) {
        if (p->ev_h2d[i]) cudaEventDestroy(p->ev_h2d[i]);
        if (p->ev_kernel[i]) cudaEventDestroy(p->ev_kernel[i]);
        if (p->ev_d2h[i]) cudaEventDestroy(p->ev_d2h[i]);
    }
    if (p->s_in) cudaStreamDestroy(p->s_in);
    if (p->s_out) cudaStreamDestroy(p->s_out);
    delete p;
}

int msat_rollout_step_host_async(msat_host_pipe* pipe, int32_t slot, const msat_plan* plan, const void* bank,
                                 int32_t P, uint32_t* state, const int32_t* actions_host, int32_t* actions_dev,
                                 const uint32_t* rng_in, uint32_t* chain_out, int32_t Bg, int32_t env_offset,
                                 int32_t* obs_dev, float* reward_dev, int32_t reward_cols, uint8_t* done_dev,
                                 int32_t done_cols, uint8_t* solved_dev, int32_t* num_unsatisfied_dev,
                                 int32_t* episode_step_dev, float* reward_host, uint8_t* done_host,
                                 uint8_t* solved_host, int32_t* num_unsatisfied_host, int32_t* episode_step_host,
                                 int32_t B, void* stream) {
    if (!pipe || slot < 0 || slot >= pipe->depth) return MSAT_EINVAL;
    HostStep h{plan, actions_host, actions_dev, reward_host, done_host, solved_host, num_unsatisfied_host,
               episode_step_host};
    if (const int rc = h.check(bank, P, state, rng_in, chain_out, Bg, env_offset, obs_dev, reward_dev, reward_cols,
                               done_dev, done_cols, solved_dev, num_unsatisfied_dev, episode_step_dev, B))
        return rc;
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaSuccess;
    // 1. upload this step's actions on the copy-in stream as soon as the kernel that last read this slot's
    //    device staging buffer has finished (it overlaps the kernels of the steps in between)
    if (pipe->kernel_valid[slot]) e = cudaStreamWaitEvent(pipe->s_in, pipe->ev_kernel[slot], 0);
    if (e == cudaSuccess) e = h.upload(0, B, pipe->s_in);
    if (e == cudaSuccess) e = cudaEventRecord(pipe->ev_h2d[slot], pipe->s_in);
    // 2. the fused step on the caller's stream: after the upload, and after the previous download out of
    //    this slot's device result buffers
    if (e == cudaSuccess) e = cudaStreamWaitEvent(s, pipe->ev_h2d[slot], 0);
    if (e == cudaSuccess && pipe->d2h_valid[slot]) e = cudaStreamWaitEvent(s, pipe->ev_d2h[slot], 0);
    if (e == cudaSuccess) e = h.step(0, B, s);
    if (e != cudaSuccess) return (int)e;
    e = cudaEventRecord(pipe->ev_kernel[slot], s);
    pipe->kernel_valid[slot] = e == cudaSuccess;
    // 3. results to the host on the copy-out stream; msat_host_wait(slot) blocks on ev_d2h
    if (e == cudaSuccess) e = cudaStreamWaitEvent(pipe->s_out, pipe->ev_kernel[slot], 0);
    if (e == cudaSuccess) e = h.download(0, B, pipe->s_out);
    if (e == cudaSuccess) e = cudaEventRecord(pipe->ev_d2h[slot], pipe->s_out);
    pipe->d2h_valid[slot] = e == cudaSuccess;
    return cuda_rc(e);
}

int msat_host_wait(msat_host_pipe* pipe, int32_t slot) {
    if (!pipe || slot < 0 || slot >= pipe->depth) return MSAT_EINVAL;
    if (!pipe->d2h_valid[slot]) return MSAT_OK;
    return cuda_rc(cudaEventSynchronize(pipe->ev_d2h[slot]));
}

int msat_shutdown(void) {
    std::lock_guard<std::mutex> lock(g_pipe_mu);
    for (auto& kv : g_pipes) {
        int cur = 0;
        if (cudaGetDevice(&cur) == cudaSuccess && cudaSetDevice(kv.first) == cudaSuccess) {
            kv.second.destroy();
            cudaSetDevice(cur);
        }
    }
    g_pipes.clear();
    return MSAT_OK;
}

int msat_rng_chain(const uint32_t* rng_in, uint32_t* chain_out, void* stream) {
    if (!rng_in || !chain_out) return MSAT_EINVAL;
    return cuda_rc(launch_rng_chain(rng_in, chain_out, (cudaStream_t)stream));
}

int msat_rng_split2(const uint32_t* key_in, uint32_t* out, void* stream) {
    if (!key_in || !out) return MSAT_EINVAL;
    return cuda_rc(launch_rng_split2(key_in, out, (cudaStream_t)stream));
}

int msat_env_keys(const uint32_t* prob_key, const uint32_t* reset_key, int32_t Bg, int32_t off, int32_t Bl, int32_t P,
                  int32_t* problem_idx, uint32_t* reset_keys, void* stream) {
    if (const int rc = shard_rule(Bg, off, Bl)) return rc;
    if (problem_idx && (!prob_key || P <= 0)) return MSAT_EINVAL;
    if (reset_keys && !reset_key) return MSAT_EINVAL;
    return cuda_rc(launch_env_keys(prob_key, reset_key, Bg, off, Bl, P, problem_idx, reset_keys, nullptr,
                                   (cudaStream_t)stream));
}

int msat_env_keys_weighted(const uint32_t* prob_key, const uint32_t* reset_key, int32_t Bg, int32_t off, int32_t Bl,
                           const int64_t* cum_weights, int32_t P, int32_t* problem_idx, uint32_t* reset_keys,
                           void* stream) {
    if (const int rc = shard_rule(Bg, off, Bl)) return rc;
    if (problem_idx && (!prob_key || !cum_weights || P <= 0)) return MSAT_EINVAL;
    if (reset_keys && !reset_key) return MSAT_EINVAL;
    if (!aligned(cum_weights, 8)) return MSAT_EALIGN;
    // without problem indices to draw, the call is msat_env_keys' reset-key half
    const long long* cum = problem_idx ? reinterpret_cast<const long long*>(cum_weights) : nullptr;
    return cuda_rc(launch_env_keys(prob_key, reset_key, Bg, off, Bl, P, problem_idx, reset_keys, cum,
                                   (cudaStream_t)stream));
}

int msat_sample_actions(const float* logits, int64_t num_rows_global, int64_t row_offset, int32_t num_rows,
                        int32_t num_classes, const uint32_t* rng_in, int32_t* actions, float* log_prob, void* stream) {
    if (num_classes < 1 || num_rows < 0 || num_rows_global < 0 || row_offset < 0) return MSAT_EINVAL;
    if (row_offset > num_rows_global - num_rows) return MSAT_EINVAL;
    if (num_rows > 0 && (!logits || !rng_in || !actions)) return MSAT_EINVAL;
    if (!aligned(logits, 4) || !aligned(log_prob, 4)) return MSAT_EALIGN;
    // one Threefry call over the whole table (JAX's single-block counter path): N + 1 must fit in 32 bits
    if (num_rows_global >= 0xFFFFFFFFll || (unsigned long long)num_rows_global * (unsigned)num_classes >= 0xFFFFFFFFull)
        return MSAT_EUNSUPPORTED;
    if (num_rows == 0) return MSAT_OK;
    const uint32_t N = (uint32_t)(num_rows_global * num_classes);
    return cuda_rc(launch_sample_actions(logits, N, (uint32_t)row_offset, num_rows, num_classes, rng_in, actions,
                                         log_prob, (cudaStream_t)stream));
}

int msat_problem_stats(const int32_t* problem_idx, int64_t pidx_stride_t, int64_t pidx_stride_b, const uint8_t* done,
                       const uint8_t* solved, const int32_t* num_unsatisfied, const int32_t* episode_step, int32_t T,
                       int32_t B, int32_t P, int64_t* stats, void* stream) {
    if (T < 0 || B < 0 || P <= 0 || !stats) return MSAT_EINVAL;
    if (T > 0 && B > 0 && (!problem_idx || !done || !solved || !num_unsatisfied || !episode_step)) return MSAT_EINVAL;
    if (!aligned(stats, 8)) return MSAT_EALIGN;
    return cuda_rc(launch_problem_stats(problem_idx, pidx_stride_t, pidx_stride_b, done, solved, num_unsatisfied,
                                        episode_step, T, B, P, reinterpret_cast<long long*>(stats),
                                        (cudaStream_t)stream));
}

int msat_gae(const float* reward, int64_t rs_t, int64_t rs_b, const uint8_t* done, const float* value,
             const float* last_val, double gamma, double gae_lambda, float* advantages, float* targets, double* stats,
             int32_t T, int32_t B, void* stream) {
    if (T < 0 || B < 0) return MSAT_EINVAL;
    if (T > 0 && B > 0 && (!reward || !done || !value || !last_val || !advantages || !targets)) return MSAT_EINVAL;
    return cuda_rc(launch_gae(reward, rs_t, rs_b, done, value, last_val, (float)gamma, (float)(gamma * gae_lambda),
                              advantages, targets, T, B, stats, (cudaStream_t)stream));
}

int msat_adv_stats(const float* adv, int64_t count, double* stats, void* stream) {
    if (count < 0 || !stats || (count > 0 && !adv)) return MSAT_EINVAL;
    return cuda_rc(launch_adv_stats(adv, count, stats, (cudaStream_t)stream));
}

int msat_adv_normalize(float* adv, int64_t count, const double* stats, void* stream) {
    if (count < 0 || !stats || (count > 0 && !adv)) return MSAT_EINVAL;
    return cuda_rc(launch_adv_normalize(adv, count, stats, (cudaStream_t)stream));
}

int msat_gnn_static(const msat_plan* plan, const void* bank, int32_t P, float* static_var_features, float* a_pos,
                    float* a_neg, void* stream) {
    if (!plan || P < 0 || (P > 0 && !bank)) return MSAT_EINVAL;
    if (2 * plan->d.n * (int)sizeof(int) > 48 * 1024) return MSAT_EUNSUPPORTED;
    return cuda_rc(launch_gnn_static(plan, static_cast<const uint8_t*>(bank), P, static_var_features, a_pos, a_neg,
                                     (cudaStream_t)stream));
}

int msat_gnn_dynamic(const msat_plan* plan, const void* bank, int32_t P, const uint32_t* state, int32_t B,
                     int32_t* assignment, float* clause_features, void* stream) {
    if (bad_env_call(plan, bank, P, B, !state)) return MSAT_EINVAL;
    return cuda_rc(launch_gnn_dynamic(plan, static_cast<const uint8_t*>(bank), P, state, B, assignment,
                                      clause_features, (cudaStream_t)stream));
}

int msat_rollout_metrics(const float* reward, int64_t rs_t, int64_t rs_b, const uint8_t* done, const uint8_t* solved,
                         const int32_t* num_unsatisfied, const int32_t* episode_step, int32_t T, int32_t B,
                         double* sums, void* stream) {
    if (T < 0 || B < 0 || !sums) return MSAT_EINVAL;
    if (T > 0 && B > 0 && (!reward || !done || !solved || !num_unsatisfied || !episode_step)) return MSAT_EINVAL;
    return cuda_rc(launch_rollout_metrics(reward, rs_t, rs_b, done, solved, num_unsatisfied, episode_step, T, B, sums,
                                          (cudaStream_t)stream));
}

int msat_flip_gains(const msat_plan* plan, const void* bank, int32_t P, const uint32_t* state, int32_t B, double tau,
                    int32_t* delta_unsat, int32_t* greedy_labels, void* stream) {
    if (bad_env_call(plan, bank, P, B, !state)) return MSAT_EINVAL;
    if (plan->d.n * (int)sizeof(int) > 48 * 1024) return MSAT_EUNSUPPORTED;
    return cuda_rc(launch_flip_gains(plan, static_cast<const uint8_t*>(bank), P, state, B, (float)tau, delta_unsat,
                                     greedy_labels, (cudaStream_t)stream));
}

int msat_eval_track(const msat_plan* plan, const uint32_t* state, const uint8_t* solved, int32_t t, int32_t B,
                    uint8_t* ever_solved, int32_t* steps_to_solve, int32_t* solution, void* stream) {
    if (!plan || B < 0 || t < 0) return MSAT_EINVAL;
    if (B > 0 && (!state || !solved || !ever_solved || !steps_to_solve || !solution)) return MSAT_EINVAL;
    return cuda_rc(launch_eval_track(plan, state, solved, t, B, ever_solved, steps_to_solve, solution,
                                     (cudaStream_t)stream));
}

}  // extern "C"
