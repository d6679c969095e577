/*
 * marl_sat_b200.h -- C ABI of the B200-native batched SATEnv hot path.
 *
 * This is the drop-in boundary for ONE path of kongqg/marl-sat: the batched
 * multi-agent SATEnv (reset / flip / clause satisfaction / reward / observation
 * / auto-reset) and the MAPPO GAE scan that consumes the rollout.  Reference
 * files (relative to the reference repo root):
 *     env     = src/envs/multi_agent_sat_env.py
 *     learner = src/learners/mappo_gnn_sat_learner.py
 *     runner  = src/runners/mappo_runner.py
 *
 * The reference has no FFI of its own (it is pure JAX); the entry points below
 * are what a `jax.ffi` custom-call layer for this path binds (one handler per
 * function, see INTEGRATION.md).  Conventions for every `msat_*` enqueue call:
 *   - plain pointers and sizes only; every buffer is owned by the caller;
 *   - all `*_dev` / unqualified data pointers are DEVICE pointers on the current
 *     device; `stream` is a `cudaStream_t` passed as `void*` (NULL = legacy
 *     default stream);
 *   - enqueue-only: no allocation, no synchronisation, no host callbacks; safe to
 *     capture in a CUDA graph; thread-safe and re-entrant (a plan is immutable);
 *   - return 0 on success, a negative MSAT_E* code on an argument error (nothing
 *     is enqueued), a positive value = the `cudaError_t` of a failed launch.
 *   - there is NO CPU fallback: without a CUDA device every enqueue call fails.
 *
 * Data layouts (DESIGN.md section 3):
 *   formula bank   P records of `rec_bytes` each: packed u16 literal codes
 *                  followed by the flat agent-mask bit stream (A*D bits);
 *   env state      B records of `state_words` u32 each: packed assignment bits,
 *                  step, problem index, #unsatisfied, done flag;
 *   observations   int32 [B, A, D], D = 2n+m, values in {-1,0,1}  (env:345-398).
 */
#ifndef MARL_SAT_B200_H
#define MARL_SAT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSAT_OK            0
#define MSAT_EINVAL       -1   /* bad shape / null pointer / out-of-range scalar      */
#define MSAT_EALIGN       -2   /* a buffer is not aligned as documented               */
#define MSAT_EUNSUPPORTED -3   /* shape exceeds what one CTA's shared memory can hold */

/* Static description of one SATEnv configuration.  Replaces the constructor
 * state of `SATEnv.__init__` (env:29-88): agent groups are the reference's
 * contiguous balanced split (env:294-338), so (n, A) determine agent_vars,
 * action_mask and variable_to_agent_idx. */
typedef struct msat_plan msat_plan;

typedef struct msat_dims {
    int32_t n, m, k;          /* variables, clauses, literals per clause (0-padded)    */
    int32_t A, V, D;          /* agents, max vars per agent, obs_dim = 2n+m            */
    int32_t action_mode;      /* 0 single-flip (Discrete(V+1)), 1 multi-flip           */
    int32_t max_steps;
    int32_t rec_bytes;        /* bytes per formula-bank record (multiple of 128)       */
    int32_t state_words;      /* u32 words per env-state record (multiple of 4)        */
    int32_t group_threads;    /* threads cooperating on one env in the step kernel     */
    int32_t smem_bytes;       /* dynamic shared memory per CTA of the step kernel      */
} msat_dims;

/* --- plan (host only, no GPU needed) ------------------------------------- */

/* Replaces SATEnv.__init__/_create_agent_groups (env:29-88, 294-338).
 * `num_agents` is the value produced by the reference's grouping rule; the
 * contiguous split base=n/A, rem=n%A is implied.  group_threads = 0 lets the
 * library choose (16/32/64/128/256 by observation size; 16 = two envs share a warp). */
int msat_plan_create(msat_plan** out, int32_t num_vars, int32_t num_clauses, int32_t lits_per_clause,
                     int32_t num_agents, int32_t action_mode, int32_t max_steps, int32_t group_threads);
void msat_plan_destroy(msat_plan* plan);
int msat_plan_dims(const msat_plan* plan, msat_dims* out);

/* Reward variant of every step entry point that uses this plan (call before the first launch):
 *   MSAT_REWARD_SPARSE (default)  the active reward of the reference, 1.0 when solved else 0.0 (env:183-198);
 *   MSAT_REWARD_SHAPED            the reference's alternative team reward (commented out at env:201-223):
 *        gamma * (-unsat') - (-unsat) + r_clause * #newly satisfied clauses + [solved] * r_sat
 *     in float32 with the reference's operation order; gamma / r_clause / r_sat are the constructor
 *     arguments the reference stores for it (env:40-42). */
#define MSAT_REWARD_SPARSE 0
#define MSAT_REWARD_SHAPED 1
int msat_plan_set_reward(msat_plan* plan, int32_t mode, double gamma, double r_clause, double r_sat);
/* Reference grouping rule (env:294-338): number of agents for (n, vars_per_agent);
 * vars_per_agent <= 0 means "auto" (n/4 if 4 | n else max(2, floor(sqrt(n)))). */
int32_t msat_num_agents_for(int32_t num_vars, int32_t vars_per_agent);
const char* msat_version(void);

/* --- formula bank ---------------------------------------------------------- */

/* Compile P raw formulas (int32 [P, m, k], DIMACS literals, 0 = padding) into bank
 * records.  Replaces the per-reset work of `_compute_observation_maps` (env:99-128)
 * and `literal_to_agent_idx` (env:160): the agent/clause and agent/neighbour
 * relations (including the "-1 == -1" padding quirk) are evaluated once per
 * formula instead of once per env per step.  `bank` needs P*rec_bytes bytes,
 * 128-byte aligned. */
int msat_compile_bank(const msat_plan* plan, const int32_t* clauses, int32_t num_problems,
                      void* bank, void* stream);

/* --- environment ----------------------------------------------------------- */

/* Replaces `jax.vmap(SATEnv.reset)(clauses[problem_idx], keys)` (env:158-181;
 * runner:137,295).  problem_idx int32[B] (indices into the bank), keys uint32[B,2]
 * (legacy JAX PRNG keys).  Writes state[B*state_words] and, if obs != NULL,
 * obs int32[B,A,D] (16-byte aligned). */
int msat_reset(const msat_plan* plan, const void* bank, int32_t num_problems,
               const int32_t* problem_idx, const uint32_t* keys,
               uint32_t* state, int32_t* obs, int32_t num_envs, void* stream);

/* Inverse of msat_export_state: packed states from reference-shaped leaves (env:13-24).
 *   problem_idx int32[B] (clamped into [0, num_problems), as msat_reset does);
 *   variable_assignments int32[B,n] (0/1; nonzero reads as 1);
 *   step int32[B] (NULL = 0, stored verbatim); done uint8[B] (NULL = 0, nonzero = done)
 * clauses_satisfied_status, num_unsatisfied (and an incremental plan's true-literal counts)
 * are recomputed from the bank record; obs (NULL = skip) as msat_get_obs of the result.
 * For warm starts, fixed starting assignments and resuming from a checkpoint: the reset path of
 * the env kernel with the assignment read from memory instead of drawn from a key. */
int msat_import_state(const msat_plan* plan, const void* bank, int32_t num_problems,
                      const int32_t* problem_idx, const int32_t* variable_assignments,
                      const int32_t* step, const uint8_t* done,
                      uint32_t* state_out, int32_t* obs, int32_t num_envs, void* stream);

/* Replaces `jax.vmap(SATEnv.step_env)` (env:225-284) and, with auto_reset != 0,
 * the reset-and-select of the rollout loop (learner:422-464) in the same launch.
 *   actions        int32 [B, A] (mode 0) or [B, A, V] (mode 1)
 *   state_in/out   may alias (in-place) or differ (functional update)
 *   new_problem_idx int32[B], reset_keys uint32[B,2]: read only for envs that
 *                  finish this step and only when auto_reset != 0 (else may be NULL)
 *   obs            int32 [B, A, D] of the state the caller continues from (the
 *                  post-reset state for finished envs when auto_reset != 0); NULL = skip
 *   reward         float [B, reward_cols]: 1.0 when solved else 0.0 (env:183-198), the same scalar
 *                  repeated reward_cols times per env (A = one per agent, env:196; 1 = the shared
 *                  team reward only, which is all the GAE reads, learner:514)
 *   done           uint8 [B, done_cols]: the episode-end flag repeated done_cols times per env
 *                  (A+1 = one per agent plus "__all__", env:260-261; 1 = Transition.global_done
 *                  only, learner:468); pre-reset values
 *   solved uint8[B], num_unsatisfied int32[B], episode_step int32[B]  (infos, env:278-282)
 *   newly_satisfied int32[B]: clauses satisfied after the step that were not before it (env:211);
 *                  only with MSAT_REWARD_SHAPED (else must be NULL)
 * Any of reward/done/solved/num_unsatisfied/episode_step/newly_satisfied may be NULL. */
int msat_step(const msat_plan* plan, const void* bank, int32_t num_problems,
              const uint32_t* state_in, uint32_t* state_out, const int32_t* actions,
              int32_t auto_reset, const int32_t* new_problem_idx, const uint32_t* reset_keys,
              int32_t* obs, float* reward, int32_t reward_cols, uint8_t* done, int32_t done_cols,
              uint8_t* solved, int32_t* num_unsatisfied, int32_t* episode_step,
              int32_t* newly_satisfied, int32_t num_envs, void* stream);

/* One whole rollout step of the learner's `_env_step` env half (learner:397-464) in ONE launch:
 * msat_rng_chain + msat_env_keys + msat_step(auto_reset=1) fused.  The kernel advances the rollout
 * rng (rng_in uint32[2] -> chain_out uint32[10] = {rng', act_key, step_key, prob_key, reset_key};
 * the two buffers must not overlap) and every env that finishes derives its own new problem index
 * and reset key from the advanced chain with its GLOBAL env index env_offset + b out of
 * num_envs_global, so any sharding of the batch reproduces the single-device values.  Other
 * arguments as msat_step. */
int msat_rollout_step(const msat_plan* plan, const void* bank, int32_t num_problems,
                      const uint32_t* state_in, uint32_t* state_out, const int32_t* actions,
                      const uint32_t* rng_in, uint32_t* chain_out,
                      int32_t num_envs_global, int32_t env_offset,
                      int32_t* obs, float* reward, int32_t reward_cols, uint8_t* done, int32_t done_cols,
                      uint8_t* solved, int32_t* num_unsatisfied, int32_t* episode_step,
                      int32_t num_envs, void* stream);

/* msat_rollout_step for a GNN-style consumer (the reference's actor/critic read the GNN input, never the
 * local observations; SURVEY.md F8): same step, but instead of obs int32[B,A,D] it emits the dynamic
 * part of the GNN input of the state the caller continues from -- assignment int32[B,n] and
 * clause_features float[B,m,3] = {is_sat, #true literals / 3.0, 1} (learner:165-195) -- straight from the
 * staged formula record.  Either may be NULL.  The static part comes from msat_gnn_static once per bank. */
int msat_rollout_step_gnn(const msat_plan* plan, const void* bank, int32_t num_problems,
                          const uint32_t* state_in, uint32_t* state_out, const int32_t* actions,
                          const uint32_t* rng_in, uint32_t* chain_out,
                          int32_t num_envs_global, int32_t env_offset,
                          int32_t* assignment, float* clause_features,
                          float* reward, int32_t reward_cols, uint8_t* done, int32_t done_cols,
                          uint8_t* solved, int32_t* num_unsatisfied, int32_t* episode_step,
                          int32_t num_envs, void* stream);

/* K rollout steps in ONE launch (1 <= K <= 64) for callers whose actions do not depend on the intermediate
 * observations -- replaying an action table, open-loop evaluation (runner:30-73 with a fixed plan), or
 * small batches where one launch per step is launch-bound.  Each env group keeps its state and formula in
 * shared memory across the K steps and re-stages the formula only after an auto-reset.
 *   actions          int32 [K, B, A] (mode 0) or [K, B, A, V] (mode 1)
 *   chain_out        the chain of the LAST step; rng_in -> K applications of learner:397-434
 *   obs / gnn_*      with emit_every_step != 0: [K, B, ...] (the policy input after every step), else
 *                    [B, ...] of the final state only; at most one of obs / gnn_* kinds per launch
 *   reward, done, solved, num_unsatisfied, episode_step, newly_satisfied: [K, B, ...] (row j = step j,
 *                    pre-reset values, learner:467-478); any may be NULL
 * Results are identical to K calls of msat_rollout_step / msat_rollout_step_gnn. */
int msat_rollout_steps(const msat_plan* plan, const void* bank, int32_t num_problems,
                       const uint32_t* state_in, uint32_t* state_out, const int32_t* actions, int32_t num_steps,
                       const uint32_t* rng_in, uint32_t* chain_out,
                       int32_t num_envs_global, int32_t env_offset,
                       int32_t* obs, int32_t* gnn_assignment, float* gnn_clause_features, int32_t emit_every_step,
                       float* reward, int32_t reward_cols, uint8_t* done, int32_t done_cols,
                       uint8_t* solved, int32_t* num_unsatisfied, int32_t* episode_step, int32_t* newly_satisfied,
                       int32_t num_envs, void* stream);

/* Replaces `SATEnv.get_obs(state)` (env:345-398): obs int32[B,A,D] from a state. */
int msat_get_obs(const msat_plan* plan, const void* bank, int32_t num_problems,
                 const uint32_t* state, int32_t* obs, int32_t num_envs, void* stream);

/* Materialise the reference-shaped `SATState` leaves (env:13-24) from packed
 * state; any output may be NULL.  variable_assignments int32[B,n];
 * clauses_satisfied_status uint8[B,m]; num_unsatisfied int32[B]; step int32[B];
 * done uint8[B,A]; clauses int32[B,m,k]; agent_clause_masks int32[B,A,m];
 * agent_neighbor_masks int32[B,A,n]; literal_to_agent_idx int32[B,m,k];
 * problem_idx int32[B]. */
int msat_export_state(const msat_plan* plan, const void* bank, int32_t num_problems,
                      const uint32_t* state, int32_t num_envs,
                      int32_t* variable_assignments, uint8_t* clauses_satisfied_status,
                      int32_t* num_unsatisfied, int32_t* step, uint8_t* done, int32_t* clauses,
                      int32_t* agent_clause_masks, int32_t* agent_neighbor_masks,
                      int32_t* literal_to_agent_idx, int32_t* problem_idx, void* stream);

/* Host-buffer entry point of one rollout step (msat_rollout_step) for callers that keep actions and
 * results in (pinned) host memory: copies `actions_host` to `actions_dev`, runs the fused step
 * (rng chain + key derivation + step + auto-reset), copies reward / done / solved / num_unsatisfied /
 * episode_step back into the `*_host` buffers (each may be NULL) and synchronises the stream.  Result
 * buffers that are adjacent in both address spaces are copied as one transfer; batches of 32768+ envs
 * are processed as four slices alternating between two internal streams so that the PCIe
 * copies overlap the kernel.  All device workspaces are caller-owned; observations stay on the device
 * (obs_dev). */
int msat_rollout_step_host(const msat_plan* plan, const void* bank, int32_t num_problems,
                           uint32_t* state, const int32_t* actions_host, int32_t* actions_dev,
                           const uint32_t* rng_in, uint32_t* chain_out,
                           int32_t num_envs_global, int32_t env_offset,
                           int32_t* obs_dev, float* reward_dev, int32_t reward_cols,
                           uint8_t* done_dev, int32_t done_cols, uint8_t* solved_dev,
                           int32_t* num_unsatisfied_dev, int32_t* episode_step_dev,
                           float* reward_host, uint8_t* done_host, uint8_t* solved_host,
                           int32_t* num_unsatisfied_host, int32_t* episode_step_host,
                           int32_t num_envs, void* stream);

/* Asynchronous, double-buffered variant of msat_rollout_step_host.  A pipe owns two copy streams and
 * `depth` (1..4) slots of events on the device that is current at creation.  msat_rollout_step_host_async
 * enqueues -- without blocking the host -- the upload of `actions_host` (pinned) on the copy-in stream,
 * the fused step on `stream`, and the download of the results into the `*_host` buffers (pinned) on the
 * copy-out stream, ordered by events; msat_host_wait(pipe, slot) blocks until that slot's results are in
 * host memory.  Calls with different slots must use different actions_dev / result buffers (device and
 * host); with depth 2 the upload of step t+1 and the download of step t-1 overlap the kernel of step t.
 * Steps execute in call order (the state is updated in place on `stream`). */
typedef struct msat_host_pipe msat_host_pipe;
int msat_host_pipe_create(msat_host_pipe** out, int32_t depth);
void msat_host_pipe_destroy(msat_host_pipe* pipe);
int msat_rollout_step_host_async(msat_host_pipe* pipe, int32_t slot,
                                 const msat_plan* plan, const void* bank, int32_t num_problems,
                                 uint32_t* state, const int32_t* actions_host, int32_t* actions_dev,
                                 const uint32_t* rng_in, uint32_t* chain_out,
                                 int32_t num_envs_global, int32_t env_offset,
                                 int32_t* obs_dev, float* reward_dev, int32_t reward_cols,
                                 uint8_t* done_dev, int32_t done_cols, uint8_t* solved_dev,
                                 int32_t* num_unsatisfied_dev, int32_t* episode_step_dev,
                                 float* reward_host, uint8_t* done_host, uint8_t* solved_host,
                                 int32_t* num_unsatisfied_host, int32_t* episode_step_host,
                                 int32_t num_envs, void* stream);
int msat_host_wait(msat_host_pipe* pipe, int32_t slot);
/* Releases the library's internal per-device streams / events (msat_rollout_step_host). */
int msat_shutdown(void);

/* Clause-satisfaction update of the step launches that write NO observations (msat_rollout_step_gnn,
 * msat_step / msat_rollout_step(s) with obs == NULL).  Call before compiling a bank or allocating state:
 * rec_bytes and state_words change with the mode (re-read them with msat_plan_dims).
 *   MSAT_CLAUSES_FULL (default)   every step re-evaluates all m clauses from the staged literal block;
 *   MSAT_CLAUSES_INCREMENTAL      the state carries a 4-bit true-literal count per clause and the bank
 *        record the var -> clause occurrence lists (CSR); a step stages the CSR block (not the literal block) in
 *        shared memory with one TMA bulk copy, touches only the clauses adjacent to the flipped variables
 *        (env:130-156 restricted to those clauses) and reads the literals only when the episode restarts.
 *        Needs lits_per_clause <= 15.  Results are bit-identical in both modes;
 *        launches that do write observations keep the counts up to date with a full evaluation. */
#define MSAT_CLAUSES_FULL        0
#define MSAT_CLAUSES_INCREMENTAL 1
int msat_plan_set_clause_update(msat_plan* plan, int32_t mode);

/* Element type of the observations written by every entry point that uses this plan (call before the first
 * launch).  The reference declares int32 (env:390-396) and that is the default and the drop-in contract;
 * values are only ever -1 / 0 / 1, so a consumer that casts them anyway (an MLP's first layer) can ask for
 *   MSAT_OBS_INT8   the same values as int8: `obs` arguments then point to int8 [.., A, D] (still 16-byte
 *                   aligned) and the step moves a quarter of the observation bytes.
 * Not offered through the XLA FFI handlers (their observation buffers are typed S32). */
#define MSAT_OBS_INT32 0
#define MSAT_OBS_INT8  1
int msat_plan_set_obs_dtype(msat_plan* plan, int32_t dtype);

/* Diagnostics: while `counter_dev` (a device uint64, 8-byte aligned, owned by the caller) is set, every
 * auto-reset performed by a step launch that uses this plan adds 1 to it.  NULL switches it off. */
int msat_plan_set_reset_counter(msat_plan* plan, uint64_t* counter_dev);

/* Process-wide measurement knobs (A/B comparisons in bench.py; not part of the drop-in surface):
 *   "gae_plain" 1 = msat_gae keeps the register-chunked scan instead of the cp.async-pipelined one. */
int msat_tune(const char* key, int32_t value);

/* --- rollout RNG chain (JAX 0.4.29 Threefry-2x32, non-partitionable) --------- */

/* One rollout step of the key chain (learner:397,416,426):
 *   rng,act = split(rng); rng,step = split(rng); rng,prob,reset = split(rng,3).
 * chain_out uint32[10] = {rng', act_key, step_key, prob_key, reset_key}.
 * rng_in and chain_out may overlap only if rng_in == chain_out. */
int msat_rng_chain(const uint32_t* rng_in, uint32_t* chain_out, void* stream);

/* Generic `a, b = jax.random.split(key)` on device: out uint32[4] = {a, b}
 * (runner:289: `key, _rng = split(key)`). */
int msat_rng_split2(const uint32_t* key_in, uint32_t* out, void* stream);

/* Per-env derivation for a shard [env_offset, env_offset + num_envs_local) of a
 * global batch of num_envs_global envs (learner:430,434; runner:291,294):
 *   problem_idx[b] = randint(prob_key, (B_global,), 0, P)[env_offset + b]
 *   reset_keys[b]  = split(reset_key, B_global)[env_offset + b]
 * Uses global indices so every sharding of the batch yields identical values. */
int msat_env_keys(const uint32_t* prob_key, const uint32_t* reset_key,
                  int32_t num_envs_global, int32_t env_offset, int32_t num_envs_local,
                  int32_t num_problems, int32_t* problem_idx, uint32_t* reset_keys, void* stream);

/* msat_env_keys with a weighted problem draw, for curricula that choose which formulas auto-reset lands on
 * (train only on formulas a solver labelled satisfiable, weight by unsolved rate, ...).  Feed its outputs to
 * msat_step(auto_reset = 1) after msat_rng_chain.
 *
 * Weighted draw contract (oracle/curriculum.py restates it word for word).  For global env g out of Bg:
 *   - take the two 32-bit words randint already uses for that env: (k1, k2) = split(prob_key),
 *     hi = bits32_at(k1, Bg, g), lo = bits32_at(k2, Bg, g); let u = hi * 2^32 + lo;
 *   - cum_weights int64[P] holds inclusive prefix sums of non-negative integer weights; W = cum_weights[P-1];
 *   - if W <= 0 the index is the uniform draw, equal to what msat_env_keys returns;
 *   - otherwise r = floor(u * W / 2^64) (umulhi) and the index is the smallest p with cum_weights[p] > r;
 *   - the index is always in [0, P), also when the table is not monotone: the binary search is bounded;
 *   - reset_keys are identical to msat_env_keys' output.
 * Each draw depends only on (prob_key, Bg, g, cum_weights), so any sharding yields the single-device values.
 * A problem of weight 0 is never drawn while W > 0.  cum_weights must be 8-byte aligned (MSAT_EALIGN) and is read
 * only when problem_idx != NULL. */
int msat_env_keys_weighted(const uint32_t* prob_key, const uint32_t* reset_key,
                           int32_t num_envs_global, int32_t env_offset, int32_t num_envs_local,
                           const int64_t* cum_weights, int32_t num_problems,
                           int32_t* problem_idx, uint32_t* reset_keys, void* stream);

/* --- MAPPO advantage path (learner:504-532) ------------------------------------ */

/* Reverse GAE scan.  reward: float, element (t,b) at reward[t*reward_stride_t +
 * b*reward_stride_b] (a [T,B,A] buffer passes strides B*A and A: agent 0 is
 * read, learner:514; a dense team reward [T,B] passes B and 1).  done uint8[T,B],
 * value float[T,B], last_val float[B] -> advantages, targets float[T,B].
 * stats (may be NULL): double[3] += {count, sum, sum of squares} of the advantages,
 * accumulated by the scan itself so that the normalisation needs no separate pass
 * (zero it first; not cleared by the call). */
int msat_gae(const float* reward, int64_t reward_stride_t, int64_t reward_stride_b,
             const uint8_t* done, const float* value, const float* last_val,
             double gamma, double gae_lambda, float* advantages, float* targets, double* stats,
             int32_t num_steps, int32_t num_envs, void* stream);

/* stats double[3] += {count, sum, sum of squares} over adv[0..count).  Zero it
 * first (msat_adv_stats does NOT clear) so shards can be all-reduced. */
int msat_adv_stats(const float* adv, int64_t count, double* stats, void* stream);
/* adv = (adv - mean) / (std + 1e-8), population std, from stats (learner:530-532). */
int msat_adv_normalize(float* adv, int64_t count, const double* stats, void* stream);

/* --- next-tier rows (SURVEY.md section 8f) ----------------------------------------------- */

/* Static part of the GNN input, once per formula (graph_constructor.py:93-114; learner:150-164):
 * static_var_features float[P,n,3] = {positive degree / m, negative degree / m, 0}; optional dense
 * occurrence-count matrices a_pos / a_neg float[P,n,m] (NULL = skip; duplicates accumulate). */
int msat_gnn_static(const msat_plan* plan, const void* bank, int32_t num_problems,
                    float* static_var_features, float* a_pos, float* a_neg, void* stream);

/* Dynamic part of the GNN input, per env (learner:165-195): assignment int32[B,n] and
 * clause_features float[B,m,3] = {is_sat, #true literals / 3.0, 1}.  Either may be NULL. */
int msat_gnn_dynamic(const msat_plan* plan, const void* bank, int32_t num_problems,
                     const uint32_t* state, int32_t num_envs,
                     int32_t* assignment, float* clause_features, void* stream);

/* Rollout metric sums (learner:661-686) over a [T,B] rollout: sums double[5] += {sum of team reward,
 * #finished episodes, #solved at finish, sum of num_unsatisfied at finish, sum of episode_step of
 * solved-at-finish}.  Not cleared by the call (zero it first; shards can be all-reduced).
 * reward element (t,b) at reward[t*reward_stride_t + b*reward_stride_b]; the other arrays dense [T,B]. */
int msat_rollout_metrics(const float* reward, int64_t reward_stride_t, int64_t reward_stride_b,
                         const uint8_t* done, const uint8_t* solved, const int32_t* num_unsatisfied,
                         const int32_t* episode_step, int32_t num_steps, int32_t num_envs,
                         double* sums, void* stream);

/* Per-problem rollout statistics over a [T,B] rollout: stats int64[P,4].  For every (t, b) with done[t,b] != 0 one
 * episode is added to row p = clamp(problem_idx[t*pidx_stride_t + b*pidx_stride_b], 0, P-1); the columns are, in the
 * order of msat_rollout_metrics' sums 1..4: #finished episodes, #solved at finish, sum of num_unsatisfied at finish,
 * sum of episode_step over the episodes solved at finish.  Not cleared by the call (zero it first; shards can be
 * all-reduced).  Strides count int32 elements, so a RolloutBuffer's state [T, B, state_words] can be passed as is,
 * pointing at the problem-index word (word ceil(n/32) + 1, DESIGN.md section 3): the pre-step state of row t belongs
 * to the episode that ends at t.  done, solved uint8 and num_unsatisfied, episode_step int32 are dense [T,B].
 * stats must be 8-byte aligned (MSAT_EALIGN).  Rows of one problem are summed per warp and, for P <= 1024, per CTA in
 * shared memory, so a hot problem (P = 1) does not serialise on one counter. */
int msat_problem_stats(const int32_t* problem_idx, int64_t pidx_stride_t, int64_t pidx_stride_b,
                       const uint8_t* done, const uint8_t* solved, const int32_t* num_unsatisfied,
                       const int32_t* episode_step, int32_t num_steps, int32_t num_envs,
                       int32_t num_problems, int64_t* stats, void* stream);

/* Per-variable flip gains and the greedy expert labels of the BC pre-training
 * (src/runners/behavioral_cloning.py:54-100): delta_unsat int32[B,n] = change of the number of
 * unsatisfied clauses if variable v alone were flipped (break - make); greedy_labels int32[B,A] = per
 * agent the local index of its owned variable with the most negative delta (first wins ties) when that
 * delta < tau, else the no-op action V.  Either output may be NULL. */
int msat_flip_gains(const msat_plan* plan, const void* bank, int32_t num_problems,
                    const uint32_t* state, int32_t num_envs, double tau,
                    int32_t* delta_unsat, int32_t* greedy_labels, void* stream);

/* Bookkeeping of the greedy evaluation loop (runner:57-70) after evaluation step t (0-based): envs
 * solved for the first time get ever_solved = 1, steps_to_solve = t+1 and solution int32[B,n] = their
 * assignment.  Initialise ever_solved = 0, steps_to_solve = max_steps, solution = 0 before step 0. */
int msat_eval_track(const msat_plan* plan, const uint32_t* state, const uint8_t* solved, int32_t t,
                    int32_t num_envs, uint8_t* ever_solved, int32_t* steps_to_solve, int32_t* solution,
                    void* stream);

/* --- local search ------------------------------------------------------------------------------------ */

/* Batched WalkSAT/SKC with noise p, in place on packed env states (a classical solver next to the env: labels
 * for a bank, a local-search baseline at an RL flip budget, near-solution starts for msat_import_state).
 *
 * Algorithm contract (oracle/walksat.py restates it word for word).  The loop is per env.  Flip iteration t
 * runs for t = 0 .. max_flips-1 and stops early as soon as num_unsat == 0; an env that is already satisfied on
 * entry makes 0 flips.  Each iteration does the following:
 *   1. Random bits.  c = flip_offset + t (uint32); (x0, x1) = threefry2x32(key[b], ctr = (c, 0)).
 *   2. Clause choice.  U = num_unsat, r = umulhi(x0, U).  The picked clause is the r-th unsatisfied clause
 *      (0-based) in increasing clause index.
 *   3. Candidates.  The clause's non-padding literal columns j = 0..k-1, in column order; duplicates stay in
 *      the list.  nc = their count.  If nc == 0 (an all-padding clause) nothing is flipped, but the iteration
 *      still counts.
 *   4. Break counts.  break(v) = the number of distinct clauses that are satisfied now and unsatisfied after
 *      flipping v alone: a satisfied clause breaks iff all of its true literals are on v and it has no false
 *      literal on v.  Literal 0 is never true (env:135-144).
 *   5. Choice of variable.  If some candidate has break 0, the first such candidate (freebie).  Otherwise, if
 *      (x1 >> 8) < thr with thr = llrint(noise * 2^24), a random walk: candidate ((x1 & 0xFF) * nc) >> 8.
 *      Otherwise the first candidate with the minimum break.
 *   6. Flip.  Flip the chosen variable and update the true-literal counts, the status and num_unsat.
 * A call with max_flips = F1 + F2 gives the same result, bit for bit, as a call with F1 followed by a call with
 * F2 and flip_offset = F1 on the returned state with the same keys.
 *
 *   state     uint32[B, state_words], read and written in place.  The problem index comes from each record
 *             (clamped into [0, num_problems)).  The call rewrites the assignment words and num_unsatisfied
 *             (plus the 4-bit true-literal counts on an MSAT_CLAUSES_INCREMENTAL plan); step, the problem index
 *             and done are left unchanged.
 *   keys      uint32[B, 2], one Threefry key per env
 *   solved    uint8[B] (NULL = skip): num_unsat == 0 after the call
 *   flips     int32[B] (NULL = skip): iterations this call used
 * MSAT_EINVAL: missing pointers while B > 0, noise outside [0, 1] or NaN, negative max_flips / flip_offset or
 * flip_offset + max_flips > 2^31 - 1.  MSAT_EALIGN as msat_import_state (bank 128 bytes, state 16 bytes).
 * MSAT_EUNSUPPORTED: lits_per_clause > 32 or the per-env working set (literal block, var -> clause occurrence
 * lists, counts and status bits) does not fit in shared memory.  B == 0 returns MSAT_OK without touching the
 * device. */
int msat_walksat(const msat_plan* plan, const void* bank, int32_t num_problems,
                 uint32_t* state, const uint32_t* keys, int32_t max_flips, int32_t flip_offset,
                 double noise, uint8_t* solved, int32_t* flips, int32_t num_envs, void* stream);

/* Native DIMACS CNF reader (host only; replaces parse_cnf, src/utils/data_parser.py:8-42).  Parses `len`
 * bytes of `text`.  Call once with clauses == NULL to obtain clause_count (rows actually present) and
 * max_width (longest clause, terminating 0 excluded), then again with clauses int32[clause_count,
 * clause_stride] (clause_stride >= max_width) to receive the literals, 0-padded on the right.  num_vars /
 * num_clauses are the header's values (either may be NULL).  strict != 0 reproduces the reference exactly
 * (a blank line is an empty clause, a '%' footer is an error); strict == 0 skips blank lines and stops at '%'.
 * Returns MSAT_EINVAL for a malformed token or header. */
int msat_dimacs_parse(const char* text, size_t len, int32_t strict, int32_t* num_vars, int32_t* num_clauses,
                      int32_t* clause_count, int32_t* max_width, int32_t* clauses, int32_t clause_stride);

/* --- observation memory (host only) --------------------------------------------------------------------
 * Device memory with the driver's generic data compression (CU_MEM_ALLOCATION_COMP_GENERIC), where the L2
 * compresses lines on their way to DRAM and expands them on the way back.  Observation buffers hold only
 * -1 / 0 / 1 and are most of a step's DRAM writes; in this memory the same bytes cost less DRAM traffic.
 * Kernels, copies and torch ops see identical contents.  Unlike the enqueue calls above, these allocate and
 * synchronise, and they are not bound in the XLA FFI layer (XLA allocates its custom calls' outputs).
 *
 * msat_obs_compression: *granted = 1 when `device` reports generic compression support and the driver
 *   honours the compressible property for a probe allocation (and for every msat_obs_alloc on it since),
 *   else 0.  MSAT_EINVAL for a NULL `granted`, a negative or unknown device.
 * msat_obs_alloc / msat_obs_free: the allocation pair torch.cuda.memory.CUDAPluggableAllocator expects
 *   (`stream` is a cudaStream_t and unused).  alloc maps `size` bytes rounded up to the driver's
 *   recommended granularity on `device` and returns NULL when the driver refuses; free waits for the
 *   device, unmaps and releases the memory.  Memory the driver hands back uncompressed is still returned
 *   and turns msat_obs_compression off for the device. */
int msat_obs_compression(int device, int* granted);
void* msat_obs_alloc(size_t size, int device, void* stream);
void msat_obs_free(void* ptr, size_t size, int device, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MARL_SAT_B200_H */
