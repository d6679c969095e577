// XLA FFI custom-call layer over the C ABI of libmarlsat_b200.so (include/marl_sat_b200.h): one handler per
// enqueue entry point.  This is the "thin XLA FFI custom-call layer" of the reference-side integration
// (call sites: src/learners/mappo_gnn_sat_learner.py:418,435; src/runners/mappo_runner.py:137): XLA calls a
// handler from its executor thread with the op's stream, device buffers it owns and the static attributes; the
// handler validates nothing itself, forwards to msat_* (enqueue only, no allocation, no synchronisation) and
// maps a non-zero return code to an ffi::Error.
//
// The observation-memory calls msat_obs_compression(), msat_obs_alloc() and msat_obs_free() have no handler:
// they allocate, and XLA allocates the outputs of a custom call itself.
//
// Built only where JAX ships the FFI headers (marl_sat_b200/build.py: `jax.ffi.include_dir()`); this image has
// no JAX, so here the file is syntax-checked against tests/ffi_stub and otherwise unused.  Registration and the
// `jax.ffi.ffi_call` wrappers live in marl_sat_b200/jax_ffi.py.
//
// Conventions: the plan handle travels as the int64 attribute "plan" (the address returned by
// msat_plan_create); scalar arguments are attributes; in-place state updates are expressed with
// input_output_aliases on the Python side, so `state_in` / `state` results may point to the same buffer.
#include <cuda_runtime_api.h>

#include <cstdint>
#include <string>

#include "../../include/marl_sat_b200.h"
#include "xla/ffi/api/ffi.h"

namespace ffi = xla::ffi;

namespace {

inline const msat_plan* plan_of(int64_t handle) { return reinterpret_cast<const msat_plan*>(handle); }

inline ffi::Error status(int rc, const char* what) {
    if (rc == MSAT_OK) return ffi::Error::Success();
    return ffi::Error(rc < 0 ? ffi::ErrorCode::kInvalidArgument : ffi::ErrorCode::kInternal,
                      std::string(what) + " failed with code " + std::to_string(rc));
}
inline int32_t dim0(const ffi::Dimensions& d) { return d.size() ? static_cast<int32_t>(d[0]) : 1; }
inline int32_t last_dim(const ffi::Dimensions& d) { return d.size() ? static_cast<int32_t>(d.back()) : 1; }

// ---- formula bank ----------------------------------------------------------------------------------------
ffi::Error CompileBank(cudaStream_t s, int64_t plan, ffi::Buffer<ffi::S32> clauses, ffi::ResultBuffer<ffi::U8> bank) {
    return status(msat_compile_bank(plan_of(plan), clauses.typed_data(), dim0(clauses.dimensions()), bank->typed_data(), s),
                  "msat_compile_bank");
}

// ---- environment -----------------------------------------------------------------------------------------
ffi::Error Reset(cudaStream_t s, int64_t plan, int64_t num_problems, ffi::Buffer<ffi::U8> bank,
                 ffi::Buffer<ffi::S32> problem_idx, ffi::Buffer<ffi::U32> keys, ffi::ResultBuffer<ffi::U32> state,
                 ffi::ResultBuffer<ffi::S32> obs) {
    return status(msat_reset(plan_of(plan), bank.typed_data(), (int32_t)num_problems, problem_idx.typed_data(),
                             keys.typed_data(), state->typed_data(), obs->typed_data(), dim0(problem_idx.dimensions()), s),
                  "msat_reset");
}

// inverse of ExportState: packed states (+ observations) from reference-shaped leaves; step / done may be given as
// zeros (msat_import_state treats them like NULL)
ffi::Error ImportState(cudaStream_t s, int64_t plan, int64_t num_problems, ffi::Buffer<ffi::U8> bank,
                       ffi::Buffer<ffi::S32> problem_idx, ffi::Buffer<ffi::S32> assignments, ffi::Buffer<ffi::S32> step,
                       ffi::Buffer<ffi::U8> done, ffi::ResultBuffer<ffi::U32> state, ffi::ResultBuffer<ffi::S32> obs) {
    return status(msat_import_state(plan_of(plan), bank.typed_data(), (int32_t)num_problems, problem_idx.typed_data(),
                                    assignments.typed_data(), step.typed_data(), done.typed_data(), state->typed_data(),
                                    obs->typed_data(), dim0(problem_idx.dimensions()), s),
                  "msat_import_state");
}

ffi::Error Step(cudaStream_t s, int64_t plan, int64_t num_problems, int64_t auto_reset, ffi::Buffer<ffi::U8> bank,
                ffi::Buffer<ffi::U32> state_in, ffi::Buffer<ffi::S32> actions, ffi::Buffer<ffi::S32> new_problem_idx,
                ffi::Buffer<ffi::U32> reset_keys, ffi::ResultBuffer<ffi::U32> state, ffi::ResultBuffer<ffi::S32> obs,
                ffi::ResultBuffer<ffi::F32> reward, ffi::ResultBuffer<ffi::U8> done, ffi::ResultBuffer<ffi::U8> solved,
                ffi::ResultBuffer<ffi::S32> num_unsatisfied, ffi::ResultBuffer<ffi::S32> episode_step) {
    return status(msat_step(plan_of(plan), bank.typed_data(), (int32_t)num_problems, state_in.typed_data(),
                            state->typed_data(), actions.typed_data(), (int32_t)auto_reset, new_problem_idx.typed_data(),
                            reset_keys.typed_data(), obs->typed_data(), reward->typed_data(),
                            last_dim(reward->dimensions()), done->typed_data(), last_dim(done->dimensions()),
                            solved->typed_data(), num_unsatisfied->typed_data(), episode_step->typed_data(), nullptr,
                            dim0(state_in.dimensions()), s),
                  "msat_step");
}

// learner:397-464 in one custom call: rng chain + per-env keys + step + auto-reset (+ K fused steps)
ffi::Error RolloutSteps(cudaStream_t s, int64_t plan, int64_t num_problems, int64_t num_steps, int64_t num_envs_global,
                        int64_t env_offset, int64_t emit_every_step, ffi::Buffer<ffi::U8> bank,
                        ffi::Buffer<ffi::U32> state_in, ffi::Buffer<ffi::S32> actions, ffi::Buffer<ffi::U32> rng_in,
                        ffi::ResultBuffer<ffi::U32> state, ffi::ResultBuffer<ffi::U32> chain_out,
                        ffi::ResultBuffer<ffi::S32> obs, ffi::ResultBuffer<ffi::F32> reward, ffi::ResultBuffer<ffi::U8> done,
                        ffi::ResultBuffer<ffi::U8> solved, ffi::ResultBuffer<ffi::S32> num_unsatisfied,
                        ffi::ResultBuffer<ffi::S32> episode_step) {
    return status(msat_rollout_steps(plan_of(plan), bank.typed_data(), (int32_t)num_problems, state_in.typed_data(),
                                     state->typed_data(), actions.typed_data(), (int32_t)num_steps, rng_in.typed_data(),
                                     chain_out->typed_data(), (int32_t)num_envs_global, (int32_t)env_offset,
                                     obs->typed_data(), nullptr, nullptr, (int32_t)emit_every_step, reward->typed_data(),
                                     last_dim(reward->dimensions()), done->typed_data(), last_dim(done->dimensions()),
                                     solved->typed_data(), num_unsatisfied->typed_data(), episode_step->typed_data(),
                                     nullptr, dim0(state_in.dimensions()), s),
                  "msat_rollout_steps");
}

// the same step for a GNN-style consumer: dynamic GNN input instead of local observations
ffi::Error RolloutStepsGnn(cudaStream_t s, int64_t plan, int64_t num_problems, int64_t num_steps,
                           int64_t num_envs_global, int64_t env_offset, int64_t emit_every_step,
                           ffi::Buffer<ffi::U8> bank, ffi::Buffer<ffi::U32> state_in, ffi::Buffer<ffi::S32> actions,
                           ffi::Buffer<ffi::U32> rng_in, ffi::ResultBuffer<ffi::U32> state,
                           ffi::ResultBuffer<ffi::U32> chain_out, ffi::ResultBuffer<ffi::S32> assignment,
                           ffi::ResultBuffer<ffi::F32> clause_features, ffi::ResultBuffer<ffi::F32> reward,
                           ffi::ResultBuffer<ffi::U8> done, ffi::ResultBuffer<ffi::U8> solved,
                           ffi::ResultBuffer<ffi::S32> num_unsatisfied, ffi::ResultBuffer<ffi::S32> episode_step) {
    return status(msat_rollout_steps(plan_of(plan), bank.typed_data(), (int32_t)num_problems, state_in.typed_data(),
                                     state->typed_data(), actions.typed_data(), (int32_t)num_steps, rng_in.typed_data(),
                                     chain_out->typed_data(), (int32_t)num_envs_global, (int32_t)env_offset, nullptr,
                                     assignment->typed_data(), clause_features->typed_data(), (int32_t)emit_every_step,
                                     reward->typed_data(), last_dim(reward->dimensions()), done->typed_data(),
                                     last_dim(done->dimensions()), solved->typed_data(), num_unsatisfied->typed_data(),
                                     episode_step->typed_data(), nullptr, dim0(state_in.dimensions()), s),
                  "msat_rollout_steps");
}

ffi::Error GetObs(cudaStream_t s, int64_t plan, int64_t num_problems, ffi::Buffer<ffi::U8> bank,
                  ffi::Buffer<ffi::U32> state, ffi::ResultBuffer<ffi::S32> obs) {
    return status(msat_get_obs(plan_of(plan), bank.typed_data(), (int32_t)num_problems, state.typed_data(),
                               obs->typed_data(), dim0(state.dimensions()), s),
                  "msat_get_obs");
}

// SATState leaves (env:13-24) for API fidelity: every leaf is a result
ffi::Error ExportState(cudaStream_t s, int64_t plan, int64_t num_problems, ffi::Buffer<ffi::U8> bank,
                       ffi::Buffer<ffi::U32> state, ffi::ResultBuffer<ffi::S32> variable_assignments,
                       ffi::ResultBuffer<ffi::U8> clauses_satisfied_status, ffi::ResultBuffer<ffi::S32> num_unsatisfied,
                       ffi::ResultBuffer<ffi::S32> step, ffi::ResultBuffer<ffi::U8> done, ffi::ResultBuffer<ffi::S32> clauses,
                       ffi::ResultBuffer<ffi::S32> agent_clause_masks, ffi::ResultBuffer<ffi::S32> agent_neighbor_masks,
                       ffi::ResultBuffer<ffi::S32> literal_to_agent_idx) {
    return status(msat_export_state(plan_of(plan), bank.typed_data(), (int32_t)num_problems, state.typed_data(),
                                    dim0(state.dimensions()), variable_assignments->typed_data(),
                                    clauses_satisfied_status->typed_data(), num_unsatisfied->typed_data(),
                                    step->typed_data(), done->typed_data(), clauses->typed_data(),
                                    agent_clause_masks->typed_data(), agent_neighbor_masks->typed_data(),
                                    literal_to_agent_idx->typed_data(), nullptr, s),
                  "msat_export_state");
}

// ---- rollout RNG chain -----------------------------------------------------------------------------------
ffi::Error RngChain(cudaStream_t s, ffi::Buffer<ffi::U32> rng_in, ffi::ResultBuffer<ffi::U32> chain_out) {
    return status(msat_rng_chain(rng_in.typed_data(), chain_out->typed_data(), s), "msat_rng_chain");
}
ffi::Error RngSplit2(cudaStream_t s, ffi::Buffer<ffi::U32> key_in, ffi::ResultBuffer<ffi::U32> out) {
    return status(msat_rng_split2(key_in.typed_data(), out->typed_data(), s), "msat_rng_split2");
}
ffi::Error EnvKeys(cudaStream_t s, int64_t num_envs_global, int64_t env_offset, int64_t num_problems,
                   ffi::Buffer<ffi::U32> prob_key, ffi::Buffer<ffi::U32> reset_key,
                   ffi::ResultBuffer<ffi::S32> problem_idx, ffi::ResultBuffer<ffi::U32> reset_keys) {
    return status(msat_env_keys(prob_key.typed_data(), reset_key.typed_data(), (int32_t)num_envs_global,
                                (int32_t)env_offset, dim0(problem_idx->dimensions()), (int32_t)num_problems,
                                problem_idx->typed_data(), reset_keys->typed_data(), s),
                  "msat_env_keys");
}

// weighted problem draw: cum_weights int64[P] are inclusive prefix sums of the problem weights
ffi::Error EnvKeysWeighted(cudaStream_t s, int64_t num_envs_global, int64_t env_offset, ffi::Buffer<ffi::U32> prob_key,
                           ffi::Buffer<ffi::U32> reset_key, ffi::Buffer<ffi::S64> cum_weights,
                           ffi::ResultBuffer<ffi::S32> problem_idx, ffi::ResultBuffer<ffi::U32> reset_keys) {
    return status(msat_env_keys_weighted(prob_key.typed_data(), reset_key.typed_data(), (int32_t)num_envs_global,
                                         (int32_t)env_offset, dim0(problem_idx->dimensions()), cum_weights.typed_data(),
                                         dim0(cum_weights.dimensions()), problem_idx->typed_data(),
                                         reset_keys->typed_data(), s),
                  "msat_env_keys_weighted");
}

// ---- MAPPO advantage path (learner:504-532) ---------------------------------------------------------------
ffi::Error Gae(cudaStream_t s, double gamma, double gae_lambda, ffi::Buffer<ffi::F32> reward, ffi::Buffer<ffi::U8> done,
               ffi::Buffer<ffi::F32> value, ffi::Buffer<ffi::F32> last_val, ffi::Buffer<ffi::F64> stats_in,
               ffi::ResultBuffer<ffi::F32> advantages, ffi::ResultBuffer<ffi::F32> targets,
               ffi::ResultBuffer<ffi::F64> stats) {
    // reward is [T, B] or [T, B, A] (agent 0 read, learner:514); stats_in is aliased to stats (zeros in, sums out)
    const ffi::Dimensions rd = reward.dimensions(), vd = value.dimensions();
    const int32_t T = dim0(vd), B = last_dim(vd);
    const int64_t A = rd.size() == 3 ? rd[2] : 1;
    (void)stats_in;
    return status(msat_gae(reward.typed_data(), (int64_t)B * A, A, done.typed_data(), value.typed_data(),
                           last_val.typed_data(), gamma, gae_lambda, advantages->typed_data(), targets->typed_data(),
                           stats->typed_data(), T, B, s),
                  "msat_gae");
}
ffi::Error AdvStats(cudaStream_t s, ffi::Buffer<ffi::F32> adv, ffi::Buffer<ffi::F64> stats_in,
                    ffi::ResultBuffer<ffi::F64> stats) {
    (void)stats_in;
    return status(msat_adv_stats(adv.typed_data(), (int64_t)adv.element_count(), stats->typed_data(), s), "msat_adv_stats");
}
ffi::Error AdvNormalize(cudaStream_t s, ffi::Buffer<ffi::F32> adv_in, ffi::Buffer<ffi::F64> stats,
                        ffi::ResultBuffer<ffi::F32> adv) {
    (void)adv_in;      // aliased to adv (in place)
    return status(msat_adv_normalize(adv->typed_data(), (int64_t)adv->element_count(), stats.typed_data(), s),
                  "msat_adv_normalize");
}

// ---- next-tier rows -----------------------------------------------------------------------------------------
ffi::Error GnnStatic(cudaStream_t s, int64_t plan, ffi::Buffer<ffi::U8> bank, ffi::ResultBuffer<ffi::F32> svf,
                     ffi::ResultBuffer<ffi::F32> a_pos, ffi::ResultBuffer<ffi::F32> a_neg) {
    return status(msat_gnn_static(plan_of(plan), bank.typed_data(), dim0(svf->dimensions()), svf->typed_data(),
                                  a_pos->typed_data(), a_neg->typed_data(), s),
                  "msat_gnn_static");
}
ffi::Error GnnDynamic(cudaStream_t s, int64_t plan, int64_t num_problems, ffi::Buffer<ffi::U8> bank,
                      ffi::Buffer<ffi::U32> state, ffi::ResultBuffer<ffi::S32> assignment,
                      ffi::ResultBuffer<ffi::F32> clause_features) {
    return status(msat_gnn_dynamic(plan_of(plan), bank.typed_data(), (int32_t)num_problems, state.typed_data(),
                                   dim0(state.dimensions()), assignment->typed_data(), clause_features->typed_data(), s),
                  "msat_gnn_dynamic");
}
ffi::Error RolloutMetrics(cudaStream_t s, ffi::Buffer<ffi::F32> reward, ffi::Buffer<ffi::U8> done,
                          ffi::Buffer<ffi::U8> solved, ffi::Buffer<ffi::S32> num_unsatisfied,
                          ffi::Buffer<ffi::S32> episode_step, ffi::Buffer<ffi::F64> sums_in,
                          ffi::ResultBuffer<ffi::F64> sums) {
    const ffi::Dimensions rd = reward.dimensions(), dd = done.dimensions();
    const int32_t T = dim0(dd), B = last_dim(dd);
    const int64_t A = rd.size() == 3 ? rd[2] : 1;
    (void)sums_in;
    return status(msat_rollout_metrics(reward.typed_data(), (int64_t)B * A, A, done.typed_data(), solved.typed_data(),
                                       num_unsatisfied.typed_data(), episode_step.typed_data(), T, B, sums->typed_data(), s),
                  "msat_rollout_metrics");
}
// per-problem statistics of a dense [T, B] rollout; stats_in (zeros or running totals) is aliased to stats
ffi::Error ProblemStats(cudaStream_t s, ffi::Buffer<ffi::S32> problem_idx, ffi::Buffer<ffi::U8> done,
                        ffi::Buffer<ffi::U8> solved, ffi::Buffer<ffi::S32> num_unsatisfied,
                        ffi::Buffer<ffi::S32> episode_step, ffi::Buffer<ffi::S64> stats_in,
                        ffi::ResultBuffer<ffi::S64> stats) {
    const ffi::Dimensions dd = done.dimensions();
    const int32_t T = dim0(dd), B = last_dim(dd);
    (void)stats_in;
    return status(msat_problem_stats(problem_idx.typed_data(), B, 1, done.typed_data(), solved.typed_data(),
                                     num_unsatisfied.typed_data(), episode_step.typed_data(), T, B,
                                     dim0(stats->dimensions()), stats->typed_data(), s),
                  "msat_problem_stats");
}
ffi::Error FlipGains(cudaStream_t s, int64_t plan, int64_t num_problems, double tau, ffi::Buffer<ffi::U8> bank,
                     ffi::Buffer<ffi::U32> state, ffi::ResultBuffer<ffi::S32> delta_unsat,
                     ffi::ResultBuffer<ffi::S32> greedy_labels) {
    return status(msat_flip_gains(plan_of(plan), bank.typed_data(), (int32_t)num_problems, state.typed_data(),
                                  dim0(state.dimensions()), tau, delta_unsat->typed_data(), greedy_labels->typed_data(), s),
                  "msat_flip_gains");
}
ffi::Error EvalTrack(cudaStream_t s, int64_t plan, int64_t t, ffi::Buffer<ffi::U32> state, ffi::Buffer<ffi::U8> solved,
                     ffi::Buffer<ffi::U8> ever_in, ffi::Buffer<ffi::S32> steps_in, ffi::Buffer<ffi::S32> solution_in,
                     ffi::ResultBuffer<ffi::U8> ever_solved, ffi::ResultBuffer<ffi::S32> steps_to_solve,
                     ffi::ResultBuffer<ffi::S32> solution) {
    (void)ever_in; (void)steps_in; (void)solution_in;      // aliased to the results (updated in place)
    return status(msat_eval_track(plan_of(plan), state.typed_data(), solved.typed_data(), (int32_t)t,
                                  dim0(state.dimensions()), ever_solved->typed_data(), steps_to_solve->typed_data(),
                                  solution->typed_data(), s),
                  "msat_eval_track");
}

// ---- local search ----------------------------------------------------------------------------------------------
// WalkSAT in place on the packed states (state_in is aliased to state); solved / flips per env
ffi::Error Walksat(cudaStream_t s, int64_t plan, int64_t num_problems, int64_t max_flips, int64_t flip_offset,
                   double noise, ffi::Buffer<ffi::U8> bank, ffi::Buffer<ffi::U32> state_in, ffi::Buffer<ffi::U32> keys,
                   ffi::ResultBuffer<ffi::U32> state, ffi::ResultBuffer<ffi::U8> solved, ffi::ResultBuffer<ffi::S32> flips) {
    (void)state_in;
    return status(msat_walksat(plan_of(plan), bank.typed_data(), (int32_t)num_problems, state->typed_data(),
                               keys.typed_data(), (int32_t)max_flips, (int32_t)flip_offset, noise, solved->typed_data(),
                               flips->typed_data(), dim0(state->dimensions()), s),
                  "msat_walksat");
}

template <ffi::DataType T> using In = ffi::Buffer<T>;
template <ffi::DataType T> using Out = ffi::Buffer<T>;
using Stream = ffi::PlatformStream<cudaStream_t>;

}  // namespace

// ---- handler symbols (looked up by marl_sat_b200/jax_ffi.py with ctypes and wrapped in PyCapsules) ----------
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatCompileBank, CompileBank,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("plan").Arg<In<ffi::S32>>().Ret<Out<ffi::U8>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatReset, Reset,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("plan").Attr<int64_t>("num_problems")
        .Arg<In<ffi::U8>>().Arg<In<ffi::S32>>().Arg<In<ffi::U32>>().Ret<Out<ffi::U32>>().Ret<Out<ffi::S32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatImportState, ImportState,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("plan").Attr<int64_t>("num_problems")
        .Arg<In<ffi::U8>>().Arg<In<ffi::S32>>().Arg<In<ffi::S32>>().Arg<In<ffi::S32>>().Arg<In<ffi::U8>>()
        .Ret<Out<ffi::U32>>().Ret<Out<ffi::S32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatStep, Step,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("plan").Attr<int64_t>("num_problems").Attr<int64_t>("auto_reset")
        .Arg<In<ffi::U8>>().Arg<In<ffi::U32>>().Arg<In<ffi::S32>>().Arg<In<ffi::S32>>().Arg<In<ffi::U32>>()
        .Ret<Out<ffi::U32>>().Ret<Out<ffi::S32>>().Ret<Out<ffi::F32>>().Ret<Out<ffi::U8>>().Ret<Out<ffi::U8>>()
        .Ret<Out<ffi::S32>>().Ret<Out<ffi::S32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatRolloutSteps, RolloutSteps,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("plan").Attr<int64_t>("num_problems").Attr<int64_t>("num_steps")
        .Attr<int64_t>("num_envs_global").Attr<int64_t>("env_offset").Attr<int64_t>("emit_every_step")
        .Arg<In<ffi::U8>>().Arg<In<ffi::U32>>().Arg<In<ffi::S32>>().Arg<In<ffi::U32>>()
        .Ret<Out<ffi::U32>>().Ret<Out<ffi::U32>>().Ret<Out<ffi::S32>>().Ret<Out<ffi::F32>>().Ret<Out<ffi::U8>>()
        .Ret<Out<ffi::U8>>().Ret<Out<ffi::S32>>().Ret<Out<ffi::S32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatRolloutStepsGnn, RolloutStepsGnn,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("plan").Attr<int64_t>("num_problems").Attr<int64_t>("num_steps")
        .Attr<int64_t>("num_envs_global").Attr<int64_t>("env_offset").Attr<int64_t>("emit_every_step")
        .Arg<In<ffi::U8>>().Arg<In<ffi::U32>>().Arg<In<ffi::S32>>().Arg<In<ffi::U32>>()
        .Ret<Out<ffi::U32>>().Ret<Out<ffi::U32>>().Ret<Out<ffi::S32>>().Ret<Out<ffi::F32>>().Ret<Out<ffi::F32>>()
        .Ret<Out<ffi::U8>>().Ret<Out<ffi::U8>>().Ret<Out<ffi::S32>>().Ret<Out<ffi::S32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatGetObs, GetObs,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("plan").Attr<int64_t>("num_problems")
        .Arg<In<ffi::U8>>().Arg<In<ffi::U32>>().Ret<Out<ffi::S32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatExportState, ExportState,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("plan").Attr<int64_t>("num_problems")
        .Arg<In<ffi::U8>>().Arg<In<ffi::U32>>().Ret<Out<ffi::S32>>().Ret<Out<ffi::U8>>().Ret<Out<ffi::S32>>()
        .Ret<Out<ffi::S32>>().Ret<Out<ffi::U8>>().Ret<Out<ffi::S32>>().Ret<Out<ffi::S32>>().Ret<Out<ffi::S32>>()
        .Ret<Out<ffi::S32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatRngChain, RngChain,
    ffi::Ffi::Bind().Ctx<Stream>().Arg<In<ffi::U32>>().Ret<Out<ffi::U32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatRngSplit2, RngSplit2,
    ffi::Ffi::Bind().Ctx<Stream>().Arg<In<ffi::U32>>().Ret<Out<ffi::U32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatEnvKeys, EnvKeys,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("num_envs_global").Attr<int64_t>("env_offset")
        .Attr<int64_t>("num_problems").Arg<In<ffi::U32>>().Arg<In<ffi::U32>>().Ret<Out<ffi::S32>>().Ret<Out<ffi::U32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatEnvKeysWeighted, EnvKeysWeighted,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("num_envs_global").Attr<int64_t>("env_offset")
        .Arg<In<ffi::U32>>().Arg<In<ffi::U32>>().Arg<In<ffi::S64>>().Ret<Out<ffi::S32>>().Ret<Out<ffi::U32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatGae, Gae,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<double>("gamma").Attr<double>("gae_lambda")
        .Arg<In<ffi::F32>>().Arg<In<ffi::U8>>().Arg<In<ffi::F32>>().Arg<In<ffi::F32>>().Arg<In<ffi::F64>>()
        .Ret<Out<ffi::F32>>().Ret<Out<ffi::F32>>().Ret<Out<ffi::F64>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatAdvStats, AdvStats,
    ffi::Ffi::Bind().Ctx<Stream>().Arg<In<ffi::F32>>().Arg<In<ffi::F64>>().Ret<Out<ffi::F64>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatAdvNormalize, AdvNormalize,
    ffi::Ffi::Bind().Ctx<Stream>().Arg<In<ffi::F32>>().Arg<In<ffi::F64>>().Ret<Out<ffi::F32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatGnnStatic, GnnStatic,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("plan").Arg<In<ffi::U8>>().Ret<Out<ffi::F32>>().Ret<Out<ffi::F32>>()
        .Ret<Out<ffi::F32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatGnnDynamic, GnnDynamic,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("plan").Attr<int64_t>("num_problems")
        .Arg<In<ffi::U8>>().Arg<In<ffi::U32>>().Ret<Out<ffi::S32>>().Ret<Out<ffi::F32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatRolloutMetrics, RolloutMetrics,
    ffi::Ffi::Bind().Ctx<Stream>().Arg<In<ffi::F32>>().Arg<In<ffi::U8>>().Arg<In<ffi::U8>>().Arg<In<ffi::S32>>()
        .Arg<In<ffi::S32>>().Arg<In<ffi::F64>>().Ret<Out<ffi::F64>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatProblemStats, ProblemStats,
    ffi::Ffi::Bind().Ctx<Stream>().Arg<In<ffi::S32>>().Arg<In<ffi::U8>>().Arg<In<ffi::U8>>().Arg<In<ffi::S32>>()
        .Arg<In<ffi::S32>>().Arg<In<ffi::S64>>().Ret<Out<ffi::S64>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatFlipGains, FlipGains,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("plan").Attr<int64_t>("num_problems").Attr<double>("tau")
        .Arg<In<ffi::U8>>().Arg<In<ffi::U32>>().Ret<Out<ffi::S32>>().Ret<Out<ffi::S32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatEvalTrack, EvalTrack,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("plan").Attr<int64_t>("t")
        .Arg<In<ffi::U32>>().Arg<In<ffi::U8>>().Arg<In<ffi::U8>>().Arg<In<ffi::S32>>().Arg<In<ffi::S32>>()
        .Ret<Out<ffi::U8>>().Ret<Out<ffi::S32>>().Ret<Out<ffi::S32>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(MsatWalksat, Walksat,
    ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("plan").Attr<int64_t>("num_problems").Attr<int64_t>("max_flips")
        .Attr<int64_t>("flip_offset").Attr<double>("noise").Arg<In<ffi::U8>>().Arg<In<ffi::U32>>().Arg<In<ffi::U32>>()
        .Ret<Out<ffi::U32>>().Ret<Out<ffi::U8>>().Ret<Out<ffi::S32>>());
