// Host-side template dispatch for one segment count N.  Each rollout_nK.cu translation unit
// instantiates launch_*_n<K> so the (N x mode) kernel matrix compiles in parallel.  Three rollout
// families: plain (swm_rollout, with the built-in screen), screened with cost forms and / or an
// ensemble (swm_rollout_costed / swm_rollout_ensemble / swm_rollout_shielded / swm_rollout_lookahead) and the model
// set (swm_rollout_models); all
// take the policy storage from with_policy_storage.
#pragma once
#include <type_traits>

#include "kernels.cuh"

namespace swm {

struct RolloutFlags {
  int variant;    // swm_variant
  bool linear;    // false: fixed actions
  bool norm, stats, screen;
  bool group_w;   // rollouts_per_policy % 32 == 0 (warp-uniform policy)
};

template <int N> int launch_step_n(const Phys& P, int variant, bool acc_only, const double* state_in,
                                   const double* action, double* out, double* reward, long long B,
                                   cudaStream_t st);
template <int N> int launch_rollout_n(const RolloutArgs& a, const RolloutFlags& f, cudaStream_t st);
// per-step screening with cost forms and / or an ensemble of simulator models: SCREEN_AFFINE without models (forms
// required), else SCREEN_ENSEMBLE (no forms: the built-in cost) or SCREEN_ENSEMBLE_AFFINE; with a backup (models
// required) SCREEN_SHIELD or SCREEN_SHIELD_AFFINE, and with a backup and lookahead > 0 SCREEN_LOOKAHEAD or
// SCREEN_LOOKAHEAD_AFFINE
template <int N> int launch_rollout_screened_n(const RolloutArgs& a, const SimModels* models, const CostForms* forms,
                                               const Backup* backup, int lookahead, const RolloutFlags& f,
                                               cudaStream_t st);
// model-set mode: cfg->B environments for each of models.M models, one CTA row per model (f as for launch_rollout_n)
template <int N> int launch_rollout_models_n(const RolloutArgs& a, const SimModels& models, const RolloutFlags& f,
                                             cudaStream_t st);
template <int N> int launch_step_models_n(const PhysSet& set, long long envs_per_model, const double* state_in,
                                          const double* action, double* out, double* reward, long long B,
                                          cudaStream_t st);

#ifdef SWM_INSTANTIATE_N

// dynamic shared memory of one rollout_body instantiation
template <int N, int VARIANT, int WMODE, bool STATS>
static size_t rollout_smem() {
  constexpr int WS = (N - 1) * (2 * N + 2);
  size_t smem = 0;
  if (WMODE == W_SMEM_THREAD) smem = sizeof(double) * WS * kRolloutBlock;
  if (WMODE == W_SMEM_GROUP) smem = sizeof(double) * WS * (kRolloutBlock / 32);
  if (STATS && (2 * N + 2) > kRegStatsMaxObs) smem += sizeof(double) * 2 * (2 * N + 2) * kRolloutBlock;
  smem += sizeof(double) * FactSmem<N, VARIANT>::doubles * kRolloutBlock;
  return smem;
}

// grid_y: CTA rows (the models of the model-set mode, else 1)
template <typename Kernel, typename... Args>
static int launch_rollout_grid(Kernel kern, size_t smem, long long B, unsigned grid_y, cudaStream_t st,
                               const Args&... args) {
  // dynamic + static shared memory (s_mu, s_piv, the moment reduction scratch: < 2 KB) above the default
  // 48 KB limit needs the opt-in attribute
  if (smem + 2048 > 48 * 1024) {
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return SWM_ERR_CUDA;
  }
  const long long blocks = (B + kRolloutBlock - 1) / kRolloutBlock;
  kern<<<dim3((unsigned)blocks, grid_y), kRolloutBlock, smem, st>>>(args...);
  return cudaPeekAtLastError() == cudaSuccess ? SWM_OK : SWM_ERR_CUDA;  // capi.cu note_launch reads + clears it
}

// Where a linear policy lives: registers up to kRegPolicyMax doubles, else shared memory, one copy per warp when
// the warp's rollouts share one policy (group_w).  Calls launch(std::integral_constant<int, WMODE>).
template <int N, typename Launch>
static int with_policy_storage(bool group_w, Launch&& launch) {
  if constexpr ((N - 1) * (2 * N + 2) <= kRegPolicyMax) {
    return launch(std::integral_constant<int, W_REG>{});
  } else {
    if (group_w) return launch(std::integral_constant<int, W_SMEM_GROUP>{});
    return launch(std::integral_constant<int, W_SMEM_THREAD>{});
  }
}

template <int N, int VARIANT, int WMODE, bool NORM, bool STATS, bool SCREEN>
static int launch_rollout_one(const RolloutArgs& a, cudaStream_t st) {
  return launch_rollout_grid(rollout_kernel<N, VARIANT, WMODE, NORM, STATS, SCREEN ? SCREEN_BUILTIN : SCREEN_NONE, false>,
                             rollout_smem<N, VARIANT, WMODE, STATS>(), a.B, 1, st, a, NoCostForms{});
}

// The screened kernels with cost forms or models exist for what per-step screening supports on the thread kernel:
// gym dynamics, linear policies, ARS V1 without statistics.
template <int N>
int launch_rollout_screened_n(const RolloutArgs& a, const SimModels* models, const CostForms* forms,
                              const Backup* backup, int lookahead, const RolloutFlags& f, cudaStream_t st) {
  if (f.variant != SWM_DYN_GYM || !f.linear || !f.screen || f.norm || f.stats) return SWM_ERR_UNSUPPORTED;
  return with_policy_storage<N>(f.group_w, [&](auto w) {
    constexpr int WMODE = decltype(w)::value;
    const size_t smem = rollout_smem<N, 0, WMODE, false>();
    if (backup && lookahead > 0 && !forms) {
      SimModelsBackupLookahead mbl;
      mbl.models = *models;
      mbl.backup = *backup;
      mbl.lookahead = lookahead;
      return launch_rollout_grid(rollout_kernel<N, 0, WMODE, false, false, SCREEN_LOOKAHEAD, false>, smem, a.B, 1, st,
                                 a, mbl);
    }
    if (backup && lookahead > 0) {
      SimModelsFormsBackupLookahead mfbl;
      mfbl.models = *models;
      mfbl.forms = *forms;
      mfbl.backup = *backup;
      mfbl.lookahead = lookahead;
      return launch_rollout_grid(rollout_kernel<N, 0, WMODE, false, false, SCREEN_LOOKAHEAD_AFFINE, false>, smem, a.B,
                                 1, st, a, mfbl);
    }
    if (backup && !forms) {
      SimModelsBackup mb;
      mb.models = *models;
      mb.backup = *backup;
      return launch_rollout_grid(rollout_kernel<N, 0, WMODE, false, false, SCREEN_SHIELD, false>, smem, a.B, 1, st, a,
                                 mb);
    }
    if (backup) {
      SimModelsFormsBackup mfb;
      mfb.models = *models;
      mfb.forms = *forms;
      mfb.backup = *backup;
      return launch_rollout_grid(rollout_kernel<N, 0, WMODE, false, false, SCREEN_SHIELD_AFFINE, false>, smem, a.B, 1,
                                 st, a, mfb);
    }
    if (!models)
      return launch_rollout_grid(rollout_kernel<N, 0, WMODE, false, false, SCREEN_AFFINE, false>, smem, a.B, 1, st, a,
                                 *forms);
    if (!forms)
      return launch_rollout_grid(rollout_kernel<N, 0, WMODE, false, false, SCREEN_ENSEMBLE, false>, smem, a.B, 1, st, a,
                                 *models);
    SimModelsForms mf;
    mf.models = *models;
    mf.forms = *forms;
    return launch_rollout_grid(rollout_kernel<N, 0, WMODE, false, false, SCREEN_ENSEMBLE_AFFINE, false>, smem, a.B, 1,
                               st, a, mf);
  });
}

// The model-set kernels exist for the simulator rollouts of ARS screening: gym dynamics, linear policies, V1 or V2
// without statistics, no per-step screening.
template <int N>
int launch_rollout_models_n(const RolloutArgs& a, const SimModels& models, const RolloutFlags& f, cudaStream_t st) {
  if (f.variant != SWM_DYN_GYM || !f.linear || f.screen || f.stats) return SWM_ERR_UNSUPPORTED;
  return with_policy_storage<N>(f.group_w, [&](auto w) {
    constexpr int WMODE = decltype(w)::value;
    const size_t smem = rollout_smem<N, 0, WMODE, false>();
    if (f.norm)
      return launch_rollout_grid(rollout_kernel<N, 0, WMODE, true, false, SCREEN_NONE, true>, smem, a.B, models.M, st,
                                 a, models);
    return launch_rollout_grid(rollout_kernel<N, 0, WMODE, false, false, SCREEN_NONE, true>, smem, a.B, models.M, st, a,
                               models);
  });
}

template <int N, int WMODE>
static int launch_rollout_linear(const RolloutArgs& a, const RolloutFlags& f, cudaStream_t st) {
  if (f.variant == SWM_DYN_RLGLUE) {
    if (f.norm || f.stats || f.screen) return SWM_ERR_UNSUPPORTED;
    return launch_rollout_one<N, 1, WMODE, false, false, false>(a, st);
  }
  if (f.screen) {
    if (f.norm || f.stats) return SWM_ERR_UNSUPPORTED;
    return launch_rollout_one<N, 0, WMODE, false, false, true>(a, st);
  }
  if (f.norm && f.stats) return launch_rollout_one<N, 0, WMODE, true, true, false>(a, st);
  if (f.norm) return launch_rollout_one<N, 0, WMODE, true, false, false>(a, st);
  if (f.stats) return SWM_ERR_UNSUPPORTED;  // statistics are an ARS-V2 feature
  return launch_rollout_one<N, 0, WMODE, false, false, false>(a, st);
}

template <int N>
int launch_rollout_n(const RolloutArgs& a, const RolloutFlags& f, cudaStream_t st) {
  if (!f.linear) {
    if (f.norm || f.stats || f.screen) return SWM_ERR_UNSUPPORTED;
    return f.variant == SWM_DYN_GYM ? launch_rollout_one<N, 0, W_NONE, false, false, false>(a, st)
                                    : launch_rollout_one<N, 1, W_NONE, false, false, false>(a, st);
  }
  return with_policy_storage<N>(f.group_w, [&](auto w) { return launch_rollout_linear<N, decltype(w)::value>(a, f, st); });
}

template <int N>
int launch_step_n(const Phys& P, int variant, bool acc_only, const double* state_in,
                  const double* action, double* out, double* reward, long long B, cudaStream_t st) {
  const unsigned blocks = (unsigned)((B + kStepBlock - 1) / kStepBlock);
  if (variant == SWM_DYN_GYM) {
    if (acc_only) step_kernel<N, 0, true><<<blocks, kStepBlock, 0, st>>>(P, state_in, action, out, reward, B);
    else step_kernel<N, 0, false><<<blocks, kStepBlock, 0, st>>>(P, state_in, action, out, reward, B);
  } else {
    if (acc_only) step_kernel<N, 1, true><<<blocks, kStepBlock, 0, st>>>(P, state_in, action, out, reward, B);
    else step_kernel<N, 1, false><<<blocks, kStepBlock, 0, st>>>(P, state_in, action, out, reward, B);
  }
  return cudaPeekAtLastError() == cudaSuccess ? SWM_OK : SWM_ERR_CUDA;  // capi.cu note_launch reads + clears it
}

template <int N>
int launch_step_models_n(const PhysSet& set, long long envs_per_model, const double* state_in,
                         const double* action, double* out, double* reward, long long B, cudaStream_t st) {
  const unsigned blocks = (unsigned)((B + kStepBlock - 1) / kStepBlock);
  step_models_kernel<N><<<blocks, kStepBlock, 0, st>>>(set, envs_per_model, state_in, action, out, reward, B);
  return cudaPeekAtLastError() == cudaSuccess ? SWM_OK : SWM_ERR_CUDA;
}

template int launch_step_models_n<SWM_INSTANTIATE_N>(const PhysSet&, long long, const double*, const double*,
                                                     double*, double*, long long, cudaStream_t);
template int launch_step_n<SWM_INSTANTIATE_N>(const Phys&, int, bool, const double*, const double*,
                                              double*, double*, long long, cudaStream_t);
template int launch_rollout_n<SWM_INSTANTIATE_N>(const RolloutArgs&, const RolloutFlags&, cudaStream_t);
template int launch_rollout_screened_n<SWM_INSTANTIATE_N>(const RolloutArgs&, const SimModels*, const CostForms*,
                                                          const Backup*, int, const RolloutFlags&, cudaStream_t);
template int launch_rollout_models_n<SWM_INSTANTIATE_N>(const RolloutArgs&, const SimModels&, const RolloutFlags&,
                                                        cudaStream_t);

#endif  // SWM_INSTANTIATE_N

}  // namespace swm
