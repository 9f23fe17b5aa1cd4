// Host-side template dispatch for one segment count N.  Each rollout_nK.cu translation unit
// instantiates launch_*_n<K> so the (N x mode) kernel matrix compiles in parallel.
#pragma once
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
template <int N> int launch_rollout_costed_n(const RolloutArgs& a, const CostForms& forms, const RolloutFlags& f,
                                             cudaStream_t st);
template <int N> int launch_rollout_ensemble_n(const RolloutArgs& a, const SimModels& models, const CostForms* forms,
                                               const RolloutFlags& f, cudaStream_t st);
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

template <int N, int VARIANT, int WMODE, bool NORM, bool STATS, bool SCREEN>
static int launch_rollout_one(const RolloutArgs& a, cudaStream_t st) {
  return launch_rollout_grid(rollout_kernel<N, VARIANT, WMODE, NORM, STATS, SCREEN ? SCREEN_BUILTIN : SCREEN_NONE, false>,
                             rollout_smem<N, VARIANT, WMODE, STATS>(), a.B, 1, st, a, NoCostForms{});
}

template <int N, int WMODE>
static int launch_rollout_costed_one(const RolloutArgs& a, const CostForms& forms, cudaStream_t st) {
  return launch_rollout_grid(rollout_kernel<N, 0, WMODE, false, false, SCREEN_AFFINE, false>,
                             rollout_smem<N, 0, WMODE, false>(), a.B, 1, st, a, forms);
}

// The costed kernel exists for what per-step screening supports on the thread kernel: gym dynamics, linear
// policies, ARS V1 without statistics.
template <int N>
int launch_rollout_costed_n(const RolloutArgs& a, const CostForms& forms, const RolloutFlags& f, cudaStream_t st) {
  constexpr int WS = (N - 1) * (2 * N + 2);
  if (f.variant != SWM_DYN_GYM || !f.linear || !f.screen || f.norm || f.stats) return SWM_ERR_UNSUPPORTED;
  if constexpr (WS <= kRegPolicyMax) {
    return launch_rollout_costed_one<N, W_REG>(a, forms, st);
  } else {
    if (f.group_w) return launch_rollout_costed_one<N, W_SMEM_GROUP>(a, forms, st);
    return launch_rollout_costed_one<N, W_SMEM_THREAD>(a, forms, st);
  }
}

// Ensemble screening: SCREEN_ENSEMBLE with the built-in cost (forms == nullptr), else SCREEN_ENSEMBLE_AFFINE.
template <int N, int WMODE>
static int launch_rollout_ensemble_one(const RolloutArgs& a, const SimModels& models, const CostForms* forms,
                                       cudaStream_t st) {
  const size_t smem = rollout_smem<N, 0, WMODE, false>();
  if (!forms) return launch_rollout_grid(rollout_kernel<N, 0, WMODE, false, false, SCREEN_ENSEMBLE, false>, smem, a.B,
                                         1, st, a, models);
  SimModelsForms mf;
  mf.models = models;
  mf.forms = *forms;
  return launch_rollout_grid(rollout_kernel<N, 0, WMODE, false, false, SCREEN_ENSEMBLE_AFFINE, false>, smem, a.B, 1, st,
                             a, mf);
}

// Same configurations as the costed kernel.
template <int N>
int launch_rollout_ensemble_n(const RolloutArgs& a, const SimModels& models, const CostForms* forms,
                              const RolloutFlags& f, cudaStream_t st) {
  constexpr int WS = (N - 1) * (2 * N + 2);
  if (f.variant != SWM_DYN_GYM || !f.linear || !f.screen || f.norm || f.stats) return SWM_ERR_UNSUPPORTED;
  if constexpr (WS <= kRegPolicyMax) {
    return launch_rollout_ensemble_one<N, W_REG>(a, models, forms, st);
  } else {
    if (f.group_w) return launch_rollout_ensemble_one<N, W_SMEM_GROUP>(a, models, forms, st);
    return launch_rollout_ensemble_one<N, W_SMEM_THREAD>(a, models, forms, st);
  }
}

template <int N, int WMODE>
static int launch_rollout_models_one(const RolloutArgs& a, const SimModels& models, bool norm, cudaStream_t st) {
  const size_t smem = rollout_smem<N, 0, WMODE, false>();
  if (norm)
    return launch_rollout_grid(rollout_kernel<N, 0, WMODE, true, false, SCREEN_NONE, true>, smem, a.B, models.M, st, a,
                               models);
  return launch_rollout_grid(rollout_kernel<N, 0, WMODE, false, false, SCREEN_NONE, true>, smem, a.B, models.M, st, a,
                             models);
}

// The model-set kernels exist for the simulator rollouts of ARS screening: gym dynamics, linear policies, V1 or V2
// without statistics, no per-step screening.
template <int N>
int launch_rollout_models_n(const RolloutArgs& a, const SimModels& models, const RolloutFlags& f, cudaStream_t st) {
  constexpr int WS = (N - 1) * (2 * N + 2);
  if (f.variant != SWM_DYN_GYM || !f.linear || f.screen || f.stats) return SWM_ERR_UNSUPPORTED;
  if constexpr (WS <= kRegPolicyMax) {
    return launch_rollout_models_one<N, W_REG>(a, models, f.norm, st);
  } else {
    if (f.group_w) return launch_rollout_models_one<N, W_SMEM_GROUP>(a, models, f.norm, st);
    return launch_rollout_models_one<N, W_SMEM_THREAD>(a, models, f.norm, st);
  }
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
  constexpr int WS = (N - 1) * (2 * N + 2);
  if (!f.linear) {
    if (f.norm || f.stats || f.screen) return SWM_ERR_UNSUPPORTED;
    return f.variant == SWM_DYN_GYM ? launch_rollout_one<N, 0, W_NONE, false, false, false>(a, st)
                                    : launch_rollout_one<N, 1, W_NONE, false, false, false>(a, st);
  }
  if constexpr (WS <= kRegPolicyMax) {
    return launch_rollout_linear<N, W_REG>(a, f, st);
  } else {
    if (f.group_w) return launch_rollout_linear<N, W_SMEM_GROUP>(a, f, st);
    return launch_rollout_linear<N, W_SMEM_THREAD>(a, f, st);
  }
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
template int launch_rollout_costed_n<SWM_INSTANTIATE_N>(const RolloutArgs&, const CostForms&, const RolloutFlags&,
                                                        cudaStream_t);
template int launch_rollout_ensemble_n<SWM_INSTANTIATE_N>(const RolloutArgs&, const SimModels&, const CostForms*,
                                                          const RolloutFlags&, cudaStream_t);
template int launch_rollout_models_n<SWM_INSTANTIATE_N>(const RolloutArgs&, const SimModels&, const RolloutFlags&,
                                                        cudaStream_t);

#endif  // SWM_INSTANTIATE_N

}  // namespace swm
