// Batched step kernel and the persistent fused H-step rollout kernel.
// One thread owns one environment; the state (2n+2 doubles), its sines/cosines and (for
// n <= 5) the environment's own perturbed policy live in registers for the whole rollout.
// Nothing but the final return (8 B/env), optional final state and optional trajectory is
// written to HBM.  Per-step screening (every ScreenMode) is one block of the step loop with one
// freeze path, and the real observation is formed once for the affine cost and the moments.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/swimmer_ars.h"
#include "dynamics.cuh"
#include "philox.cuh"

#ifndef SWM_ROLLOUT_MIN_BLOCKS
#define SWM_ROLLOUT_MIN_BLOCKS 1  // CTAs/SM the register allocator must leave room for
#endif

namespace swm {

constexpr int kStepBlock = 128;
constexpr int kRolloutBlock = 64;  // threads per CTA of the rollout kernel (2 warps)
constexpr int kRegPolicyMax = 32;  // largest policy (doubles) kept in registers: n <= 4
constexpr int kRegStatsMaxObs = 16; // V2 moment accumulators stay in registers up to n = 7; above, they
                                    // live in shared memory (one column per thread)
#ifndef SWM_FACT_SMEM_MIN_N
#define SWM_FACT_SMEM_MIN_N 8       // from this chain length on, the joint factorisation (5 doubles per joint) of
#endif                              // the gym dynamics is kept in shared memory between its two sweeps
constexpr int kFactSmemMinN = SWM_FACT_SMEM_MIN_N;
template <int N, int VARIANT> struct FactSmem {
  static constexpr bool on = (VARIANT == 0) && (N >= kFactSmemMinN);
  static constexpr int doubles = on ? (kFactSmemRhsOnly ? 2 : 5) * (N - 1) : 0;  // per thread
};

// Where the per-environment policy lives during a rollout.
enum WMode {
  W_NONE = 0,        // fixed actions
  W_REG = 1,         // registers (n <= 5: at most 48 doubles)
  W_SMEM_THREAD = 2, // shared memory, one column per thread: sW[e * BLOCK + tid]
  W_SMEM_GROUP = 3   // shared memory, one copy per warp (rollouts_per_policy % 32 == 0): broadcast
};

struct RolloutArgs {
  Phys real;
  Phys sim;  // screening model
  int H;
  int R;  // rollouts per policy
  int policy_mode;
  int clip;
  long long B;
  const double* actions;
  const double* policies;
  const double* deltas;
  const int* dir_mask;
  double nu;
  double init_perturb;
  unsigned long long seed;
  unsigned int iteration, dir0;
  const unsigned int* iter_dev;  // optional device counter added to `iteration`
  int dist;
  const double* mean;
  const double* inv_sigma;
  const double* init_state;
  long long init_count;
  double* returns;
  double* final_state;
  double* trajectory;
  double* stats_partial;
  const double* stats_pivot;
  double sim_thresh, real_thresh;
  int* violations;
  int* frozen_at;
  int accumulate;  // returns[e] += instead of =
};

// ---------------------------------------------------------------------------------------------
// step / accelerations
// ---------------------------------------------------------------------------------------------
template <int N, int VARIANT, bool ACC_ONLY>
__global__ void __launch_bounds__(kStepBlock)
step_kernel(Phys P, const double* state_in, const double* __restrict__ action,
            double* state_out, double* __restrict__ reward, long long B) {  // state_out may alias state_in
  constexpr int NO = 2 * N + 2, NA = N - 1;
  const long long e = (long long)blockIdx.x * kStepBlock + threadIdx.x;
  if (e >= B) return;
  const double2* sp = reinterpret_cast<const double2*>(state_in + e * NO);
  double gdx, gdy, th[N], thd[N], u[NA > 0 ? NA : 1];
  {
    const double2 g = sp[0];
    gdx = g.x; gdy = g.y;
#pragma unroll
    for (int i = 0; i < N; ++i) { const double2 v = sp[1 + i]; th[i] = v.x; thd[i] = v.y; }
#pragma unroll
    for (int a = 0; a < NA; ++a) u[a] = action[e * NA + a];
  }
  if (ACC_ONLY) {
    double s[N], c[N], gddx, gddy, thdd[N];
#pragma unroll
    for (int i = 0; i < N; ++i) sincos(th[i], &s[i], &c[i]);
    if (VARIANT == 0) {
#pragma unroll
      for (int a = 0; a < NA; ++a) u[a] *= P.u_scale;
      gym_accel<N>(P, s, c, gdx, gdy, thd, u, gddx, gddy, thdd);
      gddx *= P.gdd_c;
      gddy *= P.gdd_c;
    } else {
      rlglue_accelerations<N>(P, s, c, gdx, gdy, thd, u, gddx, gddy, thdd);
    }
    double* o = state_out + e * (N + 2);
    o[0] = gddx; o[1] = gddy;
#pragma unroll
    for (int i = 0; i < N; ++i) o[2 + i] = thdd[i];
    return;
  }
  const double r = swimmer_step<N, VARIANT>(P, gdx, gdy, th, thd, u);
  double2* op = reinterpret_cast<double2*>(state_out + e * NO);
  op[0] = make_double2(gdx, gdy);
#pragma unroll
  for (int i = 0; i < N; ++i) op[1 + i] = make_double2(th[i], thd[i]);
  if (reward) reward[e] = r;
}

// Several models in one launch (Estimator.I over a CMA-ES generation): the models travel in the
// kernel-argument constant bank, env e uses model e / envs_per_model.
struct PhysSet {
  Phys p[SWM_MAX_MODELS_PER_STEP];
};

template <int N>
__global__ void __launch_bounds__(kStepBlock)
step_models_kernel(const __grid_constant__ PhysSet set, long long envs_per_model,
                   const double* state_in, const double* __restrict__ action,
                   double* state_out, double* __restrict__ reward, long long B) {  // state_out may alias state_in
  constexpr int NO = 2 * N + 2, NA = N - 1;
  const long long e = (long long)blockIdx.x * kStepBlock + threadIdx.x;
  if (e >= B) return;
  const Phys& P = set.p[e / envs_per_model];
  const double2* sp = reinterpret_cast<const double2*>(state_in + e * NO);
  double gdx, gdy, th[N], thd[N], u[NA > 0 ? NA : 1];
  const double2 g = sp[0];
  gdx = g.x; gdy = g.y;
#pragma unroll
  for (int i = 0; i < N; ++i) { const double2 v = sp[1 + i]; th[i] = v.x; thd[i] = v.y; }
#pragma unroll
  for (int a = 0; a < NA; ++a) u[a] = action[e * NA + a];
  const double r = swimmer_step<N, 0>(P, gdx, gdy, th, thd, u);
  double2* op = reinterpret_cast<double2*>(state_out + e * NO);
  op[0] = make_double2(gdx, gdy);
#pragma unroll
  for (int i = 0; i < N; ++i) op[1 + i] = make_double2(th[i], thd[i]);
  if (reward) reward[e] = r;
}

// ---------------------------------------------------------------------------------------------
// fused rollout
// ---------------------------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ double cost_max_abs_thd(const double (&thd)[N]) {
  // safe_ars/experiment.py:44  np.max(|obs[3+2i]|); NaN propagates like np.max.  The sign-stripped bit
  // patterns of doubles order like their magnitudes (NaN above everything), so the maximum is taken on
  // the integer pipe and the FP64 unit only sees the final comparison with the threshold.
  long long m = 0;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const long long b = __double_as_longlong(thd[i]) & 0x7fffffffffffffffLL;
    m = b > m ? b : m;
  }
  return __longlong_as_double(m);
}

// User-defined state cost of per-step screening: cost(obs) = max_j (A_j . obs + b_j) over J forms.  Row j holds
// A_j (2n+2 entries) followed by b_j; the rows have the stride of the longest chain so that one type serves every n.
constexpr int kFormStride = 2 * SWM_MAX_SEGMENTS + 3;
struct CostForms {
  double row[SWM_MAX_COST_FORMS][kFormStride];
  int J;  // 1..SWM_MAX_COST_FORMS
};

// x(k) yields observation entry k.
template <int NO, typename Obs>
__device__ __forceinline__ double cost_max_affine(const CostForms& f, const Obs& x) {
  // NaN if any form is NaN, like np.max (fmax would drop it).  The forms are a warp-uniform kernel argument: the
  // coefficients are read from the constant bank, one form at a time.
  double m = __longlong_as_double(0xfff0000000000000LL);  // -inf
#pragma unroll 1
  for (int j = 0; j < f.J; ++j) {
    const double* r = f.row[j];
    double v = r[NO];
#pragma unroll
    for (int k = 0; k < NO; ++k) v = fma(r[k], x(k), v);
    m = (m == m && !(v <= m)) ? v : m;
  }
  return m;
}

// Screening modes of the rollout kernel: none, the built-in cost max_i |thd_i|, or max-of-affine forms, judged by
// the simulator model of RolloutArgs::sim or (ENSEMBLE*) by every model of an ensemble.
// SHIELD*: the ensemble modes with a backup action that is tried when the policy's action is judged unsafe.
// LOOKAHEAD*: the shield modes judging an action by K further simulator steps of the backup after it.
enum ScreenMode {
  SCREEN_NONE = 0, SCREEN_BUILTIN = 1, SCREEN_AFFINE = 2, SCREEN_ENSEMBLE = 3, SCREEN_ENSEMBLE_AFFINE = 4,
  SCREEN_SHIELD = 5, SCREEN_SHIELD_AFFINE = 6, SCREEN_LOOKAHEAD = 7, SCREEN_LOOKAHEAD_AFFINE = 8
};

// The simulator models of ensemble screening (M = 1..SWM_MAX_SIM_MODELS; entries from M on are not read).
struct SimModels {
  int M;
  Phys p[SWM_MAX_SIM_MODELS];
};
struct SimModelsForms {
  SimModels models;
  CostForms forms;
};

// The backup action of the shield, b = W . obs + u0 of the raw observation (row k of W: action k; entries past
// n-1 actions and 2n+2 observations are not read), and the per-environment count of steps that took it.
struct Backup {
  double W[SWM_MAX_SEGMENTS - 1][2 * SWM_MAX_SEGMENTS + 2];
  double u0[SWM_MAX_SEGMENTS - 1];
  int* overrides;  // device [B] or nullptr
};
struct SimModelsBackup {
  SimModels models;
  Backup backup;
};
struct SimModelsFormsBackup {
  SimModels models;
  CostForms forms;
  Backup backup;
};
// The lookahead shield: the shield's arguments and the number K >= 1 of backup steps after a judged action.
struct SimModelsBackupLookahead {
  SimModels models;
  Backup backup;
  int lookahead;
};
struct SimModelsFormsBackupLookahead {
  SimModels models;
  CostForms forms;
  Backup backup;
  int lookahead;
};

// Type of the rollout kernel's second argument: the cost forms and / or the simulator models of the screening
// mode, an empty struct without either.  MODELS (model-set mode, unscreened only): the models whose physics the
// rollouts run, one per CTA row blockIdx.y; the lane-split kernels take the same argument.
struct NoCostForms {};
template <int SCREEN, bool MODELS = false> struct ScreenForms { using type = NoCostForms; };
template <> struct ScreenForms<SCREEN_AFFINE> { using type = CostForms; };
template <> struct ScreenForms<SCREEN_ENSEMBLE> { using type = SimModels; };
template <> struct ScreenForms<SCREEN_ENSEMBLE_AFFINE> { using type = SimModelsForms; };
template <> struct ScreenForms<SCREEN_SHIELD> { using type = SimModelsBackup; };
template <> struct ScreenForms<SCREEN_SHIELD_AFFINE> { using type = SimModelsFormsBackup; };
template <> struct ScreenForms<SCREEN_LOOKAHEAD> { using type = SimModelsBackupLookahead; };
template <> struct ScreenForms<SCREEN_LOOKAHEAD_AFFINE> { using type = SimModelsFormsBackupLookahead; };
template <> struct ScreenForms<SCREEN_NONE, true> { using type = SimModels; };

// The physics of a rollout: RolloutArgs::real, or in the model-set mode model blockIdx.y (warp- and CTA-uniform, read
// from the constant bank through that index).  Rollout e of model m writes its outputs at row m * B + e.
template <bool MODELS, typename F>
__device__ __forceinline__ const Phys& rollout_model(const RolloutArgs& a, const F& f) {
  if constexpr (MODELS) return f.p[blockIdx.y];
  else return a.real;
}
template <bool MODELS>
__device__ __forceinline__ long long output_row(const RolloutArgs& a, long long e) {
  return MODELS ? (long long)blockIdx.y * a.B + e : e;
}

__device__ __forceinline__ const CostForms& cost_forms_of(const CostForms& f) { return f; }
__device__ __forceinline__ const CostForms& cost_forms_of(const SimModelsForms& f) { return f.forms; }
__device__ __forceinline__ const SimModels& sim_models_of(const SimModels& s) { return s; }
__device__ __forceinline__ const SimModels& sim_models_of(const SimModelsForms& s) { return s.models; }
__device__ __forceinline__ const CostForms& cost_forms_of(const SimModelsFormsBackup& f) { return f.forms; }
__device__ __forceinline__ const SimModels& sim_models_of(const SimModelsBackup& s) { return s.models; }
__device__ __forceinline__ const SimModels& sim_models_of(const SimModelsFormsBackup& s) { return s.models; }
__device__ __forceinline__ const Backup& backup_of(const SimModelsBackup& s) { return s.backup; }
__device__ __forceinline__ const Backup& backup_of(const SimModelsFormsBackup& s) { return s.backup; }
__device__ __forceinline__ const CostForms& cost_forms_of(const SimModelsFormsBackupLookahead& f) { return f.forms; }
__device__ __forceinline__ const SimModels& sim_models_of(const SimModelsBackupLookahead& s) { return s.models; }
__device__ __forceinline__ const SimModels& sim_models_of(const SimModelsFormsBackupLookahead& s) { return s.models; }
__device__ __forceinline__ const Backup& backup_of(const SimModelsBackupLookahead& s) { return s.backup; }
__device__ __forceinline__ const Backup& backup_of(const SimModelsFormsBackupLookahead& s) { return s.backup; }

// The judgement of the ensemble modes by one simulator model P: one simulator step with the action `act` from the
// state (gdx, gdy, th, w) with sines s and cosines c, unsafe unless cost <= sim_thresh (a NaN cost is unsafe).
template <int N, int FS, bool AFFINE, typename F>
__device__ __forceinline__ bool model_unsafe(const F& forms, const Phys& P, double sim_thresh, double gdx, double gdy,
                                             const double (&th)[N], const double (&s)[N], const double (&c)[N],
                                             const double (&w)[N], const double (&act)[N > 1 ? N - 1 : 1],
                                             double* sF) {
  constexpr int NA = N - 1, NO = 2 * N + 2;
  double sut[NA > 0 ? NA : 1], sgddx, sgddy, sthdd[N];
#pragma unroll
  for (int k = 0; k < NA; ++k) sut[k] = act[k] * P.u_scale;
  gym_accel<N, FS>(P, s, c, gdx, gdy, w, sut, sgddx, sgddy, sthdd, sF);
  double sim_cost;
  if constexpr (AFFINE) {
    auto so = [&](int k) {
      if (k < 2) return fma(P.h_gdd_c, k == 0 ? sgddx : sgddy, k == 0 ? gdx : gdy);
      const int i = (k - 2) / 2;
      return (k & 1) ? fma(P.h, sthdd[i], w[i]) : fma(P.h, w[i], th[i]);
    };
    sim_cost = cost_max_affine<NO>(cost_forms_of(forms), so);
  } else {
    double sthd[N];
#pragma unroll
    for (int i = 0; i < N; ++i) sthd[i] = fma(P.h, sthdd[i], w[i]);
    sim_cost = cost_max_abs_thd<N>(sthd);
  }
  return !(sim_cost <= sim_thresh);
}

// Sines and cosines of the lookahead's simulated states: 1 tracks them by the rotation of gym_step_tracked, with its
// exact re-evaluation every 64 lookahead steps; 0 evaluates them with sincos at every lookahead step (DESIGN §3.2).
#ifndef SWM_LOOKAHEAD_TRACKED_TRIG
#define SWM_LOOKAHEAD_TRACKED_TRIG 1
#endif

// The backup action b = W_b . x + u0 of the observation x = (gdx, gdy, th, thd), clipped to +-max_u if `clip`.
template <int N>
__device__ __forceinline__ void backup_action(const Backup& bk, double gdx, double gdy, const double (&th)[N],
                                              const double (&thd)[N], bool clip, double max_u,
                                              double (&b)[N > 1 ? N - 1 : 1]) {
  constexpr int NA = N - 1, NO = 2 * N + 2;
#pragma unroll
  for (int k = 0; k < NA; ++k) b[k] = 0.0;
#pragma unroll
  for (int j = 0; j < NO; ++j) {
    const double x = (j == 0) ? gdx : (j == 1) ? gdy : ((j & 1) ? thd[(j - 3) / 2] : th[(j - 2) / 2]);
#pragma unroll
    for (int k = 0; k < NA; ++k) b[k] = fma(x, bk.W[k][j], b[k]);
  }
#pragma unroll
  for (int k = 0; k < NA; ++k) {
    b[k] += bk.u0[k];
    if (clip) b[k] = fmin(fmax(b[k], -max_u), max_u);
  }
}

// The judgement of the lookahead modes by one simulator model P: x_1 = f(x_0, act) from the state x_0 = (gdx, gdy, th,
// w) with sines s and cosines c, then x_{j+1} = f(x_j, backup(x_j)) for j = 1..K; unsafe unless cost(x_j) <=
// sim_thresh for every j = 1..K+1 (a NaN cost is unsafe), and it stops at the first unsafe cost.  Its first step is
// model_unsafe's judgement, with the same operations; the K backup steps advance a private copy of the state.  The
// backup is clipped to the real model's max_u, as in the real step.
template <int N, int FS, bool AFFINE, typename F>
__device__ __forceinline__ bool model_unsafe_lookahead(const F& forms, const Phys& P, double sim_thresh, int K,
                                                       bool clip, double max_u, double gdx, double gdy,
                                                       const double (&th0)[N], const double (&s0)[N],
                                                       const double (&c0)[N], const double (&w0)[N],
                                                       const double (&act)[N > 1 ? N - 1 : 1], double* sF) {
  constexpr int NA = N - 1, NO = 2 * N + 2;
  double th[N], w[N], s[N], c[N], ut[NA > 0 ? NA : 1];
#pragma unroll
  for (int i = 0; i < N; ++i) { th[i] = th0[i]; w[i] = w0[i]; s[i] = s0[i]; c[i] = c0[i]; }
#pragma unroll
  for (int k = 0; k < NA; ++k) ut[k] = act[k] * P.u_scale;
#pragma unroll 1
  for (int j = 0;; ++j) {
    if constexpr (SWM_LOOKAHEAD_TRACKED_TRIG) {
      gym_step_tracked<N, FS>(P, gdx, gdy, th, w, s, c, ut, (j & 63) == 63, sF);
    } else {
      if (j > 0) {
#pragma unroll
        for (int i = 0; i < N; ++i) sincos(th[i], &s[i], &c[i]);
      }
      double psx, psy, thdd[N];
      gym_accel<N, FS>(P, s, c, gdx, gdy, w, ut, psx, psy, thdd, sF);
      gdx = fma(P.h_gdd_c, psx, gdx);
      gdy = fma(P.h_gdd_c, psy, gdy);
#pragma unroll
      for (int i = 0; i < N; ++i) {
        th[i] = fma(P.h, w[i], th[i]);
        w[i] = fma(P.h, thdd[i], w[i]);
      }
    }
    double cost;
    if constexpr (AFFINE)
      cost = cost_max_affine<NO>(cost_forms_of(forms), [&](int k) {
        return k == 0 ? gdx : k == 1 ? gdy : (k & 1) ? w[(k - 3) / 2] : th[(k - 2) / 2];
      });
    else
      cost = cost_max_abs_thd<N>(w);
    if (!(cost <= sim_thresh)) return true;
    if (j == K) return false;
    double b[NA > 0 ? NA : 1];
    backup_action<N>(backup_of(forms), gdx, gdy, th, w, clip, max_u, b);
#pragma unroll
    for (int k = 0; k < NA; ++k) ut[k] = b[k] * P.u_scale;
  }
}

// LINEAR: 0 fixed actions, 1 linear policy.  NORM: ARS V2 normalisation.  STATS: accumulate
// shifted first/second moments of every visited state.  SCREEN: per-step simulator screening (ScreenMode).
// With SCREEN_AFFINE the forms travel as the second kernel argument (5.9 KB of the constant bank), with
// SCREEN_ENSEMBLE the models (2.3 KB), with SCREEN_ENSEMBLE_AFFINE both (8.2 KB), and the SHIELD modes add the
// backup (1.7 KB, so at most 9.9 KB) and the LOOKAHEAD modes its length K; the other kernels' argument block grows by
// one empty byte only.  MODELS: the
// model-set mode (SCREEN_NONE, gym dynamics, no statistics, no trajectory), the models (2.3 KB) as the second
// argument.
template <int N, int VARIANT, int WMODE, bool NORM, bool STATS, int SCREEN, bool MODELS>
__global__ void __launch_bounds__(kRolloutBlock, SWM_ROLLOUT_MIN_BLOCKS)
rollout_kernel(const RolloutArgs a, const __grid_constant__ typename ScreenForms<SCREEN, MODELS>::type forms) {
  static_assert(!MODELS || (SCREEN == SCREEN_NONE && VARIANT == 0 && !STATS), "model set: unscreened gym rollouts");
  constexpr int NO = 2 * N + 2, NA = N - 1, WS = NA * NO;
  constexpr bool LINEAR = (WMODE != W_NONE);
  constexpr bool LOOKAHEAD = SCREEN == SCREEN_LOOKAHEAD || SCREEN == SCREEN_LOOKAHEAD_AFFINE;
  constexpr bool SHIELD = SCREEN == SCREEN_SHIELD || SCREEN == SCREEN_SHIELD_AFFINE || LOOKAHEAD;
  constexpr bool ENSEMBLE = SCREEN == SCREEN_ENSEMBLE || SCREEN == SCREEN_ENSEMBLE_AFFINE || SHIELD;
  constexpr bool AFFINE = SCREEN == SCREEN_AFFINE || SCREEN == SCREEN_ENSEMBLE_AFFINE || SCREEN == SCREEN_SHIELD_AFFINE ||
                          SCREEN == SCREEN_LOOKAHEAD_AFFINE;
  static_assert(!SHIELD || (VARIANT == 0 && LINEAR && !NORM && !STATS), "shield: gym dynamics, linear V1 policies");
  const Phys& P = rollout_model<MODELS>(a, forms);
  extern __shared__ __align__(16) double smem[];
  const int tid = threadIdx.x;
  const long long e0 = (long long)blockIdx.x * kRolloutBlock + tid;
  const bool active = e0 < a.B;
  const long long e = active ? e0 : a.B - 1;  // idle lanes shadow the last env, never store

  const unsigned int iteration = a.iteration + (a.iter_dev ? *a.iter_dev : 0u);

  // ---- initial state ----
  double gdx, gdy, th[N], thd[N];
  if (a.init_state) {
    const double* sp = a.init_state + (e % a.init_count) * NO;
    gdx = sp[0]; gdy = sp[1];
#pragma unroll
    for (int i = 0; i < N; ++i) { th[i] = sp[2 + 2 * i]; thd[i] = sp[3 + 2 * i]; }
  } else if (VARIANT == 0) {
    gdx = gdy = 0.0;
#pragma unroll
    for (int i = 0; i < N; ++i) { th[i] = 1.5707963267948966; thd[i] = 0.0; }
  } else {
    gdx = gdy = 0.001;
#pragma unroll
    for (int i = 0; i < N; ++i) { th[i] = 0.001; thd[i] = 0.001; }
  }

  if (a.init_perturb != 0.0) {
    // declared synthetic extension (BASELINE config 5): start = init + init_perturb * U[0,1),
    // Philox stream 1 keyed by the rollout index within the policy, so that every policy sees the
    // same R perturbed starts (common random numbers for the +/- pairs).
    const unsigned int r = (unsigned int)(e % a.R);
#pragma unroll
    for (int j = 0; j < NO; j += 2) {
      double d0, d1;
      philox_delta_pair(a.seed, iteration, r, 1u, (uint32_t)(j >> 1), SWM_DELTA_UNIFORM_01, d0, d1);
      if (j == 0) { gdx = fma(a.init_perturb, d0, gdx); gdy = fma(a.init_perturb, d1, gdy); }
      else { th[(j - 2) / 2] = fma(a.init_perturb, d0, th[(j - 2) / 2]);
             thd[(j - 2) / 2] = fma(a.init_perturb, d1, thd[(j - 2) / 2]); }
    }
  }

  // ---- policy ----
  double Wr[WMODE == W_REG ? WS : 1];
  double u[NA > 0 ? NA : 1];
  // warp-uniform vectors (V2 mean, moment pivot) are read from shared memory every step instead of
  // occupying 2(2n+2) registers per thread
  __shared__ double s_mu[NORM ? NO : 1], s_piv[STATS ? NO : 1];
  if (NORM || STATS) {
    if (NORM && tid < NO) s_mu[tid] = a.mean[tid];
    if (STATS && tid < NO) s_piv[tid] = a.stats_pivot[tid];
    __syncthreads();
  }
  double* sW = nullptr;  // W_SMEM_*: element j of this thread's policy at sW[j * wstride]
  int wstride = 1;
  if (WMODE == W_SMEM_THREAD) { sW = smem + tid; wstride = kRolloutBlock; }
  if (WMODE == W_SMEM_GROUP) { sW = smem + (tid >> 5) * WS; wstride = 1; }
  if (LINEAR) {
    const long long q = e / a.R;  // policy index
    const bool philox = a.policy_mode == SWM_POLICY_PHILOX;
    const bool from_mem = a.policy_mode == SWM_POLICY_DELTAS;
    const double* base = (philox || from_mem) ? a.policies : a.policies + q * WS;
    const double* dmem = from_mem ? a.deltas + (q >> 1) * WS : nullptr;
    const double sgn_nu = (q & 1) ? -a.nu : a.nu;
    const unsigned int dir = a.dir0 + (unsigned int)(q >> 1);
    auto make_pair = [&](int j, double& w0, double& w1) {
      w0 = base[j];
      w1 = (j + 1 < WS) ? base[j + 1] : 0.0;
      if (philox || from_mem) {
        double d0, d1 = 0.0;
        if (philox) {
          philox_delta_pair(a.seed, iteration, dir, 0u, (uint32_t)(j >> 1), a.dist, d0, d1);
        } else {
          d0 = dmem[j];
          if (j + 1 < WS) d1 = dmem[j + 1];
        }
        // policy +- nu*delta exactly as ars_agent.py:141-142 (product rounded, then added)
        w0 = __dadd_rn(w0, __dmul_rn(sgn_nu, d0));
        w1 = __dadd_rn(w1, __dmul_rn(sgn_nu, d1));
      }
      if (NORM) {  // policy @ diag(cov^-1/2), ars/environment.py:32-33
        w0 *= a.inv_sigma[j % NO];
        if (j + 1 < WS) w1 *= a.inv_sigma[(j + 1) % NO];
      }
    };
    if (WMODE == W_REG) {
#pragma unroll
      for (int j = 0; j < WS; j += 2) {
        double w0, w1;
        make_pair(j, w0, w1);
        Wr[j] = w0;
        if (j + 1 < WS) Wr[j + 1] = w1;
      }
    } else if (WMODE == W_SMEM_GROUP) {
      // the 32 lanes of the warp share the Philox calls of their common policy
#pragma unroll 1
      for (int j = 2 * (tid & 31); j < WS; j += 64) {
        double w0, w1;
        make_pair(j, w0, w1);
        sW[(j % NO) * NA + j / NO] = w0;  // [obs][action] (see the policy product in the step loop)
        if (j + 1 < WS) sW[((j + 1) % NO) * NA + (j + 1) / NO] = w1;
      }
    } else {
#pragma unroll 1
      for (int j = 0; j < WS; j += 2) {
        double w0, w1;
        make_pair(j, w0, w1);
        sW[j * wstride] = w0;
        if (j + 1 < WS) sW[(j + 1) * wstride] = w1;
      }
    }
    if (WMODE == W_SMEM_GROUP) __syncwarp();
  } else {
#pragma unroll
    for (int k = 0; k < NA; ++k) u[k] = a.actions[e * NA + k];
  }

  constexpr bool STATS_SMEM = STATS && (NO > kRegStatsMaxObs);
  constexpr bool STATS_REG = STATS && !STATS_SMEM;
  double s1[STATS_REG ? NO : 1], s2[STATS_REG ? NO : 1];
  // STATS_SMEM: accumulator j of this thread at sS[j * kRolloutBlock], j < 2*NO, after the policies
  double* sS = smem + tid;
  // gym dynamics of long chains: factorisation scratch, element k of this thread at sF[k * kRolloutBlock]
  constexpr int FS = FactSmem<N, VARIANT>::on ? kRolloutBlock : 0;
  double* sF = smem + tid;
  if (FS) {
    if (WMODE == W_SMEM_THREAD) sF += WS * kRolloutBlock;
    if (WMODE == W_SMEM_GROUP) sF += WS * (kRolloutBlock / 32);
    if (STATS_SMEM) sF += 2 * NO * kRolloutBlock;
  }
  if (STATS_SMEM) {
    if (WMODE == W_SMEM_THREAD) sS += WS * kRolloutBlock;
    if (WMODE == W_SMEM_GROUP) sS += WS * (kRolloutBlock / 32);
#pragma unroll
    for (int j = 0; j < 2 * NO; ++j) sS[j * kRolloutBlock] = 0.0;
  }
  if (STATS_REG) {
#pragma unroll
    for (int j = 0; j < NO; ++j) { s1[j] = 0.0; s2[j] = 0.0; }
  }

  // reward-constraint safe exploration (ars_agent.py:144-159): a screened-out direction is never
  // rolled out in the real world; its returns are NaN and it contributes no statistics.
  bool skipped = false;
  if (LINEAR && a.dir_mask) skipped = a.dir_mask[(e / a.R) >> 1] == 0;
  const int steps = skipped ? 0 : a.H;

  double ret = skipped ? __longlong_as_double(0x7ff8000000000000LL) : 0.0;
  double sgx = 0.0, sgy = 0.0;  // gym variant: sum_t Gdot_t
  int viol = 0, frozen = a.H, ovr = 0;
  double* traj = a.trajectory ? a.trajectory + e * NO : nullptr;
  const long long traj_step = a.B * NO;

  // gym variant: sines/cosines live in registers across steps (see gym_step_tracked)
  double sn[N], cs[N];
  double ut[NA > 0 ? NA : 1];  // torques scaled by 12/(m l^2)
  if (VARIANT == 0) {
#pragma unroll
    for (int i = 0; i < N; ++i) sincos(th[i], &sn[i], &cs[i]);
    if (!LINEAR) {
#pragma unroll
      for (int k = 0; k < NA; ++k) ut[k] = u[k] * P.u_scale;
    }
  }

  // SHIELD: this step is re-run with the backup action because the models rejected the policy's action
  bool backup_turn = false;
  for (int t = 0; t < steps; ++t) {
    if (LINEAR) {
      // action_k = sum_j W[k][j] * obs_j, observation-major: the NA accumulators advance together so
      // that consecutive DFMAs share the obs_j operand (served by the operand-reuse cache: a DFMA
      // with three fresh register sources issues every 3 cycles on B200, see profiles/r01b_summary.md)
      // and only one (normalised) observation is live at a time.  Each action still sums j = 0..NO-1
      // in order, exactly like np.matmul's row dot product in ars/environment.py:27-35.
      double acc[NA > 0 ? NA : 1];
#pragma unroll
      for (int k = 0; k < NA; ++k) acc[k] = 0.0;
      if constexpr (SHIELD) {
        if (backup_turn) {
          // the backup action b = W_b . obs + u0 of the raw observation, in the order of the policy's product; the
          // coefficients are warp-uniform kernel arguments, read from the constant bank like the cost forms
          const Backup& bk = backup_of(forms);
#pragma unroll
          for (int j = 0; j < NO; ++j) {
            const double x = (j == 0) ? gdx : (j == 1) ? gdy : ((j & 1) ? thd[(j - 3) / 2] : th[(j - 2) / 2]);
#pragma unroll
            for (int k = 0; k < NA; ++k) acc[k] = fma(x, bk.W[k][j], acc[k]);
          }
#pragma unroll
          for (int k = 0; k < NA; ++k) acc[k] += bk.u0[k];
        }
      }
#pragma unroll
      for (int j = 0; j < NO && !(SHIELD && backup_turn); ++j) {
        double x = (j == 0) ? gdx : (j == 1) ? gdy : ((j & 1) ? thd[(j - 3) / 2] : th[(j - 2) / 2]);
        if (NORM) x -= s_mu[j];
#pragma unroll
        for (int k = 0; k < NA; ++k) {
          double w;
          if (WMODE == W_REG) w = Wr[k * NO + j];
          else if (WMODE == W_SMEM_GROUP) w = sW[j * NA + k];  // warp-uniform broadcast, [obs][action]
          else w = sW[(k * NO + j) * wstride];
          acc[k] = fma(x, w, acc[k]);
        }
        // shared-memory policies: keep at most one column of coefficients in flight, otherwise the
        // scheduler hoists all (n-1)(2n+2) loads and spills
        if (WMODE == W_SMEM_THREAD || WMODE == W_SMEM_GROUP) asm volatile("" ::: "memory");
      }
#pragma unroll
      for (int k = 0; k < NA; ++k) {
        double v = acc[k];
        if (a.clip) v = fmin(fmax(v, -P.max_u), P.max_u);
        u[k] = v;
        if (VARIANT == 0) ut[k] = v * P.u_scale;
      }
    }
    if constexpr (SCREEN != SCREEN_NONE) {
      // Safe_ARS.isSafe (safe_ars/ars.py:111-122): one simulator step from the current state.  The
      // simulator starts from the same angles, so it shares this step's sines/cosines and needs only
      // its own accelerations.
      bool unsafe = false;
      if constexpr (!ENSEMBLE) {
        double sut[NA > 0 ? NA : 1], sgddx, sgddy, sthdd[N];
#pragma unroll
        for (int k = 0; k < NA; ++k) sut[k] = u[k] * a.sim.u_scale;
        gym_accel<N, FS>(a.sim, sn, cs, gdx, gdy, thd, sut, sgddx, sgddy, sthdd, sF);
        double sim_cost;
        if constexpr (AFFINE) {
          // the whole simulated observation, explicit Euler as in gym_step_tracked.  Held in 2n+2 registers for
          // n = 7 and formed per use otherwise: either way round, ptxas spills (8 B at n = 6, 36-56 B at n = 7).
          double sob[N == 7 ? NO : 1];
          auto sim_obs = [&](int k) {
            if (k < 2) return fma(a.sim.h_gdd_c, k == 0 ? sgddx : sgddy, k == 0 ? gdx : gdy);
            const int i = (k - 2) / 2;
            return (k & 1) ? fma(a.sim.h, sthdd[i], thd[i]) : fma(a.sim.h, thd[i], th[i]);
          };
          if constexpr (N == 7) {
#pragma unroll
            for (int k = 0; k < NO; ++k) sob[k] = sim_obs(k);
          }
          auto so = [&](int k) { return N == 7 ? sob[k] : sim_obs(k); };
          sim_cost = cost_max_affine<NO>(forms, so);
        } else {
          // the built-in cost only looks at the new angular velocities
          double sthd[N];
#pragma unroll
          for (int i = 0; i < N; ++i) sthd[i] = fma(a.sim.h, sthdd[i], thd[i]);
          sim_cost = cost_max_abs_thd<N>(sthd);
        }
        unsafe = !(sim_cost <= a.sim_thresh);
      } else {
        // The judgement above once per simulator model: every model must judge the step safe.  The decisions are
        // OR-ed (not the costs maxed), so that the order of the models cannot matter.  No early exit: a safe step
        // needs all M evaluations, and an unsafe one ends the rollout.  Models 1..M-1 run in a loop, reading their
        // constants from the constant bank through the runtime index m; model 0 runs last, in straight-line code
        // directly before the real step, as in the single-model kernels.  That keeps one model bit-identical to
        // them: there the compiler shares the model-independent products of the simulator's accelerations (of the
        // sines, cosines and velocities) with the real step, which then keeps them as separately rounded multiplies;
        // without the shared copy the real step fuses one of them into an FMA instead (one ulp in the real
        // trajectory).  The loop works on opaque copies of the sines, cosines and velocities, so that none of its
        // products is hoisted and shared with the code after it (which would keep them live across the loop).
        // The single-model modes keep the judgement inline: called through model_unsafe their kernels compile to the
        // same instructions and spills but other registers and another order.
        // LOOKAHEAD: each model judges by K backup steps after the action (model_unsafe_lookahead), and the first
        // unsafe model ends the judgement: the decision is an OR, so skipping the other models cannot change it.
        const SimModels& sm = sim_models_of(forms);
#pragma unroll 1
        for (int m = 1; m < sm.M && !(LOOKAHEAD && unsafe); ++m) {
          double s[N], c[N], w[N];
#pragma unroll
          for (int i = 0; i < N; ++i) { s[i] = opaque(sn[i]); c[i] = opaque(cs[i]); w[i] = opaque(thd[i]); }
          if constexpr (LOOKAHEAD)
            unsafe = model_unsafe_lookahead<N, FS, AFFINE>(forms, sm.p[m], a.sim_thresh, forms.lookahead, a.clip,
                                                           P.max_u, gdx, gdy, th, s, c, w, u, sF);
          else
            unsafe |= model_unsafe<N, FS, AFFINE>(forms, sm.p[m], a.sim_thresh, gdx, gdy, th, s, c, w, u, sF);
        }
        if constexpr (LOOKAHEAD) {
          if (!unsafe)
            unsafe = model_unsafe_lookahead<N, FS, AFFINE>(forms, sm.p[0], a.sim_thresh, forms.lookahead, a.clip,
                                                           P.max_u, gdx, gdy, th, sn, cs, thd, u, sF);
        } else {
          unsafe |= model_unsafe<N, FS, AFFINE>(forms, sm.p[0], a.sim_thresh, gdx, gdy, th, sn, cs, thd, u, sF);
        }
        if constexpr (SHIELD) {
          // The shield: a rejected policy action re-runs this step with the backup action (the state has not moved),
          // judged by the same code; the real step takes it if it is safe, and a rejected backup freezes.  The code
          // of the policy's steps is that of SCREEN_ENSEMBLE*, so an environment that never takes the backup
          // computes what those kernels compute.
          if (unsafe && !backup_turn) {
            backup_turn = true;
            --t;
            continue;
          }
          if (!unsafe && backup_turn) {
            backup_turn = false;
            ++ovr;
          }
        }
      }
      if (unsafe) {
        // unsafe: nothing advances, and since obs and policy never change it never will again
        // (safe_ars/ars.py:151-152) -- the remaining H-t steps are this state repeated.
        frozen = t;
        if (traj && active) {
          for (int tt = t; tt < a.H; ++tt) {
            double* o = traj + (long long)tt * traj_step;
            o[0] = gdx; o[1] = gdy;
#pragma unroll
            for (int i = 0; i < N; ++i) { o[2 + 2 * i] = th[i]; o[3 + 2 * i] = thd[i]; }
          }
        }
        break;
      }
    }
    if (VARIANT == 0) {
      // reward_t = Gdot_t . direction (remy_swimmer_env.py:238-243); the two components are summed
      // separately and dotted with the direction once, after the loop
      gym_step_tracked<N, FS>(P, gdx, gdy, th, thd, sn, cs, ut, (t & 63) == 63, sF);
      sgx += gdx;
      sgy += gdy;
    } else {
      ret += swimmer_step<N, 1>(P, gdx, gdy, th, thd, u);
    }
    if (SCREEN == SCREEN_BUILTIN || SCREEN == SCREEN_ENSEMBLE || SCREEN == SCREEN_SHIELD || SCREEN == SCREEN_LOOKAHEAD)
      viol += (cost_max_abs_thd<N>(thd) > a.real_thresh) ? 1 : 0;
    if constexpr (AFFINE || STATS) {
      double x[NO];  // the real observation after the step
      x[0] = gdx; x[1] = gdy;
#pragma unroll
      for (int i = 0; i < N; ++i) { x[2 + 2 * i] = th[i]; x[3 + 2 * i] = thd[i]; }
      if constexpr (AFFINE)
        viol += (cost_max_affine<NO>(cost_forms_of(forms), [&](int k) { return x[k]; }) > a.real_thresh) ? 1 : 0;
      if constexpr (STATS) {
#pragma unroll
        for (int j = 0; j < NO; ++j) {
          const double d = x[j] - s_piv[j];
          if (STATS_SMEM) {
            sS[j * kRolloutBlock] += d;
            sS[(NO + j) * kRolloutBlock] = fma(d, d, sS[(NO + j) * kRolloutBlock]);
          } else {
            s1[j] += d;
            s2[j] = fma(d, d, s2[j]);
          }
        }
      }
    }
    if (traj && active) {
      double2* o = reinterpret_cast<double2*>(traj + (long long)t * traj_step);
      o[0] = make_double2(gdx, gdy);
#pragma unroll
      for (int i = 0; i < N; ++i) o[1 + i] = make_double2(th[i], thd[i]);
    }
  }

  if (VARIANT == 0) ret += fma(sgx, P.dirx, sgy * P.diry);
  if (active) {
    const long long eo = output_row<MODELS>(a, e);
    a.returns[eo] = a.accumulate ? a.returns[eo] + ret : ret;
    if (a.final_state) {
      double2* o = reinterpret_cast<double2*>(a.final_state + eo * NO);
      o[0] = make_double2(gdx, gdy);
#pragma unroll
      for (int i = 0; i < N; ++i) o[1 + i] = make_double2(th[i], thd[i]);
    }
    if (SCREEN != SCREEN_NONE) {
      if (a.violations) a.violations[e] = viol;
      if (a.frozen_at) a.frozen_at[e] = frozen;
    }
    if constexpr (SHIELD) {
      if (backup_of(forms).overrides) backup_of(forms).overrides[e] = ovr;
    }
  }

  if (STATS) {
    // fixed-order block reduction: lanes by xor-butterfly, then warps in index order
    __shared__ double red[kRolloutBlock / 32][2 * NO];
#pragma unroll
    for (int j = 0; j < NO; ++j) {
      double v1 = STATS_SMEM ? sS[j * kRolloutBlock] : s1[j];
      double v2 = STATS_SMEM ? sS[(NO + j) * kRolloutBlock] : s2[j];
      if (!active) { v1 = 0.0; v2 = 0.0; }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        v1 += __shfl_xor_sync(0xffffffffu, v1, off);
        v2 += __shfl_xor_sync(0xffffffffu, v2, off);
      }
      if ((tid & 31) == 0) { red[tid >> 5][j] = v1; red[tid >> 5][NO + j] = v2; }
    }
    __syncthreads();
    if (tid < 2 * NO) {
      double v = 0.0;
#pragma unroll
      for (int w = 0; w < kRolloutBlock / 32; ++w) v += red[w][tid];
      a.stats_partial[(long long)blockIdx.x * 2 * NO + tid] = v;
    }
  }
}

}  // namespace swm
