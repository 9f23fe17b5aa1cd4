// extern "C" entry points of libswimmer_ars.so (see include/swimmer_ars.h): argument checks,
// precomputation of the physical constants (swm::make_phys) and dispatch on the segment count.
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>

#include <mutex>

#include "errors.cuh"
#include "lane_launch.cuh"

using namespace swm;

namespace {

thread_local char g_cuda_err[256] = "";

int cuda_fail(cudaError_t e) {
  snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", cudaGetErrorName(e), cudaGetErrorString(e));
  return SWM_ERR_CUDA;
}

int note_launch(int rc) {
  if (rc == SWM_ERR_CUDA) {
    cudaError_t e = cudaPeekAtLastError();
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", cudaGetErrorName(e), cudaGetErrorString(e));
    cudaGetLastError();
  }
  return rc;
}

}  // namespace

int swm::check_launch() {
  const cudaError_t e = cudaGetLastError();  // reads and clears
  if (e == cudaSuccess) return SWM_OK;
  return cuda_fail(e);
}

namespace {

bool params_ok(const swm_params_t* p) {
  return p && p->n >= SWM_MIN_SEGMENTS && p->n <= SWM_MAX_SEGMENTS && p->l_i > 0.0 && p->m_i > 0.0;
}

#define SWM_DISPATCH_N(n, CALL)                 \
  switch (n) {                                  \
    case 2: return note_launch(CALL(2));        \
    case 3: return note_launch(CALL(3));        \
    case 4: return note_launch(CALL(4));        \
    case 5: return note_launch(CALL(5));        \
    case 6: return note_launch(CALL(6));        \
    case 7: return note_launch(CALL(7));        \
    case 8: return note_launch(CALL(8));        \
    case 9: return note_launch(CALL(9));        \
    case 10: return note_launch(CALL(10));      \
    default: return SWM_ERR_UNSUPPORTED;        \
  }

int step_common(const swm_params_t* params, int variant, bool acc_only, const double* state_in,
                const double* action, double* out, double* reward, int64_t B, void* stream) {
  if (!params_ok(params) || B < 0) return SWM_ERR_BAD_ARG;
  if (variant != SWM_DYN_GYM && variant != SWM_DYN_RLGLUE) return SWM_ERR_BAD_ARG;
  if (B == 0) return SWM_OK;  // empty batch: nothing to do, pointers may be NULL
  if (!state_in || !action || !out) return SWM_ERR_BAD_ARG;
  const Phys P = make_phys(*params);
  cudaStream_t st = (cudaStream_t)stream;
#define CALL(K) launch_step_n<K>(P, variant, acc_only, state_in, action, out, reward, (long long)B, st)
  SWM_DISPATCH_N(params->n, CALL)
#undef CALL
}

}  // namespace

extern "C" int swm_abi_version(void) { return SWM_ABI_VERSION; }

extern "C" const char* swm_strerror(int status) {
  switch (status) {
    case SWM_OK: return "ok";
    case SWM_ERR_BAD_ARG: return "bad argument";
    case SWM_ERR_UNSUPPORTED: return "unsupported configuration";
    case SWM_ERR_CUDA: return "CUDA error (see swm_last_cuda_error)";
    case SWM_ERR_NO_DEVICE: return "no CUDA device";
    default: return "unknown status";
  }
}

extern "C" const char* swm_last_cuda_error(void) { return g_cuda_err; }

extern "C" int swm_device_info(int* sm_count, int* cc_major, int* cc_minor) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) { cuda_fail(e); return SWM_ERR_NO_DEVICE; }
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) return cuda_fail(e);
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  return SWM_OK;
}

extern "C" int swm_step_batched(const swm_params_t* params, int variant, const double* state_in,
                                const double* action, double* state_out, double* reward,
                                int64_t B, void* stream) {
  return step_common(params, variant, false, state_in, action, state_out, reward, B, stream);
}

extern "C" int swm_step_batched_models(const swm_params_t* params, int n_models, int64_t envs_per_model,
                                       const double* state_in, const double* action, double* state_out,
                                       double* reward, void* stream) {
  if (!params || n_models < 1 || n_models > SWM_MAX_MODELS_PER_STEP || envs_per_model < 0) return SWM_ERR_BAD_ARG;
  PhysSet set;
  for (int i = 0; i < n_models; ++i) {
    if (!params_ok(&params[i]) || params[i].n != params[0].n) return SWM_ERR_BAD_ARG;
    set.p[i] = make_phys(params[i]);
  }
  for (int i = n_models; i < SWM_MAX_MODELS_PER_STEP; ++i) set.p[i] = set.p[0];
  const long long B = (long long)n_models * envs_per_model;
  if (B == 0) return SWM_OK;
  if (!state_in || !action || !state_out) return SWM_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
#define CALL(K) launch_step_models_n<K>(set, (long long)envs_per_model, state_in, action, state_out, reward, B, st)
  SWM_DISPATCH_N(params[0].n, CALL)
#undef CALL
}

extern "C" int swm_accelerations_batched(const swm_params_t* params, int variant,
                                         const double* state, const double* action, double* acc,
                                         int64_t B, void* stream) {
  return step_common(params, variant, true, state, action, acc, nullptr, B, stream);
}

namespace {

int sm_count_cached() {
  static int sms[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (sms[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) return 148;
    sms[dev] = v;
  }
  return sms[dev];
}

// Validates cfg and fills the kernel arguments; returns SWM_OK or an error.
int build_rollout_args(const swm_params_t* params, const swm_rollout_t* cfg, RolloutArgs& a, RolloutFlags& f) {
  if (!params_ok(params) || !cfg) return SWM_ERR_BAD_ARG;
  if (cfg->B < 0 || cfg->H < 0 || cfg->rollouts_per_policy < 1) return SWM_ERR_BAD_ARG;
  if (cfg->variant != SWM_DYN_GYM && cfg->variant != SWM_DYN_RLGLUE) return SWM_ERR_BAD_ARG;
  if (cfg->kernel < SWM_KERNEL_AUTO || cfg->kernel > SWM_KERNEL_LANES3) return SWM_ERR_BAD_ARG;
  if (cfg->B > (int64_t)kRolloutBlock * 0x7fffffffLL) return SWM_ERR_BAD_ARG;
  memset(&a, 0, sizeof(a));
  f.variant = cfg->variant;
  f.norm = cfg->normalize != 0;
  f.stats = cfg->stats_partial != nullptr;
  f.screen = cfg->screen.enabled != 0;
  f.group_w = (cfg->rollouts_per_policy % 32) == 0;
  switch (cfg->policy_mode) {
    case SWM_POLICY_FIXED_ACTION:
      f.linear = false;
      break;
    case SWM_POLICY_EXPLICIT:
    case SWM_POLICY_PHILOX:
    case SWM_POLICY_DELTAS:
      if (cfg->B % cfg->rollouts_per_policy != 0) return SWM_ERR_BAD_ARG;
      if (cfg->policy_mode != SWM_POLICY_EXPLICIT && ((cfg->B / cfg->rollouts_per_policy) % 2) != 0)
        return SWM_ERR_BAD_ARG;  // +delta / -delta pairs
      if (cfg->policy_mode == SWM_POLICY_EXPLICIT && cfg->dir_mask) return SWM_ERR_BAD_ARG;
      f.linear = true;
      break;
    default:
      return SWM_ERR_BAD_ARG;
  }
  if (!f.linear && cfg->dir_mask) return SWM_ERR_BAD_ARG;
  if (cfg->init_state && cfg->init_state_count < 1) return SWM_ERR_BAD_ARG;
  if (f.screen) {
    if (!params_ok(&cfg->screen.sim) || cfg->screen.sim.n != params->n) return SWM_ERR_BAD_ARG;
    a.sim = make_phys(cfg->screen.sim);
  }
  a.real = make_phys(*params);
  a.H = cfg->H;
  a.R = cfg->rollouts_per_policy;
  a.policy_mode = cfg->policy_mode;
  a.clip = cfg->clip_actions;
  a.B = cfg->B;
  a.actions = cfg->actions;
  a.policies = cfg->policies;
  a.deltas = cfg->deltas;
  a.dir_mask = cfg->dir_mask;
  a.init_perturb = cfg->init_perturb;
  a.nu = cfg->nu;
  a.seed = cfg->philox.seed;
  a.iteration = cfg->philox.iteration;
  a.iter_dev = cfg->philox.iteration_dev;
  a.dir0 = cfg->philox.dir0;
  a.dist = cfg->philox.dist;
  a.mean = cfg->mean;
  a.inv_sigma = cfg->inv_sigma;
  a.init_state = cfg->init_state;
  a.init_count = cfg->init_state ? cfg->init_state_count : 1;
  a.returns = cfg->returns;
  a.final_state = cfg->final_state;
  a.trajectory = cfg->trajectory;
  a.stats_partial = cfg->stats_partial;
  a.stats_pivot = cfg->stats_pivot;
  a.sim_thresh = cfg->screen.sim_thresh;
  a.real_thresh = cfg->screen.real_thresh;
  a.violations = cfg->screen.violations;
  a.frozen_at = cfg->screen.frozen_at;
  a.accumulate = cfg->accumulate_returns;
  return SWM_OK;
}

// AUTO (measured crossovers, tools/lane_split_sweep.py, profiles/r02_summary.md), for chains of up to 7 segments
// (8 lanes per environment):
//   lane groups <= 1 per SM, n >= 6       -> LANES3: main warp + two operator warps taking alternate steps (the
//                                            operator warp is the slower one of the pair from 6 segments on;
//                                            n = 7: 683 against 802 cycles per step, n <= 5: no gain)
//   lane groups <= 2 per SM               -> LANES2: main warp + operator warp per group, every warp on a
//                                            sub-partition of its own (n = 5: 0.30 ms against 0.40 / 0.72 ms)
//   lane-split warps <= 2 per sub-partition -> LANES (n = 5, 2,048 envs: 0.42 ms against 0.72 ms)
//   larger batches                        -> THREAD (one environment per thread fills the FP64 units)
constexpr double kLaneSplitMaxWarpsPerSmsp = 2.0;
constexpr double kLane2MaxGroupsPerSm = 2.0;
constexpr int kLane3MinSegments = 6;

inline bool is_lane_kernel(int k) { return k == SWM_KERNEL_LANES || k == SWM_KERNEL_LANES2 || k == SWM_KERNEL_LANES3; }

int choose_kernel(int n, const swm_rollout_t* cfg, const RolloutArgs& a, const RolloutFlags& f) {
  // per-step screening exists in the warp-specialised kernels only
  const bool ok = lane_split_supported(a, f, cfg->kernel == SWM_KERNEL_LANES ? 0 : 1);
  if (is_lane_kernel(cfg->kernel)) return ok ? cfg->kernel : SWM_ERR_UNSUPPORTED;
  if (cfg->kernel == SWM_KERNEL_THREAD || !ok || n > 7) return SWM_KERNEL_THREAD;
  const int per_warp = 32 / lane_split_lanes(n);
  const double groups = (double)((cfg->B + per_warp - 1) / per_warp);
  if (n >= kLane3MinSegments && groups <= sm_count_cached()) return SWM_KERNEL_LANES3;
  if (groups <= kLane2MaxGroupsPerSm * sm_count_cached()) return SWM_KERNEL_LANES2;
  if (f.screen) return SWM_KERNEL_THREAD;
  return groups <= kLaneSplitMaxWarpsPerSmsp * 4.0 * sm_count_cached() ? SWM_KERNEL_LANES : SWM_KERNEL_THREAD;
}

}  // namespace

extern "C" int swm_rollout_kernel_choice(const swm_params_t* params, const swm_rollout_t* cfg) {
  RolloutArgs a;
  RolloutFlags f;
  const int rc = build_rollout_args(params, cfg, a, f);
  if (rc != SWM_OK) return rc;
  return choose_kernel(params->n, cfg, a, f);
}

namespace {

// ---- chunked schedule of one rollout: sub-batches x 64-step-aligned time chunks on internal streams -------
// One thread owns one environment for all H steps, so a batch that leaves a fractional number of warps per SM
// sub-partition between 3 and 4 (65,536 three-segment envs on 148 SMs: 3.46, the busiest holds 4) runs at the
// pace of the busiest sub-partition.  Cutting the rollout into short launches on several streams (state chained
// through final_state -> init_state, returns accumulated, chunk boundaries on the exact re-evaluation of the
// tracked sines/cosines so that every state is bit-identical) lets the hardware re-balance every 64 steps.
constexpr int kPlanMaxSub = 32;

struct Plan {
  int n_sub = 0, chunk = 0;  // n_sub == 0: one plain launch
};

struct PlanStreams {
  cudaStream_t s[kPlanMaxSub];
  cudaEvent_t fork, join[kPlanMaxSub];
  bool ready = false;
};

PlanStreams* plan_streams() {
  static PlanStreams table[64];
  static std::mutex mu;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  std::lock_guard<std::mutex> lock(mu);
  PlanStreams& ps = table[dev];
  if (!ps.ready) {
    for (int i = 0; i < kPlanMaxSub; ++i) {
      if (cudaStreamCreateWithFlags(&ps.s[i], cudaStreamNonBlocking) != cudaSuccess) return nullptr;
      if (cudaEventCreateWithFlags(&ps.join[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
    }
    if (cudaEventCreateWithFlags(&ps.fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    ps.ready = true;
  }
  return &ps;
}

long long plan_unit(const swm_rollout_t* cfg) {  // environments that must stay in one launch
  const bool perturbed = cfg->policy_mode == SWM_POLICY_PHILOX || cfg->policy_mode == SWM_POLICY_DELTAS;
  return (long long)cfg->rollouts_per_policy * (perturbed ? 2 : 1);
}

// contiguous sub-batches of whole units; cut[i] .. cut[i+1]
int plan_cuts(long long B, long long unit, int n_sub, long long* cut) {
  const long long groups = B / unit;
  if (n_sub > groups) n_sub = (int)groups;
  if (n_sub < 1) n_sub = 1;
  for (int i = 0; i <= n_sub; ++i) cut[i] = unit * ((groups * i) / n_sub);
  return n_sub;
}

bool plan_feasible(const swm_rollout_t* cfg, const RolloutFlags& f, int n_sub, int chunk) {
  if (n_sub < 1 || n_sub > kPlanMaxSub || chunk < 64 || chunk % 64 != 0) return false;
  if (!cfg->final_state || cfg->trajectory || f.screen || cfg->H <= chunk) return false;
  const long long unit = plan_unit(cfg);
  if (cfg->B % unit != 0) return false;
  if (cfg->init_state && cfg->init_state_count != cfg->B) {
    long long cut[kPlanMaxSub + 1];
    const int ns = plan_cuts(cfg->B, unit, n_sub, cut);
    for (int i = 0; i < ns; ++i)
      if (cut[i] % cfg->init_state_count != 0) return false;  // e % count must not change with the offset
  }
  return true;
}

Plan choose_plan(int n, const swm_rollout_t* cfg, const RolloutFlags& f, int kernel, cudaStream_t st) {
  Plan p;
  if (kernel != SWM_KERNEL_THREAD || cfg->schedule_sub < 0) return p;
  if (cfg->schedule_sub > 0) {  // forced by the caller
    if (plan_feasible(cfg, f, cfg->schedule_sub, cfg->schedule_chunk)) { p.n_sub = cfg->schedule_sub; p.chunk = cfg->schedule_chunk; }
    return p;
  }
  // AUTO: only where it was measured to pay (tools/chunk_sweep.py, profiles/r02_chunk_sweep.txt): between 3 and 4
  // warps per sub-partition, kernels that keep >= 2 warps per sub-partition resident (n <= 5)
  if (n > 5) return p;
  const double w = (double)((cfg->B + 31) / 32) / (4.0 * sm_count_cached());
  if (w <= 3.05 || w >= 3.95) return p;
  // Fine chunks balance best (16 x 64: +20 % for the fixed-action kernel) but are 256 launches per rollout: that
  // only pays when the caller is capturing a CUDA graph (replay has no per-launch host cost).  Enqueued
  // eagerly -- and for policy kernels, which regenerate their policy in every launch -- 8 x 256 (+14 %).
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  const bool capturing = cudaStreamIsCapturing(st, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusActive;
  const bool fine = capturing && !f.linear;
  const int n_sub = fine ? 16 : 8, chunk = fine ? 64 : 256;
  if (plan_feasible(cfg, f, n_sub, chunk)) { p.n_sub = n_sub; p.chunk = chunk; }
  return p;
}

long long plan_stats_rows(const swm_rollout_t* cfg, const Plan& p) {
  long long cut[kPlanMaxSub + 1];
  const int ns = plan_cuts(cfg->B, plan_unit(cfg), p.n_sub, cut);
  long long rows = 0;
  for (int i = 0; i < ns; ++i) rows += (cut[i + 1] - cut[i] + kRolloutBlock - 1) / kRolloutBlock;
  return rows * ((cfg->H + p.chunk - 1) / p.chunk);
}

int launch_thread_kernel(int n, const RolloutArgs& a, const RolloutFlags& f, cudaStream_t st) {
#define CALL(K) launch_rollout_n<K>(a, f, st)
  SWM_DISPATCH_N(n, CALL)
#undef CALL
}

int launch_planned(int n, const swm_rollout_t* cfg, const RolloutArgs& a0, const RolloutFlags& f, const Plan& p,
                   cudaStream_t st) {
  PlanStreams* ps = plan_streams();
  if (!ps) return SWM_ERR_CUDA;
  const int NO = 2 * n + 2, NA = n - 1, WS = NA * NO;
  const long long unit = plan_unit(cfg);
  long long cut[kPlanMaxSub + 1];
  const int ns = plan_cuts(a0.B, unit, p.n_sub, cut);
  const bool perturbed = cfg->policy_mode == SWM_POLICY_PHILOX || cfg->policy_mode == SWM_POLICY_DELTAS;
  if (cudaEventRecord(ps->fork, st) != cudaSuccess) return SWM_ERR_CUDA;
  for (int i = 0; i < ns; ++i)
    if (cudaStreamWaitEvent(ps->s[i], ps->fork, 0) != cudaSuccess) return SWM_ERR_CUDA;
  long long row = 0;
  int rc = SWM_OK;
  for (int t0 = 0, c = 0; t0 < a0.H && rc == SWM_OK; t0 += p.chunk, ++c) {
    for (int i = 0; i < ns && rc == SWM_OK; ++i) {
      const long long lo = cut[i], Bs = cut[i + 1] - cut[i];
      RolloutArgs a = a0;
      a.B = Bs;
      a.H = (a0.H - t0 < p.chunk) ? a0.H - t0 : p.chunk;
      a.returns = a0.returns + lo;
      a.final_state = a0.final_state + lo * NO;
      if (a0.actions) a.actions = a0.actions + lo * NA;
      if (f.linear) {
        const long long pol = lo / a0.R;  // first policy of this sub-batch
        if (cfg->policy_mode == SWM_POLICY_EXPLICIT) a.policies = a0.policies + pol * WS;
        if (perturbed) a.dir0 = a0.dir0 + (unsigned int)(pol >> 1);
        if (a0.deltas) a.deltas = a0.deltas + (pol >> 1) * WS;
        if (a0.dir_mask) a.dir_mask = a0.dir_mask + (pol >> 1);
      }
      if (c == 0) {
        if (a0.init_state && a0.init_count == a0.B) { a.init_state = a0.init_state + lo * NO; a.init_count = Bs; }
      } else {
        a.init_state = a.final_state;  // continue from the state the previous chunk left
        a.init_count = Bs;
        a.init_perturb = 0.0;
        a.accumulate = 1;
      }
      if (a0.stats_partial) {
        a.stats_partial = a0.stats_partial + row * 2 * NO;
        row += (Bs + kRolloutBlock - 1) / kRolloutBlock;
      }
      rc = launch_thread_kernel(n, a, f, ps->s[i]);
    }
  }
  for (int i = 0; i < ns; ++i) {
    if (cudaEventRecord(ps->join[i], ps->s[i]) != cudaSuccess || cudaStreamWaitEvent(st, ps->join[i], 0) != cudaSuccess)
      return SWM_ERR_CUDA;
  }
  return rc;
}

}  // namespace

extern "C" int swm_rollout_schedule(const swm_params_t* params, const swm_rollout_t* cfg, void* stream, int* n_sub,
                                    int* chunk) {
  RolloutArgs a;
  RolloutFlags f;
  const int rc = build_rollout_args(params, cfg, a, f);
  if (rc != SWM_OK) return rc;
  const int kernel = choose_kernel(params->n, cfg, a, f);
  if (kernel < 0) return kernel;
  const Plan p = choose_plan(params->n, cfg, f, kernel, (cudaStream_t)stream);
  if (n_sub) *n_sub = p.n_sub;
  if (chunk) *chunk = p.chunk;
  return SWM_OK;
}

extern "C" int64_t swm_rollout_stats_blocks(const swm_params_t* params, const swm_rollout_t* cfg, void* stream) {
  if (!cfg || cfg->B < 1) return 0;
  // the row count depends on the kernel and the schedule swm_rollout will choose, which never look at the
  // statistics pointers themselves
  swm_rollout_t probe = *cfg;
  static double dummy;
  probe.stats_partial = &dummy;
  RolloutArgs a;
  RolloutFlags f;
  if (build_rollout_args(params, &probe, a, f) != SWM_OK) return 0;
  const int kernel = choose_kernel(params->n, &probe, a, f);
  if (is_lane_kernel(kernel)) {
    const int per_warp = 32 / lane_split_lanes(params->n);
    return (cfg->B + per_warp - 1) / per_warp;
  }
  const Plan p = choose_plan(params->n, &probe, f, kernel, (cudaStream_t)stream);
  if (p.n_sub > 0) return plan_stats_rows(&probe, p);
  return (cfg->B + kRolloutBlock - 1) / kRolloutBlock;
}

extern "C" int swm_rollout(const swm_params_t* params, const swm_rollout_t* cfg, void* stream) {
  RolloutArgs a;
  RolloutFlags f;
  if (params_ok(params) && cfg && cfg->B == 0 && cfg->H >= 0 && cfg->rollouts_per_policy >= 1 &&
      (cfg->variant == SWM_DYN_GYM || cfg->variant == SWM_DYN_RLGLUE))
    return SWM_OK;  // empty batch: nothing to do, pointers may be NULL
  const int rc = build_rollout_args(params, cfg, a, f);
  if (rc != SWM_OK) return rc;
  if (!cfg->returns) return SWM_ERR_BAD_ARG;
  if (!f.linear && !cfg->actions) return SWM_ERR_BAD_ARG;
  if (f.linear && !cfg->policies) return SWM_ERR_BAD_ARG;
  if (cfg->policy_mode == SWM_POLICY_DELTAS && !cfg->deltas) return SWM_ERR_BAD_ARG;
  if (f.norm && (!cfg->mean || !cfg->inv_sigma)) return SWM_ERR_BAD_ARG;
  if (f.stats && !cfg->stats_pivot) return SWM_ERR_BAD_ARG;
  const int kernel = choose_kernel(params->n, cfg, a, f);
  if (kernel < 0) return kernel;
  cudaStream_t st = (cudaStream_t)stream;
  if (is_lane_kernel(kernel)) {
#define CALL(K) launch_lane_rollout_n<K>(a, f, kernel == SWM_KERNEL_LANES3 ? 2 : kernel == SWM_KERNEL_LANES2 ? 1 : 0, st)
    SWM_DISPATCH_N(params->n, CALL)
#undef CALL
  }
  const Plan p = choose_plan(params->n, cfg, f, kernel, st);
  if (cfg->schedule_sub > 0 && p.n_sub == 0) return SWM_ERR_UNSUPPORTED;  // a forced schedule that cannot run
  if (p.n_sub > 0) return note_launch(launch_planned(params->n, cfg, a, f, p, st));
  return launch_thread_kernel(params->n, a, f, st);
}

// Layout self-check for language bindings: sizes of the ABI structs as this build sees them.
extern "C" int swm_abi_struct_sizes(int* params, int* philox, int* screen, int* rollout) {
  if (params) *params = (int)sizeof(swm_params_t);
  if (philox) *philox = (int)sizeof(swm_philox_t);
  if (screen) *screen = (int)sizeof(swm_screen_t);
  if (rollout) *rollout = (int)sizeof(swm_rollout_t);
  return SWM_OK;
}
