// The RL-Glue ARS experiment at STEP granularity, with the reference's literal state machine:
// rlglue/agent/SwimmerAgent.py:79-130 (agent_start / agent_step), :181-201 (clipped linear policy),
// :203-212 (delta ~ U[0,1)), :214-241 (index order, sample standard deviation, first b directions) driven by
// rlglue/experiment/SwimmerExperiment.cpp:65-84 (2 N H training steps with "load state" every H steps, then
// "freeze training" + one H-step evaluation rollout whose total is the line of plot/results.txt) against
// rlglue/environment/SwimmerEnvironment.cpp (env_start state 0.001, semi-implicit step, reward Gdot . dir).
//
// The reference's bookkeeping couples consecutive rollouts (the first environment step after each "load
// state" applies the action chosen from the previous rollout's last observation with the previous rollout's
// policy; the agent acts on the stored initial observation at the first step of a rollout; a rollout's
// return is shifted by one step and the last slot of the reward table is filled one iteration late), so the
// 2N rollouts of an iteration are NOT independent and cannot be batched: this kernel runs the state machine
// sequentially, one thread per experiment replica (seeds are the parallel dimension).  The batched
// engine (ArsEngine with semantics ARS_RLGLUE) implements the intended algorithm -- independent rollouts --
// and is what RlglueArsExperiment uses by default; this kernel is its `protocol="reference"` mode, pinned
// against the unmodified agent + environment (tests/golden/rlglue_agent.npz).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "../../include/swimmer_ars.h"
#include "dynamics.cuh"
#include "errors.cuh"
#include "philox.cuh"

namespace swm {

struct ProtoArgs {
  int N, b, H, n_it;
  double alpha, nu;
  const double* deltas;     // [n_it + 1, N, WS] shared by all replicas, or NULL: Philox U[0,1)
  uint64_t seed;            // Philox: key = seed + replica, counter = (pair, direction, iteration, 0)
  uint32_t iteration0;
  double* state;            // [replicas, WS + NA + 2]: policy, pending action, running total, iterations done
  double* results;          // [replicas, n_it] evaluation totals
  double* table;            // [replicas, n_it, 2N] reward table at each update (also the kernel's scratch)
  long long replicas;
};

template <int N>
__global__ void __launch_bounds__(32) rlglue_protocol_kernel(const Phys P, const ProtoArgs a) {
  constexpr int NO = 2 * N + 2, NA = N - 1, WS = NA * NO;
  const long long rep = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (rep >= a.replicas) return;
  double* S = a.state + rep * (WS + NA + 2);
  double W[WS], Wp[WS], act[NA > 0 ? NA : 1];
  const int done0 = (int)S[WS + NA + 1];
  double total = S[WS + NA];
#pragma unroll 1
  for (int j = 0; j < WS; ++j) W[j] = S[j];
  auto delta = [&](int it, int k, int j) -> double {
    if (a.deltas) return a.deltas[((size_t)it * a.N + k) * WS + j];
    double d0, d1;
    philox_delta_pair(a.seed + (uint64_t)rep, a.iteration0 + (uint32_t)it, (uint32_t)k, 0u, (uint32_t)(j >> 1),
                      SWM_DELTA_UNIFORM_01, d0, d1);
    return (j & 1) ? d1 : d0;
  };
  // deltaPolicies[q] = agentPolicy +- nu * deltas[q / 2]  (:209-212), q < 0: the unperturbed policy
  auto set_policy = [&](int it, int q) {
#pragma unroll 1
    for (int j = 0; j < WS; ++j)
      Wp[j] = q < 0 ? W[j] : __dadd_rn(W[j], ((q & 1) ? -1.0 : 1.0) * __dmul_rn(a.nu, delta(it, q >> 1, j)));
  };
  auto select_action = [&](const double* obs) {  // np.matmul + clip (:181-196)
#pragma unroll
    for (int k = 0; k < NA; ++k) {
      double acc = 0.0;
#pragma unroll
      for (int j = 0; j < NO; ++j) acc = fma(Wp[k * NO + j], obs[j], acc);
      act[k] = fmin(fmax(acc, -P.max_u), P.max_u);
    }
  };
  double o0[NO];
#pragma unroll
  for (int j = 0; j < NO; ++j) o0[j] = 0.001;  // env_start (cpp:39-42), also the agent's initial_state
  if (done0 == 0) {                            // agent_start: first action from deltaPolicies[0] on o0
    set_policy(0, 0);
    select_action(o0);
    total = 0.0;
  } else {
#pragma unroll
    for (int k = 0; k < NA; ++k) act[k] = S[WS + k];
  }
  double gdx, gdy, th[N], thd[N];
  auto load_state = [&]() {
    gdx = gdy = 0.001;
#pragma unroll
    for (int i = 0; i < N; ++i) { th[i] = 0.001; thd[i] = 0.001; }
  };
  load_state();
  const int rollouts = 2 * a.N;
  for (int it = 0; it < a.n_it; ++it) {
    const int git = done0 + it;  // index into the delta sequence
    double* rewards = a.table + ((size_t)rep * a.n_it + it) * rollouts;
    for (int q = 0; q < rollouts; ++q) rewards[q] = 0.0;
    int cur = -2;                // rollout whose perturbed policy is in Wp
    for (int i = 0; i < rollouts * a.H + a.H; ++i) {
      const bool training = i < rollouts * a.H;
      if (i % a.H == 0) load_state();  // RL_env_message("load state") every H steps and before the evaluation
      const double r = swimmer_step<N, 1>(P, gdx, gdy, th, thd, act);
      total += r;
      double obs[NO];
      obs[0] = gdx; obs[1] = gdy;
#pragma unroll
      for (int s = 0; s < N; ++s) { obs[2 + 2 * s] = th[s]; obs[3 + 2 * s] = thd[s]; }
      bool first = false;
      if (training) {
        if (i % a.H == 0) {      // "New rollout": the total collected so far belongs to the PREVIOUS slot
          rewards[(i / a.H - 1 + rollouts) % rollouts] = total;
          total = 0.0;
          first = true;
        }
        const int q = i / a.H;
        if (q != cur) { set_policy(git, q); cur = q; }
      } else {
        if (i == rollouts * a.H) { total = 0.0; first = true; set_policy(git, -1); cur = -1; }
      }
      select_action(first ? o0 : obs);
      if (training && i == rollouts * a.H - 1) {
        // update_policy (:223-241): first b directions, sample standard deviation of their 2b rewards
        double mean = 0.0;
        for (int k = 0; k < 2 * a.b; ++k) mean += rewards[k];
        mean /= (2.0 * a.b);
        double var = 0.0;
        for (int k = 0; k < 2 * a.b; ++k) var = fma(rewards[k] - mean, rewards[k] - mean, var);
        const double sigma = sqrt(var / (2.0 * a.b - 1.0));
        const double scale = a.alpha / ((double)a.b * sigma);
#pragma unroll 1
        for (int j = 0; j < WS; ++j) {
          double g = 0.0;
          for (int k = 0; k < a.b; ++k) g = fma(rewards[2 * k] - rewards[2 * k + 1], delta(git, k, j), g);
          W[j] = fma(scale, g, W[j]);
        }
        cur = -2;  // sample_deltas: the next iteration perturbs the updated policy with new directions
      }
    }
    a.results[rep * a.n_it + it] = total;
  }
#pragma unroll 1
  for (int j = 0; j < WS; ++j) S[j] = W[j];
#pragma unroll
  for (int k = 0; k < NA; ++k) S[WS + k] = act[k];
  S[WS + NA] = total;
  S[WS + NA + 1] = (double)(done0 + a.n_it);
}

template <int N>
static int launch_protocol(const Phys& P, const ProtoArgs& a, cudaStream_t st) {
  rlglue_protocol_kernel<N><<<(unsigned)((a.replicas + 31) / 32), 32, 0, st>>>(P, a);
  return swm::check_launch();
}

}  // namespace swm

using namespace swm;

extern "C" int64_t swm_rlglue_protocol_state_doubles(int n) {
  if (n < SWM_MIN_SEGMENTS || n > SWM_MAX_SEGMENTS) return 0;
  return (int64_t)(n - 1) * (2 * n + 2) + (n - 1) + 2;
}

extern "C" int swm_rlglue_protocol(const swm_params_t* params, const swm_rlglue_protocol_t* cfg, void* stream) {
  if (!params || !cfg || params->n < SWM_MIN_SEGMENTS || params->n > SWM_MAX_SEGMENTS) return SWM_ERR_BAD_ARG;
  if (cfg->N < 1 || cfg->b < 1 || cfg->b > cfg->N || cfg->H < 1 || cfg->n_it < 0 || cfg->replicas < 0) return SWM_ERR_BAD_ARG;
  if (cfg->n_it == 0 || cfg->replicas == 0) return SWM_OK;
  if (!cfg->state || !cfg->results || !cfg->table) return SWM_ERR_BAD_ARG;
  if (2 * cfg->b < 2) return SWM_ERR_BAD_ARG;
  ProtoArgs a;
  memset(&a, 0, sizeof(a));
  a.N = cfg->N; a.b = cfg->b; a.H = cfg->H; a.n_it = cfg->n_it;
  a.alpha = cfg->alpha; a.nu = cfg->nu;
  a.deltas = cfg->deltas;
  a.seed = cfg->seed; a.iteration0 = cfg->iteration0;
  a.state = cfg->state; a.results = cfg->results; a.table = cfg->table;
  a.replicas = cfg->replicas;
  const Phys P = make_phys(*params);
  cudaStream_t st = (cudaStream_t)stream;
  switch (params->n) {
    case 2: return launch_protocol<2>(P, a, st);
    case 3: return launch_protocol<3>(P, a, st);
    case 4: return launch_protocol<4>(P, a, st);
    case 5: return launch_protocol<5>(P, a, st);
    case 6: return launch_protocol<6>(P, a, st);
    case 7: return launch_protocol<7>(P, a, st);
    case 8: return launch_protocol<8>(P, a, st);
    case 9: return launch_protocol<9>(P, a, st);
    case 10: return launch_protocol<10>(P, a, st);
    default: return SWM_ERR_UNSUPPORTED;
  }
}
