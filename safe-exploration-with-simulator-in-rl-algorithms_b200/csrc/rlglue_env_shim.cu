// RL-Glue environment plugin ABI (env_init / env_start / env_step / env_cleanup / env_message)
// backed by the sm_100a kernels: the B200-native counterpart of
// rlglue/environment/SwimmerEnvironment.cpp:14-97.  Same symbols, same ownership rules (the callee
// owns every returned pointer; pointers stay valid until the next call; arrays are allocated in
// env_init and released in env_cleanup), same messages, same start state (all entries 0.001,
// cpp:39-42), same parameter-file format (cpp:297-326).  One environment = a batch of 1 through
// swm_step_batched(variant = SWM_DYN_RLGLUE); the batched entry points are the fast path, this shim
// exists so that an RL-Glue experiment can link the new library unchanged.
// Differences, on purpose: no per-step printing of the state (cpp:61), and an out-of-range action
// returns the previous observation with terminal = 1 instead of assert-aborting (cpp:56-58) when
// SWM_RLGLUE_NO_ABORT is set in the environment (default: abort like the reference).
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>

#include "../../include/swimmer_rlglue_env.h"

namespace {

observation_t this_observation;
observation_t saved_observation;
reward_observation_terminal_t this_reward_observation;
swm_params_t g_params = {3, 0, 1.0, 1.0, 10.0, 0.01, 5.0, {1.0, 0.0}};
// One step = one upload, one launch, one download on a private stream, through pinned staging buffers:
double* d_in = nullptr;      // device [2n+2 state | n-1 action]
double* d_out = nullptr;     // device [2n+2 next state | reward]
double* h_in = nullptr;      // pinned mirror of d_in
double* h_out = nullptr;     // pinned mirror of d_out
cudaStream_t g_stream = nullptr;
int g_sized_n = 0;           // chain length the buffers above are sized for (0: before env_init / after env_cleanup)
std::string g_task_spec, g_param_msg;

// private stand-ins for RLStruct_util.h (not exported: librlutils owns those names)
void shim_alloc(rl_abstract_type_t* dst, unsigned int numDoubles) {
  dst->numInts = 0; dst->numDoubles = numDoubles; dst->numChars = 0;
  dst->intArray = nullptr;
  dst->doubleArray = numDoubles ? (double*)calloc(numDoubles, sizeof(double)) : nullptr;
  dst->charArray = nullptr;
}
void shim_clear(rl_abstract_type_t* dst) {
  free(dst->doubleArray);
  dst->intArray = nullptr; dst->doubleArray = nullptr; dst->charArray = nullptr;
  dst->numInts = dst->numDoubles = dst->numChars = 0;
}

void die(const char* what) {
  fprintf(stderr, "swimmer rlglue shim: %s (%s)\n", what, swm_last_cuda_error());
  abort();
}

// Returns "" or why a requested n_seg was not applied: outside SWM_MIN_SEGMENTS..SWM_MAX_SEGMENTS, or a change
// after env_init, whose observation, pinned and device buffers hold 2n+2 doubles of the chain they were sized for.
std::string set_parameters(const char* path) {
  FILE* f = fopen(path, "r");
  if (!f) { fprintf(stderr, "Unable to open file for setting environment parameters\n"); return ""; }
  std::string refused;
  char name[128];
  char line[512];
  while (fgets(line, sizeof(line), f)) {
    double a = 0, b = 0;
    const int got = sscanf(line, "%127s %lf %lf", name, &a, &b);
    if (got < 2) continue;
    if (!strcmp(name, "n_seg")) {
      if (!(a >= SWM_MIN_SEGMENTS && a <= SWM_MAX_SEGMENTS && a == (int)a))
        refused = "n_seg must be an integer in " + std::to_string(SWM_MIN_SEGMENTS) + ".." +
                  std::to_string(SWM_MAX_SEGMENTS);
      else if (g_sized_n && (int)a != g_sized_n)
        refused = "n_seg cannot change between env_init and env_cleanup";
      else
        g_params.n = (int)a;
    } else if (!strcmp(name, "max_u")) g_params.max_u = a;
    else if (!strcmp(name, "l_i")) g_params.l_i = a;
    else if (!strcmp(name, "k")) g_params.k = a;
    else if (!strcmp(name, "m_i")) g_params.m_i = a;
    else if (!strcmp(name, "h_global")) g_params.h = a;
    else if (!strcmp(name, "direction") && got == 3) { g_params.direction[0] = a; g_params.direction[1] = b; }
  }
  fclose(f);
  return refused;
}

void copy_obs(observation_t& dst, const observation_t& src) {
  dst.numInts = src.numInts; dst.numDoubles = src.numDoubles; dst.numChars = src.numChars;
  for (unsigned i = 0; i < src.numDoubles; ++i) dst.doubleArray[i] = src.doubleArray[i];
}

}  // namespace

extern "C" {

/* Programmatic alternative to the "set parameters" message (the reference has file globals). */
int swm_rlglue_set_params(const swm_params_t* p) {
  if (!p || p->n < SWM_MIN_SEGMENTS || p->n > SWM_MAX_SEGMENTS) return SWM_ERR_BAD_ARG;
  if (g_sized_n && p->n != g_sized_n) return SWM_ERR_BAD_ARG;
  g_params = *p;
  return SWM_OK;
}

const char* env_init(void) {
  const int n_obs = 2 + 2 * g_params.n, n_action = g_params.n - 1;
  shim_alloc(&this_observation, n_obs);
  shim_alloc(&saved_observation, n_obs);
  this_reward_observation.observation = &this_observation;
  this_reward_observation.reward = 0;
  this_reward_observation.terminal = 0;
  if (cudaMalloc(&d_in, sizeof(double) * (n_obs + n_action)) != cudaSuccess ||
      cudaMalloc(&d_out, sizeof(double) * (n_obs + 1)) != cudaSuccess ||
      cudaMallocHost(&h_in, sizeof(double) * (n_obs + n_action)) != cudaSuccess ||
      cudaMallocHost(&h_out, sizeof(double) * (n_obs + 1)) != cudaSuccess ||
      cudaStreamCreateWithFlags(&g_stream, cudaStreamNonBlocking) != cudaSuccess)
    die("device / pinned allocation failed");
  g_sized_n = g_params.n;
  g_task_spec = "VERSION RL-Glue-3.0 PROBLEMTYPE continuing DISCOUNTFACTOR 0.9 OBSERVATIONS DOUBLES (" +
                std::to_string(n_obs) + " UNSPEC UNSPEC) ACTIONS DOUBLES (" + std::to_string(n_action) +
                " " + std::to_string(-g_params.max_u) + " " + std::to_string(g_params.max_u) +
                ") REWARDS (UNSPEC UNSPEC) EXTRA SwimmerEnvironment(B200) swimmer_ars";
  return g_task_spec.c_str();
}

const observation_t* env_start(void) {
  for (unsigned i = 0; i < this_observation.numDoubles; ++i) this_observation.doubleArray[i] = 0.001;
  copy_obs(saved_observation, this_observation);
  return &this_observation;
}

const reward_observation_terminal_t* env_step(const action_t* this_action) {
  const int n_obs = 2 + 2 * g_params.n, n_action = g_params.n - 1;
  bool valid = (int)this_action->numDoubles == n_action;
  for (int i = 0; valid && i < n_action; ++i)
    valid = fabs(this_action->doubleArray[i]) <= g_params.max_u;
  if (!valid) {
    if (!getenv("SWM_RLGLUE_NO_ABORT")) { fprintf(stderr, "env_step: invalid action\n"); abort(); }
    this_reward_observation.terminal = 1;
    return &this_reward_observation;
  }
  memcpy(h_in, this_observation.doubleArray, sizeof(double) * n_obs);
  memcpy(h_in + n_obs, this_action->doubleArray, sizeof(double) * n_action);
  if (cudaMemcpyAsync(d_in, h_in, sizeof(double) * (n_obs + n_action), cudaMemcpyHostToDevice, g_stream) != cudaSuccess)
    die("H2D copy failed");
  if (swm_step_batched(&g_params, SWM_DYN_RLGLUE, d_in, d_in + n_obs, d_out, d_out + n_obs, 1, g_stream) != SWM_OK)
    die("swm_step_batched failed");
  if (cudaMemcpyAsync(h_out, d_out, sizeof(double) * (n_obs + 1), cudaMemcpyDeviceToHost, g_stream) != cudaSuccess ||
      cudaStreamSynchronize(g_stream) != cudaSuccess)
    die("D2H copy failed");
  memcpy(this_observation.doubleArray, h_out, sizeof(double) * n_obs);
  this_reward_observation.observation = &this_observation;
  this_reward_observation.reward = h_out[n_obs];
  this_reward_observation.terminal = 0;
  return &this_reward_observation;
}

void env_cleanup(void) {
  shim_clear(&this_observation);
  shim_clear(&saved_observation);
  cudaFree(d_in); cudaFree(d_out); cudaFreeHost(h_in); cudaFreeHost(h_out);
  if (g_stream) cudaStreamDestroy(g_stream);
  d_in = d_out = h_in = h_out = nullptr;
  g_stream = nullptr;
  g_sized_n = 0;
}

const char* env_message(const char* message) {
  if (strcmp(message, "what is your name?") == 0) return "My name is swimmer_environment, B200 edition!";
  if (strcmp(message, "save state") == 0) {
    copy_obs(saved_observation, this_observation);
    return "saved_observation has the value of this_observation";
  }
  if (strcmp(message, "load state") == 0) {
    copy_obs(this_observation, saved_observation);
    return "this_observation has the value of saved_observation";
  }
  if (strncmp(message, "set parameters", 14) == 0) {
    const char* path = message[14] == ' ' ? message + 15 : getenv("SWM_PARAMETERS_FILE");
    const std::string refused = set_parameters(path ? path : "../parameters.txt");
    g_param_msg = (refused.empty() ? "" : "Refused: " + refused + "; n_seg unchanged. ") +
                  "Environment parameters are: n_seg=" + std::to_string(g_params.n) +
                  "; max_u=" + std::to_string(g_params.max_u) + "; l_i=" + std::to_string(g_params.l_i) +
                  "; k=" + std::to_string(g_params.k) + "; m_i=" + std::to_string(g_params.m_i) +
                  "; h_global=" + std::to_string(g_params.h);
    return g_param_msg.c_str();
  }
  return "SwimmerEnvironment(B200) does not respond to that message.";
}

}  // extern "C"
