// ARS bookkeeping kernels: direction ranking (top-b), the delta-weighted policy update with
// in-kernel Philox regeneration, deterministic Welford statistics, return reduction and the FP64
// pipe probe.  Everything here is a fixed-order computation: given identical inputs every rank
// produces bit-identical outputs, which is what lets all ranks update W redundantly.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/swimmer_ars.h"
#include "errors.cuh"
#include "philox.cuh"

namespace swm {

constexpr int kArsBlock = 256;

// Ascending total order: by key, NaN last, ties by ascending index.  The descending order the
// reference wants (np.argsort(max_r)[::-1], ars_agent.py:107-108) is its reverse.
__device__ __forceinline__ bool asc_less(double a, int ia, double b, int ib) {
  const bool an = a != a, bn = b != b;
  if (an || bn) return (an && bn) ? (ia < ib) : bn;
  if (a < b) return true;
  if (a > b) return false;
  return ia < ib;
}

// order[rank_i] = i, rank_i = #directions that precede i in descending order.  Rank by counting:
// one warp per direction i, lanes stride over j, integer warp reduction -- O(N^2) comparisons spread
// over 32 N threads, no data-dependent control flow, exact for any N.
__global__ void __launch_bounds__(kArsBlock)
ars_rank_kernel(const double* __restrict__ returns, const int* __restrict__ mask, int N,
                int* __restrict__ order) {
  extern __shared__ double keys[];  // N keys followed by N validity flags (int)
  int* valid = reinterpret_cast<int*>(keys + N);
  for (int i = threadIdx.x; i < N; i += kArsBlock) {
    const double a = returns[2 * i], b = returns[2 * i + 1];
    keys[i] = (b > a) ? b : a;  // Python max(a, b)
    valid[i] = mask ? (mask[i] != 0) : 1;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * (kArsBlock / 32) + (threadIdx.x >> 5);
  if (i >= N) return;
  const double ki = keys[i];
  const int vi = valid[i];
  int rank = 0;
  for (int j = lane; j < N; j += 32) {
    // j precedes i iff (j valid, i not) or (same validity and i <asc j)
    const int vj = valid[j];
    const bool before = (vj != vi) ? (vj > vi) : asc_less(ki, i, keys[j], j);
    rank += (j != i && before) ? 1 : 0;
  }
  rank = __reduce_add_sync(0xffffffffu, rank);
  if (lane == 0) order[rank] = i;
}

__device__ __forceinline__ double block_sum(double v, double* red) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
#pragma unroll
  for (int w = 0; w < kArsBlock / 32; ++w) t += red[w];
  return t;
}

// One CTA per pair of policy elements (2j, 2j+1) = one Philox call per (direction, CTA).
__global__ void __launch_bounds__(kArsBlock)
ars_update_kernel(double* __restrict__ W, int wsize, const double* __restrict__ returns, int N,
                  const int* __restrict__ order, int n_order, const int* __restrict__ mask,
                  double divisor, int ddof, double alpha, uint64_t seed, uint32_t iteration,
                  const uint32_t* __restrict__ iter_dev, uint32_t dir0, int dist,
                  const double* __restrict__ deltas, double* __restrict__ sigma_out) {
  __shared__ double red[kArsBlock / 32];
  const int tid = threadIdx.x;
  if (iter_dev) iteration += *iter_dev;
  int used = min(n_order, N);
  if (mask) {  // only directions that were actually rolled out (sorted first by ars_rank_kernel)
    double c = 0.0;
    for (int i = tid; i < N; i += kArsBlock) c += (mask[i] != 0) ? 1.0 : 0.0;
    used = min(used, (int)block_sum(c, red));
  }
  if (used <= 0) return;
  // sigma_R over the 2*used returns (np.std / statistics.stdev), two passes
  double sacc = 0.0;
  for (int q = tid; q < used; q += kArsBlock) {
    const int k = order ? order[q] : q;
    sacc += returns[2 * k] + returns[2 * k + 1];
  }
  const double mean = block_sum(sacc, red) / (2.0 * used);
  double vacc = 0.0;
  for (int q = tid; q < used; q += kArsBlock) {
    const int k = order ? order[q] : q;
    const double d0 = returns[2 * k] - mean, d1 = returns[2 * k + 1] - mean;
    vacc += d0 * d0 + d1 * d1;
  }
  const double sigma = sqrt(block_sum(vacc, red) / (2.0 * used - (double)ddof));
  // sum_k (r+ - r-) delta_k for this CTA's element pair
  const int j = blockIdx.x;
  double g0 = 0.0, g1 = 0.0;
  for (int q = tid; q < used; q += kArsBlock) {
    const int k = order ? order[q] : q;
    const double coef = returns[2 * k] - returns[2 * k + 1];
    double d0, d1 = 0.0;
    if (deltas) {
      d0 = deltas[(size_t)k * wsize + 2 * j];
      if (2 * j + 1 < wsize) d1 = deltas[(size_t)k * wsize + 2 * j + 1];
    } else {
      philox_delta_pair(seed, iteration, dir0 + (uint32_t)k, 0u, (uint32_t)j, dist, d0, d1);
    }
    g0 = fma(coef, d0, g0);
    g1 = fma(coef, d1, g1);
  }
  g0 = block_sum(g0, red);
  g1 = block_sum(g1, red);
  if (tid == 0) {
    // grad /= (b * sigma_r); policy += alpha * grad   (ars_agent.py:128-130)
    const double scale = (divisor > 0.0 ? divisor : (double)used) * sigma;
    W[2 * j] += alpha * (g0 / scale);
    if (2 * j + 1 < wsize) W[2 * j + 1] += alpha * (g1 / scale);
    if (j == 0 && sigma_out) *sigma_out = sigma;
  }
}

// mask[k] = both simulated returns of direction k exceed the simulator threshold under every one of the M models
// (rows of 2N returns) (ars_agent.py:150-157: `reward <= sim_threshold` => no real rollout).
__global__ void screen_mask_kernel(const double* __restrict__ sim_returns, int M, int N, double threshold,
                                   int* __restrict__ mask, int* __restrict__ n_pass,
                                   long long* __restrict__ n_pass_total) {
  __shared__ double red[kArsBlock / 32];
  double c = 0.0;
  for (int k = threadIdx.x; k < N; k += kArsBlock) {
    // The reference skips on `reward <= sim_threshold`; a NaN simulator return (diverged simulation) compares
    // false there and would be rolled out in the real world.  Declared deviation: NaN is screened out too.
    bool pass = true;
    for (int m = 0; m < M; ++m) {
      const double* r = sim_returns + (long long)m * 2 * N;
      pass = pass && (r[2 * k] > threshold) && (r[2 * k + 1] > threshold);
    }
    const bool skip = !pass;
    mask[k] = skip ? 0 : 1;
    c += skip ? 0.0 : 1.0;
  }
  c = block_sum(c, red);
  if (threadIdx.x == 0 && n_pass) *n_pass = (int)c;
  if (threadIdx.x == 0 && n_pass_total) *n_pass_total += (long long)c;
}

// select_action for a batch (ars/environment.py:19-35)
__global__ void policy_actions_kernel(int n, double max_u, const double* __restrict__ obs,
                                      const double* __restrict__ policies, int R,
                                      const double* __restrict__ mean,
                                      const double* __restrict__ inv_sigma, int clip,
                                      double* __restrict__ actions, long long B) {
  const int no = 2 * n + 2, na = n - 1;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * na) return;
  const long long e = idx / na;
  const int a = (int)(idx % na);
  const double* W = policies + ((e / R) * na + a) * no;
  const double* o = obs + e * no;
  double acc = 0.0;
  for (int j = 0; j < no; ++j) {
    if (mean) acc = fma(W[j] * inv_sigma[j], o[j] - mean[j], acc);
    else acc = fma(W[j], o[j], acc);
  }
  if (clip) acc = fmin(fmax(acc, -max_u), max_u);
  actions[idx] = acc;
}

__global__ void philox_deltas_kernel(uint64_t seed, uint32_t iteration, const uint32_t* iter_dev,
                                     uint32_t dir0, int dist, int count, int wsize,
                                     double* __restrict__ out) {
  if (iter_dev) iteration += *iter_dev;
  const int pairs = (wsize + 1) / 2;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)count * pairs) return;
  const int k = (int)(idx / pairs), j = (int)(idx % pairs);
  double d0, d1;
  philox_delta_pair(seed, iteration, dir0 + (uint32_t)k, 0u, (uint32_t)j, dist, d0, d1);
  out[(size_t)k * wsize + 2 * j] = d0;
  if (2 * j + 1 < wsize) out[(size_t)k * wsize + 2 * j + 1] = d1;
}

// ---- statistics -------------------------------------------------------------------------------
// column c of partial[n_blocks, 2F] summed in a fixed order into record[1 + c]
__global__ void __launch_bounds__(kArsBlock)
stats_colsum_kernel(const double* __restrict__ partial, long long n_blocks, int twoF,
                    double* __restrict__ record) {
  __shared__ double red[kArsBlock / 32];
  const int c = blockIdx.x;
  double acc = 0.0;
  for (long long r = threadIdx.x; r < n_blocks; r += kArsBlock) acc += partial[r * twoF + c];
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) record[1 + c] = acc;
}

// shifted sums -> (count, mean, M2):  mean = pivot + S1/n,  M2 = S2 - S1^2/n
__global__ void stats_convert_kernel(double* __restrict__ record, int F, double samples,
                                     const int* __restrict__ units, const double* __restrict__ pivot) {
  const int f = threadIdx.x;
  if (units) samples *= (double)(*units);
  double s1 = 0.0, s2 = 0.0;
  if (f < F) { s1 = record[1 + f]; s2 = record[1 + F + f]; }
  __syncthreads();
  if (f < F) {
    record[1 + f] = samples > 0.0 ? pivot[f] + s1 / samples : 0.0;
    record[1 + F + f] = samples > 0.0 ? fmax(s2 - s1 * (s1 / samples), 0.0) : 0.0;
  }
  if (f == 0) record[0] = samples;
}

// running <- merge(running, records[0], records[1], ...) in index order (Chan et al. 1979)
__global__ void stats_merge_kernel(double* __restrict__ running, const double* __restrict__ records,
                                   int n_records, int F, double* __restrict__ mean_out,
                                   double* __restrict__ inv_sigma_out) {
  const int f = threadIdx.x;
  if (f >= F) return;
  const int stride = 1 + 2 * F;
  double na = running[0], ma = running[1 + f], Ma = running[1 + F + f];
  for (int r = 0; r < n_records; ++r) {
    const double* rec = records + (size_t)r * stride;
    const double nb = rec[0], mb = rec[1 + f], Mb = rec[1 + F + f];
    if (nb <= 0.0) continue;
    if (na <= 0.0) { na = nb; ma = mb; Ma = Mb; continue; }
    const double n = na + nb, d = mb - ma;
    ma = ma + d * (nb / n);
    Ma = Ma + Mb + d * d * (na * (nb / n));
    na = n;
  }
  __syncthreads();
  running[1 + f] = ma;
  running[1 + F + f] = Ma;
  if (f == 0) running[0] = na;
  // ars_agent.py:179-182 only recomputes mean / cov `if len(rewards) > 0`: while nothing has been observed
  // (every direction screened out so far) the initial mean = 0, cov = I stay in place; np.cov needs >= 2 samples
  if (na >= 2.0) {
    if (mean_out) mean_out[f] = ma;
    if (inv_sigma_out) inv_sigma_out[f] = 1.0 / sqrt(Ma / (na - 1.0));  // diag(np.cov)**(-1/2)
  }
}

__global__ void reduce_returns_kernel(const double* __restrict__ returns, long long n_groups, int R,
                                      double* __restrict__ out) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_groups) return;
  double acc = 0.0;
  for (int r = 0; r < R; ++r) acc += returns[g * R + r];
  out[g] = acc / R;
}

// ---- FP64 pipe probe --------------------------------------------------------------------------
__global__ void fp64_probe_kernel(int iters, double* __restrict__ sink) {
  double x0 = 1.0 + threadIdx.x * 1e-9, x1 = x0 + 1e-3, x2 = x0 + 2e-3, x3 = x0 + 3e-3;
  double x4 = x0 + 4e-3, x5 = x0 + 5e-3, x6 = x0 + 6e-3, x7 = x0 + 7e-3;
  const double a = 0.999999999, b = 1e-9;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
      x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
  }
  const double s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
  if (s == 123.456) sink[0] = s;  // never true; keeps the chains alive
}

__global__ void counter_add_kernel(uint32_t* counter, uint32_t inc) { *counter += inc; }

// mean of the non-NaN entries, fixed-order block reduction (one CTA)
__global__ void __launch_bounds__(kArsBlock)
record_nanmean_kernel(const double* __restrict__ x, int n, double* __restrict__ curve,
                      const uint32_t* __restrict__ index, uint32_t capacity) {
  __shared__ double red[kArsBlock / 32];
  double s = 0.0, c = 0.0;
  for (int i = threadIdx.x; i < n; i += kArsBlock) {
    const double v = x[i];
    if (v == v) { s += v; c += 1.0; }
  }
  s = block_sum(s, red);
  __syncthreads();
  c = block_sum(c, red);
  if (threadIdx.x == 0) {
    uint32_t at = index ? *index : 0u;
    if (at >= capacity) at = capacity - 1;
    curve[at] = (c > 0.0) ? s / c : __longlong_as_double(0x7ff8000000000000LL);
  }
}

}  // namespace swm

using namespace swm;

#define SWM_CHECK_LAUNCH() swm::check_launch()

extern "C" int swm_ars_topb(const double* returns, const int32_t* mask, int N, int32_t* order,
                            void* stream) {
  if (!returns || !order || N < 1) return SWM_ERR_BAD_ARG;
  const size_t smem = (size_t)N * (sizeof(double) + sizeof(int));
  if (smem > 200 * 1024) return SWM_ERR_UNSUPPORTED;
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(ars_rank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return SWM_ERR_CUDA;
  const int per_block = kArsBlock / 32;
  ars_rank_kernel<<<(N + per_block - 1) / per_block, kArsBlock, smem, (cudaStream_t)stream>>>(
      returns, mask, N, order);
  return SWM_CHECK_LAUNCH();
}

extern "C" int swm_ars_update(double* W, int wsize, const double* returns, int N,
                              const int32_t* order, int n_order, const int32_t* mask, double divisor,
                              int ddof, double alpha, const swm_philox_t* philox,
                              const double* deltas, double* sigma_out, void* stream) {
  if (!W || !returns || wsize < 1 || N < 1 || n_order < 0) return SWM_ERR_BAD_ARG;
  if (ddof != 0 && ddof != 1) return SWM_ERR_BAD_ARG;
  if (mask && !order) return SWM_ERR_BAD_ARG;
  if (!deltas && !philox) return SWM_ERR_BAD_ARG;
  if (n_order == 0) return SWM_OK;
  const uint64_t seed = philox ? philox->seed : 0;
  const uint32_t it = philox ? philox->iteration : 0, d0 = philox ? philox->dir0 : 0;
  const int dist = philox ? philox->dist : 0;
  ars_update_kernel<<<(wsize + 1) / 2, kArsBlock, 0, (cudaStream_t)stream>>>(
      W, wsize, returns, N, order, n_order, mask, divisor, ddof, alpha, seed, it,
      philox ? philox->iteration_dev : nullptr, d0, dist, deltas, sigma_out);
  return SWM_CHECK_LAUNCH();
}

extern "C" int swm_screen_mask(const double* sim_returns, int N, double threshold, int32_t* mask,
                               int32_t* n_pass, int64_t* n_pass_total, void* stream) {
  return swm_screen_mask_models(sim_returns, 1, N, threshold, mask, n_pass, n_pass_total, stream);
}

extern "C" int swm_screen_mask_models(const double* sim_returns, int n_models, int N, double threshold, int32_t* mask,
                                      int32_t* n_pass, int64_t* n_pass_total, void* stream) {
  if (!sim_returns || !mask || N < 1 || n_models < 1 || n_models > SWM_MAX_SIM_MODELS) return SWM_ERR_BAD_ARG;
  screen_mask_kernel<<<1, kArsBlock, 0, (cudaStream_t)stream>>>(sim_returns, n_models, N, threshold, mask, n_pass,
                                                              reinterpret_cast<long long*>(n_pass_total));
  return SWM_CHECK_LAUNCH();
}

extern "C" int swm_policy_actions(const swm_params_t* params, const double* obs,
                                  const double* policies, int rollouts_per_policy,
                                  const double* mean, const double* inv_sigma, int clip,
                                  double* actions, int64_t B, void* stream) {
  if (!params || params->n < SWM_MIN_SEGMENTS || params->n > SWM_MAX_SEGMENTS) return SWM_ERR_BAD_ARG;
  if (!obs || !policies || !actions || B < 0 || rollouts_per_policy < 1) return SWM_ERR_BAD_ARG;
  if ((mean == nullptr) != (inv_sigma == nullptr)) return SWM_ERR_BAD_ARG;
  if (B == 0) return SWM_OK;
  const long long total = B * (params->n - 1);
  policy_actions_kernel<<<(unsigned)((total + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      params->n, params->max_u, obs, policies, rollouts_per_policy, mean, inv_sigma, clip, actions, B);
  return SWM_CHECK_LAUNCH();
}

extern "C" int swm_philox_deltas(const swm_philox_t* philox, int count, int wsize, double* out,
                                 void* stream) {
  if (!philox || !out || count < 1 || wsize < 1) return SWM_ERR_BAD_ARG;
  const long long total = (long long)count * ((wsize + 1) / 2);
  philox_deltas_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      philox->seed, philox->iteration, philox->iteration_dev, philox->dir0, philox->dist, count, wsize, out);
  return SWM_CHECK_LAUNCH();
}

extern "C" int swm_stats_finalize(const double* partial, int64_t n_blocks, int n_features,
                                  double samples, const int32_t* units, const double* pivot,
                                  double* out_record, void* stream) {
  if (!partial || !pivot || !out_record || n_blocks < 1 || n_features < 1 || n_features > 512)
    return SWM_ERR_BAD_ARG;
  stats_colsum_kernel<<<2 * n_features, kArsBlock, 0, (cudaStream_t)stream>>>(
      partial, n_blocks, 2 * n_features, out_record);
  stats_convert_kernel<<<1, ((n_features + 31) / 32) * 32, 0, (cudaStream_t)stream>>>(
      out_record, n_features, samples, units, pivot);
  return SWM_CHECK_LAUNCH();
}

extern "C" int swm_stats_merge(double* running, const double* records, int n_records,
                               int n_features, double* mean_out, double* inv_sigma_out,
                               void* stream) {
  if (!running || (!records && n_records > 0) || n_features < 1 || n_features > 512 || n_records < 0)
    return SWM_ERR_BAD_ARG;
  stats_merge_kernel<<<1, ((n_features + 31) / 32) * 32, 0, (cudaStream_t)stream>>>(
      running, records, n_records, n_features, mean_out, inv_sigma_out);
  return SWM_CHECK_LAUNCH();
}

extern "C" int swm_reduce_returns(const double* returns, int64_t n_groups, int R, double* out,
                                  void* stream) {
  if (!returns || !out || n_groups < 1 || R < 1) return SWM_ERR_BAD_ARG;
  reduce_returns_kernel<<<(unsigned)((n_groups + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      returns, n_groups, R, out);
  return SWM_CHECK_LAUNCH();
}

extern "C" int swm_fp64_probe(int blocks, int threads, int iters, double* sink, double* flops_out,
                              void* stream) {
  if (blocks < 1 || threads < 1 || threads > 1024 || iters < 1 || !sink) return SWM_ERR_BAD_ARG;
  fp64_probe_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(iters, sink);
  if (flops_out) *flops_out = 2.0 * 64.0 * (double)iters * (double)blocks * (double)threads;
  return SWM_CHECK_LAUNCH();
}

extern "C" int swm_counter_add(uint32_t* counter, uint32_t inc, void* stream) {
  if (!counter) return SWM_ERR_BAD_ARG;
  counter_add_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(counter, inc);
  return SWM_CHECK_LAUNCH();
}

extern "C" int swm_record_nanmean(const double* x, int n, double* curve, const uint32_t* index,
                                  uint32_t capacity, void* stream) {
  if (!x || !curve || n < 1 || capacity < 1) return SWM_ERR_BAD_ARG;
  record_nanmean_kernel<<<1, kArsBlock, 0, (cudaStream_t)stream>>>(x, n, curve, index, capacity);
  return SWM_CHECK_LAUNCH();
}
