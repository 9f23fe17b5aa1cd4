// Simulator-model estimation on the device (include/swimmer_ars.h, "Simulator-model estimation"):
//   - the prediction-error objective of Estimator.I (ars/estimator.py:36-62) for a whole population of
//     candidate models in one launch (+ a small fixed-order reduction launch);
//   - CMA-ES (Hansen's tutorial, default strategy parameters, no active update) with all of its state in one
//     device buffer: a sampling kernel, the objective and a one-CTA update kernel per generation, so that a
//     run is a replayable CUDA graph with no host round trip (replaces the `cma` package call of
//     ars/estimator.py:103).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/swimmer_ars.h"
#include "dynamics.cuh"
#include "errors.cuh"
#include "kernels.cuh"
#include "philox.cuh"

namespace swm {
namespace {

constexpr int kEstBlock = 128;  // threads per CTA of the objective: one recorded transition each
constexpr int kEstWarps = kEstBlock / 32;
constexpr int kPhysDoubles = sizeof(Phys) / sizeof(double);
constexpr int kJacobiSweeps = 12;    // d <= 3 converges to rounding in ~4 sweeps; a fixed count keeps it deterministic
constexpr double kMaxCondition = 1e14;
constexpr uint32_t kCmaesStream = 2;  // Philox stream (0: ARS directions, 1: initial-state perturbations)

struct EstArgs {
  swm_params_t base;
  const double* traj;
  const double* pol;
  int K, H, d;
  int fields[3];
  const double* cand;
  int M;
  double* partial;       // [gridDim.x, M]
  const double* status;  // CMA-ES status word (generation call) or NULL
};

__host__ __device__ inline swm_params_t candidate_params(const swm_params_t& base, const int* fields, int d,
                                                         const double* x) {
  swm_params_t p = base;
  for (int i = 0; i < d; ++i) {
    if (fields[i] == SWM_FIELD_M_I) p.m_i = x[i];
    else if (fields[i] == SWM_FIELD_L_I) p.l_i = x[i];
    else p.k = x[i];
  }
  return p;
}

// A mass or length that is not positive and finite is non-physical.  NaN fails every comparison; an infinite
// mass must be refused explicitly, since it zeroes the torque and friction constants of make_phys and would
// otherwise step to a finite error.
__host__ __device__ inline bool physical(double m, double l) {
  return m > 0.0 && l > 0.0 && isfinite(m) && isfinite(l);
}

// One thread = one recorded transition (k, t).  The state, its sines/cosines and the V1 action W_k s do not
// depend on the model, so they are formed once; the loop then steps every candidate model (constants in shared
// memory, a warp-uniform broadcast) and reduces each candidate's error over the warp with a fixed butterfly.
template <int N>
__global__ void __launch_bounds__(kEstBlock) prediction_kernel(const EstArgs a) {
  if (a.status && *a.status != 0.0) return;
  constexpr int NO = 2 * N + 2, NA = N - 1, WS = NA * NO;
  constexpr int FS = FactSmem<N, 0>::on ? kEstBlock : 0;
  extern __shared__ __align__(16) double smem[];
  Phys* sP = reinterpret_cast<Phys*>(smem);
  double* red = smem + (size_t)a.M * kPhysDoubles;  // [kEstWarps, M]
  double* fs = red + (size_t)kEstWarps * a.M + threadIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int c = tid; c < a.M; c += kEstBlock)
    sP[c] = make_phys(candidate_params(a.base, a.fields, a.d, a.cand + (size_t)c * a.d));

  const long long T = (long long)a.K * (a.H - 1);
  const long long i0 = (long long)blockIdx.x * kEstBlock + tid;
  const bool active = i0 < T;
  const long long i = active ? i0 : T - 1;  // idle lanes shadow the last transition and add 0
  const long long k = i / (a.H - 1), t = i % (a.H - 1);
  const double* s0 = a.traj + (k * a.H + t) * NO;
  const double* s1 = s0 + NO;
  double gdx = s0[0], gdy = s0[1], th[N], thd[N], sn[N], cs[N], u[NA > 0 ? NA : 1];
#pragma unroll
  for (int q = 0; q < N; ++q) { th[q] = s0[2 + 2 * q]; thd[q] = s0[3 + 2 * q]; }
  // select_action V1 (ars/environment.py:27-30), summed like swm_policy_actions
  const double* W = a.pol + k * WS;
#pragma unroll
  for (int r = 0; r < NA; ++r) {
    double acc = 0.0;
#pragma unroll
    for (int j = 0; j < NO; ++j) acc = fma(W[r * NO + j], s0[j], acc);
    u[r] = acc;
  }
#pragma unroll
  for (int q = 0; q < N; ++q) sincos(th[q], &sn[q], &cs[q]);
  __syncthreads();

#pragma unroll 1
  for (int c = 0; c < a.M; ++c) {
    const Phys& P = sP[c];
    double e = 0.0;
    if (physical(P.m, P.l)) {  // uniform over the CTA
      // swimmer_step<N, 0> from the precomputed sines/cosines
      double ut[NA > 0 ? NA : 1], gddx, gddy, thdd[N];
#pragma unroll
      for (int r = 0; r < NA; ++r) ut[r] = u[r] * P.u_scale;
      gym_accel<N, FS>(P, sn, cs, gdx, gdy, thd, ut, gddx, gddy, thdd, fs);
      gddx *= P.gdd_c;
      gddy *= P.gdd_c;
      const double ex = fma(P.h, gddx, gdx) - s1[0], ey = fma(P.h, gddy, gdy) - s1[1];
      double ss = fma(ex, ex, ey * ey);
#pragma unroll
      for (int q = 0; q < N; ++q) {
        const double et = fma(P.h, thd[q], th[q]) - s1[2 + 2 * q];
        const double ed = fma(P.h, thdd[q], thd[q]) - s1[3 + 2 * q];
        ss = fma(et, et, ss);
        ss = fma(ed, ed, ss);
      }
      e = active ? sqrt(ss) : 0.0;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) e += __shfl_xor_sync(0xffffffffu, e, off);
    if (lane == 0) red[warp * a.M + c] = e;
  }
  __syncthreads();
  for (int c = tid; c < a.M; c += kEstBlock) {
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < kEstWarps; ++w) v += red[w * a.M + c];
    a.partial[(size_t)blockIdx.x * a.M + c] = v;
  }
}

// err[c] = sum of the CTA partials in CTA order; non-physical candidates and non-finite sums -> +inf
__global__ void prediction_reduce_kernel(const EstArgs a, long long n_blocks, double* __restrict__ err) {
  if (a.status && *a.status != 0.0) return;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= a.M) return;
  double v = 0.0;
  for (long long b = 0; b < n_blocks; ++b) v += a.partial[b * a.M + c];
  const swm_params_t p = candidate_params(a.base, a.fields, a.d, a.cand + (size_t)c * a.d);
  err[c] = (physical(p.m_i, p.l_i) && isfinite(v)) ? v : __longlong_as_double(0x7ff0000000000000LL);
}

// ---- CMA-ES -----------------------------------------------------------------------------------------------
struct Layout {  // offsets into the state buffer (include/swimmer_ars.h)
  int d, lam, L;
  int mean, best_x, ps, pc, D, C, B, hist, z, total;
  __host__ __device__ Layout(int d_, int lam_) : d(d_), lam(lam_) {
    L = 10 + (30 * d + lam - 1) / lam;
    mean = 7; best_x = mean + d; ps = best_x + d; pc = ps + d; D = pc + d; C = D + d; B = C + d * d;
    hist = B + d * d; z = hist + L; total = z + lam * d;
  }
};
enum { kGen = 0, kStatus = 1, kSigma = 2, kBestF = 3, kMaxGen = 4, kTolfun = 5, kTolx = 6 };

struct InitArgs {
  double x0[3], sigma0, tolfun, tolx, max_gen;
};

__global__ void cmaes_init_kernel(double* __restrict__ S, int d, int lam, InitArgs a) {
  const Layout Ly(d, lam);
  for (int j = threadIdx.x; j < Ly.total; j += blockDim.x) S[j] = 0.0;
  __syncthreads();
  if (threadIdx.x != 0) return;
  S[kSigma] = a.sigma0;
  S[kBestF] = __longlong_as_double(0x7ff0000000000000LL);
  S[kMaxGen] = a.max_gen;
  S[kTolfun] = a.tolfun;
  S[kTolx] = a.tolx;
  for (int i = 0; i < d; ++i) {
    S[Ly.mean + i] = a.x0[i];
    S[Ly.best_x + i] = a.x0[i];
    S[Ly.D + i] = 1.0;
    S[Ly.C + i * d + i] = 1.0;
    S[Ly.B + i * d + i] = 1.0;
  }
}

// y = B (D .* z), the same arithmetic in the sampling and in the update kernel
__device__ __forceinline__ void scale_rotate(const double* S, const Layout& Ly, const double* z, double* y) {
  for (int i = 0; i < Ly.d; ++i) {
    double v = 0.0;
    for (int j = 0; j < Ly.d; ++j) v = fma(S[Ly.B + i * Ly.d + j], S[Ly.D + j] * z[j], v);
    y[i] = v;
  }
}

__global__ void cmaes_sample_kernel(double* __restrict__ S, int d, int lam, uint64_t seed,
                                    double* __restrict__ cand) {
  if (S[kStatus] != 0.0) return;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= lam) return;
  const Layout Ly(d, lam);
  const uint32_t gen = (uint32_t)S[kGen];
  double z[4], y[3];
  for (int j = 0; 2 * j < d; ++j) {
    uint32_t o[4];
    philox4x32_10((uint32_t)j, (uint32_t)c, gen, kCmaesStream, (uint32_t)seed, (uint32_t)(seed >> 32), o);
    const double u1 = 1.0 - u53(o[0], o[1]), u2 = u53(o[2], o[3]);  // u1 in (0, 1]: log never sees 0
    const double r = sqrt(-2.0 * log(u1));
    double sa, ca;
    sincospi(2.0 * u2, &sa, &ca);
    z[2 * j] = r * ca;
    z[2 * j + 1] = r * sa;
  }
  scale_rotate(S, Ly, z, y);
  const double sigma = S[kSigma];
  for (int i = 0; i < d; ++i) {
    S[Ly.z + c * d + i] = z[i];
    cand[c * d + i] = fma(sigma, y[i], S[Ly.mean + i]);
  }
}

// ascending by fitness, NaN / +inf last (-inf is an ordinary value and ranks first), ties by lower index
__device__ __forceinline__ bool fit_less(double a, int ia, double b, int ib) {
  const bool an = !(a < __longlong_as_double(0x7ff0000000000000LL)), bn = !(b < __longlong_as_double(0x7ff0000000000000LL));
  if (an || bn) return (an && bn) ? (ia < ib) : bn;
  if (a < b) return true;
  if (a > b) return false;
  return ia < ib;
}

// symmetric A (d x d, row-major) -> eigenvalues on its diagonal, eigenvectors in the columns of V
__device__ void jacobi_eigen(int d, double* A, double* V) {
  for (int i = 0; i < d * d; ++i) V[i] = (i % (d + 1) == 0) ? 1.0 : 0.0;
  for (int sweep = 0; sweep < kJacobiSweeps; ++sweep) {
    for (int p = 0; p < d - 1; ++p) {
      for (int q = p + 1; q < d; ++q) {
        const double apq = A[p * d + q];
        if (apq == 0.0) continue;
        const double theta = (A[q * d + q] - A[p * d + p]) / (2.0 * apq);
        const double t = fabs(theta) > 1e150 ? 0.5 / theta
                                              : copysign(1.0, theta) / (fabs(theta) + sqrt(fma(theta, theta, 1.0)));
        const double c = 1.0 / sqrt(fma(t, t, 1.0)), s = t * c;
        A[p * d + p] -= t * apq;
        A[q * d + q] += t * apq;
        A[p * d + q] = A[q * d + p] = 0.0;
        for (int r = 0; r < d; ++r) {
          if (r != p && r != q) {
            const double arp = A[r * d + p], arq = A[r * d + q];
            A[r * d + p] = A[p * d + r] = c * arp - s * arq;
            A[r * d + q] = A[q * d + r] = s * arp + c * arq;
          }
          const double vrp = V[r * d + p], vrq = V[r * d + q];
          V[r * d + p] = c * vrp - s * vrq;
          V[r * d + q] = s * vrp + c * vrq;
        }
      }
    }
  }
}

// One CTA: every thread ranks one candidate by counting, then thread 0 runs the d <= 3 arithmetic.  The CTA has
// up to SWM_MAX_CANDIDATES threads: the launch bound keeps the kernel within the register file at that size.
__global__ void __launch_bounds__(SWM_MAX_CANDIDATES) cmaes_update_kernel(double* __restrict__ S, int d, int lam, const double* __restrict__ cand,
                                    const double* __restrict__ fit) {
  __shared__ int order[SWM_MAX_CANDIDATES];
  if (S[kStatus] != 0.0) return;
  for (int c = threadIdx.x; c < lam; c += blockDim.x) {
    const double fc = fit[c];
    int rank = 0;
    for (int j = 0; j < lam; ++j) rank += fit_less(fit[j], j, fc, c) ? 1 : 0;
    order[rank] = c;
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  const Layout Ly(d, lam);
  const double n = (double)d;
  const int mu = lam / 2;
  // strategy parameters (tutorial, Table 1, positive weights only)
  double wsum = 0.0, w2sum = 0.0;
  for (int i = 1; i <= mu; ++i) {
    const double w = log((lam + 1) / 2.0) - log((double)i);
    wsum += w;
    w2sum += w * w;
  }
  const double mueff = wsum * wsum / w2sum;
  const double cs = (mueff + 2.0) / (n + mueff + 5.0);
  const double ds = 1.0 + 2.0 * fmax(0.0, sqrt((mueff - 1.0) / (n + 1.0)) - 1.0) + cs;
  const double cc = (4.0 + mueff / n) / (n + 4.0 + 2.0 * mueff / n);
  const double c1 = 2.0 / ((n + 1.3) * (n + 1.3) + mueff);
  const double cmu = fmin(1.0 - c1, 2.0 * (mueff - 2.0 + 1.0 / mueff) / ((n + 2.0) * (n + 2.0) + mueff));
  const double chiN = sqrt(n) * (1.0 - 1.0 / (4.0 * n) + 1.0 / (21.0 * n * n));
  const double sigma = S[kSigma];
  const double gen = S[kGen] + 1.0;

  // recombination: <y>_w, <z>_w and the rank-mu matrix sum_i w_i y_i y_i^T
  double yw[3] = {0, 0, 0}, zw[3] = {0, 0, 0}, rmu[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int i = 1; i <= mu; ++i) {
    const double w = (log((lam + 1) / 2.0) - log((double)i)) / wsum;
    const double* z = S + Ly.z + order[i - 1] * d;
    double y[3];
    scale_rotate(S, Ly, z, y);
    for (int a = 0; a < d; ++a) {
      yw[a] = fma(w, y[a], yw[a]);
      zw[a] = fma(w, z[a], zw[a]);
      for (int b = 0; b < d; ++b) rmu[a * d + b] = fma(w * y[a], y[b], rmu[a * d + b]);
    }
  }
  for (int a = 0; a < d; ++a) S[Ly.mean + a] = fma(sigma, yw[a], S[Ly.mean + a]);
  // step-size path: C^{-1/2} <y>_w = B <z>_w
  const double fs = sqrt(cs * (2.0 - cs) * mueff);
  double ps2 = 0.0;
  for (int a = 0; a < d; ++a) {
    double bz = 0.0;
    for (int b = 0; b < d; ++b) bz = fma(S[Ly.B + a * d + b], zw[b], bz);
    const double v = fma(1.0 - cs, S[Ly.ps + a], fs * bz);
    S[Ly.ps + a] = v;
    ps2 = fma(v, v, ps2);
  }
  const double psn = sqrt(ps2);
  const bool hsig = psn / sqrt(1.0 - pow(1.0 - cs, 2.0 * gen)) < (1.4 + 2.0 / (n + 1.0)) * chiN;
  const double fc = hsig ? sqrt(cc * (2.0 - cc) * mueff) : 0.0;
  for (int a = 0; a < d; ++a) S[Ly.pc + a] = fma(1.0 - cc, S[Ly.pc + a], fc * yw[a]);
  const double dh = hsig ? 0.0 : cc * (2.0 - cc);
  const double keep = 1.0 + c1 * dh - c1 - cmu;
  double A[9], V[9];
  for (int a = 0; a < d; ++a) {
    for (int b = a; b < d; ++b) {
      const double pa = S[Ly.pc + a], pb = S[Ly.pc + b];
      const double v = keep * S[Ly.C + a * d + b] + c1 * (pa * pb) + cmu * rmu[a * d + b];
      S[Ly.C + a * d + b] = S[Ly.C + b * d + a] = v;
      A[a * d + b] = A[b * d + a] = v;
    }
  }
  const double sigma_new = sigma * exp((cs / ds) * (psn / chiN - 1.0));
  S[kSigma] = sigma_new;
  jacobi_eigen(d, A, V);
  double ev_min = A[0], ev_max = A[0];
  for (int a = 0; a < d; ++a) {
    const double ev = A[a * d + a];
    ev_min = fmin(ev_min, ev);
    ev_max = fmax(ev_max, ev);
    S[Ly.D + a] = sqrt(fmax(ev, 0.0));
    for (int b = 0; b < d; ++b) S[Ly.B + a * d + b] = V[a * d + b];
  }

  // best ever, best-f history, stop tests
  const double fbest = fit[order[0]];
  if (fbest < S[kBestF]) {
    S[kBestF] = fbest;
    for (int a = 0; a < d; ++a) S[Ly.best_x + a] = cand[order[0] * d + a];
  }
  const long long g0 = (long long)S[kGen];
  S[Ly.hist + (int)(g0 % Ly.L)] = fbest;
  S[kGen] = gen;
  int status = SWM_CMAES_RUNNING;
  if (gen >= Ly.L) {
    double lo = fbest, hi = fit[order[lam - 1]];
    for (int j = 0; j < Ly.L; ++j) { lo = fmin(lo, S[Ly.hist + j]); hi = fmax(hi, S[Ly.hist + j]); }
    if (hi - lo < S[kTolfun]) status = SWM_CMAES_STOP_TOLFUN;
  }
  if (status == SWM_CMAES_RUNNING) {
    bool small = true;
    for (int a = 0; a < d; ++a)
      small = small && sigma_new * sqrt(S[Ly.C + a * d + a]) < S[kTolx] && sigma_new * fabs(S[Ly.pc + a]) < S[kTolx];
    if (small) status = SWM_CMAES_STOP_TOLX;
  }
  if (status == SWM_CMAES_RUNNING && !(ev_min > 0.0 && ev_max / ev_min <= kMaxCondition))
    status = SWM_CMAES_STOP_CONDITIONCOV;
  if (status == SWM_CMAES_RUNNING && gen >= S[kMaxGen]) status = SWM_CMAES_STOP_MAXITER;
  S[kStatus] = (double)status;
}

// ---- host side --------------------------------------------------------------------------------------------
bool fields_ok(int d, const int* f) {
  if (d < 1 || d > 3) return false;
  for (int i = 0; i < d; ++i) {
    if (f[i] < SWM_FIELD_M_I || f[i] > SWM_FIELD_K) return false;
    for (int j = 0; j < i; ++j)
      if (f[i] == f[j]) return false;
  }
  return true;
}

long long objective_blocks(int K, int H) { return ((long long)K * (H - 1) + kEstBlock - 1) / kEstBlock; }

size_t objective_smem(int n, int M) {
  const size_t fs = n >= kFactSmemMinN ? (kFactSmemRhsOnly ? 2 : 5) * (size_t)(n - 1) * kEstBlock : 0;
  return ((size_t)M * (kPhysDoubles + kEstWarps) + fs) * sizeof(double);
}

template <int N>
int launch_prediction(const EstArgs& a, long long blocks, double* err, cudaStream_t st) {
  const size_t smem = objective_smem(N, a.M);
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(prediction_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch();
  prediction_kernel<N><<<(unsigned)blocks, kEstBlock, smem, st>>>(a);
  prediction_reduce_kernel<<<(a.M + 127) / 128, 128, 0, st>>>(a, blocks, err);
  return check_launch();
}

bool objective_args_ok(const swm_params_t* base, const swm_estimate_data_t* data) {
  if (!base || !data || base->n < SWM_MIN_SEGMENTS || base->n > SWM_MAX_SEGMENTS) return false;
  if (!fields_ok(data->d, data->fields)) return false;
  if (data->K < 1 || data->H < 2 || (long long)data->K * (data->H - 1) > 0x7fffffffLL * kEstBlock) return false;
  return data->trajectories && data->policies && data->workspace;
}

int prediction_error(const swm_params_t* base, const swm_estimate_data_t* data, const double* cand, int M,
                     double* err, const double* status, cudaStream_t st) {
  if (!objective_args_ok(base, data) || M < 1 || M > SWM_MAX_CANDIDATES || !cand || !err) return SWM_ERR_BAD_ARG;
  EstArgs a;
  a.base = *base;
  a.traj = data->trajectories;
  a.pol = data->policies;
  a.K = data->K;
  a.H = data->H;
  a.d = data->d;
  for (int i = 0; i < 3; ++i) a.fields[i] = i < data->d ? data->fields[i] : 0;
  a.cand = cand;
  a.M = M;
  a.partial = data->workspace;
  a.status = status;
  const long long blocks = objective_blocks(a.K, a.H);
  switch (base->n) {
    case 2: return launch_prediction<2>(a, blocks, err, st);
    case 3: return launch_prediction<3>(a, blocks, err, st);
    case 4: return launch_prediction<4>(a, blocks, err, st);
    case 5: return launch_prediction<5>(a, blocks, err, st);
    case 6: return launch_prediction<6>(a, blocks, err, st);
    case 7: return launch_prediction<7>(a, blocks, err, st);
    case 8: return launch_prediction<8>(a, blocks, err, st);
    case 9: return launch_prediction<9>(a, blocks, err, st);
    default: return launch_prediction<10>(a, blocks, err, st);
  }
}

bool cmaes_dims_ok(int d, int lam) {
  return d >= 1 && d <= 3 && lam >= SWM_CMAES_MIN_POPSIZE && lam <= SWM_MAX_CANDIDATES;
}

int cmaes_sample(double* state, int d, int lam, uint64_t seed, double* cand, cudaStream_t st) {
  cmaes_sample_kernel<<<(lam + 127) / 128, 128, 0, st>>>(state, d, lam, seed, cand);
  return check_launch();
}

int cmaes_update(double* state, int d, int lam, const double* cand, const double* fit, cudaStream_t st) {
  cmaes_update_kernel<<<1, ((lam + 31) / 32) * 32, 0, st>>>(state, d, lam, cand, fit);
  return check_launch();
}

}  // namespace
}  // namespace swm

using namespace swm;

extern "C" int64_t swm_prediction_error_workspace_doubles(int K, int H, int M) {
  if (K < 1 || H < 2 || M < 1) return 0;
  return (int64_t)objective_blocks(K, H) * M;
}

extern "C" int swm_prediction_error(const swm_params_t* base, const swm_estimate_data_t* data,
                                    const double* candidates, int M, double* err, void* stream) {
  return prediction_error(base, data, candidates, M, err, nullptr, (cudaStream_t)stream);
}

extern "C" int64_t swm_cmaes_state_doubles(int d, int lambda) {
  if (!cmaes_dims_ok(d, lambda)) return 0;
  return Layout(d, lambda).total;
}

extern "C" int swm_cmaes_init(double* state, int d, int lambda, const double* x0, double sigma0, double tolfun,
                              double tolx, int64_t max_generations, void* stream) {
  if (!state || !x0 || !cmaes_dims_ok(d, lambda) || !(sigma0 > 0.0) || !(tolfun >= 0.0) || !(tolx >= 0.0))
    return SWM_ERR_BAD_ARG;
  InitArgs a;
  for (int i = 0; i < 3; ++i) a.x0[i] = i < d ? x0[i] : 0.0;
  a.sigma0 = sigma0;
  a.tolfun = tolfun;
  a.tolx = tolx;
  // the cma package's default maxiter: 100 + 150 * (N+3)**2 // popsize**0.5
  a.max_gen = max_generations > 0 ? (double)max_generations
                                   : 100.0 + floor(150.0 * (d + 3) * (d + 3) / sqrt((double)lambda));
  cmaes_init_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(state, d, lambda, a);
  return check_launch();
}

extern "C" int swm_cmaes_sample(double* state, int d, int lambda, uint64_t seed, double* candidates,
                                void* stream) {
  if (!state || !candidates || !cmaes_dims_ok(d, lambda)) return SWM_ERR_BAD_ARG;
  return cmaes_sample(state, d, lambda, seed, candidates, (cudaStream_t)stream);
}

extern "C" int swm_cmaes_update(double* state, int d, int lambda, const double* candidates, const double* fitness,
                                void* stream) {
  if (!state || !candidates || !fitness || !cmaes_dims_ok(d, lambda)) return SWM_ERR_BAD_ARG;
  return cmaes_update(state, d, lambda, candidates, fitness, (cudaStream_t)stream);
}

extern "C" int swm_cmaes_generation(double* state, int d, int lambda, uint64_t seed, const swm_params_t* base,
                                    const swm_estimate_data_t* data, double* candidates, double* fitness,
                                    void* stream) {
  if (!state || !candidates || !fitness || !data || !cmaes_dims_ok(d, lambda) || data->d != d)
    return SWM_ERR_BAD_ARG;
  if (!objective_args_ok(base, data)) return SWM_ERR_BAD_ARG;  // before anything is enqueued
  cudaStream_t st = (cudaStream_t)stream;
  int rc = cmaes_sample(state, d, lambda, seed, candidates, st);
  if (rc == SWM_OK) rc = prediction_error(base, data, candidates, lambda, fitness, state + kStatus, st);
  if (rc == SWM_OK) rc = cmaes_update(state, d, lambda, candidates, fitness, st);
  return rc;
}
