// Per-environment swimmer dynamics as register-resident device functions (one thread = one env).
//
// gym variant  -- same equations as envs/gym_swimmer/swimmer/remy_swimmer_env.py:95-214, but NOT
// the reference's formulation.  The reference carries every joint acceleration/force as an affine
// row over the n+2 unknowns and solves a dense (n+2)x(n+2) system (O(n^3) flops, O(n^2) storage).
// Here the same Newton/Euler equations are reduced analytically:
//   * f_n = 0 sums all segment equations:  Gdd = sum_i Phi_i / (n m)        (Phi_i = friction force)
//   * eliminating thdd_i leaves a block-tridiagonal SPD system in the n-1 interior joint forces
//       Q_{j-1} f_{j-1} + P_j f_j + Q_j f_{j+1} = r_j ,   P_j = 2I + 3(N_{j-1}+N_j), Q_j = 3N_j - I,
//       N_i = n_i n_i^T,  r_j = Phi_j - Phi_{j-1} - w_{j-1} - w_j,
//       w_i = (6 tau_i / l) n_i - (l m thd_i^2 / 2) p_i,   tau_i = k thd_i l^3/12 + u_{i-1} - u_i
//     solved by an unpivoted 2x2-block LDL^T sweep (one reciprocal per joint),
//   * thdd_i = (6/(m l)) n_i.(f_i + f_{i+1}) + 12 tau_i/(m l^2).
// The code works in a non-dimensional form of these equations (see gym_accelerations) so that the
// physical constants fold into four precomputed numbers.
// O(n) flops and O(n) registers, no pivoting, no local memory.  Agrees with the reference's
// pivoted dense solve to ~1e-15 relative (tests/test_parity_step.py).
//
// rlglue variant -- rlglue/environment/SwimmerEnvironment.cpp:139-271 including its literal
// column/weight quirks (SURVEY appendix B).  The (5n+2) system is reduced algebraically to the
// n+2 unknowns [Gdd_1, thdd_1..n] (the f_j and Gdd_i are affine in those), then solved with a
// partially pivoted LU.
#pragma once
#include <cuda_runtime.h>

#include "../../include/swimmer_ars.h"

namespace swm {

// Physical constants of one model, precomputed once per model (kernel argument -> constant bank, or shared
// memory for the per-candidate models of the estimation objective).
struct Phys {
  double l, m, k, h, max_u, dirx, diry;
  // gym variant, non-dimensional form (lengths in units of l, forces in units of m*l/2)
  double inv_l;      // 1/l
  double kappa;      // k*l/m       (friction torque coefficient: tau_i/I = kappa*thd_i + ...)
  double m2kappa;    // -2*k*l/m    (psi_i = F_i n_i, F_i = m2kappa * (v_i.n_i))
  double u_scale;    // 12/(m*l^2)  (torques enter as u/I)
  double gdd_c;      // m2kappa*l/(2n)    (Gdd = gdd_c * sum_i (v_i.n_i) n_i: the friction coefficient is folded in)
  double h_gdd_c;    // h*m2kappa*l/(2n)  (Euler update of Gdot straight from sum_i (v_i.n_i) n_i)
  double inv_n;      // 1/n
  // rlglue variant
  double kl;         // k*l
  double tau_c;      // k*l^3/12
  double half_l;     // l/2
  double I;          // m*l^2/12
};

// Host and device build the same constants bit for bit: only correctly rounded products and quotients, no
// sum that the device compiler could contract into an FMA.
__host__ __device__ inline Phys make_phys(const swm_params_t& p) {
  Phys P;
  const double l = p.l_i, m = p.m_i, k = p.k, n = (double)p.n;
  P.l = l; P.m = m; P.k = k; P.h = p.h; P.max_u = p.max_u;
  P.dirx = p.direction[0]; P.diry = p.direction[1];
  P.inv_l = 1.0 / l;
  P.kappa = k * l / m;
  P.m2kappa = -2.0 * (k * l / m);
  P.u_scale = 12.0 / (m * l * l);
  P.gdd_c = P.m2kappa * (l / (2.0 * n));
  P.h_gdd_c = p.h * P.gdd_c;
  P.inv_n = 1.0 / n;
  P.kl = k * l;
  P.tau_c = k * (l * l * l) / 12.0;
  P.half_l = l / 2.0;
  P.I = m * (l * l) / 12.0;
  return P;
}

// ~1-ulp reciprocal for well-scaled positive arguments (2x2 block determinants >= 4, joint-form pivots >= 1):
// hardware seed (>= 20 bits) + one cubically convergent step x(1 + e + e^2), e = 1 - d x
// (3 FMAs, residual e^3 < 2^-60), no special-case path.
__device__ __forceinline__ double fast_rcp(double d) {
  double x;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
  const double e = fma(-d, x, 1.0);
  return fma(x, fma(e, e, e), x);
}

// Hides a value from common-subexpression elimination (the compiler would otherwise keep 2N products
// alive across the whole sweep to save 2N multiplies, and spill for long chains).
__device__ __forceinline__ double opaque(double x) {
  asm volatile("" : "+d"(x));
  return x;
}
constexpr int kKeepTsTc = 7;
#ifndef SWM_FACT_SMEM_RHS_ONLY
#define SWM_FACT_SMEM_RHS_ONLY 1
#endif
constexpr bool kFactSmemRhsOnly = SWM_FACT_SMEM_RHS_ONLY != 0;
constexpr int kRegLuMax = 90;  // rlglue variant: largest augmented system (doubles) factorised in registers (n <= 7)

// ---------------------------------------------------------------------------------------------
// gym variant, non-dimensional O(n) form.  With v = Gdot_i / l, g_j = 2 f_j / (m l),
// ut = u * 12/(m l^2), kappa = k l / m:
//   tau~_i = kappa thd_i + ut_{i-1} - ut_i                       (= tau_i / I)
//   psi_i  = -2 kappa (v_i . n_i) n_i                            (= 2 Phi_i / (m l))
//   w^_i   = tau~_i n_i - thd_i^2 p_i
//   Q_{j-1} g_{j-1} + P_j g_j + Q_j g_{j+1} = psi_j - psi_{j-1} - w^_{j-1} - w^_j
//        P_j = 2I + 3(N_{j-1}+N_j),  Q_j = 3N_j - I,  N_i = n_i n_i^T
//   thdd_i = 3 n_i.(g_i + g_{i+1}) + tau~_i,    Gdd = l/(2n) sum_i psi_i
// s[i] = sin(th_i), c[i] = cos(th_i); ut has N-1 entries (already scaled by u_scale).
// ---------------------------------------------------------------------------------------------
// FS: where the factorisation (5 doubles per joint) lives between the forward and the backward sweep:
// 0 = registers, > 0 = shared memory, element k of this thread at fs[k * FS] (FS = threads per CTA).  Long
// chains (n >= 8) keep 45 doubles there instead of 90 registers that the 255-register limit cannot hold.
template <int N, int FS = 0>
__device__ __forceinline__ void gym_accelerations(const Phys& P, const double (&s)[N],
                                                  const double (&c)[N], double gdx, double gdy,
                                                  const double (&thd)[N], const double* ut,
                                                  double& psx, double& psy, double (&thdd)[N],
                                                  double* fs = nullptr) {
  // Outputs: thdd, and (psx, psy) = sum_i (v_i.n_i) n_i = sum_i psi_i / m2kappa; the caller scales it
  // (Gdd = gdd_c * sum, gdd_c carries m2kappa), so the friction force itself is never formed: it enters the
  // right-hand sides as F -+ tau~ = fma(m2kappa, v.n, -+tau~), one operation less per segment.
  // Streaming formulation: apart from the factorisation (5 doubles per joint) everything is a
  // rolling value, so the live state is O(N) with a small constant (registers, no local memory).
  //
  // pass 0 -- barycentric shift.  Head-frame centre velocity of segment i (units of l) is
  //   v'_i = sum_{q<i} thd_q n_q + thd_i n_i / 2, so mean_i v'_i = sum_q (N-q-1/2)/N thd_q n_q.
  // The weights are compile-time constants, so with ts = thd*s, tc = thd*c (needed by pass 1 anyway)
  // the two sums are constant-operand FMAs.  Up to kKeepTsTc segments ts/tc stay in registers; for
  // longer chains pass 1 recomputes them (2 multiplies) rather than holding 2N more doubles live.
  constexpr bool KEEP = (N <= kKeepTsTc);
  double tsa[KEEP ? N : 1], tca[KEEP ? N : 1];
  double sx = gdx * P.inv_l, sy = gdy * P.inv_l;
#pragma unroll
  for (int q = 0; q < N; ++q) {
    const double w = (N - q - 0.5) / N;
    const double ts = thd[q] * s[q], tc = thd[q] * c[q];
    if (KEEP) { tsa[q] = ts; tca[q] = tc; }
    sx = fma(w, ts, sx);
    sy = fma(-w, tc, sy);
  }
  // pass 1 -- per segment: friction, right-hand sides, and the forward block elimination of the
  // joint between segment i-1 and i.
  constexpr int J = N - 1;
  constexpr int JR = (FS == 0 && J > 0) ? J : 1;
  // FS > 0 with kFactSmemRhsOnly: only the eliminated right-hand sides (2 doubles per joint) go to shared
  // memory, the inverse pivot blocks stay in registers -- enough to remove the last spills of n = 10 at 40 % of
  // the shared-memory traffic
  constexpr int JX = ((FS == 0 || kFactSmemRhsOnly) && J > 0) ? J : 1;
  double Xa[JX], Xb[JX], Xd[JX];  // inverse pivot blocks
  double rx[JR], ry[JR];          // eliminated right-hand sides
  double pXa = 0.0, pXb = 0.0, pXd = 0.0, prx = 0.0, pry = 0.0;  // FS > 0: the previous joint's values (registers)
  double ax = sx, ay = sy;          // velocity of the joint at the head of segment i
  double sumx = 0.0, sumy = 0.0;    // sum_i (v_i.n_i) n_i
  double Bpx = 0.0, Bpy = 0.0;      // B_{i-1}
  double ssp = 0.0, scp = 0.0;      // s^2, s c of segment i-1
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const double ts = KEEP ? tsa[i] : opaque(thd[i]) * s[i], tc = KEEP ? tca[i] : opaque(thd[i]) * c[i];
    const double vx = fma(-0.5, ts, ax), vy = fma(0.5, tc, ay);
    if (i + 1 < N) { ax -= ts; ay += tc; }
    const double vn = fma(vy, c[i], -vx * s[i]);  // F_i = m2kappa * vn
    sumx = fma(-vn, s[i], sumx);
    sumy = fma(vn, c[i], sumy);
    double du = 0.0;
    if (i >= 1 && i <= N - 2) du = ut[i - 1] - ut[i];
    else if (i >= 1) du = ut[i - 1];
    else if (i <= N - 2) du = -ut[i];
    const double tau = fma(P.kappa, thd[i], du);
    thdd[i] = tau;  // completed in pass 2
    const double ss = s[i] * s[i], sc = s[i] * c[i];
    if (i >= 1) {
      // A_i = psi_i - w^_i = (F - tau~) n_i + thd^2 p_i
      const double a = fma(P.m2kappa, vn, -tau);
      const double Ax = fma(-a, s[i], thd[i] * tc), Ay = fma(a, c[i], thd[i] * ts);
      // joint j = i: P_j = 2I + 3(N_{i-1} + N_i); cc = 1 - ss  =>  pd = 10 - pa, qd = 1 - qa
      double pa = fma(3.0, ssp + ss, 2.0);
      double pb = -3.0 * (scp + sc);
      double pd = 10.0 - pa;
      double r0 = Ax - Bpx, r1 = Ay - Bpy;
      if (i >= 2) {
        const double qa = fma(3.0, ssp, -1.0), qb = -3.0 * scp, qd = 1.0 - qa;  // Q_{i-1}
        const double xa = FS ? pXa : Xa[FS ? 0 : i - 2], xb = FS ? pXb : Xb[FS ? 0 : i - 2];
        const double xd = FS ? pXd : Xd[FS ? 0 : i - 2];
        const double rpx = FS ? prx : rx[FS ? 0 : i - 2], rpy = FS ? pry : ry[FS ? 0 : i - 2];
        const double t00 = fma(qa, xa, qb * xb);
        const double t01 = fma(qa, xb, qb * xd);
        const double t10 = fma(qb, xa, qd * xb);
        const double t11 = fma(qb, xb, qd * xd);
        pa = fma(-t01, qb, fma(-t00, qa, pa));
        pb = fma(-t01, qd, fma(-t00, qb, pb));
        pd = fma(-t11, qd, fma(-t10, qb, pd));
        r0 = fma(-t01, rpy, fma(-t00, rpx, r0));
        r1 = fma(-t11, rpy, fma(-t10, rpx, r1));
      }
      const double idet = fast_rcp(fma(pa, pd, -pb * pb));
      if (FS && kFactSmemRhsOnly) {
        pXa = pd * idet; pXb = -pb * idet; pXd = pa * idet; prx = r0; pry = r1;
        Xa[JX > 1 ? i - 1 : 0] = pXa; Xb[JX > 1 ? i - 1 : 0] = pXb; Xd[JX > 1 ? i - 1 : 0] = pXd;
        double* f = fs + (size_t)(2 * (i - 1)) * FS;
        f[0] = r0; f[FS] = r1;
      } else if (FS) {
        pXa = pd * idet; pXb = -pb * idet; pXd = pa * idet; prx = r0; pry = r1;
        double* f = fs + (size_t)(5 * (i - 1)) * FS;
        f[0] = pXa; f[FS] = pXb; f[2 * FS] = pXd; f[3 * FS] = r0; f[4 * FS] = r1;
      } else {
        Xa[FS ? 0 : i - 1] = pd * idet;
        Xb[FS ? 0 : i - 1] = -pb * idet;
        Xd[FS ? 0 : i - 1] = pa * idet;
        rx[FS ? 0 : i - 1] = r0;
        ry[FS ? 0 : i - 1] = r1;
      }
    }
    if (i <= N - 2) {
      // B_i = psi_i + w^_i = (F + tau~) n_i - thd^2 p_i
      const double b = fma(P.m2kappa, vn, tau);
      Bpx = -fma(b, s[i], thd[i] * tc);
      Bpy = fma(b, c[i], -thd[i] * ts);
    }
    ssp = ss;
    scp = sc;
  }
  psx = sumx;
  psy = sumy;
  // pass 2 -- back substitution g_j = X_j (r'_j - Q_j g_{j+1}) and thdd_i = 3 n_i.(g_i+g_{i+1}) + tau~_i
  double gnx = 0.0, gny = 0.0;  // g_{j+1}
#pragma unroll
  for (int j = J; j >= 1; --j) {
    double y0, y1, xa, xb, xd;
    if (FS && kFactSmemRhsOnly) {
      const double* f = fs + (size_t)(2 * (j - 1)) * FS;
      xa = Xa[JX > 1 ? j - 1 : 0]; xb = Xb[JX > 1 ? j - 1 : 0]; xd = Xd[JX > 1 ? j - 1 : 0];
      y0 = f[0]; y1 = f[FS];
    } else if (FS) {
      const double* f = fs + (size_t)(5 * (j - 1)) * FS;
      xa = f[0]; xb = f[FS]; xd = f[2 * FS]; y0 = f[3 * FS]; y1 = f[4 * FS];
    } else {
      xa = Xa[FS ? 0 : j - 1]; xb = Xb[FS ? 0 : j - 1]; xd = Xd[FS ? 0 : j - 1];
      y0 = rx[FS ? 0 : j - 1]; y1 = ry[FS ? 0 : j - 1];
    }
    if (j < J) {
      // same expressions as pass 1: the compiler keeps or rebuilds them as register pressure allows
      const double qa = fma(3.0, s[j] * s[j], -1.0), qb = -3.0 * (s[j] * c[j]), qd = 1.0 - qa;
      y0 = fma(-qb, gny, fma(-qa, gnx, y0));
      y1 = fma(-qd, gny, fma(-qb, gnx, y1));
    }
    const double gjx = fma(xa, y0, xb * y1);
    const double gjy = fma(xb, y0, xd * y1);
    // segment j lies between joints j and j+1
    const double ex = (j == J) ? gjx : gjx + gnx, ey = (j == J) ? gjy : gjy + gny;
    thdd[j] = fma(3.0, fma(c[j], ey, -s[j] * ex), thdd[j]);
    gnx = gjx;
    gny = gjy;
  }
  if (J >= 1) thdd[0] = fma(3.0, fma(c[0], gny, -s[0] * gnx), thdd[0]);  // free head: g_0 = 0
}

// ---------------------------------------------------------------------------------------------
// gym variant, joint-angle form for short chains (DESIGN.md §3.1).  With G at the origin the segment
// centres are x_i - G = l sum_q A_iq p_q, A_iq = [q < i] + 1/2 [q = i] - (N - q - 1/2)/N, whose columns sum
// to zero, so Gdd drops out of the angle equations.  Projecting Newton's equations on dx_i/dth_r gives,
// divided by I = m l^2/12 and with C_rq = cos(th_q - th_r), S_rq = sin(th_q - th_r), K = A^T A:
//   (1 + 12 K o C) thdd = tau~ + m2kappa F + 12 (K o S) thd^2,       F_r = sum_i 6 A_ir C_ir vn_i
//   vn_i = v.n_i + sum_q A_iq thd_q C_qi   (v = Gdot / l: the centre velocity along n_i, units of l)
// K o C is a Schur product of two PSD matrices, so the matrix is >= I: every LDL^T pivot is >= 1 and the
// unpivoted elimination with fast_rcp is safe.  The first pivot is a compile-time constant.
// Same interface and outputs as gym_accelerations; O(N^2) operations, fewer than the block-tridiagonal
// sweep up to kJointFormMaxN segments.
// ---------------------------------------------------------------------------------------------
#ifndef SWM_JOINT_FORM_MAX_N
#define SWM_JOINT_FORM_MAX_N 5
#endif
constexpr int kJointFormMaxN = SWM_JOINT_FORM_MAX_N;

template <int N>
struct JointForm {
  double A[N][N];    // A[i][q]
  double A6[N][N];   // 6 A
  double K12[N][N];  // 12 K
  __host__ __device__ constexpr JointForm() : A(), A6(), K12() {
    for (int i = 0; i < N; ++i)
      for (int q = 0; q < N; ++q) {
        A[i][q] = (q < i ? 1.0 : 0.0) + (q == i ? 0.5 : 0.0) - (N - q - 0.5) / N;
        A6[i][q] = 6.0 * A[i][q];
      }
    for (int r = 0; r < N; ++r)
      for (int q = 0; q < N; ++q) {
        double k = 0.0;
        for (int i = 0; i < N; ++i) k += A[i][r] * A[i][q];
        K12[r][q] = 12.0 * k;
      }
  }
};

// k * x for a compile-time constant k, without the multiply when k is 1
__device__ __forceinline__ double scaled(double k, double x) { return k == 1.0 ? x : k * x; }

template <int N>
__device__ __forceinline__ void gym_accelerations_joint(const Phys& P, const double (&s)[N],
                                                        const double (&c)[N], double gdx, double gdy,
                                                        const double (&thd)[N], const double* ut,
                                                        double& psx, double& psy, double (&thdd)[N]) {
  constexpr JointForm<N> T{};
  // pair terms r < q: C[r][q] = cos(th_q - th_r), S[r][q] = sin(th_q - th_r) (C symmetric, S antisymmetric)
  double C[N][N], S[N][N];
#pragma unroll
  for (int r = 0; r < N; ++r)
#pragma unroll
    for (int q = r + 1; q < N; ++q) {
      C[r][q] = fma(c[r], c[q], s[r] * s[q]);
      S[r][q] = fma(s[q], c[r], -c[q] * s[r]);
    }
  const double vx = gdx * P.inv_l, vy = gdy * P.inv_l;
  double vn[N];
  psx = 0.0;
  psy = 0.0;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    double a = fma(vy, c[i], -vx * s[i]);
#pragma unroll
    for (int q = 0; q < N; ++q) {
      if (T.A[i][q] == 0.0) continue;
      const double t = (q == i) ? thd[i] : thd[q] * (q < i ? C[q][i] : C[i][q]);
      a = fma(T.A[i][q], t, a);
    }
    vn[i] = a;
    psx = fma(-a, s[i], psx);
    psy = fma(a, c[i], psy);
  }
  double th2[N];
#pragma unroll
  for (int q = 0; q < N; ++q) th2[q] = thd[q] * thd[q];
  // right-hand side b and the symmetric matrix M (upper triangle, diagonal constant)
  double b[N], M[N][N];
#pragma unroll
  for (int r = 0; r < N; ++r) {
    double du = 0.0;
    if (r >= 1 && r <= N - 2) du = ut[r - 1] - ut[r];
    else if (r >= 1) du = ut[r - 1];
    else if (r <= N - 2) du = -ut[r];
    // A6[r][r] is 0 for the middle segment of odd N: no multiply by a compile-time zero
    double f = 0.0;
    bool first = true;
#pragma unroll
    for (int i = 0; i < N; ++i) {
      if (T.A6[i][r] == 0.0) continue;
      const double t = (i == r) ? vn[i] : (i < r ? C[i][r] : C[r][i]) * vn[i];
      f = first ? T.A6[i][r] * t : fma(T.A6[i][r], t, f);
      first = false;
    }
    double br = fma(P.m2kappa, f, fma(P.kappa, thd[r], du));
#pragma unroll
    for (int q = 0; q < N; ++q) {
      if (q == r || T.K12[r][q] == 0.0) continue;
      br = fma(T.K12[r][q], (r < q ? S[r][q] : -S[q][r]) * th2[q], br);
    }
    b[r] = br;
#pragma unroll
    for (int q = r + 1; q < N; ++q) M[r][q] = scaled(T.K12[r][q], C[r][q]);
  }
  // unpivoted LDL^T, right-looking: after step k, M[i][j] (k < i <= j) holds the Schur complement and
  // L[k][i] = M[k][i] / d_k
  double inv_d[N], L[N][N];
#pragma unroll
  for (int k = 0; k < N; ++k) {
    double dk = 1.0 + T.K12[k][k];
#pragma unroll
    for (int j = 0; j < k; ++j) dk = fma(-L[j][k], M[j][k], dk);
    inv_d[k] = (k == 0) ? 1.0 / (1.0 + T.K12[0][0]) : fast_rcp(dk);
#pragma unroll
    for (int i = k + 1; i < N; ++i) {
      double mki = M[k][i];
#pragma unroll
      for (int j = 0; j < k; ++j) mki = fma(-L[j][k], M[j][i], mki);
      M[k][i] = mki;
      // first pivot a compile-time constant: L[0][i] = C[0][i] * (K12[0][i] / d_0), one multiply (none for n = 3,
      // where the quotient is 1 for i = 1) instead of two
      L[k][i] = (k == 0) ? scaled(T.K12[0][i] / (1.0 + T.K12[0][0]), C[0][i]) : mki * inv_d[k];
      b[i] = fma(-L[k][i], b[k], b[i]);
    }
  }
#pragma unroll
  for (int k = N - 1; k >= 0; --k) {
    double x = b[k] * inv_d[k];
#pragma unroll
    for (int i = k + 1; i < N; ++i) x = fma(-L[k][i], thdd[i], x);
    thdd[k] = x;
  }
}

// The gym accelerations in the cheaper of the two forms for N segments (same outputs either way).
template <int N, int FS = 0>
__device__ __forceinline__ void gym_accel(const Phys& P, const double (&s)[N], const double (&c)[N],
                                          double gdx, double gdy, const double (&thd)[N], const double* ut,
                                          double& psx, double& psy, double (&thdd)[N], double* fs = nullptr) {
  if constexpr (N <= kJointFormMaxN)
    gym_accelerations_joint<N>(P, s, c, gdx, gdy, thd, ut, psx, psy, thdd);
  else
    gym_accelerations<N, FS>(P, s, c, gdx, gdy, thd, ut, psx, psy, thdd, fs);
}

// (sin, cos) of th + d from (sin, cos) of th for a small increment d: polynomials of sin d and
// cos d - 1, then one 2x2 rotation -- no range reduction, no integer work (a full double-precision
// sincos is ~27 FP64 + ~50 other instructions).
//
// Per-thread rollout step (gym_step_tracked) for N <= kRotateOneTierMaxN: one polynomial for |d| <= 1/8, z = d^2,
//   sin d = d + d^3 P(z),  cos d - 1 = z Q(z),  P and Q of degree 3
// with P and Q Chebyshev-economised in z on [0, 1/64] (rotation_poly.py derives the coefficients in
// exact rational arithmetic): truncation <= 2.8e-20 for sin d and <= 2.3e-18 for cos d - 1 over the
// whole range, below one ulp of the rotated value.  Approximating P and Q rather than sin d itself
// keeps the sine's error proportional to d^3.
// It costs 3 FP64 operations per segment more than the base tier below and removes the per-lane tail branch:
// measured on B200 (profiles/r04_summary.md) that wins for n = 3 with fast segments (config[1]: the tail ran on
// about half of the warp-steps) and loses for n = 5 and n = 10 V2 rollouts, whose segments rarely leave the base
// tier; longer chains keep the two tiers.
constexpr int kRotateOneTierMaxN = 3;
constexpr double kRotateP[4] = {-0.16666666666666666, 0.008333333333309446, -0.0001984126907688373,
                                2.75494915427022e-06};
constexpr double kRotateQ[4] = {-0.4999999999999999, 0.04166666666640392, -0.0013888888048092878,
                                2.4792977072672542e-05};
__device__ __forceinline__ void small_sincos(double d, double& sn, double& cm1) {
  const double z = d * d;
  const double p = fma(z, fma(z, fma(z, kRotateP[3], kRotateP[2]), kRotateP[1]), kRotateP[0]);
  const double q = fma(z, fma(z, fma(z, kRotateQ[3], kRotateQ[2]), kRotateQ[1]), kRotateQ[0]);
  sn = fma(d * z, p, d);
  cm1 = z * q;
}

// Longer chains in the per-thread step and the lane-split kernels (lane_rollout.cuh, lane2_rollout.cuh): Taylor
// polynomials in two additive tiers,
//   base, |d| <= 1/32: sin to d^5, cos to d^6     truncation <= 5.8e-15 at the limit and ~(32 d)^7 of
//                                                 that below it (1e-19 at |thd| = 7 rad/s, h = 1e-3)
//   tail, |d| <= 1/8 : + the d^7, d^9 terms of sin and the d^8, d^10 terms of cos (truncation < 3e-17)
// The tail is added under a per-lane branch in the per-thread step, and out of line or under a warp vote,
// once per segment lane, in the lane-split kernels; no lane's result depends on its neighbours.  Every
// rollout kernel re-evaluates (s, c) exactly from th every 64th step, so truncation never accumulates over
// more than 63 steps.
constexpr double kRotateShort = 0.03125, kRotateLong = 0.125;
constexpr int kRotateShortHi = 0x3FA00000, kRotateLongHi = 0x3FC00000;  // high words of 1/32 and 1/8
__device__ __forceinline__ void small_sincos_base(double d, double& z, double& sn, double& cm1) {
  z = d * d;
  const double ps = fma(z, 8.3333333333333332e-03, -1.6666666666666666e-01);  // 1/5!, -1/3!
  double pc = fma(z, -1.3888888888888889e-03, 4.1666666666666664e-02);        // -1/6!, 1/4!
  pc = fma(z, pc, -0.5);
  sn = fma(d * z, ps, d);  // sin d
  cm1 = z * pc;            // cos d - 1
}
__device__ __forceinline__ void small_sincos_tail(double d, double z, double& sn, double& cm1) {
  const double z2 = z * z;
  const double ts = fma(z, 2.7557319223985893e-06, -1.9841269841269841e-04);   // 1/9!, -1/7!
  const double tc = fma(z, -2.7557319223985888e-07, 2.4801587301587302e-05);   // -1/10!, 1/8!
  sn = fma(d * (z2 * z), ts, sn);
  cm1 = fma(z2 * z2, tc, cm1);
}
__device__ __forceinline__ void rotate_by(double sn, double cm1, double& s, double& c) {
  const double c2 = fma(-s, sn, fma(c, cm1, c));
  const double s2 = fma(c, sn, fma(s, cm1, s));
  c = c2;
  s = s2;
}

// ---------------------------------------------------------------------------------------------
// rlglue variant (reduced form of SwimmerEnvironment.cpp:139-271).
// Unknowns z = [g1x, g1y, thdd_0..thdd_{N-1}] with g1 = Gdd of the first segment; affine rows have
// N+3 slots (last = constant).
// ---------------------------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ void rlglue_accelerations(const Phys& P, const double (&s)[N],
                                                     const double (&c)[N], double gdx, double gdy,
                                                     const double (&thd)[N], const double* u,
                                                     double& gddx, double& gddy,
                                                     double (&thdd)[N]) {
  constexpr int M = N + 2, S = N + 3;
  // --- compute_friction (cpp:238-271); n_i = (-s, c) ---
  double g1x = gdx, g1y = gdy;
  {
    // G1_dot -= l/n * sum_{i=1..n} sum_{j<i} e_ij thd_j n_j, e = 0.5 for j==0 or j==i-1 else 1
    double accx = 0.0, accy = 0.0;
#pragma unroll
    for (int i = 1; i <= N; ++i) {
      double sx = 0.0, sy = 0.0;
#pragma unroll
      for (int j = 0; j < i; ++j) {
        const double e = (j == 0 || j == i - 1) ? 0.5 : 1.0;
        sx += e * thd[j] * (-s[j]);
        sy += e * thd[j] * c[j];
      }
      accx += sx;
      accy += sy;
    }
    g1x -= P.l * P.inv_n * accx;
    g1y -= P.l * P.inv_n * accy;
  }
  double Fx[N], Fy[N];
  {
    double cx = g1x, cy = g1y;
#pragma unroll
    for (int i = 0; i < N; ++i) {
      if (i >= 1) {
        cx += P.half_l * (thd[i - 1] * (-s[i - 1]) + thd[i] * (-s[i]));
        cy += P.half_l * (thd[i - 1] * c[i - 1] + thd[i] * c[i]);
      }
      const double dot = fma(cy, c[i], -cx * s[i]);
      const double F = -P.kl * dot;
      Fx[i] = -F * s[i];
      Fy[i] = F * c[i];
    }
  }
  // --- affine forms: segment accelerations G_i (cpp:187-207 solved for Gdd_{i+1}) and joint
  //     forces f_j = f_{j-1} + m Gdd_j - F_j (cpp:172-181) ---
  double A[M][S];
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q < S; ++q) A[r][q] = 0.0;
  double Gx[S], Gy[S], fxa[S], fya[S], fxp[S], fyp[S];
#pragma unroll
  for (int q = 0; q < S; ++q) { Gx[q] = Gy[q] = fxa[q] = fya[q] = fxp[q] = fyp[q] = 0.0; }
  Gx[0] = 1.0;
  Gy[1] = 1.0;
  // walk segments; after processing segment i (0-based) fxa/fya hold f_{i+1}, fxp/fyp hold f_i.
#pragma unroll
  for (int i = 0; i < N; ++i) {
    if (i >= 1) {
      // Gdd_i = Gdd_{i-1} + (l/2)[(thdd n - thd^2 p)_{i-1} + (thdd n - thd^2 p)_i]
      Gx[2 + i - 1] += P.half_l * (-s[i - 1]);
      Gy[2 + i - 1] += P.half_l * c[i - 1];
      Gx[2 + i] += P.half_l * (-s[i]);
      Gy[2 + i] += P.half_l * c[i];
      Gx[S - 1] -= P.half_l * (thd[i - 1] * thd[i - 1] * c[i - 1] + thd[i] * thd[i] * c[i]);
      Gy[S - 1] -= P.half_l * (thd[i - 1] * thd[i - 1] * s[i - 1] + thd[i] * thd[i] * s[i]);
    }
#pragma unroll
    for (int q = 0; q < S; ++q) {
      fxp[q] = fxa[q];
      fyp[q] = fya[q];
      fxa[q] = fma(P.m, Gx[q], fxa[q]);
      fya[q] = fma(P.m, Gy[q], fya[q]);
    }
    fxa[S - 1] -= Fx[i];
    fya[S - 1] -= Fy[i];
    // torque row of segment i-1 (1-based i): I thdd - (l/2) n.(f_i + f_{i+1}) = B   (cpp:152-161,
    // literal column choice f_i, f_{i+1}); available once f_{i+1} is known.
    if (i >= 1) {
      const int sgm = i - 1;
#pragma unroll
      for (int q = 0; q < S; ++q) {
        const double vx = fxp[q] + fxa[q], vy = fyp[q] + fya[q];
        // for sgm == N-2 the second force is f_N, which the system pins to zero (cpp:183-184)
        const double ux = (sgm == N - 2) ? fxp[q] : vx, uy = (sgm == N - 2) ? fyp[q] : vy;
        A[2 + sgm][q] = -P.half_l * fma(c[sgm], uy, -s[sgm] * ux);
      }
    }
  }
  // rows 0,1: f_N = 0
#pragma unroll
  for (int q = 0; q < S; ++q) { A[0][q] = fxa[q]; A[1][q] = fya[q]; }
  // torque row of the last segment: forces f_N (=0) and "f_{N+1}" which aliases Gdd_1 (cpp:155,157)
  {
    const int sgm = N - 1;
    A[2 + sgm][0] = -P.half_l * (-s[sgm]);
    A[2 + sgm][1] = -P.half_l * c[sgm];
  }
#pragma unroll
  for (int i = 0; i < N; ++i) {
    A[2 + i][2 + i] += P.I;
    double Bi = -P.tau_c * thd[i];  // M_friction (cpp:267)
    if (i >= 1) Bi += u[i - 1];
    if (i <= N - 2) Bi -= u[i];
    A[2 + i][S - 1] -= Bi;
  }
  // --- partially pivoted LU on [A | -const] ---
  double z[M];
  if constexpr (M * S <= kRegLuMax) {
    // Small systems (n <= 7) stay in registers.  Every loop runs over a compile-time range with the
    // triangular bounds as guards: loops whose trip count depends on the unrolled outer index were
    // left rolled by the compiler, which put the whole system into local memory.
#pragma unroll
    for (int col = 0; col < M; ++col) {
      int best = col;
      double bv = fabs(A[col][col]);
#pragma unroll
      for (int r = 0; r < M; ++r) {
        if (r > col) {
          const double v = fabs(A[r][col]);
          if (v > bv) { bv = v; best = r; }
        }
      }
#pragma unroll
      for (int r = 0; r < M; ++r) {
        if (r > col) {
          const bool sw = (r == best);
#pragma unroll
          for (int q = 0; q < S; ++q) {
            if (q >= col) {
              const double up = A[col][q], lo = A[r][q];
              A[col][q] = sw ? lo : up;
              A[r][q] = sw ? up : lo;
            }
          }
        }
      }
      const double inv = 1.0 / A[col][col];
#pragma unroll
      for (int r = 0; r < M; ++r) {
        if (r > col) {
          const double f = A[r][col] * inv;
#pragma unroll
          for (int q = 0; q < S; ++q)
            if (q > col) A[r][q] = fma(-f, A[col][q], A[r][q]);
        }
      }
    }
#pragma unroll
    for (int r = M - 1; r >= 0; --r) {
      double acc = -A[r][S - 1];
#pragma unroll
      for (int q = 0; q < M; ++q)
        if (q > r) acc = fma(-A[r][q], z[q], acc);
      z[r] = acc / A[r][r];
    }
  } else {
    // Larger systems (n >= 8: more than 255 registers' worth) live in local memory; the pivot row is
    // swapped in by predicated moves over the unrolled rows.
#pragma unroll
    for (int col = 0; col < M; ++col) {
      int best = col;
      double bv = fabs(A[col][col]);
#pragma unroll
      for (int r = col + 1; r < M; ++r) {
        const double v = fabs(A[r][col]);
        if (v > bv) { bv = v; best = r; }
      }
#pragma unroll
      for (int r = col + 1; r < M; ++r) {
        if (r == best) {
#pragma unroll
          for (int q = col; q < S; ++q) { const double t = A[col][q]; A[col][q] = A[r][q]; A[r][q] = t; }
        }
      }
      const double inv = 1.0 / A[col][col];
#pragma unroll
      for (int r = col + 1; r < M; ++r) {
        const double f = A[r][col] * inv;
#pragma unroll
        for (int q = col + 1; q < S; ++q) A[r][q] = fma(-f, A[col][q], A[r][q]);
      }
    }
#pragma unroll
    for (int r = M - 1; r >= 0; --r) {
      double acc = -A[r][S - 1];
#pragma unroll
      for (int q = r + 1; q < M; ++q) acc = fma(-A[r][q], z[q], acc);
      z[r] = acc / A[r][r];
    }
  }
#pragma unroll
  for (int i = 0; i < N; ++i) thdd[i] = z[2 + i];
  // Gdd = mean_i Gdd_i (cpp:222-225); Gdd_i = g1 + (l/2) sum_{q} w_iq v_q
  {
    double sx = 0.0, sy = 0.0, cx = z[0], cy = z[1];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      if (i >= 1) {
        const double vx0 = fma(z[2 + i - 1], -s[i - 1], -(thd[i - 1] * thd[i - 1]) * c[i - 1]);
        const double vy0 = fma(z[2 + i - 1], c[i - 1], -(thd[i - 1] * thd[i - 1]) * s[i - 1]);
        const double vx1 = fma(z[2 + i], -s[i], -(thd[i] * thd[i]) * c[i]);
        const double vy1 = fma(z[2 + i], c[i], -(thd[i] * thd[i]) * s[i]);
        cx += P.half_l * (vx0 + vx1);
        cy += P.half_l * (vy0 + vy1);
      }
      sx += cx;
      sy += cy;
    }
    gddx = sx * P.inv_n;
    gddy = sy * P.inv_n;
  }
}

// One integration step in registers with freshly evaluated sines/cosines (batched single step,
// RL-Glue rollouts).  VARIANT 0: explicit Euler (remy_swimmer_env.py:88-91), VARIANT 1:
// semi-implicit Euler (SwimmerEnvironment.cpp:228-236).  u = torques (unscaled, n-1 entries).
// Returns the reward Gdot_new . direction (remy_swimmer_env.py:238-243 / cpp:273-277).
template <int N, int VARIANT>
__device__ __forceinline__ double swimmer_step(const Phys& P, double& gdx, double& gdy,
                                               double (&th)[N], double (&thd)[N],
                                               const double* u) {
  double s[N], c[N];
#pragma unroll
  for (int i = 0; i < N; ++i) sincos(th[i], &s[i], &c[i]);
  double gddx, gddy, thdd[N];
  if (VARIANT == 0) {
    double ut[N > 1 ? N - 1 : 1];
#pragma unroll
    for (int k = 0; k < N - 1; ++k) ut[k] = u[k] * P.u_scale;
    gym_accel<N>(P, s, c, gdx, gdy, thd, ut, gddx, gddy, thdd);
    gddx *= P.gdd_c;
    gddy *= P.gdd_c;
  } else {
    rlglue_accelerations<N>(P, s, c, gdx, gdy, thd, u, gddx, gddy, thdd);
  }
  gdx = fma(P.h, gddx, gdx);
  gdy = fma(P.h, gddy, gdy);
#pragma unroll
  for (int i = 0; i < N; ++i) {
    if (VARIANT == 0) {
      th[i] = fma(P.h, thd[i], th[i]);
      thd[i] = fma(P.h, thdd[i], thd[i]);
    } else {
      thd[i] = fma(P.h, thdd[i], thd[i]);
      th[i] = fma(P.h, thd[i], th[i]);
    }
  }
  return fma(gdx, P.dirx, gdy * P.diry);
}

// Rollout form of the gym step: (s, c) = (sin th, cos th) are carried in registers from step to
// step and advanced by the rotation of the angle increment h*thd instead of being re-evaluated.
// `resync` (warp-uniform; the rollout kernel sets it every 64th step) or an increment above 1/8 rad
// on any segment re-evaluates them exactly from th.  ut = torques already scaled by P.u_scale.
template <int N, int FS = 0>
__device__ __forceinline__ void gym_step_tracked(const Phys& P, double& gdx, double& gdy,
                                                 double (&th)[N], double (&thd)[N],
                                                 double (&s)[N], double (&c)[N],
                                                 const double* ut, bool resync, double* fs = nullptr) {
  double psx, psy, thdd[N];
  gym_accel<N, FS>(P, s, c, gdx, gdy, thd, ut, psx, psy, thdd, fs);
  gdx = fma(P.h_gdd_c, psx, gdx);
  gdy = fma(P.h_gdd_c, psy, gdy);
  double d[N];
  // Tier selection on the integer pipe: for non-negative doubles the high word orders like the value, so
  // max_i |d_i| is taken as the maximum of the sign-stripped high words (NaN / Inf have the largest ones
  // and fall through to sincos).  Thresholds are powers of two (low word 0): hi <= hi(threshold) admits
  // |d| < threshold * (1 + 2^-20), which the polynomial bounds cover.
  int dmax_hi = 0;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    d[i] = P.h * thd[i];
    dmax_hi = max(dmax_hi, __double2hiint(d[i]) & 0x7fffffff);
    th[i] = fma(P.h, thd[i], th[i]);
    thd[i] = fma(P.h, thdd[i], thd[i]);
  }
  // Decided per lane from the lane's own data only, so that an environment's trajectory does not
  // depend on which other environments share its warp.  NaN falls through to sincos.
  double sn[N], cm1[N];
  if constexpr (N <= kRotateOneTierMaxN) {
#pragma unroll
    for (int i = 0; i < N; ++i) small_sincos(d[i], sn[i], cm1[i]);
  } else {
    double z[N];
#pragma unroll
    for (int i = 0; i < N; ++i) small_sincos_base(d[i], z[i], sn[i], cm1[i]);
#ifndef SWM_ANALYZE_TIER
    // One branch for all segments of a lane.  (A branch per segment would skip the tail for segments that are
    // slow in every lane, ~7 FP64 operations per step fewer for n = 3 -- measured 1.7 % SLOWER there and 18 %
    // slower for n = 10: N divergent regions per step cost more than they save, profiles/r02_summary.md.)
    if (dmax_hi > kRotateShortHi)
#else  // static SASS analysis of one fast path only (tools/fastpath_mix.sh); never shipped
    if (SWM_ANALYZE_TIER == 1)
#endif
    {
#pragma unroll
      for (int i = 0; i < N; ++i) small_sincos_tail(d[i], z[i], sn[i], cm1[i]);
    }
  }
#ifdef SWM_ANALYZE_TIER
#pragma unroll
  for (int i = 0; i < N; ++i) rotate_by(sn[i], cm1[i], s[i], c[i]);
  return;
#endif
  if (resync || dmax_hi > kRotateLongHi) {
#pragma unroll
    for (int i = 0; i < N; ++i) sincos(th[i], &s[i], &c[i]);
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i) rotate_by(sn[i], cm1[i], s[i], c[i]);
  }
}

}  // namespace swm
