// Lane-split fused rollout: ONE environment is spread over L lanes of a warp (lane i = segment i, one more
// lane carries the barycentre-velocity pair of the observation), for batches that are too small to fill
// the chip with one environment per thread.
//
// Why: the FP64 unit of an SM sub-partition issues one warp instruction every 2-3 cycles whatever the
// number of active lanes (profiles/r01b_microbench.txt), so a rollout of 2,048 five-segment environments
// (BASELINE config[2]) as 64 full warps costs ~480 FP64 instructions per warp-step = ~1,440 cycles per step
// on 64 of the 592 sub-partitions (profiles/r01c_summary.md).  Here the per-segment work (observation
// normalisation, friction, joint right-hand sides, the tracked sine/cosine, V2 moments) is executed once
// per warp instruction for ALL segments of 32/L environments, which leaves ~215 FP64 instructions per
// warp-step for n = 5 and uses 8x as many sub-partitions.
//
// Per step (same equations as gym_accelerations in dynamics.cuh; remy_swimmer_env.py:69-214):
//   round 1  every lane publishes its (normalised) observation pair and thd*(sin, cos) in shared memory;
//            after a __syncwarp every lane reads all of them and forms, with per-lane constant weights,
//              du_i = u_{i-1} - u_i   directly as a dot product with the DIFFERENCE of two policy rows
//                                     (no cross-lane reduction of the policy product), and
//              v_i                    the velocity of its segment's centre (barycentric frame);
//            then friction, tau, the joint right-hand side r_i (one shuffle from the neighbour).
//   round 2  publishes r_i, the friction force and -- one step ahead, they only depend on th(t+1), which
//            explicit Euler forms from thd(t) -- the blocks P_i, Q_i of the NEXT step's joint system.
//            Every lane then runs the block-tridiagonal solve redundantly (identical instructions, so it
//            costs one instruction stream): right-hand sides with the factorisation of this step, then
//            the first half of the next step's factorisation; its second half runs after round 1 of the
//            next step.  A warp issues in order, so the reciprocal chain of the factorisation is placed
//            where its latency hides behind independent work instead of in front of a __syncwarp.
//   The factorisation keeps X_j = D_j^-1 and T_j = Q_{j-1} X_{j-1}; forward elimination is r'_j = r_j -
//   T_j r'_{j-1}, back-substitution g_j = X_j r'_j - T_{j+1}^T g_{j+1}: two dependent FMAs per joint.
//
// Every decision (sine/cosine tier) depends on the lane's own data only, and every cross-lane sum runs in
// a fixed order inside the environment's own lane group, so a trajectory does not depend on which other
// environments share the warp.  Results differ from the one-thread-per-environment kernel by rounding
// only (different summation order): both meet the same parity tolerances (tests/test_lane_split.py).
#pragma once
#include <type_traits>

#include "kernels.cuh"


namespace swm {

template <int N>
struct LaneSplit {
  static constexpr int L = (N + 1 <= 4) ? 4 : (N + 1 <= 8) ? 8 : 16;  // lanes per environment
  static constexpr int G = 32 / L;                                     // environments per warp
};

constexpr int kLaneBlock = 32;  // one warp per CTA: the block scheduler spreads warps over all SMs

// 16-byte shared-memory accesses through a 32-bit shared-window address (the generic-pointer form made
// the compiler rebuild the window base inside the step loop); constant offsets fold into the instruction
__device__ __forceinline__ void sts2(uint32_t addr, int off, double2 v) {
  asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(addr + (uint32_t)off), "d"(v.x), "d"(v.y) : "memory");
}
__device__ __forceinline__ double2 lds2(uint32_t addr, int off) {
  double2 v;
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr + (uint32_t)off) : "memory");
  return v;
}

// Rare tiers of the tracked sine/cosine (tail polynomial, exact re-evaluation), out of line, for the main warp of
// the two-warp kernel (lane2_rollout.cuh): its step loop takes them under a warp-uniform vote, and inlined they put
// a reconvergence barrier and a taken branch over ~100 instructions into EVERY step (~37 of 570 cycles, ncu source
// page; n = 3: 498 -> 450 cycles per step).  All lanes call it together; the caller keeps the result only on the
// lanes that need it.  (The single-warp kernel below keeps them inline: measured 1-3 % faster there.)
static __device__ __noinline__ double2 tracked_sincos_slow(double th_new, double d, double s, double c, bool exact) {
  double sN = s, cN = c;
  if (exact) {
    sincos(th_new, &sN, &cN);
  } else {
    double z, sn, cm1;
    small_sincos_base(d, z, sn, cm1);
    small_sincos_tail(d, z, sn, cm1);
    rotate_by(sn, cm1, sN, cN);
  }
  return make_double2(sN, cN);
}

// Sum of v over the L lanes of an environment by xor butterfly.  Both partners of a level add the same two
// values, so every lane ends with the bitwise identical sum (Gdot is replicated per lane and must stay so).
template <int L>
__device__ __forceinline__ double group_sum(double v) {
#pragma unroll
  for (int off = 1; off < L; off <<= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

// max |v| over the L lanes of an environment, NaN above everything (np.max semantics, as cost_max_abs_thd in
// kernels.cuh): the sign-stripped bit patterns of doubles order like their magnitudes, so the butterfly runs on the
// integer pipe; both partners of a level keep the same value, every lane ends with the same result
template <int L>
__device__ __forceinline__ double group_max_abs(double v) {
  long long b = __double_as_longlong(v) & 0x7fffffffffffffffLL;
#pragma unroll
  for (int off = 1; off < L; off <<= 1) {
    const long long o = __shfl_xor_sync(0xffffffffu, b, off);
    b = o > b ? o : b;
  }
  return __longlong_as_double(b);
}

// MODELS: the model-set mode of rollout_kernel (CTA row blockIdx.y runs model blockIdx.y; no statistics)
template <int N, bool LINEAR, bool NORM, bool STATS, bool MODELS>
__global__ void __launch_bounds__(kLaneBlock)
lane_rollout_kernel(const RolloutArgs a, const __grid_constant__ typename ScreenForms<SCREEN_NONE, MODELS>::type models) {
  static_assert(!MODELS || !STATS, "model set: no statistics");
  constexpr int L = LaneSplit<N>::L, G = LaneSplit<N>::G;
  constexpr int NO = 2 * N + 2, NA = N - 1, WS = NA * NO, J = N - 1;
  constexpr unsigned FULL = 0xffffffffu;
  // Exchange rows (one double2 per lane each): observation pair, thd*(sin, cos), joint right-hand side,
  // friction force, and two buffers (step parity) of the joint blocks P and Q.  Addressed through 32-bit
  // shared-window addresses computed once: row r of this lane's environment starts at gbase + r * kRow.
  constexpr int kRow = 32 * 16;
  enum { ROW_OBS = 0, ROW_T = 1, ROW_R = 2, ROW_P = 3, ROW_Q = 5 };  // P, Q: + parity
  __shared__ __align__(16) double2 sh[7][32];

  const int lane = threadIdx.x;
  const int seg = lane & (L - 1), grp = lane / L;
  const uint32_t sh_base = (uint32_t)__cvta_generic_to_shared(&sh[0][0]);
  const uint32_t gbase = sh_base + (uint32_t)(grp * L * 16);
  const uint32_t mine = gbase + (uint32_t)(seg * 16);
  const bool is_seg = seg < N;
  const long long e0 = (long long)blockIdx.x * G + grp;
  const bool active = e0 < a.B;
  const long long e = active ? e0 : a.B - 1;  // idle groups shadow the last env, never store
  const unsigned int iteration = a.iteration + (a.iter_dev ? *a.iter_dev : 0u);
  const Phys& P = rollout_model<MODELS>(a, models);

  // ---- initial state: this lane's pair of the observation, Gdot replicated on every lane ----
  const int jpair = is_seg ? 2 + 2 * seg : 0;  // observation index of this lane's pair (lanes > N: unused)
  double gdx, gdy, th = 0.0, thd = 0.0;
  if (a.init_state) {
    const double* sp = a.init_state + (e % a.init_count) * NO;
    gdx = sp[0]; gdy = sp[1];
    if (is_seg) { th = sp[jpair]; thd = sp[jpair + 1]; }
  } else {
    gdx = gdy = 0.0;
    if (is_seg) th = 1.5707963267948966;
  }
  if (a.init_perturb != 0.0) {  // same Philox addressing as rollout_kernel
    const unsigned int r = (unsigned int)(e % a.R);
    double d0, d1;
    philox_delta_pair(a.seed, iteration, r, 1u, 0u, SWM_DELTA_UNIFORM_01, d0, d1);
    gdx = fma(a.init_perturb, d0, gdx);
    gdy = fma(a.init_perturb, d1, gdy);
    if (is_seg) {
      philox_delta_pair(a.seed, iteration, r, 1u, (uint32_t)(1 + seg), SWM_DELTA_UNIFORM_01, d0, d1);
      th = fma(a.init_perturb, d0, th);
      thd = fma(a.init_perturb, d1, thd);
    }
  }

  // ---- policy: D = u_scale * (row seg-1  -  row seg) of the environment's own effective policy, stored
  //      per slot (slot q < N: (th_q, thd_q), slot N: (Gdot_x, Gdot_y)) ----
  double D[LINEAR ? 2 * (N + 1) : 1];
  double du_fixed = 0.0;
  const bool has_ka = is_seg && seg >= 1, has_kb = is_seg && seg <= N - 2;  // torques u_{seg-1}, u_seg exist
  if (LINEAR) {
    const long long q = e / a.R;  // policy index
    const bool philox = a.policy_mode == SWM_POLICY_PHILOX;
    const bool from_mem = a.policy_mode == SWM_POLICY_DELTAS;
    const double* base = (philox || from_mem) ? a.policies : a.policies + q * WS;
    const double* dmem = from_mem ? a.deltas + (q >> 1) * WS : nullptr;
    const double sgn_nu = (q & 1) ? -a.nu : a.nu;
    const unsigned int dir = a.dir0 + (unsigned int)(q >> 1);
    auto weight_pair = [&](int k, int slot, double& w0, double& w1) {
      const int j = (slot == N) ? 0 : 2 + 2 * slot;
      const int flat = k * NO + j;  // even: one Philox call yields both elements
      w0 = base[flat];
      w1 = base[flat + 1];
      if (philox || from_mem) {
        double d0, d1;
        if (philox) {
          philox_delta_pair(a.seed, iteration, dir, 0u, (uint32_t)(flat >> 1), a.dist, d0, d1);
        } else {
          d0 = dmem[flat];
          d1 = dmem[flat + 1];
        }
        // policy +- nu*delta exactly as ars_agent.py:141-142 (product rounded, then added)
        w0 = __dadd_rn(w0, __dmul_rn(sgn_nu, d0));
        w1 = __dadd_rn(w1, __dmul_rn(sgn_nu, d1));
      }
      if (NORM) {  // policy @ diag(cov^-1/2), ars/environment.py:32-33
        w0 *= a.inv_sigma[j];
        w1 *= a.inv_sigma[j + 1];
      }
    };
#pragma unroll
    for (int slot = 0; slot <= N; ++slot) {
      double a0 = 0.0, a1 = 0.0, b0 = 0.0, b1 = 0.0;
      if (has_ka) weight_pair(seg - 1, slot, a0, a1);
      if (has_kb) weight_pair(seg, slot, b0, b1);
      D[2 * slot] = P.u_scale * (a0 - b0);
      D[2 * slot + 1] = P.u_scale * (a1 - b1);
    }
  } else {
    const double ua = has_ka ? a.actions[e * NA + seg - 1] : 0.0;
    const double ub = has_kb ? a.actions[e * NA + seg] : 0.0;
    du_fixed = P.u_scale * ua - P.u_scale * ub;
  }

  // V2 mean / moment pivot of this lane's pair
  double mu_a = 0.0, mu_b = 0.0, pv_a = 0.0, pv_b = 0.0;
  if (NORM && seg <= N) { mu_a = a.mean[jpair]; mu_b = a.mean[jpair + 1]; }
  if (STATS && seg <= N) { pv_a = a.stats_pivot[jpair]; pv_b = a.stats_pivot[jpair + 1]; }
  double s1a = 0.0, s1b = 0.0, s2a = 0.0, s2b = 0.0;

  // weights of thd_q n_q in the velocity of this segment's centre (barycentric frame, units of l):
  //   v_i = Gdot/l + sum_q om_q thd_q n_q,   om_q = (N - q - 1/2)/N - [q < i] - [q == i]/2
  double om[N];
#pragma unroll
  for (int q = 0; q < N; ++q) om[q] = (N - q - 0.5) / N - (q < seg ? 1.0 : 0.0) - (q == seg ? 0.5 : 0.0);

  bool skipped = false;  // reward-constraint safe exploration: a screened-out direction is not rolled out
  if (LINEAR && a.dir_mask) skipped = a.dir_mask[(e / a.R) >> 1] == 0;
  const bool live = active && !skipped;
  if (active && skipped && a.final_state && seg <= N) {
    double2* o = reinterpret_cast<double2*>(a.final_state + output_row<MODELS>(a, e) * NO + jpair);
    *o = is_seg ? make_double2(th, thd) : make_double2(gdx, gdy);
  }

  double s, c;
  sincos(th, &s, &c);  // lanes >= N: th = 0
  double Xa[J > 0 ? J : 1], Xb[J > 0 ? J : 1], Xd[J > 0 ? J : 1];  // X_j = D_j^-1, joint j = 1..J at [j-1]
  double T0[J > 1 ? J - 1 : 1], T1[J > 1 ? J - 1 : 1], T2[J > 1 ? J - 1 : 1], T3[J > 1 ? J - 1 : 1];  // T_j, j = 2..J at [j-2]

  // blocks of the joint system owned by this lane: P_i = 2I + 3(N_{i-1} + N_i) (joint i, needs the
  // neighbour's sines), Q_i = 3 N_i - I; only (pa, pb) and (qa, qb) travel: pd = 10 - pa, qd = 1 - qa
  auto make_blocks = [&](double sn, double cn, double2& bP, double2& bQ) {
    const double ss = sn * sn, sc = sn * cn;
    const double ssp = __shfl_up_sync(FULL, ss, 1, L), scp = __shfl_up_sync(FULL, sc, 1, L);
    bP = make_double2(fma(3.0, ssp + ss, 2.0), -3.0 * (scp + sc));
    bQ = make_double2(fma(3.0, ss, -1.0), -3.0 * sc);
  };
  // joints j0..j1 of the factorisation, from the blocks in buffer `buf` (compile-time parity)
  auto factorise = [&](int j0, int j1, int buf) {
#pragma unroll
    for (int j = 1; j <= J; ++j) {
      if (j < j0 || j > j1) continue;
      const double2 Pj = lds2(gbase, (ROW_P + buf) * kRow + j * 16);
      double pa = Pj.x, pb = Pj.y, pd = 10.0 - pa;
      if (j >= 2) {
        const double2 Qp = lds2(gbase, (ROW_Q + buf) * kRow + (j - 1) * 16);
        const double qa = Qp.x, qb = Qp.y, qd = 1.0 - qa;
        const double t00 = fma(qa, Xa[j - 2], qb * Xb[j - 2]);
        const double t01 = fma(qa, Xb[j - 2], qb * Xd[j - 2]);
        const double t10 = fma(qb, Xa[j - 2], qd * Xb[j - 2]);
        const double t11 = fma(qb, Xb[j - 2], qd * Xd[j - 2]);
        pa = fma(-t01, qb, fma(-t00, qa, pa));
        pb = fma(-t01, qd, fma(-t00, qb, pb));
        pd = fma(-t11, qd, fma(-t10, qb, pd));
        T0[j - 2] = t00; T1[j - 2] = t01; T2[j - 2] = t10; T3[j - 2] = t11;
      }
      const double idet = fast_rcp(fma(pa, pd, -pb * pb));
      Xa[j - 1] = pd * idet;
      Xb[j - 1] = -pb * idet;
      Xd[j - 1] = pa * idet;
    }
  };
  // The dependent chain of the factorisation (one reciprocal per joint) is cut in two so that neither half
  // delays a __syncwarp: joints 1..JM of step t+1 run behind the solve of step t, joints JM+1..J behind
  // the friction / right-hand-side phase of step t+1.  Blocks of step t live in buffer t & 1.
  constexpr int JM = (J + 1) / 2;
  {
    double2 bP, bQ;
    make_blocks(s, c, bP, bQ);
    sts2(mine, ROW_P * kRow, bP);
    sts2(mine, ROW_Q * kRow, bQ);
    __syncwarp();
    factorise(1, JM, 0);
  }

  double sgx = 0.0, sgy = 0.0;  // sum_t Gdot_t
  double* traj = (a.trajectory && live && seg <= N) ? a.trajectory + e * NO + jpair : nullptr;
  const long long traj_step = a.B * NO;
  // this lane's pair of the current observation: (th_i, thd_i), or (Gdot_x, Gdot_y) on lane N
  double oa = is_seg ? th : gdx, ob = is_seg ? thd : gdy;

  // one step; BUF = t & 1 as a compile-time constant (the time loop is unrolled by two)
  auto step = [&](const int t, auto buf_c) {
    constexpr int buf = decltype(buf_c)::value;
    // ---- round 1 ----
    const double ts = thd * s, tc = thd * c;
    if (LINEAR) sts2(mine, ROW_OBS * kRow, NORM ? make_double2(oa - mu_a, ob - mu_b) : make_double2(oa, ob));
    sts2(mine, ROW_T * kRow, make_double2(ts, tc));
    __syncwarp();
    double2 xo[LINEAR ? N + 1 : 1], tq[N];
    if (LINEAR) {
#pragma unroll
      for (int q = 0; q <= N; ++q) xo[q] = lds2(gbase, ROW_OBS * kRow + q * 16);
    }
#pragma unroll
    for (int q = 0; q < N; ++q) tq[q] = lds2(gbase, ROW_T * kRow + q * 16);

    // ---- sine/cosine and joint blocks of step t+1 while the loads are in flight: th(t+1) = th + h thd(t)
    //      only needs this step's velocity.  Base tier unconditionally; the rare tiers (tail polynomial,
    //      exact sincos, the re-evaluation every 64th step) under a warp-uniform branch that only repairs
    //      the lanes that need it. ----
    double sN = s, cN = c;
    double2 bP, bQ;
    {
      const double d = P.h * thd;
      const int hi = __double2hiint(d) & 0x7fffffff;
      th = fma(P.h, thd, th);
      double z, sn, cm1;
      small_sincos_base(d, z, sn, cm1);
      rotate_by(sn, cm1, sN, cN);
      make_blocks(sN, cN, bP, bQ);
      const bool resync = (t & 63) == 63;
      const bool slow = resync || hi > kRotateShortHi;
      if (__any_sync(FULL, slow)) {
        if (slow) {
          if (resync || hi > kRotateLongHi) {
            sincos(th, &sN, &cN);
          } else {
            small_sincos_tail(d, z, sn, cm1);
            sN = s; cN = c;
            rotate_by(sn, cm1, sN, cN);
          }
        }
        make_blocks(sN, cN, bP, bQ);
      }
    }
    sts2(mine, (ROW_P + (buf ^ 1)) * kRow, bP);
    sts2(mine, (ROW_Q + (buf ^ 1)) * kRow, bQ);

    factorise(JM + 1, J, buf);
    double du = du_fixed;
    if (LINEAR) {
      double d0 = 0.0, d1 = 0.0;
#pragma unroll
      for (int q = 0; q <= N; ++q) {
        d0 = fma(D[2 * q], xo[q].x, d0);
        d1 = fma(D[2 * q + 1], xo[q].y, d1);
      }
      du = d0 + d1;
    }
    double vx = gdx * P.inv_l, vy = gdy * P.inv_l;
#pragma unroll
    for (int q = 0; q < N; ++q) {
      vx = fma(om[q], tq[q].x, vx);
      vy = fma(-om[q], tq[q].y, vy);
    }
    const double vn = fma(vy, c, -vx * s);  // F = m2kappa * vn; h_gdd_c carries m2kappa for the sum below
    const double tau = fma(P.kappa, thd, du);
    const double ttc = thd * tc, tts = thd * ts;
    const double am = fma(P.m2kappa, vn, -tau), bp = fma(P.m2kappa, vn, tau);
    // A_i = psi_i - w^_i = (F - tau~) n_i + thd^2 p_i;  B_i = psi_i + w^_i = (F + tau~) n_i - thd^2 p_i
    const double Ax = fma(-am, s, ttc), Ay = fma(am, c, tts);
    const double Bx = -fma(bp, s, ttc), By = fma(bp, c, -tts);
    const double Bpx = __shfl_up_sync(FULL, Bx, 1, L), Bpy = __shfl_up_sync(FULL, By, 1, L);
    // sum_q (v_q.n_q) n_q over the environment's lanes: log2(L) shuffle levels instead of a shared-memory row
    // read back by every lane (N additions per component and N + 1 wavefronts of the SM-wide shared-memory
    // pipe); independent of round 2, it overlaps the exchange below
    const double psx = group_sum<L>(is_seg ? -vn * s : 0.0), psy = group_sum<L>(is_seg ? vn * c : 0.0);

    // ---- round 2 ----
    sts2(mine, ROW_R * kRow, make_double2(Ax - Bpx, Ay - Bpy));  // r_i, meaningful for joints 1..J
    __syncwarp();
    // right-hand sides with this step's factorisation: r'_j = r_j - T_j r'_{j-1}, w_j = X_j r'_j
    double wx[J > 0 ? J : 1], wy[J > 0 ? J : 1];
    {
      double rx = 0.0, ry = 0.0;
#pragma unroll
      for (int j = 1; j <= J; ++j) {
        const double2 rj = lds2(gbase, ROW_R * kRow + j * 16);
        double r0 = rj.x, r1 = rj.y;
        if (j >= 2) {
          r0 = fma(-T1[j - 2], ry, fma(-T0[j - 2], rx, r0));
          r1 = fma(-T3[j - 2], ry, fma(-T2[j - 2], rx, r1));
        }
        rx = r0; ry = r1;
        wx[j - 1] = fma(Xa[j - 1], r0, Xb[j - 1] * r1);
        wy[j - 1] = fma(Xb[j - 1], r0, Xd[j - 1] * r1);
      }
    }
    // g_j = w_j - T_{j+1}^T g_{j+1}; this lane needs e = g_seg + g_{seg+1} (free head / tail: g_0 = g_N = 0)
    double ex = 0.0, ey = 0.0;
    {
      double gx = 0.0, gy = 0.0;
#pragma unroll
      for (int j = J; j >= 1; --j) {
        double x = wx[j - 1], y = wy[j - 1];
        if (j < J) {
          x = fma(-T2[j - 1], gy, fma(-T0[j - 1], gx, x));
          y = fma(-T3[j - 1], gy, fma(-T1[j - 1], gx, y));
        }
        gx = x; gy = y;
        // (picking g_seg, g_{seg+1} with selects instead of 2J predicated additions: 6 FP64 instructions fewer
        // for n = 5, measured slower for n = 3 and 7, profiles/r02_summary.md)
        if (seg == j || seg == j - 1) { ex += gx; ey += gy; }
      }
    }
    const double thdd = fma(3.0, fma(c, ey, -s * ex), tau);
    // ---- explicit Euler (remy_swimmer_env.py:88-91), reward = Gdot_new . direction ----
    gdx = fma(P.h_gdd_c, psx, gdx);
    gdy = fma(P.h_gdd_c, psy, gdy);
    thd = fma(P.h, thdd, thd);
    s = sN; c = cN;
    sgx += gdx;
    sgy += gdy;
    oa = is_seg ? th : gdx;
    ob = is_seg ? thd : gdy;
    if (STATS) {
      const double da = oa - pv_a, db = ob - pv_b;
      s1a += da; s2a = fma(da, da, s2a);
      s1b += db; s2b = fma(db, db, s2b);
    }
    if (traj) *reinterpret_cast<double2*>(traj + (long long)t * traj_step) = make_double2(oa, ob);
    factorise(1, JM, buf ^ 1);  // first half of step t+1's chain, from the blocks published before round 2
  };
  {
    int t = 0;
    for (; t + 1 < a.H; t += 2) {
      step(t, std::integral_constant<int, 0>());
      step(t + 1, std::integral_constant<int, 1>());
    }
    if (t < a.H) step(t, std::integral_constant<int, 0>());
  }

  if (live) {
    if (seg == 0) {
      const double ret = fma(sgx, P.dirx, sgy * P.diry);
      const long long eo = output_row<MODELS>(a, e);
      a.returns[eo] = a.accumulate ? a.returns[eo] + ret : ret;
    }
    if (a.final_state && seg <= N) {
      *reinterpret_cast<double2*>(a.final_state + output_row<MODELS>(a, e) * NO + jpair) =
          is_seg ? make_double2(th, thd) : make_double2(gdx, gdy);
    }
  } else if (active && seg == 0) {
    a.returns[output_row<MODELS>(a, e)] = __longlong_as_double(0x7ff8000000000000LL);  // screened out: NaN (see rollout_kernel)
  }

  if (STATS) {
    // fixed-order sum over the environments of this warp (xor butterfly over the group index)
    if (!live) { s1a = s1b = s2a = s2b = 0.0; }
#pragma unroll
    for (int off = L; off < 32; off <<= 1) {
      s1a += __shfl_xor_sync(FULL, s1a, off);
      s1b += __shfl_xor_sync(FULL, s1b, off);
      s2a += __shfl_xor_sync(FULL, s2a, off);
      s2b += __shfl_xor_sync(FULL, s2b, off);
    }
    if (grp == 0 && seg <= N) {
      double* o = a.stats_partial + (long long)blockIdx.x * 2 * NO;
      o[jpair] = s1a; o[jpair + 1] = s1b;
      o[NO + jpair] = s2a; o[NO + jpair + 1] = s2b;
    }
  }
}

}  // namespace swm
