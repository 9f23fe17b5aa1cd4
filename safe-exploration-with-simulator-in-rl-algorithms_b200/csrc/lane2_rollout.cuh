// Warp-specialised lane-split rollout: the lane-split kernel of lane_rollout.cuh cut into TWO warps per
// group of 32/L environments, for batches so small that SM sub-partitions would otherwise sit idle (the
// per-GPU share of BASELINE config[2] on >= 2 GPUs: <= 1,024 five-segment environments = 256 lane groups for
// 592 sub-partitions).
//
//   warp M ("main")      holds the state and runs the recurrence of a step: observation / velocity exchange
//                        (round 1), policy-row dot product, friction, joint right-hand sides (round 2),
//                        thdd_i = tau_i + y_i . r, Euler, V2 moments, trajectory output, and its own segment's
//                        tracked sine/cosine;
//   warp F ("operator")  a pure function of the ANGLES of a step (th(t+1) = th + h thd(t) needs nothing of step
//                        t but its velocity, so they are known a step ahead): the 2x2 blocks of the joint system,
//                        its factorisation, and for every lane the row y_i of the solution operator
//                        (thdd_i - tau_i = 3 n_i . (g_i + g_{i+1}) with M g = r  ==  y_i . r with M y_i = c_i).
//
// In the one-warp kernel those two instruction streams share one in-order issue port (214 FP64 instructions and
// ~800 cycles per step for n = 5); here each has its own sub-partition: M issues ~100 FP64 instructions per step and
// its dependent chain no longer contains the block-tridiagonal solve (2J FMAs instead), F issues ~185.  F uses a
// division-free recurrence for the pivot blocks (E_{j+1} = kappa_{j+1} P_{j+1} - Q_j adj(E_j) Q_j with
// kappa_{j+1} = det(E_j) / kappa_j, X_j = (kappa_j / det E_j) adj(E_j)): the reciprocals leave the dependent
// chain (40 instead of ~105 cycles per joint), so that F keeps pace with M.
//
// Hand-over through shared memory, double-buffered by step parity, ordered by named barriers (bar.arrive on the
// producer, bar.sync on the consumer, 64 threads each; one barrier id per (signal, parity), so a producer that
// runs ahead can never complete a barrier phase on its own):
//   M -> F  (sin, cos)(t+1) of every segment    during M's step t (after round 1)
//   F -> M  y_i(t+1), 2J doubles per lane        before M's dot product of step t+1
// Same equations, same per-lane decisions and fixed-order sums as lane_rollout.cuh (whose header explains the
// per-step algorithm): trajectories do not depend on which environments share a CTA.  Results differ from the
// other two rollout kernels by rounding only (tests/test_lane_split.py).
#pragma once
#include "lane_rollout.cuh"


namespace swm {

constexpr int kLane2Block = 64;

__device__ __forceinline__ void named_bar_sync(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(int id) { asm volatile("bar.arrive %0, 64;" ::"r"(id) : "memory"); }

// NF = number of operator warps (1 or 2).  With two, warp 1 forms the rows of the even steps and warp 2 those of
// the odd steps (each owns one parity of the (sin, cos) / row buffers and of the barrier ids, so nothing else
// changes): a row set is then due every second step of M instead of every step.
// SCREEN = per-step state-constraint screening (Safe_ARS.rollout, safe_ars/ars.py:124-153; see rollout_kernel): before
// a step is taken, one step of the simulator model from the same state is judged by max_i |thd_i| <= sim_thresh.  In
// the non-dimensional form the joint matrix only depends on the angles, so the simulator's accelerations are a second
// right-hand side dotted with the SAME solution rows; an environment judged unsafe freezes for the rest of the horizon
// (its lanes keep taking part in the exchanges, nothing of it advances).
// MODELS: the model-set mode of rollout_kernel (CTA row blockIdx.y runs model blockIdx.y; warp F needs no model).
template <int N, bool LINEAR, bool NORM, bool STATS, int NF, bool SCREEN, bool MODELS>
__global__ void __launch_bounds__(32 * (1 + NF))
lane2_rollout_kernel(const RolloutArgs a, const __grid_constant__ typename ScreenForms<SCREEN_NONE, MODELS>::type models) {
  static_assert(!MODELS || (!STATS && !SCREEN), "model set: no statistics, no screening");
  static_assert(NF == 1 || NF == 2, "one or two operator warps");
  static_assert(!SCREEN || (LINEAR && !NORM && !STATS), "screening: plain linear policies only");
  constexpr int L = LaneSplit<N>::L, G = LaneSplit<N>::G;
  constexpr int NO = 2 * N + 2, NA = N - 1, WS = NA * NO, J = N - 1;
  constexpr int NV = 7 * J - 4 > 0 ? 7 * J - 4 : 3;  // X_j (3 each, j = 1..J) then T_j (4 each, j = 2..J)
  constexpr unsigned FULL = 0xffffffffu;
  constexpr int kRow = 32 * 16;
  // rows of one double2 per lane; + parity where noted
  enum { ROW_OBS = 0, ROW_T = 1, ROW_R = 2, ROW_PSI = 3, ROW_SC = 4, ROW_RS = 6, ROWS = SCREEN ? 7 : 6 };  // SC: + parity
  // barrier ids: signal base + parity  (0 is __syncthreads)
  enum { BAR_SC = 1, BAR_XT = 3 };
  __shared__ __align__(16) double2 sh[ROWS][32];
  __shared__ __align__(16) double2 sh_y[2][J > 0 ? J : 1][32];  // [parity][joint][lane]: this lane's y_i at joint j

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int seg = lane & (L - 1), grp = lane / L;
  const uint32_t sh_base = (uint32_t)__cvta_generic_to_shared(&sh[0][0]);
  const uint32_t gbase = sh_base + (uint32_t)(grp * L * 16);
  const uint32_t mine = gbase + (uint32_t)(seg * 16);
  const uint32_t y_mine = (uint32_t)__cvta_generic_to_shared(&sh_y[0][0][0]) + (uint32_t)(lane * 16);
  constexpr int kYBuf = (J > 0 ? J : 1) * kRow;
  const bool is_seg = seg < N;
  const long long e0 = (long long)blockIdx.x * G + grp;
  const bool active = e0 < a.B;
  const long long e = active ? e0 : a.B - 1;
  const unsigned int iteration = a.iteration + (a.iter_dev ? *a.iter_dev : 0u);
  const Phys& P = rollout_model<MODELS>(a, models);

  // ---- initial state (both warps): this lane's pair of the observation ----
  const int jpair = is_seg ? 2 + 2 * seg : 0;
  double gdx, gdy, th = 0.0, thd = 0.0;
  if (a.init_state) {
    const double* sp = a.init_state + (e % a.init_count) * NO;
    gdx = sp[0]; gdy = sp[1];
    if (is_seg) { th = sp[jpair]; thd = sp[jpair + 1]; }
  } else {
    gdx = gdy = 0.0;
    if (is_seg) th = 1.5707963267948966;
  }
  if (a.init_perturb != 0.0) {
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

  if (warp >= 1) {
    // =========================================== warp F ===========================================
    // A pure function of the angles: (sin, cos) of every segment at step u  ->  this lane's row y_i(u) of the
    // solution operator.  Every lane reads all N (sin, cos) pairs M published (no exchange inside this warp),
    // forms the blocks and the factorisation redundantly and solves for its own row.
    if (a.H <= 0) return;
    auto frow = [&](auto buf_c) {
      constexpr int buf = decltype(buf_c)::value;
      named_bar_sync(BAR_SC + buf);                        // (sin, cos)(u) of all segments published by M
      const double2 own = lds2(mine, (ROW_SC + buf) * kRow);             // (sin, cos) of this lane's segment
      const double sn = own.x, cn = own.y;
      double V[NV + 1];
      double ss[N], sc[N];
#pragma unroll
      for (int q = 0; q < N; ++q) {
        const double2 v = lds2(gbase, (ROW_SC + buf) * kRow + q * 16);
        ss[q] = v.x * v.x;
        sc[q] = v.x * v.y;
      }
      // division-free factorisation: E_{j+1} = kappa_{j+1} P_{j+1} - Q_j adj(E_j) Q_j, kappa_{j+1} = det E_j / kappa_j,
      // X_j = (kappa_j / det E_j) adj(E_j), T_{j+1} = Q_j X_j;  P_j = 2I + 3(N_{j-1} + N_j), Q_j = 3 N_j - I
      double ea = fma(3.0, ss[0] + ss[J > 0 ? 1 : 0], 2.0), eb = -3.0 * (sc[0] + sc[J > 0 ? 1 : 0]), ed = 10.0 - ea;
      double kap = 1.0, ikap = 1.0;
#pragma unroll
      for (int j = 1; j <= J; ++j) {
        const double delta = fma(ea, ed, -eb * eb);
        const double rho = kap * fast_rcp(delta);
        V[3 * (j - 1)] = rho * ed;
        V[3 * (j - 1) + 1] = -rho * eb;
        V[3 * (j - 1) + 2] = rho * ea;
        if (j < J) {
          const double qa = fma(3.0, ss[j], -1.0), qb = -3.0 * sc[j], qd = 1.0 - qa;
          const double pa = fma(3.0, ss[j] + ss[j + 1], 2.0), pb = -3.0 * (sc[j] + sc[j + 1]);
          // M = Q adj(E), adj(E) = (ed, -eb; -eb, ea)
          const double m00 = fma(qa, ed, -qb * eb), m01 = fma(qb, ea, -qa * eb);
          const double m10 = fma(qb, ed, -qd * eb), m11 = fma(qd, ea, -qb * eb);
          V[3 * J + 4 * (j - 1)] = rho * m00;      // T_{j+1} = Q_j X_j
          V[3 * J + 4 * (j - 1) + 1] = rho * m01;
          V[3 * J + 4 * (j - 1) + 2] = rho * m10;
          V[3 * J + 4 * (j - 1) + 3] = rho * m11;
          const double s00 = fma(m00, qa, m01 * qb), s01 = fma(m00, qb, m01 * qd), s11 = fma(m10, qb, m11 * qd);
          const double kn = delta * ikap;
          ea = fma(kn, pa, -s00);
          eb = fma(kn, pb, -s01);
          ed = fma(kn, 10.0 - pa, -s11);
          ikap = rho;
          kap = kn;
        }
      }
      // this lane's row: thdd_i - tau_i = 3 n_i . (g_i + g_{i+1}) with M g = r, i.e. y_i . r with M y_i = c_i
      // (M symmetric), c_i = 3 n_i at the blocks of joints i and i+1.
      // forward: c'_j = c_j - T_j c'_{j-1},  w_j = X_j c'_j
      const double nx = -3.0 * sn, ny = 3.0 * cn;
      double wx[J > 0 ? J : 1], wy[J > 0 ? J : 1];
      {
        double rx = 0.0, ry = 0.0;
#pragma unroll
        for (int j = 1; j <= J; ++j) {
          const bool on = is_seg && (seg == j || seg == j - 1);
          double r0 = on ? nx : 0.0, r1 = on ? ny : 0.0;
          if (j >= 2) {
            const int o = 3 * J + 4 * (j - 2);
            r0 = fma(-V[o + 1], ry, fma(-V[o], rx, r0));
            r1 = fma(-V[o + 3], ry, fma(-V[o + 2], rx, r1));
          }
          rx = r0; ry = r1;
          wx[j - 1] = fma(V[3 * (j - 1)], r0, V[3 * (j - 1) + 1] * r1);
          wy[j - 1] = fma(V[3 * (j - 1) + 1], r0, V[3 * (j - 1) + 2] * r1);
        }
      }
      // back: y_j = w_j - T_{j+1}^T y_{j+1}; stored as soon as known (row j of this lane)
      {
        double gx = 0.0, gy = 0.0;
#pragma unroll
        for (int j = J; j >= 1; --j) {
          double x = wx[j - 1], y = wy[j - 1];
          if (j < J) {
            const int o = 3 * J + 4 * (j - 1);
            x = fma(-V[o + 2], gy, fma(-V[o], gx, x));
            y = fma(-V[o + 3], gy, fma(-V[o + 1], gx, y));
          }
          gx = x; gy = y;
          sts2(y_mine, buf * kYBuf + (j - 1) * kRow, make_double2(gx, gy));
        }
      }
      named_bar_arrive(BAR_XT + buf);                      // rows y_i(u) ready
    };
    // one row set per step u = 0 .. H-1 (M publishes the angles of step u+1 during step u, those of step 0
    // before its loop)
    if (NF == 1) {
      int u = 0;
      for (; u + 1 < a.H; u += 2) {
        frow(std::integral_constant<int, 0>());
        frow(std::integral_constant<int, 1>());
      }
      if (u < a.H) frow(std::integral_constant<int, 0>());
    } else if (warp == 1) {
      for (int u = 0; u < a.H; u += 2) frow(std::integral_constant<int, 0>());
    } else {
      for (int u = 1; u < a.H; u += 2) frow(std::integral_constant<int, 1>());
    }
    return;
  }

  // ============================================= warp M =============================================
  double D[LINEAR ? 2 * (N + 1) : 1];
  double du_fixed = 0.0;
  const bool has_ka = is_seg && seg >= 1, has_kb = is_seg && seg <= N - 2;
  if (LINEAR) {
    const long long q = e / a.R;
    const bool philox = a.policy_mode == SWM_POLICY_PHILOX;
    const bool from_mem = a.policy_mode == SWM_POLICY_DELTAS;
    const double* base = (philox || from_mem) ? a.policies : a.policies + q * WS;
    const double* dmem = from_mem ? a.deltas + (q >> 1) * WS : nullptr;
    const double sgn_nu = (q & 1) ? -a.nu : a.nu;
    const unsigned int dir = a.dir0 + (unsigned int)(q >> 1);
    auto weight_pair = [&](int k, int slot, double& w0, double& w1) {
      const int j = (slot == N) ? 0 : 2 + 2 * slot;
      const int flat = k * NO + j;
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
        w0 = __dadd_rn(w0, __dmul_rn(sgn_nu, d0));
        w1 = __dadd_rn(w1, __dmul_rn(sgn_nu, d1));
      }
      if (NORM) {
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
  double mu_a = 0.0, mu_b = 0.0, pv_a = 0.0, pv_b = 0.0;
  if (NORM && seg <= N) { mu_a = a.mean[jpair]; mu_b = a.mean[jpair + 1]; }
  if (STATS && seg <= N) { pv_a = a.stats_pivot[jpair]; pv_b = a.stats_pivot[jpair + 1]; }
  double s1a = 0.0, s1b = 0.0, s2a = 0.0, s2b = 0.0;
  double om[N];
#pragma unroll
  for (int q = 0; q < N; ++q) om[q] = (N - q - 0.5) / N - (q < seg ? 1.0 : 0.0) - (q == seg ? 0.5 : 0.0);

  bool skipped = false;
  if (LINEAR && a.dir_mask) skipped = a.dir_mask[(e / a.R) >> 1] == 0;
  const bool live = active && !skipped;
  if (active && skipped && a.final_state && seg <= N) {
    double2* o = reinterpret_cast<double2*>(a.final_state + output_row<MODELS>(a, e) * NO + jpair);
    *o = is_seg ? make_double2(th, thd) : make_double2(gdx, gdy);
  }
  double sgx = 0.0, sgy = 0.0;
  // screening state (per environment, replicated on its lanes)
  const Phys& PS = a.sim;
  bool alive = true;
  int viol = 0, frozen = a.H;
  const double u_ratio = SCREEN ? PS.u_scale / P.u_scale : 1.0, dinv_l = SCREEN ? PS.inv_l - P.inv_l : 0.0;
  double* traj = (a.trajectory && live && seg <= N) ? a.trajectory + e * NO + jpair : nullptr;
  const long long traj_step = a.B * NO;
  double oa = is_seg ? th : gdx, ob = is_seg ? thd : gdy;

  // tracked (sin, cos) of this lane's segment; the angles of step 0 go to warp F before the loop
  double s, c;
  sincos(th, &s, &c);
  if (a.H > 0) {
    sts2(mine, (ROW_SC + 0) * kRow, make_double2(s, c));
    named_bar_arrive(BAR_SC + 0);
  }

  auto mstep = [&](const int t, auto buf_c) {
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
    // ---- sine/cosine of step t+1 while the loads are in flight (th(t+1) = th + h thd(t)); base tier
    //      unconditionally, rare tiers under a warp-uniform branch (see lane_rollout.cuh); warp F turns the
    //      angles of step t+1 into the solution rows of step t+1 while M finishes step t ----
    double sN = s, cN = c;
    const double th_prev = th;
    {
      const double d = P.h * thd;
      const int hi = __double2hiint(d) & 0x7fffffff;
      th = fma(P.h, thd, th);
      double z, sn, cm1;
      small_sincos_base(d, z, sn, cm1);
      rotate_by(sn, cm1, sN, cN);
      const bool resync = (t & 63) == 63;
      const bool slow = resync || hi > kRotateShortHi;
      if (__any_sync(FULL, slow)) {  // out of line: see tracked_sincos_slow
        const double2 r = tracked_sincos_slow(th, d, s, c, resync || hi > kRotateLongHi);
        if (slow) { sN = r.x; cN = r.y; }
      }
    }
    if (t + 1 < a.H) {
      sts2(mine, (ROW_SC + (buf ^ 1)) * kRow, make_double2(sN, cN));
      named_bar_arrive(BAR_SC + (buf ^ 1));                // angles of step t+1 for F
    }
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
    const double Ax = fma(-am, s, ttc), Ay = fma(am, c, tts);
    const double Bx = -fma(bp, s, ttc), By = fma(bp, c, -tts);
    const double Bpx = __shfl_up_sync(FULL, Bx, 1, L), Bpy = __shfl_up_sync(FULL, By, 1, L);
    double taus = 0.0;
    if (SCREEN) {
      // the simulator's right-hand side from the same state: its own l (velocities in units of l), kappa, torque scale
      const double vxs = fma(gdx, dinv_l, vx), vys = fma(gdy, dinv_l, vy);
      const double vns = fma(vys, c, -vxs * s);
      taus = fma(PS.kappa, thd, du * u_ratio);
      const double ams = fma(PS.m2kappa, vns, -taus), bps = fma(PS.m2kappa, vns, taus);
      const double Axs = fma(-ams, s, ttc), Ays = fma(ams, c, tts);
      const double Bxs = -fma(bps, s, ttc), Bys = fma(bps, c, -tts);
      const double Bpxs = __shfl_up_sync(FULL, Bxs, 1, L), Bpys = __shfl_up_sync(FULL, Bys, 1, L);
      sts2(mine, ROW_RS * kRow, make_double2(Axs - Bpxs, Ays - Bpys));
    }
    // ---- round 2 ----
    sts2(mine, ROW_PSI * kRow, is_seg ? make_double2(-vn * s, vn * c) : make_double2(0.0, 0.0));
    sts2(mine, ROW_R * kRow, make_double2(Ax - Bpx, Ay - Bpy));
    __syncwarp();
    // thdd_i = tau_i + y_i . r  (the block-tridiagonal solve was folded into y_i by warp F, which forms the rows
    // of this step while M runs rounds 1 and 2)
    named_bar_sync(BAR_XT + buf);
    double2 yrow[J > 0 ? J : 1];
#pragma unroll
    for (int j = 1; j <= J; ++j) yrow[j - 1] = lds2(y_mine, buf * kYBuf + (j - 1) * kRow);
    double acc0 = tau, acc1 = 0.0;
#pragma unroll
    for (int j = 1; j <= J; ++j) {
      const double2 rj = lds2(gbase, ROW_R * kRow + j * 16);
      acc0 = fma(yrow[j - 1].x, rj.x, acc0);
      acc1 = fma(yrow[j - 1].y, rj.y, acc1);
    }
    const double thdd = acc0 + acc1;
    if (SCREEN) {
      double b0 = taus, b1 = 0.0;
#pragma unroll
      for (int j = 1; j <= J; ++j) {
        const double2 rj = lds2(gbase, ROW_RS * kRow + j * 16);
        b0 = fma(yrow[j - 1].x, rj.x, b0);
        b1 = fma(yrow[j - 1].y, rj.y, b1);
      }
      const double sthd = fma(PS.h, b0 + b1, thd);
      const double cost = group_max_abs<L>(is_seg ? sthd : 0.0);
      // unsafe (or NaN): nothing advances, and since observation and policy never change again it never will
      if (alive && !(cost <= a.sim_thresh)) { alive = false; frozen = t; }
    }
    // (the shuffle butterfly of lane_rollout.cuh instead of this row: 6-12 % slower here for n = 3 and 5, M's
    // step is a latency chain and the row read hides behind the barrier wait; profiles/r02_summary.md)
    double psx = 0.0, psy = 0.0;
#pragma unroll
    for (int q = 0; q < N; ++q) {
      const double2 pq = lds2(gbase, ROW_PSI * kRow + q * 16);
      psx += pq.x;
      psy += pq.y;
    }
    if (!SCREEN || alive) {
      gdx = fma(P.h_gdd_c, psx, gdx);
      gdy = fma(P.h_gdd_c, psy, gdy);
      thd = fma(P.h, thdd, thd);
      s = sN; c = cN;
      sgx += gdx;
      sgy += gdy;
    } else {
      th = th_prev;
    }
    if (SCREEN) {
      const double cost = group_max_abs<L>(is_seg ? thd : 0.0);
      viol += (alive && cost > a.real_thresh) ? 1 : 0;
    }
    oa = is_seg ? th : gdx;
    ob = is_seg ? thd : gdy;
    if (STATS) {
      const double da = oa - pv_a, db = ob - pv_b;
      s1a += da; s2a = fma(da, da, s2a);
      s1b += db; s2b = fma(db, db, s2b);
    }
    if (traj) *reinterpret_cast<double2*>(traj + (long long)t * traj_step) = make_double2(oa, ob);
  };
  {
    int t = 0;
    for (; t + 1 < a.H; t += 2) {
      mstep(t, std::integral_constant<int, 0>());
      mstep(t + 1, std::integral_constant<int, 1>());
    }
    if (t < a.H) mstep(t, std::integral_constant<int, 0>());
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
    if (SCREEN && seg == 0) {
      if (a.violations) a.violations[e] = viol;
      if (a.frozen_at) a.frozen_at[e] = frozen;
    }
  } else if (active && seg == 0) {
    a.returns[output_row<MODELS>(a, e)] = __longlong_as_double(0x7ff8000000000000LL);
    if (SCREEN) {  // masked out: never judged unsafe, no real step taken (as rollout_kernel)
      if (a.violations) a.violations[e] = 0;
      if (a.frozen_at) a.frozen_at[e] = a.H;
    }
  }
  if (STATS) {
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
