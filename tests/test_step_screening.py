"""Per-step simulator screening (Safe_ARS.rollout, safe_ars/ars.py:124-153) against the CPU oracle's
orc_rollout_safe_step on every kernel that implements it: the one-thread-per-environment rollout_kernel and the
warp-specialised lane2_rollout_kernel with one (LANES2) or two (LANES3) operator warps.

Before every real step one simulator step is taken from the same state; the real step is taken only if
max_i |thd_i| of the simulated state is <= sim_thresh, otherwise the environment freezes for good.  Real steps
whose cost is > real_thresh are counted as violations.  The freeze step and the violation count must equal the
oracle's exactly.  GPU and oracle differ by rounding, so every threshold is placed between neighbouring costs of
the oracle's own rollouts, and every cost a decision depends on is asserted to be at least
MARGIN * max(1, |threshold|) away from it: an exact check can then not flip on rounding.  Returns, final states
and trajectories (frozen tail included) are held to the parity bars of the other rollout tests."""
import ctypes
import functools

import numpy as np
import pytest
import torch

from conftest import rand_states, rel_err

pytestmark = pytest.mark.gpu
RET_TOL = 1e-6
STATE_TOL = 1e-8
MARGIN = 1e-9
KERNELS = ["THREAD", "LANES2", "LANES3"]


def _cuda(a):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _ret_err(got, want):
    got, want = np.asarray(got), np.asarray(want)
    return float(np.max(np.abs(got - want) / np.maximum(1e-3, np.abs(want))))


def _k(S, name):
    return getattr(S, "KERNEL_" + name)


def _models(mod, n):
    """Real model and a simulator that differs from it in l, m, k and h."""
    real = mod.make_params(n=n, l_i=.9, m_i=1.1, k=9.5, h=0.001, direction=(.6, .8))
    sim = mod.make_params(n=n, l_i=.93, m_i=1.05, k=9.9, h=0.0012, direction=(.6, .8))
    return real, sim


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _kernel_choice(S, real, sim, B, kernel, policy_mode, R=1):
    cfg = S._lib.SwmRollout()
    cfg.variant, cfg.policy_mode, cfg.H, cfg.B, cfg.rollouts_per_policy = S.GYM, policy_mode, 10, B, R
    cfg.kernel = kernel
    cfg.screen.enabled = 1
    cfg.screen.sim = sim
    return S._lib.lib().swm_rollout_kernel_choice(ctypes.byref(real), ctypes.byref(cfg))


def _screened(S, kern, real, sim, H, sim_thr, real_thr, policy_mode=None, **kw):
    """Screened rollout on a forced kernel (final state and trajectory wanted); asserts that kernel ran."""
    B = kw.get("B")
    if B is None:
        B = kw["policies"].shape[0] * kw.get("rollouts_per_policy", 1)
    mode = policy_mode if policy_mode is not None else (
        S.ops.POLICY_EXPLICIT if "policies" in kw else S.ops.POLICY_PHILOX)
    assert _kernel_choice(S, real, sim, B, _k(S, kern), mode, kw.get("rollouts_per_policy", 1)) == _k(S, kern)
    return S.ops.rollout(real, H, want_final=True, want_trajectory=True, kernel=_k(S, kern),
                         screen=dict(sim_params=sim, sim_thresh=sim_thr, real_thresh=real_thr), **kw)


def _host(res):
    return (res.returns.cpu().numpy(), res.final_state.cpu().numpy(), res.trajectory.cpu().numpy(),
            res.frozen_at.cpu().numpy(), res.violations.cpu().numpy())


def _self_consistent(res, starts, H, real_thr):
    """Exact properties of the kernel's own output: the violation count is the number of stored states before the
    freeze whose max |thd| exceeds real_thr, and from the freeze on every stored state is the state before it."""
    _, fin, traj, fz, viol = _host(res)
    B = fin.shape[0]
    assert ((fz >= 0) & (fz <= H)).all()
    for e in range(B):
        f = int(fz[e])
        cost = np.max(np.abs(traj[:f, e, 3::2]), axis=1) if f else np.zeros(0)
        assert int(np.sum(cost > real_thr)) == viol[e], e
        held = starts[e] if f == 0 else traj[f - 1, e]
        assert np.array_equal(_bits(traj[f:, e]), np.broadcast_to(_bits(held), traj[f:, e].shape)), e
        assert np.array_equal(_bits(fin[e]), _bits(traj[-1, e] if H else starts[e])), e


def _oracle_costs(O, real, sim, W, start, H):
    """Simulator cost before every step and real cost after it along the UNSCREENED oracle rollout: the screened
    rollout follows it up to and including its freeze step."""
    n = real.n
    W = np.asarray(W).reshape(n - 1, 2 * n + 2)
    _, _, traj = O.rollout(real, O.GYM, H, policy=W, init_state=start, want_traj=True)
    pre = np.vstack([start[None], traj[:-1]])
    nxt, _ = O.step_batch(sim, O.GYM, pre, pre @ W.T)
    return np.max(np.abs(nxt[:, 3::2]), axis=1), np.max(np.abs(traj[:, 3::2]), axis=1)


def _freeze_steps(sim_cost, thr):
    unsafe = ~(sim_cost <= thr)
    return np.where(unsafe.any(axis=1), unsafe.argmax(axis=1), sim_cost.shape[1])


def _margins_ok(sim_cost, real_cost, sim_thr, real_thr):
    """Every cost a decision depends on -- simulator costs up to and including the freeze step, real costs before
    it -- is at least MARGIN * max(1, |thr|) away from its threshold (non-finite thresholds need no margin)."""
    fz = _freeze_steps(sim_cost, sim_thr)
    H = sim_cost.shape[1]
    for e in range(len(fz)):
        f = int(fz[e])
        if np.isfinite(sim_thr):
            d = np.abs(sim_cost[e, :min(f + 1, H)] - sim_thr)
            if not d.min(initial=np.inf) >= MARGIN * max(1.0, abs(sim_thr)):
                return False
        if np.isfinite(real_thr) and f:
            d = np.abs(real_cost[e, :f] - real_thr)
            if not d.min() >= MARGIN * max(1.0, abs(real_thr)):
                return False
    return True


def _midpoint(costs, q):
    """A threshold halfway between two neighbouring sorted costs near quantile q, with a gap of >= 4 MARGIN."""
    c = np.unique(costs[np.isfinite(costs)])
    i0 = int(q * (len(c) - 2))
    for d in range(len(c)):
        for i in (i0 + d, i0 - d):
            if 0 <= i < len(c) - 1 and c[i + 1] - c[i] >= 4 * MARGIN * max(1.0, c[i + 1]):
                return 0.5 * (c[i] + c[i + 1])
    raise AssertionError("no threshold with a decision margin")


def _spread(fz, viol, H, zero=3, mid=5, mid_steps=5, never=5, violated=3):
    m = fz[(fz > 0) & (fz < H)]
    return ((fz == 0).sum() >= zero and len(m) >= mid and len(set(m.tolist())) >= mid_steps
            and (fz == H).sum() >= never and (viol > 0).sum() >= violated)


def _thresholds(sim_cost, real_cost, quantiles=np.linspace(0.05, 0.995, 200), **need):
    """Thresholds for which the oracle's decisions give the required spread, with their margins asserted; the
    simulator threshold is the first of the given cost quantiles that does."""
    H = sim_cost.shape[1]
    for q in quantiles:
        s = _midpoint(sim_cost, q)
        fz = _freeze_steps(sim_cost, s)
        taken = np.concatenate([real_cost[e, :fz[e]] for e in range(len(fz))])
        if taken.size < 2:
            continue
        for rq in (0.8, 0.9, 0.7, 0.95, 0.6, 0.5):
            r = _midpoint(taken, rq)
            viol = np.array([(real_cost[e, :fz[e]] > r).sum() for e in range(len(fz))])
            if _spread(fz, viol, H, **need):
                assert _margins_ok(sim_cost, real_cost, s, r)
                return s, r
    raise AssertionError("this population does not give the required spread of freeze steps")


def _starts(rng, n, count):
    """Start states whose angular velocities are scaled from 0.01 to 5 (in a random order)."""
    init = rand_states(rng, n, count, scale=1.0)
    init[:, 3::2] *= 10.0 ** np.linspace(-2.0, 0.7, count)[rng.permutation(count), None]
    return init


def _population(n, B, seed):
    """B explicit policies and start states: policy scales spread over 2.5 decades, start velocities over 2.7, in
    independent orders; six environments have near-zero policies and velocities.  At the thresholds chosen by
    _thresholds some are unsafe from the start, some become unsafe on the way and some never do."""
    rng = np.random.default_rng(seed)
    no = 2 * n + 2
    a = 10.0 ** np.linspace(-2.0, 0.5, B)[rng.permutation(B)]
    init = _starts(rng, n, B)
    calm = rng.permutation(B)[:6]
    a[calm] = 1e-3
    init[calm, 3::2] *= 1e-3
    W = rng.uniform(-1, 1, (B, n - 1, no)) * a[:, None, None]
    return W, init


def _compare_with_oracle(O, real, sim, pols, starts, H, sim_thr, real_thr, res):
    """Exact freeze steps and violation counts, returns / states / trajectories at the parity bars;
    -> largest (return, final-state, trajectory) errors."""
    got_r, got_f, traj, fz, viol = _host(res)
    er = ef = et = 0.0
    for e in range(len(got_r)):
        r, f, t, v, z = O.rollout_safe_step(real, sim, pols[e], H, sim_thr, real_thr, init_state=starts[e],
                                            want_traj=True)
        assert (fz[e], viol[e]) == (z, v), (e, fz[e], z, viol[e], v)
        er = max(er, _ret_err(got_r[e], r))
        ef = max(ef, rel_err(got_f[e], f))
        et = max(et, rel_err(traj[:, e], t) if H else 0.0)
    assert er < RET_TOL and ef < STATE_TOL and et < STATE_TOL, (er, ef, et)
    return er, ef, et


def _report(tag, errs):
    print("\n[step screening] %s: max return err %.2e, final state %.2e, trajectory %.2e" % ((tag,) + tuple(errs)))


# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kern", KERNELS)
@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 7, 8, 9, 10])
def test_screening_matches_oracle(S, O, n, kern):
    """Explicit policies, B = 37 (the last warp / CTA holds idle environments or lane groups), H = 201 (odd: the
    unroll-by-two tail; crosses the sine/cosine re-evaluations at steps 63, 127 and 191).  n >= 8 runs the
    shared-memory factorisation scratch of the thread kernel for both models and 16 lanes per environment."""
    B, H = 37, 201
    (real, sim), (ro, so) = _models(S, n), _models(O, n)
    W, init = _population(n, B, seed=100 + n)
    costs = [_oracle_costs(O, ro, so, W[e], init[e], H) for e in range(B)]
    sc, rc = np.array([c[0] for c in costs]), np.array([c[1] for c in costs])
    sim_thr, real_thr = _thresholds(sc, rc)
    res = _screened(S, kern, real, sim, H, sim_thr, real_thr, policies=_cuda(W), init_state=_cuda(init))
    errs = _compare_with_oracle(O, ro, so, W, init, H, sim_thr, real_thr, res)
    _self_consistent(res, init, H, real_thr)
    fz, viol = res.frozen_at.cpu().numpy(), res.violations.cpu().numpy()
    assert _spread(fz, viol, H)
    _report("%s n=%d" % (kern, n), errs)


@pytest.mark.parametrize("kern", KERNELS)
@pytest.mark.parametrize("n,R,D", [(3, 1, 16), (5, 3, 8), (5, 32, 2), (8, 3, 8), (10, 32, 2)])
def test_screening_policy_sources_match_oracle(S, O, n, R, D, kern):
    """W +- nu delta_k from in-kernel Philox, and the same perturbations read from memory (bit-identical).
    R > 1 rollouts per direction with R start states: R = 32 keeps one policy per warp in the thread kernel's shared
    memory (n = 5, 10), R = 3 one per thread (n = 5, 8)."""
    H, nu, seed, it, dir0 = 201, 0.3, 31 + n, 2, 5
    B, ws, no = 2 * D * R, (n - 1) * (2 * n + 2), 2 * n + 2
    (real, sim), (ro, so) = _models(S, n), _models(O, n)
    rng = np.random.default_rng(7 * n + R)
    Wb = rng.uniform(-1, 1, ws) * 0.05
    # R = 1: one start state per environment; R > 1: rollout r of every direction starts from init[r]
    count = B if R == 1 else R
    init = _starts(rng, n, count)
    pols, starts = [], []
    for e in range(B):
        q = e // R
        d = O.philox_delta(seed, it, dir0 + (q >> 1), ws)
        pols.append(Wb + (-nu if q & 1 else nu) * d)
        starts.append(init[e % count])
    pols, starts = np.array(pols), np.array(starts)
    costs = [_oracle_costs(O, ro, so, pols[e], starts[e], H) for e in range(B)]
    sc, rc = np.array([c[0] for c in costs]), np.array([c[1] for c in costs])
    need = dict(zero=1, mid=3, mid_steps=3, never=2, violated=2)
    sim_thr, real_thr = _thresholds(sc, rc, **need)
    kw = dict(B=B, base_policy=_cuda(Wb), nu=nu, seed=seed, iteration=it, dir0=dir0, rollouts_per_policy=R,
              init_state=_cuda(init))
    res = _screened(S, kern, real, sim, H, sim_thr, real_thr, **kw)
    errs = _compare_with_oracle(O, ro, so, pols, starts, H, sim_thr, real_thr, res)
    _self_consistent(res, starts, H, real_thr)
    assert _spread(res.frozen_at.cpu().numpy(), res.violations.cpu().numpy(), H, **need)
    mem = _screened(S, kern, real, sim, H, sim_thr, real_thr, policy_mode=S.ops.POLICY_DELTAS,
                    deltas=S.ops.philox_deltas(seed, it, dir0, D, ws), **kw)
    for name in ("returns", "frozen_at", "violations", "final_state", "trajectory"):
        assert torch.equal(getattr(mem, name), getattr(res, name)), name
    _report("%s n=%d R=%d philox" % (kern, n, R), errs)


@functools.lru_cache(maxsize=None)
def _freeze_pool(O, n):
    """64 random policies and starts with the oracle's simulator / real costs along 129 unscreened steps."""
    ro, so = _models(O, n)
    W, init = _population(n, 64, seed=500 + n)
    W *= 10.0 ** np.linspace(-0.5, 0.5, 64)[:, None, None]
    init[:, 3::2] *= 0.1
    costs = [_oracle_costs(O, ro, so, W[e], init[e], 129) for e in range(64)]
    return W, init, np.array([c[0] for c in costs]), np.array([c[1] for c in costs])


@pytest.mark.parametrize("kern", KERNELS)
@pytest.mark.parametrize("n", [3, 6, 9])
@pytest.mark.parametrize("H", [1, 2, 3, 63, 64, 65, 129])
def test_screening_freeze_position_and_horizon_edges(S, O, n, H, kern):
    """One launch per target step t* in {0, 1, 62, 63, 64, H-1}: the threshold sits between the running maximum of
    one environment's simulator cost before t* and its cost at t*, so that environment freezes exactly at t*.  Odd and
    even t* meet both operator warps of LANES3; t* = 63 is a step with the exact sine/cosine re-evaluation."""
    (real, sim), (ro, so) = _models(S, n), _models(O, n)
    W, init, sc, rc = _freeze_pool(O, n)
    sc, rc = sc[:, :H], rc[:, :H]
    for ts in sorted({t for t in (0, 1, 62, 63, 64, H - 1) if t < H}):
        run_max = np.max(sc[:, :ts], axis=1, initial=0.0)
        lo, hi = run_max, sc[:, ts]
        ok = np.isfinite(hi) & (hi - lo > 4 * MARGIN * np.maximum(1.0, hi))
        assert ok.any(), "no environment of the pool sets a new running maximum at step %d" % ts
        tgt = int(np.flatnonzero(ok)[np.argmax((hi - lo)[ok] / np.maximum(1.0, hi[ok]))])
        sim_thr = 0.5 * (lo[tgt] + hi[tgt])
        fz_all = _freeze_steps(sc, sim_thr)
        taken = np.concatenate([rc[e, :fz_all[e]] for e in range(len(fz_all))])
        real_thr = _midpoint(taken, 0.7) if taken.size >= 2 else 0.5 * sim_thr

        def clear(e):  # margins of every decision of environment e at these thresholds
            return _margins_ok(sc[e:e + 1], rc[e:e + 1], sim_thr, real_thr)

        assert clear(tgt) and fz_all[tgt] == ts
        # the target in the middle of a warp / lane group, fillers around it
        fill = [e for e in range(len(sc)) if e != tgt and clear(e)][:20]
        sel = fill[:5] + [tgt] + fill[5:]
        res = _screened(S, kern, real, sim, H, sim_thr, real_thr, policies=_cuda(W[sel]), init_state=_cuda(init[sel]))
        _compare_with_oracle(O, ro, so, W[sel], init[sel], H, sim_thr, real_thr, res)
        _self_consistent(res, init[sel], H, real_thr)
        assert int(res.frozen_at[5]) == ts


@pytest.mark.parametrize("kern", KERNELS)
@pytest.mark.parametrize("n", [2, 5, 8])
def test_screening_threshold_semantics(S, O, n, kern):
    """Non-finite and signed-zero thresholds decide as `cost <= sim_thresh` and `cost > real_thresh` do in the
    reference: NaN compares false, the cost is never negative."""
    B, H = 37, 65
    (real, sim), (ro, so) = _models(S, n), _models(O, n)
    W, init = _population(n, B, seed=300 + n)
    Wc, ic = _cuda(W), _cuda(init)
    kw = dict(policies=Wc, init_state=ic)
    inf, nan = float("inf"), float("nan")
    # never unsafe: the unscreened rollout of the same kernel
    plain = S.ops.rollout(real, H, want_final=True, want_trajectory=True, kernel=_k(S, kern), **kw)
    a = _screened(S, kern, real, sim, H, inf, inf, **kw)
    assert (a.frozen_at.cpu().numpy() == H).all() and (a.violations.cpu().numpy() == 0).all()
    assert _ret_err(a.returns.cpu().numpy(), plain.returns.cpu().numpy()) < 1e-12
    assert rel_err(a.final_state.cpu().numpy(), plain.final_state.cpu().numpy()) < 1e-12
    assert rel_err(a.trajectory.cpu().numpy(), plain.trajectory.cpu().numpy()) < 1e-12
    # unsafe from the start: nothing advances
    for thr in (nan, -inf):
        b = _screened(S, kern, real, sim, H, thr, -inf, **kw)
        assert (b.frozen_at.cpu().numpy() == 0).all() and (b.violations.cpu().numpy() == 0).all()
        assert (b.returns.cpu().numpy() == 0.0).all()
        _self_consistent(b, init, H, -inf)
    # real thresholds: +inf / NaN count nothing, -inf counts every step taken
    costs = [_oracle_costs(O, ro, so, W[e], init[e], H) for e in range(B)]
    sc, rc = np.array([c[0] for c in costs]), np.array([c[1] for c in costs])
    sim_thr, _ = _thresholds(sc, rc, zero=1, mid=1, mid_steps=1, never=1, violated=1)
    for rthr in (inf, nan, -inf):
        c = _screened(S, kern, real, sim, H, sim_thr, rthr, **kw)
        fz, viol = c.frozen_at.cpu().numpy(), c.violations.cpu().numpy()
        assert np.array_equal(viol, fz if rthr == -inf else np.zeros_like(fz))
        assert ((fz > 0) & (fz < H)).any() and (fz == H).any()
        _compare_with_oracle(O, ro, so, W, init, H, sim_thr, rthr, c)
    # reset state, zero policy: thd stays exactly 0, so a zero threshold is safe and the smallest negative one is not
    Z = np.zeros((B, n - 1, 2 * n + 2))
    z = S.ops.rollout(real, H, policies=_cuda(Z), want_trajectory=True, kernel=_k(S, kern))
    assert (z.trajectory[:, :, 3::2] == 0).all()
    start = S.ops.reset_state(n).cpu().numpy()
    for thr, frozen in ((0.0, H), (-0.0, H), (-5e-324, 0)):
        d = _screened(S, kern, real, sim, H, thr, 0.0, policies=_cuda(Z))
        assert (d.frozen_at.cpu().numpy() == frozen).all() and (d.violations.cpu().numpy() == 0).all()
        _self_consistent(d, np.broadcast_to(start, (B, len(start))), H, 0.0)
        _, _, _, v, f = O.rollout_safe_step(ro, so, Z[0], H, thr, 0.0)
        assert (f, v) == (frozen, 0)


@pytest.mark.parametrize("n", [3, 8])
def test_thread_kernel_screening_nan_isolation(S, O, n):
    """A NaN in one start state makes that environment unsafe at step 0 (the cost propagates NaN like np.max); the
    environments sharing its warp are bit-identical to the launch without it."""
    B, H = 37, 201
    (real, sim), (ro, so) = _models(S, n), _models(O, n)
    W, init = _population(n, B, seed=100 + n)
    costs = [_oracle_costs(O, ro, so, W[e], init[e], H) for e in range(B)]
    sim_thr, real_thr = _thresholds(np.array([c[0] for c in costs]), np.array([c[1] for c in costs]))
    init2 = init.copy()
    init2[3, 3] = np.nan
    a = _screened(S, "THREAD", real, sim, H, sim_thr, real_thr, policies=_cuda(W), init_state=_cuda(init))
    b = _screened(S, "THREAD", real, sim, H, sim_thr, real_thr, policies=_cuda(W), init_state=_cuda(init2))
    ha, hb = _host(a), _host(b)
    assert hb[3][3] == 0 and hb[4][3] == 0 and hb[0][3] == 0.0
    _self_consistent(b, init2, H, real_thr)
    keep = np.arange(B) != 3
    for x, y in zip(ha, hb):
        sel = (slice(None), keep) if x.ndim == 3 else keep
        assert np.array_equal(_bits(x[sel]) if x.dtype == np.float64 else x[sel],
                              _bits(y[sel]) if y.dtype == np.float64 else y[sel])


@pytest.mark.parametrize("kern", KERNELS)
@pytest.mark.parametrize("n", [3, 8])
def test_screening_dir_mask(S, n, kern):
    """Directions skipped by dir_mask: returns NaN, final state = start state, frozen_at = H, violations = 0 on
    every kernel, whatever the output buffers held before.  The surviving directions are bit-identical to the
    launch without a mask.  (Trajectory rows of skipped directions are not written.)"""
    D, R, H = 6, 2, 130
    B, ws, no = 2 * D * R, (n - 1) * (2 * n + 2), 2 * n + 2
    real, sim = _models(S, n)
    rng = np.random.default_rng(40 + n)
    init = rand_states(rng, n, R, scale=0.5)
    mask = torch.tensor([1, 0, 1, 1, 0, 1], dtype=torch.int32, device="cuda")
    kw = dict(B=B, base_policy=_cuda(rng.uniform(-1, 1, ws) * 0.05), nu=0.8, seed=3, iteration=1,
              rollouts_per_policy=R, init_state=_cuda(init))
    probe = S.ops.rollout(real, H, want_trajectory=True, kernel=S.KERNEL_THREAD, **kw)
    peak = probe.trajectory[:, :, 3::2].abs().amax(dim=(0, 2)).cpu().numpy()
    thr = float(np.median(peak))
    full = _screened(S, kern, real, sim, H, thr, 0.8 * thr, **kw)

    def sentinels():
        f64 = dict(dtype=torch.float64, device="cuda")
        return {"returns": torch.full((B,), 12345.0, **f64), "final_state": torch.full((B, no), 777.0, **f64),
                "frozen_at": torch.full((B,), -7, dtype=torch.int32, device="cuda"),
                "violations": torch.full((B,), -9, dtype=torch.int32, device="cuda")}

    out = sentinels()
    m = _screened(S, kern, real, sim, H, thr, 0.8 * thr, dir_mask=mask, out=out, **kw)
    live = np.repeat(mask.cpu().numpy().astype(bool), 2 * R)
    fz, viol = m.frozen_at.cpu().numpy(), m.violations.cpu().numpy()
    assert (fz[~live] == H).all() and (viol[~live] == 0).all()
    assert np.isnan(m.returns.cpu().numpy()[~live]).all()
    starts = init[np.arange(B) % R]
    assert np.array_equal(_bits(m.final_state.cpu().numpy()[~live]), _bits(starts[~live]))
    lv = torch.as_tensor(live, device="cuda")
    for name in ("returns", "frozen_at", "violations", "final_state"):
        assert torch.equal(getattr(m, name)[lv], getattr(full, name)[lv]), name
    assert torch.equal(m.trajectory[:, lv], full.trajectory[:, lv])
    fzl = fz[live]
    assert ((fzl > 0) & (fzl < H)).any() and (fzl == H).any()


@pytest.mark.parametrize("n,kern", [(3, "LANES2"), (8, "THREAD")])
def test_engine_step_screening_matches_oracle_loop(S, O, n, kern):
    """ArsEngine(step_screen=...) for three ARS iterations (true top-b): every +- direction against
    orc_rollout_safe_step on W +- nu delta_k, the policy against the oracle's update."""
    N, b, H, nu, alpha, seed = 8, 4, 150, 0.3, 0.02, 21
    (real, sim), (ro, so) = _models(S, n), _models(O, n)
    ws = (n - 1) * (2 * n + 2)
    assert _kernel_choice(S, real, sim, 2 * N, S.KERNEL_AUTO, S.ops.POLICY_PHILOX) == _k(S, kern)
    W = np.random.default_rng(n).uniform(-1, 1, ws) * 0.3
    start = S.ops.reset_state(n).cpu().numpy()

    def directions(W, it):
        deltas = np.stack([O.philox_delta(seed, it, k, ws) for k in range(N)])
        return deltas, [W + s * nu * deltas[k] for k in range(N) for s in (+1, -1)]

    # thresholds from the first iteration's directions; margins asserted for every rollout of the loop
    _, pols = directions(W, 0)
    costs = [_oracle_costs(O, ro, so, p, start, H) for p in pols]
    sim_thr, real_thr = _thresholds(np.array([c[0] for c in costs]), np.array([c[1] for c in costs]),
                                    zero=0, mid=2, mid_steps=2, never=1, violated=1)
    eng = S.ArsEngine(real, N=N, b=b, alpha=alpha, nu=nu, H=H, semantics=S.ARS_TOPB, seed=seed, distributed=False,
                      initial_policy=W, step_screen=dict(sim_params=sim, sim_thresh=sim_thr, real_thresh=real_thr))
    frozen = []
    for it in range(3):
        got = eng.run_iteration().cpu().numpy()
        fz, viol = eng.last.frozen_at.cpu().numpy(), eng.last.violations.cpu().numpy()
        deltas, pols = directions(W, it)
        rets = []
        for e, p in enumerate(pols):
            sc, rc = _oracle_costs(O, ro, so, p, start, H)
            assert _margins_ok(sc[None], rc[None], sim_thr, real_thr), (it, e)
            r, _, _, v, z = O.rollout_safe_step(ro, so, p, H, sim_thr, real_thr)
            assert (fz[e], viol[e]) == (z, v), (it, e)
            rets.append(r)
        assert _ret_err(got, rets) < RET_TOL
        W, _ = O.update_policy(W, deltas, np.array(rets), b=b, alpha=alpha, semantics=1)
        assert rel_err(eng.W.cpu().numpy(), W) < 1e-6
        frozen.append(fz)
    frozen = np.concatenate(frozen)
    assert (frozen < H).any() and (frozen == H).any()
