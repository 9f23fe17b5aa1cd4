"""The tracked sine/cosine of every rollout kernel, tier by tier, against the CPU oracle.

No rollout kernel evaluates sincos on every step: each carries (sin th_i, cos th_i) in registers and rotates it by the
increment d = h thd_i, with a Taylor polynomial for |d| <= 1/32 (base), extra terms for |d| <= 1/8 (tail) and an exact
sincos above that and on every 64th step (csrc/dynamics.cuh).  The thread kernel decides once per environment from
max_i |d_i| (gym_step_tracked), LANES once per segment lane, inline under a warp vote (lane_rollout.cuh), and
LANES2 / LANES3 call the out-of-line tracked_sincos_slow on every lane and keep its result on the slow lanes only
(lane2_rollout.cuh).

A wrong tier is invisible to whole-trajectory comparisons: a missing tail term changes the next state by 5e-12 to
5e-10, while fast rollouts amplify rounding by up to 1e13 over a few hundred steps.  So the main check is per step:
every state the kernel visited is stepped once by the oracle (exact sincos, dense solve) and compared with the
kernel's next state.  A correct kernel differs there only by the drift of its tracked angles since the last exact
re-evaluation and by the O(n) solve, both around 1e-14; chaos does not enter because every step starts from the
kernel's own state.  Whole trajectories are compared only up to the step where an oracle twin started 1e-14 away
still agrees with the oracle to 1e-10."""
import ctypes
import functools
import struct

import numpy as np
import pytest
import torch

from conftest import rel_err
import test_step_screening as scr

pytestmark = pytest.mark.gpu
KERNELS = ["THREAD", "LANES", "LANES2", "LANES3"]
NS = [2, 3, 4, 5, 6, 7, 8, 9, 10]
STEP_TOL = 1e-12      # per-step check against the oracle (norm-relative, floor 1)
EXACT_TOL = 1e-12     # returns / moments against the kernel's own trajectory
RET_TOL, STATE_TOL = 1e-6, 1e-8
TWIN_REL, TWIN_TOL = 1e-14, 1e-10
K_TIER = 50           # segment-steps required in every tier band
SHORT, LONG = 1.0 / 32, 1.0 / 8
BLOWN = 1e4           # the per-step check stops at the first state with |x| >= BLOWN (or non-finite)


def _cuda(a):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _k(S, name):
    return getattr(S, "KERNEL_" + name)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _params(mod, n, h):
    return mod.make_params(n=n, l_i=.9, m_i=1.1, k=9.5, h=h, direction=(.6, .8))


def _launch(S, kern, p, H, mode, B, **kw):
    """Rollout with final state and trajectory on a forced kernel; asserts that kernel ran, and that the same launch
    without a trajectory gives bit-identical returns and final states."""
    cfg = S._lib.SwmRollout()
    cfg.variant, cfg.policy_mode, cfg.H, cfg.B, cfg.rollouts_per_policy = S.GYM, mode, H, B, 1
    cfg.kernel = _k(S, kern)
    assert S._lib.lib().swm_rollout_kernel_choice(ctypes.byref(p), ctypes.byref(cfg)) == _k(S, kern)
    res = S.ops.rollout(p, H, B=B, want_final=True, want_trajectory=True, kernel=_k(S, kern), **kw)
    bare = S.ops.rollout(p, H, B=B, want_final=True, kernel=_k(S, kern), **kw)
    assert np.array_equal(_bits(bare.returns.cpu().numpy()), _bits(res.returns.cpu().numpy()))
    assert np.array_equal(_bits(bare.final_state.cpu().numpy()), _bits(res.final_state.cpu().numpy()))
    return res


def _valid(x):
    """Number of leading states that are finite and below BLOWN in magnitude."""
    ok = np.isfinite(x).all(axis=1) & (np.abs(x).max(axis=1) < BLOWN)
    return len(x) if ok.all() else int(np.argmin(ok))


def _visited(starts, traj, e, stop=None):
    """States x_0 = start, x_{t+1} = trajectory[t] of environment e (up to `stop` steps), cut at the first bad one."""
    x = np.vstack([starts[e][None], traj[:stop, e]])
    return x[:_valid(x)]


def _per_step(starts, traj, step, stops=None):
    """Oracle step from every visited state against the kernel's next state.  step(e, x) -> oracle next state.
    -> (largest norm-relative error, visited states per environment)."""
    worst, seen = 0.0, []
    for e in range(len(starts)):
        x = _visited(starts, traj, e, None if stops is None else stops[e])
        seen.append(x)
        if len(x) < 2:
            continue
        want = np.array([step(e, x[t]) for t in range(len(x) - 1)])
        err = np.max(np.abs(x[1:] - want), axis=1) / np.maximum(1.0, np.max(np.abs(want), axis=1))
        assert err.max() <= STEP_TOL, (e, int(np.argmax(err)), float(err.max()))
        worst = max(worst, float(err.max()))
    return worst, seen


def _tier_counts(seen, h, kern):
    """Tier decisions the per-step check verified -- step t sets the angles that step t+1 uses -- per band (base,
    tail, exact), leaving out the exact re-evaluation steps and increments within 1e-6 (relative) of a band edge; and
    the environment-steps with segments in two different bands.  The lane kernels decide per segment, so the counts
    are segment-steps; the thread kernel decides once per environment from max_i |d_i|, so they are environment-steps
    binned by that maximum."""
    counts, mixed = np.zeros(3, dtype=np.int64), 0
    for x in seen:
        t = np.arange(max(0, len(x) - 2))
        t = t[(t & 63) != 63]
        d = np.abs(h * x[t][:, 3::2])
        far = (np.abs(d - SHORT) > 1e-6 * SHORT) & (np.abs(d - LONG) > 1e-6 * LONG)
        band = np.where(d < SHORT, 0, np.where(d < LONG, 1, 2))
        lo = np.where(far, band, 3).min(axis=1)
        hi = np.where(far, band, -1).max(axis=1)
        mixed += int(np.sum(hi > lo))
        if kern == "THREAD":
            dm = d.max(axis=1)
            far = (np.abs(dm - SHORT) > 1e-6 * SHORT) & (np.abs(dm - LONG) > 1e-6 * LONG)
            band = np.where(dm < SHORT, 0, np.where(dm < LONG, 1, 2))
        for b in range(3):
            counts[b] += np.sum(far & (band == b))
    return counts, mixed


def _assert_coverage(kern, counts, mixed, bands=(0, 1, 2)):
    assert (counts[list(bands)] >= K_TIER).all(), counts
    if kern != "THREAD":  # per-lane decisions: one environment's segments in different tiers on the same step
        assert mixed >= K_TIER, mixed


def _returns_consistent(res, traj, p):
    """returns = sum_t Gdot_t . direction over the kernel's own trajectory, to EXACT_TOL of sum_t |Gdot_t . dir|."""
    got = res.returns.cpu().numpy()
    (dx, dy), gx, gy = p.direction, traj[:, :, 0], traj[:, :, 1]
    want = dx * gx.sum(axis=0) + dy * gy.sum(axis=0)
    scale = abs(dx) * np.abs(gx).sum(axis=0) + abs(dy) * np.abs(gy).sum(axis=0)
    fin = np.isfinite(want)
    assert np.array_equal(fin, np.isfinite(got))
    assert (np.abs(got - want)[fin] <= EXACT_TOL * np.maximum(1.0, scale[fin])).all()


def _twin(x, rng):
    return x + TWIN_REL * max(1.0, np.abs(x).max()) * rng.choice([-1.0, 1.0], x.shape)


def _horizon(want, twin):
    """Leading steps over which the twin stays within TWIN_TOL of the oracle's trajectory."""
    err = np.max(np.abs(twin - want), axis=1) / np.maximum(1.0, np.max(np.abs(want), axis=1))
    ok = err <= TWIN_TOL
    return len(ok) if ok.all() else int(np.argmin(ok))


def _compare_within_horizon(res, traj, p, oracle, spun):
    """Whole trajectories against the oracle up to each environment's twin horizon (returns: partial sums where the
    horizon stops short of H); half of the spun environments must carry the comparison past the step-63
    re-evaluation.  -> (largest return error, largest state error)."""
    got_r = res.returns.cpu().numpy()
    er = es = 0.0
    for e, (want_r, want_t, hz) in enumerate(oracle):
        H = len(want_t)
        es = max(es, rel_err(traj[:hz, e], want_t[:hz]) if hz else 0.0)
        if hz == H:
            er = max(er, scr._ret_err(got_r[e], want_r))
        elif hz:
            part = lambda t: p.direction[0] * t[:hz, 0].sum() + p.direction[1] * t[:hz, 1].sum()
            er = max(er, scr._ret_err(part(traj[:, e]), part(want_t)))
    hz = np.array([o[2] for o in oracle])
    assert np.sum(hz[spun] >= 64) * 2 >= len(spun), hz[spun]
    assert er < RET_TOL and es < STATE_TOL, (er, es)
    return er, es


def _report(tag, worst, counts, mixed, extra=""):
    print("\n[trig tiers] %s: max per-step err %.2e, verified tier decisions base/tail/exact %d/%d/%d, mixed %d%s"
          % (tag, worst, counts[0], counts[1], counts[2], mixed, extra))


# ---- populations ------------------------------------------------------------------------------------------------
def _calm(rng, n, B):
    init = np.zeros((B, 2 * n + 2))
    init[:, :2] = rng.normal(size=(B, 2)) * 0.3
    init[:, 2::2] = rng.uniform(-3, 3, (B, n))
    init[:, 3::2] = rng.normal(size=(B, n)) * 0.5
    return init


def _random_fast(n):
    """(a) h = 1e-2, thd ~ N(0, 25): every tier on most steps (the oracle puts 5-25 / 20-50 / 30-70 % of segment-steps
    in base / tail / exact); a few n >= 7 environments blow up, where the per-step check stops."""
    rng = np.random.default_rng(n)
    B, H = 32, 200
    init = _calm(rng, n, B)
    init[:, :2] = rng.normal(size=(B, 2))
    init[:, 2::2] = rng.uniform(-4, 4, (B, n))
    init[:, 3::2] = rng.normal(size=(B, n)) * 5.0
    return 1e-2, H, init, rng.uniform(-5, 5, (B, n - 1)), np.arange(0)


def _spun(n, B=32, top=300.0, seed=0):
    """(b) h = 1e-3, calm and spun environments alternating (so both share every warp: 8 / 4 / 2 environments per warp
    for L = 4 / 8 / 16 lanes): a spun environment has one segment at +-20 ... `top` rad/s, the others calm."""
    rng = np.random.default_rng(1000 * seed + n)
    init = _calm(rng, n, B)
    spun = np.arange(1, B, 2)
    speed = 10.0 ** np.linspace(np.log10(20.0), np.log10(top), len(spun))[rng.permutation(len(spun))]
    for j, e in enumerate(spun):
        init[e, 3 + 2 * rng.integers(n)] = speed[j] * rng.choice([-1.0, 1.0])
    return init, rng.uniform(-5, 5, (B, n - 1)), spun


def _from_words(hi, lo):
    return struct.unpack("<d", struct.pack("<II", lo, hi))[0]


def _edge_increments():
    """Increments at the two band edges 2^-5 and 2^-3: one high word below, the edge itself, the edge's high word with
    the largest low word (still not above it: the kernels compare high words), one high word above."""
    out = []
    for edge in (SHORT, LONG):
        hi = struct.unpack("<II", struct.pack("<d", edge))[1]
        out += [_from_words(hi - 1, 0), edge, _from_words(hi, 0xFFFFFFFF), _from_words(hi + 1, 0)]
    return np.array(out)


def _edges(n):
    """(c) h = 2^-10, so that d = h thd is exact: step-0 speeds put one segment of every other environment on an edge
    increment (both signs).  The tiers on the two sides of an edge differ by at most ~6e-15 (at 1/32) and ~3e-18 (at
    1/8) in angle, far below the per-step bar: this catches gross errors at the edges (the base polynomial run near
    1/8, a comparison that sends an edge value to the wrong branch family), not which side of an edge was taken."""
    h = 2.0 ** -10
    rng = np.random.default_rng(300 + n)
    B, H = 32, 130
    init = _calm(rng, n, B)
    dd = np.concatenate([_edge_increments(), -_edge_increments()])
    spun = np.arange(1, B, 2)
    for j, e in enumerate(spun):
        init[e, 3 + 2 * (j % n)] = dd[j] / h
    assert np.array_equal(h * init[spun, 3 + 2 * (np.arange(len(spun)) % n)], dd)  # exact increments
    return h, H, init, rng.uniform(-5, 5, (B, n - 1)), spun


def _population(name, n):
    if name == "a":
        return _random_fast(n)
    if name == "b":
        init, ac, spun = _spun(n)
        return 1e-3, 300, init, ac, spun
    return _edges(n)


@functools.lru_cache(maxsize=None)
def _oracle_fixed(O, n, name):
    """Oracle rollouts and twin horizons of a fixed-action population (independent of the kernel)."""
    h, H, init, ac, _ = _population(name, n)
    po = _params(O, n, h)
    rng = np.random.default_rng(7 + n)
    out = []
    for e in range(len(init)):
        r, _, t = O.rollout(po, O.GYM, H, action=ac[e], init_state=init[e], want_traj=True)
        _, _, tw = O.rollout(po, O.GYM, H, action=ac[e], init_state=_twin(init[e], rng), want_traj=True)
        out.append((r, t, _horizon(t, tw)))
    return out


# -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pop", ["a", "b", "c"])
@pytest.mark.parametrize("kern", KERNELS)
@pytest.mark.parametrize("n", NS)
def test_tracked_trig_tiers_match_oracle(S, O, n, kern, pop):
    """Fixed actions.  (a) h = 1e-2 random fast starts, (b) h = 1e-3 calm and spun environments sharing warps, (c)
    exact increments on and next to the band edges (see _edges for what that can show).  Every visited state stepped by the oracle; every tier band reached (a, b);
    returns equal to the sum over the kernel's own trajectory; (b) whole trajectories within the twin horizon, and a
    NaN environment that leaves its warp neighbours bit-identical."""
    h, H, init, ac, spun = _population(pop, n)
    ps, po = _params(S, n, h), _params(O, n, h)
    B = len(init)
    kw = dict(actions=_cuda(ac), init_state=_cuda(init))
    res = _launch(S, kern, ps, H, S.ops.POLICY_FIXED_ACTION, B, **kw)
    traj = res.trajectory.cpu().numpy()
    worst, seen = _per_step(init, traj, lambda e, x: O.step(po, O.GYM, x, ac[e])[0])
    counts, mixed = _tier_counts(seen, h, kern)
    _returns_consistent(res, traj, ps)
    extra = ""
    if pop == "a":  # nearly every environment has a fast segment: the thread kernel's base tier is covered by (b)
        _assert_coverage(kern, counts, mixed, (1, 2) if kern == "THREAD" else (0, 1, 2))
    elif pop == "b":
        _assert_coverage(kern, counts, mixed)
    else:  # every edge environment is checked past its first step, where the edge increment set the angles
        assert all(len(seen[e]) >= 3 for e in spun)
    if pop == "b":
        extra = ", whole trajectory: return %.2e, state %.2e" % _compare_within_horizon(
            res, traj, ps, _oracle_fixed(O, n, pop), spun)
        bad = init.copy()
        bad[spun[2], 3] = np.nan
        nan = S.ops.rollout(ps, H, want_final=True, kernel=_k(S, kern), actions=kw["actions"], init_state=_cuda(bad))
        r2, f2 = nan.returns.cpu().numpy(), nan.final_state.cpu().numpy()
        keep = np.arange(B) != spun[2]
        assert np.isnan(r2[spun[2]])
        assert np.array_equal(_bits(r2[keep]), _bits(res.returns.cpu().numpy()[keep]))
        assert np.array_equal(_bits(f2[keep]), _bits(res.final_state.cpu().numpy()[keep]))
    _report("%s n=%d (%s)" % (kern, n, pop), worst, counts, mixed, extra)


def _v2_setup(n):
    """(d) V2 Philox policies W +- nu delta_k with a normalising mean / inv_sigma and moments, on population (b) with
    spins up to 220 rad/s over 200 steps (every environment stays finite, so the moments are)."""
    init, _, spun = _spun(n, top=220.0, seed=2)
    B, H, no, ws = len(init), 200, 2 * n + 2, (n - 1) * (2 * n + 2)
    rng = np.random.default_rng(50 + n)
    Wb, nu, seed, it, dir0 = rng.uniform(-1, 1, ws) * 0.05, 0.03, 3, 1, 2
    mean, inv = rng.normal(size=no) * 0.1, rng.uniform(0.5, 2.0, no)
    return dict(init=init, spun=spun, B=B, H=H, Wb=Wb, nu=nu, seed=seed, it=it, dir0=dir0, mean=mean, inv=inv)


def _v2_policies(O, c, n):
    """Environment e runs direction e >> 1 with sign + (even e) or - (odd e)."""
    ws = (n - 1) * (2 * n + 2)
    return np.array([c["Wb"] + (-c["nu"] if e & 1 else c["nu"]) * O.philox_delta(c["seed"], c["it"], c["dir0"] + (e >> 1), ws)
                     for e in range(c["B"])])


@functools.lru_cache(maxsize=None)
def _oracle_v2(O, n):
    c = _v2_setup(n)
    po, pols = _params(O, n, 1e-3), _v2_policies(O, c, n)
    rng = np.random.default_rng(70 + n)
    out = []
    for e in range(c["B"]):
        kw = dict(policy=pols[e], mean=c["mean"], inv_sigma=c["inv"], want_traj=True)
        r, _, t = O.rollout(po, O.GYM, c["H"], init_state=c["init"][e], **kw)
        _, _, tw = O.rollout(po, O.GYM, c["H"], init_state=_twin(c["init"][e], rng), **kw)
        out.append((r, t, _horizon(t, tw)))
    return out


@pytest.mark.parametrize("kern", KERNELS)
@pytest.mark.parametrize("n", NS)
def test_v2_policies_in_slow_tiers_match_oracle(S, O, n, kern):
    """(d): the NORM and STATS paths under the slow tiers.  Per-step check with the oracle's one-step V2 rollout, tier
    coverage, returns and moments (stats_finalize) equal to those of the kernel's own trajectory, whole trajectories
    within the twin horizon."""
    c = _v2_setup(n)
    ps, po = _params(S, n, 1e-3), _params(O, n, 1e-3)
    B, H, init = c["B"], c["H"], c["init"]
    pivot = S.ops.reset_state(n)
    res = _launch(S, kern, ps, H, S.ops.POLICY_PHILOX, B, base_policy=_cuda(c["Wb"]), nu=c["nu"], seed=c["seed"],
                  iteration=c["it"], dir0=c["dir0"], mean=_cuda(c["mean"]), inv_sigma=_cuda(c["inv"]),
                  stats_pivot=pivot, init_state=_cuda(init))
    traj = res.trajectory.cpu().numpy()
    pols = _v2_policies(O, c, n)
    step = lambda e, x: O.rollout(po, O.GYM, 1, policy=pols[e], mean=c["mean"], inv_sigma=c["inv"], init_state=x)[1]
    worst, seen = _per_step(init, traj, step)
    assert all(len(x) == H + 1 for x in seen)
    counts, mixed = _tier_counts(seen, 1e-3, kern)
    _assert_coverage(kern, counts, mixed)
    _returns_consistent(res, traj, ps)
    # moments of the kernel's own visited states: mean to EXACT_TOL of mean |x - pivot|, M2 to EXACT_TOL of
    # sum (x - pivot)^2 (the sums the kernel accumulates)
    rec = S.ops.stats_finalize(res.stats_partial, res.samples, pivot).cpu().numpy()
    no = 2 * n + 2
    x = traj.reshape(-1, no)
    dev = x - pivot.cpu().numpy()
    assert rec[0] == B * H
    assert (np.abs(rec[1:1 + no] - x.mean(axis=0)) <= EXACT_TOL * np.maximum(1.0, np.abs(dev).mean(axis=0))).all()
    m2 = ((x - x.mean(axis=0)) ** 2).sum(axis=0)
    assert (np.abs(rec[1 + no:] - m2) <= EXACT_TOL * np.maximum(1.0, (dev ** 2).sum(axis=0))).all()
    er, es = _compare_within_horizon(res, traj, ps, _oracle_v2(O, n), c["spun"])
    _report("%s n=%d (d, V2)" % (kern, n), worst, counts, mixed, ", whole trajectory: return %.2e, state %.2e" % (er, es))


@pytest.mark.parametrize("kern", KERNELS)
@pytest.mark.parametrize("n", [3, 5, 9])
def test_neighbour_isolation_is_bitwise(S, n, kern):
    """An environment whose increments sit near the top of the base band, |h thd| in [1/64, 1/32) -- where the tail
    terms change bits -- has the same trajectory bit for bit among calm warp neighbours and among neighbours in the
    tail and exact tiers: the slow path of one lane never leaks into another.  n = 3, 5, 9: 4, 8, 16 lanes."""
    h, H, B, subject = 1e-3, 200, 32, 5
    p = _params(S, n, h)
    rng = np.random.default_rng(900 + n)
    calm = _calm(rng, n, B)
    fast = _calm(rng, n, B)
    fast[:, 3::2] = rng.uniform(40.0, 300.0, (B, n)) * rng.choice([-1.0, 1.0], (B, n))
    x0 = calm[subject].copy()
    x0[3::2] = rng.uniform(1.0 / 64, 1.0 / 32, n) / h * rng.choice([-1.0, 1.0], n)
    ac = rng.uniform(-5, 5, (B, n - 1))
    runs = []
    for nb in (calm, fast):
        init = nb.copy()
        init[subject] = x0
        res = _launch(S, kern, p, H, S.ops.POLICY_FIXED_ACTION, B, actions=_cuda(ac), init_state=_cuda(init))
        runs.append((res.trajectory.cpu().numpy()[:, subject], res.returns.cpu().numpy()[subject],
                     res.final_state.cpu().numpy()[subject]))
    near_top = np.abs(h * np.vstack([x0[None], runs[0][0]])[:, 3::2])
    assert np.sum((near_top >= 1.0 / 64) & (near_top < SHORT)) >= K_TIER
    for a, b in zip(*runs):
        assert np.array_equal(_bits(a), _bits(b))


# ---- per-step screening in the slow tiers ------------------------------------------------------------------------
def _screen_population(n):
    """Explicit policies and starts of test_step_screening with two thirds of the environments spun (one segment at
    +-20 ... 250 rad/s): the unscreened real rollouts reach the tail and exact tiers."""
    B = 37
    W, init = scr._population(n, B, seed=700 + n)
    rng = np.random.default_rng(701 + n)
    spun = rng.permutation(B)[:2 * B // 3]
    speed = 10.0 ** np.linspace(np.log10(20.0), np.log10(250.0), len(spun))
    for j, e in enumerate(spun):
        init[e, 3 + 2 * rng.integers(n)] = speed[j] * rng.choice([-1.0, 1.0])
    return W, init


@functools.lru_cache(maxsize=None)
def _screen_thresholds(O, n):
    ro, so = scr._models(O, n)
    W, init = _screen_population(n)
    costs = [scr._oracle_costs(O, ro, so, W[e], init[e], 201) for e in range(len(W))]
    # the highest simulator threshold that gives the spread: the environments that keep going are the fast ones
    return scr._thresholds(np.array([c[0] for c in costs]), np.array([c[1] for c in costs]),
                           quantiles=np.linspace(0.995, 0.05, 200))


@pytest.mark.parametrize("kern", scr.KERNELS)
@pytest.mark.parametrize("n", NS)
def test_step_screening_in_slow_tiers_matches_oracle(S, O, n, kern):
    """Per-step simulator screening (h_real = 1e-3, h_sim = 1.2e-3) on environments whose real steps run in the tail
    and exact tiers: freeze steps and violation counts exact, returns and states at the parity bars, and before each
    freeze the per-step check of every real step."""
    H = 201
    (real, sim), (ro, so) = scr._models(S, n), scr._models(O, n)
    W, init = _screen_population(n)
    sim_thr, real_thr = _screen_thresholds(O, n)
    res = scr._screened(S, kern, real, sim, H, sim_thr, real_thr, policies=_cuda(W), init_state=_cuda(init))
    errs = scr._compare_with_oracle(O, ro, so, W, init, H, sim_thr, real_thr, res)
    scr._self_consistent(res, init, H, real_thr)
    fz = res.frozen_at.cpu().numpy()
    assert scr._spread(fz, res.violations.cpu().numpy(), H)
    traj = res.trajectory.cpu().numpy()
    step = lambda e, x: O.rollout(ro, O.GYM, 1, policy=W[e], init_state=x)[1]
    worst, seen = _per_step(init, traj, step, stops=fz)
    counts, mixed = _tier_counts(seen, real.h, kern)
    assert (counts[1:] >= K_TIER).all(), counts
    _report("%s n=%d (screened)" % (kern, n), worst, counts, mixed,
            ", oracle return %.2e, final state %.2e, trajectory %.2e" % errs)
