"""Per-step simulator screening with a user-defined max-of-affine state cost (swm_rollout_costed, MaxAffineCost)
against a CPU reference: orc_rollout_safe_step's loop restated here with the cost as a parameter, every step taken
by the oracle's own one-step rollout.

cost(obs) = max_j (A_j . obs + b_j).  Before every real step one simulator step is taken from the same state and
the real step is taken only if the cost of the simulator's whole next observation is <= sim_thresh; otherwise the
environment freezes for good.  Real steps whose post-step cost is > real_thresh are violations.  As in
test_step_screening.py, every threshold sits between neighbouring costs of the oracle's own rollouts and every
deciding cost is asserted to be at least MARGIN * max(1, |thr|) away from it, so the exact checks of freeze steps
and violation counts cannot flip on rounding."""
import contextlib
import ctypes
import functools
import io

import numpy as np
import pytest
import torch

from conftest import rel_err
from test_step_screening import (MARGIN, RET_TOL, STATE_TOL, _bits, _cuda, _midpoint, _models, _population,
                                 _ret_err, _spread, _starts)

gpu = pytest.mark.gpu
COSTS = ["bend", "gdot", "dense1", "dense32"]


# ---- costs -------------------------------------------------------------------------------------------------------
def builtin_rows(n):
    """max_i |thd_i| as 2n forms +-e_{3+2i}."""
    no = 2 * n + 2
    A = np.zeros((2 * n, no))
    for i in range(n):
        A[2 * i, 3 + 2 * i], A[2 * i + 1, 3 + 2 * i] = 1.0, -1.0
    return A, np.zeros(2 * n)


def cost_rows(kind, n):
    no = 2 * n + 2
    rng = np.random.default_rng(1000 + n)
    if kind == "builtin":
        return builtin_rows(n)
    if kind == "bend":  # |th_i - th_{i+1}|
        A = np.zeros((2 * (n - 1), no))
        for i in range(n - 1):
            A[2 * i, 2 + 2 * i], A[2 * i, 4 + 2 * i] = 1.0, -1.0
            A[2 * i + 1] = -A[2 * i]
        return A, np.zeros(2 * (n - 1))
    if kind == "gdot":  # signed bounds on Gdot with offsets, mixed with the angular velocities
        A = np.zeros((4, no))
        A[0, 0], A[1, 0], A[2, 1], A[3, 1] = 1.0, -1.0, 1.0, -1.0
        A[:, 3::2] = 0.5 * rng.uniform(-1, 1, (4, n))
        return A, np.array([-0.1, 0.2, 0.05, -0.15])
    J = {"dense1": 1, "dense32": 32}[kind]
    return rng.uniform(-1, 1, (J, no)), rng.uniform(-0.5, 0.5, J)


def _cost_of(A, b, X):
    """max_j (A_j . x + b_j) for every row x of X."""
    return np.max(np.asarray(X) @ A.T + b, axis=-1)


# ---- oracle-side helpers ---------------------------------------------------------------------------------------------
def _oracle_costs(O, real, sim, W, start, H, A, b):
    """Simulator cost before every step and real cost after it along the UNSCREENED oracle rollout."""
    n = real.n
    W = np.asarray(W).reshape(n - 1, 2 * n + 2)
    _, _, traj = O.rollout(real, O.GYM, H, policy=W, init_state=start, want_traj=True)
    pre = np.vstack([start[None], traj[:-1]])
    nxt, _ = O.step_batch(sim, O.GYM, pre, pre @ W.T)
    return _cost_of(A, b, nxt), _cost_of(A, b, traj)


def _freeze_steps(sim_cost, thr):
    unsafe = ~(sim_cost <= thr)
    return np.where(unsafe.any(axis=1), unsafe.argmax(axis=1), sim_cost.shape[1])


def _margins_ok(sim_cost, real_cost, sim_thr, real_thr):
    fz = _freeze_steps(sim_cost, sim_thr)
    H = sim_cost.shape[1]
    for e in range(len(fz)):
        f = int(fz[e])
        if np.isfinite(sim_thr) and np.abs(sim_cost[e, :min(f + 1, H)] - sim_thr).min(initial=np.inf) < \
                MARGIN * max(1.0, abs(sim_thr)):
            return False
        if np.isfinite(real_thr) and f and np.abs(real_cost[e, :f] - real_thr).min() < MARGIN * max(1.0, abs(real_thr)):
            return False
    return True


def _thresholds(sim_cost, real_cost, quantiles=np.linspace(0.05, 0.995, 200), **need):
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


NEED = dict(zero=2, mid=4, mid_steps=3, never=2, violated=2)


@functools.lru_cache(maxsize=None)
def _case(O, n, kind, B=37, H=201):
    """Explicit policies, starts, the cost and thresholds with the required spread (oracle only): the first of a
    few seeded populations that gives it."""
    ro, so = _models(O, n)
    A, b = cost_rows(kind, n)
    for seed in range(8):
        W, init = _population(n, B, seed=100 + n + 1000 * seed)
        init[:, :2] *= 0.1  # Gdot starts small and builds up under the policy
        costs = [_oracle_costs(O, ro, so, W[e], init[e], H, A, b) for e in range(B)]
        sc, rc = np.array([c[0] for c in costs]), np.array([c[1] for c in costs])
        try:
            sim_thr, real_thr = _thresholds(sc, rc, **NEED)
        except AssertionError:
            continue
        return W, init, A, b, sim_thr, real_thr
    raise AssertionError("no population gives the required spread for n=%d, %s" % (n, kind))


def _affine_cost(A, b, x):
    """max_j (sum_k A[j,k] x_k + b_j), the products summed in index order, then b_j; NaN if any form is NaN."""
    v = np.zeros(A.shape[0])
    for k in range(A.shape[1]):
        v = v + A[:, k] * x[k]
    return float(np.max(v + b))


def rollout_safe_step_affine(O, real_p, sim_p, policy, H, A, b, sim_thresh, real_thresh, init_state=None,
                             want_traj=False):
    """Safe_ARS.rollout (safe_ars/ars.py:124-153) with the cost _affine_cost: orc_rollout_safe_step's loop, each
    simulator and real step an oracle rollout of one step from the current state (its select_action, then
    orc_gym_step).  -> (return, final state, trajectory [H, 2n+2] or None, violations, freeze step)."""
    n = real_p.n
    W = np.ascontiguousarray(policy, dtype=np.float64).reshape(n - 1, 2 * n + 2)
    if init_state is None:
        st = O.rollout(real_p, O.GYM, 0, policy=W)[1]  # reset()
    else:
        st = np.array(init_state, dtype=np.float64)
    traj = np.zeros((H, 2 * n + 2)) if want_traj else None
    total, viol, frozen = 0.0, 0, H
    for t in range(H):
        sim_next = O.rollout(sim_p, O.GYM, 1, policy=W, init_state=st)[1]
        if _affine_cost(A, b, sim_next) <= sim_thresh:
            r, st, _ = O.rollout(real_p, O.GYM, 1, policy=W, init_state=st)
            total += r
            if _affine_cost(A, b, st) > real_thresh:
                viol += 1
        elif frozen == H:
            frozen = t
        if want_traj:
            traj[t] = st
    return total, st, traj, viol, frozen


def _oracle_loop(O, ro, so, pols, starts, H, A, b, sim_thr, real_thr):
    return [rollout_safe_step_affine(O, ro, so, pols[e], H, A, b, sim_thr, real_thr, init_state=starts[e],
                                     want_traj=True) for e in range(len(pols))]


# ---- CPU tests -------------------------------------------------------------------------------------------------------
def test_max_affine_cost_validation(S):
    A, b = builtin_rows(3)
    c = S.MaxAffineCost(A, b)
    assert c.n == 3 and c.forms.shape == (6, 9) and c.forms.flags.c_contiguous
    x = np.arange(8.0) - 3.5
    assert c(x) == S.builtin_cost(x) and c(list(x)) == c(x)
    assert S.MaxAffineCost(A).b.tolist() == [0.0] * 6
    assert np.isnan(c(np.full(8, np.nan)))
    for bad in (np.zeros(8), np.zeros((2, 7)), np.zeros((2, 4)), np.zeros((2, 24)), np.zeros((0, 8)),
                np.zeros((33, 8))):
        with pytest.raises(ValueError):
            S.MaxAffineCost(bad)
    with pytest.raises(ValueError):
        S.MaxAffineCost(A, np.zeros(5))
    for v in (np.nan, np.inf, -np.inf):
        A2 = A.copy(); A2[1, 2] = v
        with pytest.raises(ValueError):
            S.MaxAffineCost(A2)
        with pytest.raises(ValueError):
            S.MaxAffineCost(A, np.full(6, v))
    assert S.MaxAffineCost(np.ones((32, 22))).n == 10


def test_safe_ars_cost_dispatch(S):
    sim = S.SwimmerEnv("Simulator", n=3)
    A, b = cost_rows("bend", 3)
    ag = S.Safe_ARS(S.MaxAffineCost(A, b), 1.0, 0.5, sim)
    scr = ag._screen(S.SwimmerEnv("RealWorld", n=3))
    assert scr["cost"] is ag.cost and scr["sim_thresh"] == 0.5 and scr["real_thresh"] == 1.0
    assert "cost" not in S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sim)._screen(S.SwimmerEnv("RealWorld", n=3))
    with pytest.raises(ValueError):
        S.Safe_ARS(S.MaxAffineCost(*cost_rows("bend", 4)), 1.0, 0.5, sim)
    with pytest.raises(NotImplementedError):
        S.Safe_ARS(lambda x: np.sum(np.abs(x)), 1.0, 0.5, sim)


def test_rollout_costed_argument_checks(S):
    """Rejected before anything is launched: no device needed."""
    L = S._lib.lib()
    n = 3
    real, sim = _models(S, n)
    A, b = builtin_rows(n)
    F = np.ascontiguousarray(np.hstack([A, b[:, None]]))
    fp = F.ctypes.data_as(ctypes.c_void_p)

    def cfg(**kw):
        c = S._lib.SwmRollout()
        c.variant, c.policy_mode, c.H, c.B, c.rollouts_per_policy = S.GYM, S.ops.POLICY_EXPLICIT, 10, 64, 1
        c.screen.enabled, c.screen.sim = 1, sim
        for k, v in kw.items():
            if k == "enabled":
                c.screen.enabled = v
            else:
                setattr(c, k, v)
        return c

    def call(c, forms=fp, J=len(F)):
        return L.swm_rollout_costed(ctypes.byref(real), ctypes.byref(c), forms, J, None)

    bad, unsup = -1, -2
    assert call(cfg(enabled=0)) == bad
    assert call(cfg(), J=0) == bad and call(cfg(), J=33) == bad and call(cfg(), forms=None) == bad
    for v in (np.nan, np.inf):
        G = F.copy(); G[2, 4] = v
        assert call(cfg(), forms=G.ctypes.data_as(ctypes.c_void_p)) == bad
    for k in (S.KERNEL_LANES, S.KERNEL_LANES2, S.KERNEL_LANES3):
        assert call(cfg(kernel=k)) == unsup
    assert call(cfg(variant=S.RLGLUE)) == unsup
    assert call(cfg(normalize=1)) == unsup
    dummy = (ctypes.c_double * 64)()
    assert call(cfg(stats_partial=ctypes.cast(dummy, ctypes.c_void_p))) == unsup
    assert call(cfg(policy_mode=S.ops.POLICY_FIXED_ACTION)) == unsup
    assert call(cfg(schedule_sub=2, schedule_chunk=64)) == unsup


@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 7, 8, 9, 10])
def test_reference_affine_builtin_rows_equal_builtin(O, n):
    """The reference max-of-affine rollout with rows +-e_{3+2i} is the oracle's built-in one bit for bit, on a
    population with freezes and violations."""
    ro, so = _models(O, n)
    W, init, A, b, sim_thr, real_thr = _case(O, n, "builtin")
    H = 201
    fz_all, viol_all = [], []
    for e in range(len(W)):
        r1, f1, t1, v1, z1 = O.rollout_safe_step(ro, so, W[e], H, sim_thr, real_thr, init_state=init[e],
                                                 want_traj=True)
        r2, f2, t2, v2, z2 = rollout_safe_step_affine(O, ro, so, W[e], H, A, b, sim_thr, real_thr,
                                                      init_state=init[e], want_traj=True)
        assert (v1, z1) == (v2, z2) and _bits([r1]) == _bits([r2])
        assert np.array_equal(_bits(f1), _bits(f2)) and np.array_equal(_bits(t1), _bits(t2))
        fz_all.append(z1); viol_all.append(v1)
    fz_all = np.array(fz_all)
    assert (fz_all == 0).any() and ((fz_all > 0) & (fz_all < H)).any() and (fz_all == H).any()
    assert (np.array(viol_all) > 0).any()


@pytest.mark.parametrize("kind", COSTS)
@pytest.mark.parametrize("n", [2, 5, 10])
def test_reference_affine_cost_equals_max_affine_cost(S, O, n, kind):
    """The reference rollout's cost equals MaxAffineCost on every state it visits."""
    W, init, A, b, sim_thr, real_thr = _case(O, n, kind)
    ro, so = _models(O, n)
    c = S.MaxAffineCost(A, b)
    for e in range(0, len(W), 4):
        _, _, traj, _, _ = rollout_safe_step_affine(O, ro, so, W[e], 201, A, b, sim_thr, real_thr,
                                                    init_state=init[e], want_traj=True)
        for x in traj[::5]:
            want = c(x)
            scale = max(1.0, float(np.max(np.abs(A) @ np.abs(x) + np.abs(b))))  # summation order is free
            assert abs(_affine_cost(A, b, x) - want) <= 1e-15 * scale, (_affine_cost(A, b, x), want)
    assert np.isnan(_affine_cost(A, b, np.full(2 * n + 2, np.nan)))


# ---- GPU tests -------------------------------------------------------------------------------------------------------
def _costed(S, real, sim, H, cost, sim_thr, real_thr, kernel=0, **kw):
    return S.ops.rollout(real, H, want_final=True, want_trajectory=True, kernel=kernel,
                         screen=dict(sim_params=sim, sim_thresh=sim_thr, real_thresh=real_thr, cost=cost), **kw)


def _host(res):
    return (res.returns.cpu().numpy(), res.final_state.cpu().numpy(), res.trajectory.cpu().numpy(),
            res.frozen_at.cpu().numpy(), res.violations.cpu().numpy())


def _compare(O, ro, so, pols, starts, H, A, b, sim_thr, real_thr, res):
    got_r, got_f, traj, fz, viol = _host(res)
    er = ef = et = 0.0
    for e, (r, f, t, v, z) in enumerate(_oracle_loop(O, ro, so, pols, starts, H, A, b, sim_thr, real_thr)):
        assert (fz[e], viol[e]) == (z, v), (e, fz[e], z, viol[e], v)
        er = max(er, _ret_err(got_r[e], r))
        ef = max(ef, rel_err(got_f[e], f))
        et = max(et, rel_err(traj[:, e], t) if H else 0.0)
    assert er < RET_TOL and ef < STATE_TOL and et < STATE_TOL, (er, ef, et)
    return er, ef, et


def _frozen_tail(res, starts, H):
    """From the freeze on every stored state is the state before it."""
    _, fin, traj, fz, _ = _host(res)
    for e in range(fin.shape[0]):
        f = int(fz[e])
        held = starts[e] if f == 0 else traj[f - 1, e]
        assert np.array_equal(_bits(traj[f:, e]), np.broadcast_to(_bits(held), traj[f:, e].shape)), e


@gpu
@pytest.mark.parametrize("kind", COSTS)
@pytest.mark.parametrize("kern", ["THREAD", "AUTO"])
@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 7, 8, 9, 10])
def test_costed_screening_matches_oracle(S, O, n, kern, kind):
    """Explicit policies, B = 37, H = 201 (odd; crosses the sine/cosine re-evaluations at steps 63, 127, 191)."""
    H = 201
    (real, sim), (ro, so) = _models(S, n), _models(O, n)
    W, init, A, b, sim_thr, real_thr = _case(O, n, kind)
    res = _costed(S, real, sim, H, S.MaxAffineCost(A, b), sim_thr, real_thr, kernel=getattr(S, "KERNEL_" + kern),
                  policies=_cuda(W), init_state=_cuda(init))
    errs = _compare(O, ro, so, W, init, H, A, b, sim_thr, real_thr, res)
    _frozen_tail(res, init, H)
    assert _spread(res.frozen_at.cpu().numpy(), res.violations.cpu().numpy(), H, **NEED)
    print("\n[costed screening] %s n=%d %s: return %.2e, final %.2e, trajectory %.2e" % ((kern, n, kind) + errs))


@gpu
@pytest.mark.parametrize("kind", COSTS)
@pytest.mark.parametrize("kern", ["THREAD", "AUTO"])
@pytest.mark.parametrize("n,R,D", [(3, 1, 16), (5, 3, 8), (5, 32, 2), (8, 3, 8), (10, 32, 2)])
def test_costed_policy_sources_match_oracle(S, O, n, R, D, kern, kind):
    """In-kernel Philox perturbations, the same read from memory (bit-identical), R = 1, 3 and 32."""
    H, nu, seed, it, dir0 = 201, 0.3, 31 + n, 2, 5
    B, ws = 2 * D * R, (n - 1) * (2 * n + 2)
    (real, sim), (ro, so) = _models(S, n), _models(O, n)
    A, b = cost_rows(kind, n)
    rng = np.random.default_rng(7 * n + R)
    Wb = rng.uniform(-1, 1, ws) * 0.05
    count = B if R == 1 else R
    init = _starts(rng, n, count)
    pols = np.array([Wb + (-nu if (e // R) & 1 else nu) * O.philox_delta(seed, it, dir0 + ((e // R) >> 1), ws)
                     for e in range(B)])
    starts = np.array([init[e % count] for e in range(B)])
    costs = [_oracle_costs(O, ro, so, pols[e], starts[e], H, A, b) for e in range(B)]
    need = dict(zero=0, mid=2, mid_steps=2, never=1, violated=1)
    sim_thr, real_thr = _thresholds(np.array([c[0] for c in costs]), np.array([c[1] for c in costs]), **need)
    cost = S.MaxAffineCost(A, b)
    kw = dict(B=B, base_policy=_cuda(Wb), nu=nu, seed=seed, iteration=it, dir0=dir0, rollouts_per_policy=R,
              init_state=_cuda(init), kernel=getattr(S, "KERNEL_" + kern))
    res = _costed(S, real, sim, H, cost, sim_thr, real_thr, **kw)
    _compare(O, ro, so, pols, starts, H, A, b, sim_thr, real_thr, res)
    _frozen_tail(res, starts, H)
    mem = _costed(S, real, sim, H, cost, sim_thr, real_thr, deltas=S.ops.philox_deltas(seed, it, dir0, D, ws), **kw)
    for name in ("returns", "frozen_at", "violations", "final_state", "trajectory"):
        assert torch.equal(getattr(mem, name), getattr(res, name)), name


@gpu
@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 7, 8, 9, 10])
def test_builtin_rows_match_builtin_kernel(S, O, n):
    """The built-in cost as 2n forms on swm_rollout_costed against swm_rollout's built-in cost (THREAD)."""
    H = 201
    real, sim = _models(S, n)
    W, init, A, b, thr, rthr = _case(O, n, "builtin")
    cost = S.MaxAffineCost(A, b)
    kw = dict(policies=_cuda(W), init_state=_cuda(init), kernel=S.KERNEL_THREAD, want_final=True,
              want_trajectory=True)
    a = S.ops.rollout(real, H, screen=dict(sim_params=sim, sim_thresh=thr, real_thresh=rthr), **kw)
    c = S.ops.rollout(real, H, screen=dict(sim_params=sim, sim_thresh=thr, real_thresh=rthr, cost=cost), **kw)
    assert torch.equal(a.frozen_at, c.frozen_at) and torch.equal(a.violations, c.violations)
    fz = a.frozen_at.cpu().numpy()
    assert (fz == 0).any() and ((fz > 0) & (fz < H)).any() and (fz == H).any()
    assert rel_err(c.final_state.cpu().numpy(), a.final_state.cpu().numpy()) < STATE_TOL
    assert rel_err(c.trajectory.cpu().numpy(), a.trajectory.cpu().numpy()) < STATE_TOL
    same = all(torch.equal(getattr(a, k), getattr(c, k)) for k in ("returns", "final_state", "trajectory"))
    print("\n[costed screening] built-in rows n=%d: bit-identical to the built-in cost: %s" % (n, same))


@gpu
@pytest.mark.parametrize("n", [2, 5, 8])
def test_costed_threshold_semantics(S, O, n):
    B, H = 37, 65
    real, sim = _models(S, n)
    W, init, A, b, sim_thr, _ = _case(O, n, "bend")
    cost = S.MaxAffineCost(A, b)
    inf, nan = float("inf"), float("nan")
    kw = dict(policies=_cuda(W), init_state=_cuda(init))
    plain = S.ops.rollout(real, H, want_final=True, kernel=S.KERNEL_THREAD, **kw)
    never = _costed(S, real, sim, H, cost, inf, inf, **kw)
    assert (never.frozen_at.cpu().numpy() == H).all() and (never.violations.cpu().numpy() == 0).all()
    assert rel_err(never.final_state.cpu().numpy(), plain.final_state.cpu().numpy()) < 1e-12
    for thr in (-inf, nan):
        always = _costed(S, real, sim, H, cost, thr, -inf, **kw)
        assert (always.frozen_at.cpu().numpy() == 0).all() and (always.violations.cpu().numpy() == 0).all()
        assert (always.returns.cpu().numpy() == 0.0).all()
        assert np.array_equal(_bits(always.final_state.cpu().numpy()), _bits(init))
    for rthr in (inf, nan):
        r = _costed(S, real, sim, H, cost, sim_thr, rthr, **kw)
        assert (r.violations.cpu().numpy() == 0).all()
        assert ((r.frozen_at.cpu().numpy() > 0) & (r.frozen_at.cpu().numpy() < H)).any()
    # a NaN start state is unsafe at step 0; its neighbours are unaffected
    init2 = init.copy()
    init2[3, 2] = np.nan
    ref = _costed(S, real, sim, H, cost, sim_thr, 1.0, **kw)
    got = _costed(S, real, sim, H, cost, sim_thr, 1.0, policies=_cuda(W), init_state=_cuda(init2))
    assert int(got.frozen_at[3]) == 0 and int(got.violations[3]) == 0 and float(got.returns[3]) == 0.0
    keep = torch.arange(B, device="cuda") != 3
    for k in ("returns", "frozen_at", "violations", "final_state"):
        assert torch.equal(getattr(got, k)[keep], getattr(ref, k)[keep]), k


@functools.lru_cache(maxsize=None)
def _pool(O, n, kind):
    ro, so = _models(O, n)
    A, b = cost_rows(kind, n)
    W, init = _population(n, 64, seed=500 + n)
    W *= 10.0 ** np.linspace(-0.5, 0.5, 64)[:, None, None]
    init[:, 3::2] *= 0.1
    costs = [_oracle_costs(O, ro, so, W[e], init[e], 129, A, b) for e in range(64)]
    return W, init, A, b, np.array([c[0] for c in costs]), np.array([c[1] for c in costs])


@gpu
@pytest.mark.parametrize("n,kind", [(3, "dense32"), (6, "bend"), (9, "dense1")])
@pytest.mark.parametrize("H", [1, 63, 64, 65, 129])
def test_costed_freeze_position_and_horizon_edges(S, O, n, kind, H):
    """One launch per target step t* in {0, 1, 62, 63, 64, H-1}: the threshold sits between one environment's running
    maximum of simulator costs before t* and its cost at t*, so that it freezes exactly at t*."""
    (real, sim), (ro, so) = _models(S, n), _models(O, n)
    W, init, A, b, sc, rc = _pool(O, n, kind)
    sc, rc = sc[:, :H], rc[:, :H]
    cost = S.MaxAffineCost(A, b)
    for ts in sorted({t for t in (0, 1, 62, 63, 64, H - 1) if t < H}):
        lo, hi = np.max(sc[:, :ts], axis=1, initial=-np.inf), sc[:, ts]
        gap = hi - lo
        ok = np.isfinite(hi) & (gap > 4 * MARGIN * np.maximum(1.0, np.abs(hi))) & (np.isfinite(lo) | (ts == 0))
        assert ok.any(), ts
        tgt = int(np.flatnonzero(ok)[np.argmax(np.where(np.isfinite(gap), gap, 1.0)[ok])])
        sim_thr = 0.5 * (lo[tgt] + hi[tgt]) if ts else hi[tgt] - 0.5 * max(1.0, abs(hi[tgt])) * 1e-3
        fz_all = _freeze_steps(sc, sim_thr)
        taken = np.concatenate([rc[e, :fz_all[e]] for e in range(len(fz_all))])
        real_thr = _midpoint(taken, 0.7) if taken.size >= 2 else sim_thr

        def clear(e):
            return _margins_ok(sc[e:e + 1], rc[e:e + 1], sim_thr, real_thr)

        assert clear(tgt) and fz_all[tgt] == ts
        fill = [e for e in range(len(sc)) if e != tgt and clear(e)][:20]
        sel = fill[:5] + [tgt] + fill[5:]
        res = _costed(S, real, sim, H, cost, sim_thr, real_thr, policies=_cuda(W[sel]), init_state=_cuda(init[sel]))
        _compare(O, ro, so, W[sel], init[sel], H, A, b, sim_thr, real_thr, res)
        _frozen_tail(res, init[sel], H)
        assert int(res.frozen_at[5]) == ts


@gpu
@pytest.mark.parametrize("n", [3, 8])
def test_costed_batch_order_invariance(S, O, n):
    H = 201
    real, sim = _models(S, n)
    W, init, A, b, sim_thr, real_thr = _case(O, n, "dense32")
    cost = S.MaxAffineCost(A, b)
    a = _costed(S, real, sim, H, cost, sim_thr, real_thr, policies=_cuda(W), init_state=_cuda(init))
    p = np.random.default_rng(n).permutation(len(W))
    c = _costed(S, real, sim, H, cost, sim_thr, real_thr, policies=_cuda(W[p]), init_state=_cuda(init[p]))
    pt = torch.as_tensor(p, device="cuda")
    for k in ("returns", "frozen_at", "violations", "final_state"):
        assert torch.equal(getattr(c, k), getattr(a, k)[pt]), k
    assert torch.equal(c.trajectory, a.trajectory[:, pt])


@gpu
@pytest.mark.parametrize("n", [3, 8])
def test_costed_dir_mask(S, n):
    D, R, H = 6, 2, 130
    B, ws = 2 * D * R, (n - 1) * (2 * n + 2)
    real, sim = _models(S, n)
    rng = np.random.default_rng(40 + n)
    init = _starts(rng, n, R)
    cost = S.MaxAffineCost(*cost_rows("bend", n))
    kw = dict(B=B, base_policy=_cuda(rng.uniform(-1, 1, ws) * 0.05), nu=0.8, seed=3, iteration=1,
              rollouts_per_policy=R, init_state=_cuda(init))
    thr = float(np.median([cost(x) for x in init])) + 0.05
    full = _costed(S, real, sim, H, cost, thr, 0.8 * thr, **kw)
    mask = torch.tensor([1, 0, 1, 1, 0, 1], dtype=torch.int32, device="cuda")
    out = {"frozen_at": torch.full((B,), -7, dtype=torch.int32, device="cuda"),
           "violations": torch.full((B,), -9, dtype=torch.int32, device="cuda")}
    m = _costed(S, real, sim, H, cost, thr, 0.8 * thr, dir_mask=mask, out=out, **kw)
    live = np.repeat(mask.cpu().numpy().astype(bool), 2 * R)
    assert (m.frozen_at.cpu().numpy()[~live] == H).all() and (m.violations.cpu().numpy()[~live] == 0).all()
    assert np.isnan(m.returns.cpu().numpy()[~live]).all()
    lv = torch.as_tensor(live, device="cuda")
    for k in ("returns", "frozen_at", "violations", "final_state"):
        assert torch.equal(getattr(m, k)[lv], getattr(full, k)[lv]), k


@gpu
def test_costed_kernel_choice(S, O):
    n = 3
    real, sim = _models(S, n)
    W, init, A, b, sim_thr, real_thr = _case(O, n, "bend")
    cost = S.MaxAffineCost(A, b)
    for k in (S.KERNEL_LANES, S.KERNEL_LANES2, S.KERNEL_LANES3):
        with pytest.raises(S.SwimmerLibError):
            _costed(S, real, sim, 50, cost, sim_thr, real_thr, kernel=k, policies=_cuda(W), init_state=_cuda(init))
    # 512 environments: AUTO would pick a lane kernel for the built-in cost; the costed path runs THREAD
    rng = np.random.default_rng(5)
    pols = rng.uniform(-1, 1, (512, n - 1, 2 * n + 2)) * 0.3
    kw = dict(policies=_cuda(pols), init_state=_cuda(init[np.arange(512) % len(init)]))
    a = _costed(S, real, sim, 300, cost, sim_thr, real_thr, kernel=S.KERNEL_AUTO, **kw)
    t = _costed(S, real, sim, 300, cost, sim_thr, real_thr, kernel=S.KERNEL_THREAD, **kw)
    for k in ("returns", "frozen_at", "violations", "final_state", "trajectory"):
        assert torch.equal(getattr(a, k), getattr(t, k)), k


@gpu
@pytest.mark.parametrize("n", [3, 8])
def test_engine_costed_screening_matches_oracle_loop(S, O, n):
    """ArsEngine(step_screen=dict(..., cost=...)) for three iterations against the oracle loop; eager and graph
    replay bit-identical."""
    N, b, H, nu, alpha, seed = 8, 4, 150, 0.3, 0.02, 21
    (real, sim), (ro, so) = _models(S, n), _models(O, n)
    ws = (n - 1) * (2 * n + 2)
    A, bb = cost_rows("bend", n)
    W0 = np.random.default_rng(n).uniform(-1, 1, ws) * 0.3
    start = S.ops.reset_state(n).cpu().numpy()

    def directions(W, it):
        deltas = np.stack([O.philox_delta(seed, it, k, ws) for k in range(N)])
        return deltas, [W + s * nu * deltas[k] for k in range(N) for s in (+1, -1)]

    _, pols = directions(W0, 0)
    costs = [_oracle_costs(O, ro, so, p, start, H, A, bb) for p in pols]
    sim_thr, real_thr = _thresholds(np.array([c[0] for c in costs]), np.array([c[1] for c in costs]),
                                    zero=0, mid=2, mid_steps=2, never=1, violated=1)
    screen = dict(sim_params=sim, sim_thresh=sim_thr, real_thresh=real_thr, cost=S.MaxAffineCost(A, bb))
    engines = [S.ArsEngine(real, N=N, b=b, alpha=alpha, nu=nu, H=H, semantics=S.ARS_TOPB, seed=seed,
                           distributed=False, initial_policy=W0, step_screen=screen, use_graph=g) for g in (False, True)]
    W, frozen = W0, []
    for it in range(3):
        got = [e.run_iteration().clone() for e in engines]
        fz, viol = engines[0].last.frozen_at.cpu().numpy(), engines[0].last.violations.cpu().numpy()
        deltas, pols = directions(W, it)
        rets = []
        for e, p in enumerate(pols):
            sc, rc = _oracle_costs(O, ro, so, p, start, H, A, bb)
            assert _margins_ok(sc[None], rc[None], sim_thr, real_thr), (it, e)
            r, _, _, v, z = rollout_safe_step_affine(O, ro, so, p, H, A, bb, sim_thr, real_thr)
            assert (fz[e], viol[e]) == (z, v), (it, e)
            rets.append(r)
        assert _ret_err(got[0].cpu().numpy(), rets) < RET_TOL
        assert torch.equal(got[0], got[1]) and torch.equal(engines[0].W, engines[1].W)
        W, _ = O.update_policy(W, deltas, np.array(rets), b=b, alpha=alpha, semantics=1)
        assert rel_err(engines[0].W.cpu().numpy(), W) < 1e-6
        frozen.append(fz)
    assert engines[1]._graph is not None
    frozen = np.concatenate(frozen)
    assert (frozen < H).any() and (frozen == H).any()


@gpu
def test_safe_ars_train_with_max_affine_cost(S, O):
    """Safe_ARS(MaxAffineCost).train with numpy deltas against the same oracle loop."""
    n, N, b, alpha, nu, H, n_iter = 3, 3, 2, 0.02, 0.3, 150, 2
    real = S.SwimmerEnv("RealWorld", n=n)
    sim = S.SwimmerEnv("Simulator", n=n, m_i=1.05, l_i=0.95, k=9.5)
    ro = O.make_params(n=n)
    so = O.make_params(n=n, m_i=1.05, l_i=0.95, k=9.5)
    A, bb = cost_rows("bend", n)
    start = S.ops.reset_state(n).cpu().numpy()
    np.random.seed(2)
    d0 = np.stack([2 * np.random.rand(n - 1, 2 * n + 2) - 1 for _ in range(N)]).reshape(N, -1)
    costs = [_oracle_costs(O, ro, so, s * nu * d0[k], start, H, A, bb) for k in range(N) for s in (1, -1)]
    sim_thr, real_thr = _thresholds(np.array([c[0] for c in costs]), np.array([c[1] for c in costs]),
                                    zero=0, mid=1, mid_steps=1, never=0, violated=1)
    ag = S.Safe_ARS(S.MaxAffineCost(A, bb), real_thr, sim_thr, sim)
    np.random.seed(2)
    with contextlib.redirect_stdout(io.StringIO()):
        curve, _ = ag.train(n_iter, real, N, b, alpha, nu, H)
    np.random.seed(2)
    W, want = np.zeros((n - 1) * (2 * n + 2)), []
    for it in range(n_iter):
        d = np.stack([2 * np.random.rand(n - 1, 2 * n + 2) - 1 for _ in range(N)]).reshape(N, -1)
        rets = []
        for k in range(N):
            for s in (1, -1):
                sc, rc = _oracle_costs(O, ro, so, W + s * nu * d[k], start, H, A, bb)
                assert _margins_ok(sc[None], rc[None], sim_thr, real_thr)
                rets.append(rollout_safe_step_affine(O, ro, so, W + s * nu * d[k], H, A, bb, sim_thr, real_thr)[0])
        want.append(np.mean(rets))
        W, _ = O.update_policy(W, d, np.array(rets), b=b, alpha=alpha, semantics=1)
    np.testing.assert_allclose(curve, want, rtol=1e-6, atol=1e-10)
    assert rel_err(ag.policy.reshape(-1), W) < 1e-6
