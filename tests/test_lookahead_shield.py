"""The lookahead shield (swm_rollout_lookahead; ops.rollout with screen["lookahead"]; Safe_ARS(..., lookahead=K))
against a CPU reference: rollout_safe_step_shielded's loop with each judgement composed from the oracle's own single
steps.

An action a is safe from the real state s only if, for every model m, x_1 = f_m(s, a), x_{j+1} = f_m(x_j, backup(x_j))
for j = 1..K and cost(x_j) <= sim_thresh for j = 1..K+1.  The step takes the policy's action if it is safe, else the
backup b_0 = backup(s) if that is safe by the same rule (one override), else it freezes for good.  A judgement may stop
at its first unsafe cost; its deciding maximum is the largest cost it evaluated (the first unsafe one, or every cost of
a safe judgement).  Every threshold is accepted only if every deciding maximum along the reference's own path, and
every real cost of a step taken, is at least MARGIN * max(1, |thr|) away from it: the exact checks of freeze steps,
override and violation counts then cannot flip on rounding, whatever order the kernel judges the models in."""
import contextlib
import ctypes
import functools
import io

import numpy as np
import pytest
import torch

from conftest import rel_err
from test_costed_screening import _affine_cost, builtin_rows, cost_rows
from test_ensemble_screening import _costs, _ensemble, _same
from test_shield_screening import _backup, _compare, _ok, _rows, rollout_safe_step_shielded
from test_step_screening import _bits, _cuda, _midpoint, _population, _starts

gpu = pytest.mark.gpu


# ---- reference -------------------------------------------------------------------------------------------------------
def _judge(O, sims, st, A, b, thr, Wb, u0, K, max_u, clip, **act):
    """One judgement from the state st of the action given by `act` (policy= or action=, as O.rollout takes it)
    -> (safe, deciding maximum).  The backup of the lookahead is clipped to +-max_u (the real model's) with `clip`."""
    dec = -np.inf
    for s in sims:
        x = O.rollout(s, O.GYM, 1, init_state=st, clip=clip, **act)[1]
        for j in range(K + 1):
            if j:
                bu = Wb @ x + u0
                if clip:
                    bu = np.clip(bu, -max_u, max_u)
                x = O.rollout(s, O.GYM, 1, action=np.ascontiguousarray(bu), init_state=x)[1]
            c = _affine_cost(A, b, x)
            if np.isnan(c) or c > dec:
                dec = c
            if not c <= thr:
                return False, dec
    return True, dec


def rollout_safe_step_lookahead(O, real_p, sims, policy, H, A, b, sim_thresh, real_thresh, Wb, u0, K, init_state=None,
                                want_traj=False, clip=False):
    """rollout_safe_step_shielded with the K-step judgement.  -> (return, final state, trajectory [H, 2n+2] or None,
    violations, freeze step, overrides, deciding maxima of every judgement, real costs of the steps taken, first
    rejection's backup rejected, decisions: one of 'p' (policy), 'b' (backup), 'f' (freeze) per step)."""
    n = real_p.n
    W = np.ascontiguousarray(policy, dtype=np.float64).reshape(n - 1, 2 * n + 2)
    st = O.rollout(real_p, O.GYM, 0, policy=W)[1] if init_state is None else np.array(init_state, dtype=np.float64)
    traj = np.zeros((H, 2 * n + 2)) if want_traj else None
    total, viol, frozen, over = 0.0, 0, H, 0
    sim_costs, real_costs, first_rejected, dec = [], [], None, ""
    judge = functools.partial(_judge, O, sims, A=A, b=b, thr=sim_thresh, Wb=Wb, u0=u0, K=K, max_u=real_p.max_u,
                              clip=clip)
    for t in range(H):
        safe, c = judge(st, policy=W)
        sim_costs.append(c)
        if safe:
            r, st, _ = O.rollout(real_p, O.GYM, 1, policy=W, init_state=st, clip=clip)
            dec += "p"
        else:
            bu = Wb @ st + u0
            if clip:  # the oracle clips policy actions only
                bu = np.clip(bu, -real_p.max_u, real_p.max_u)
            bu = np.ascontiguousarray(bu)
            safe, c = judge(st, action=bu)
            sim_costs.append(c)
            if first_rejected is None:
                first_rejected = not safe
            if not safe:
                frozen = t
                dec += "f"
                if want_traj:
                    traj[t:] = st
                break
            r, st, _ = O.rollout(real_p, O.GYM, 1, action=bu, init_state=st, clip=clip)
            over += 1
            dec += "b"
        total += r
        real_costs.append(_affine_cost(A, b, st))
        if real_costs[-1] > real_thresh:
            viol += 1
        if want_traj:
            traj[t] = st
    return (total, st, traj, viol, frozen, over, np.array(sim_costs), np.array(real_costs), bool(first_rejected), dec)


def _refs_at(O, ro, sims, pols, starts, H, A, b, thr, rthr, Wb, u0, K, clip=False, check=True):
    """References of a population, or None as soon as one deciding maximum is within the margin (with `check`)."""
    refs = []
    for e in range(len(pols)):
        r = rollout_safe_step_lookahead(O, ro, sims, pols[e], H, A, b, thr, rthr, Wb, u0, K, starts[e], True, clip)
        if check and not _ok(r[6], thr):
            return None
        refs.append(r)
    return refs


def _thresholds(O, ro, sims, pols, starts, H, A, b, Wb, u0, K, sc, clip=False, need_over=True,
                quantiles=(0.5, 0.3, 0.7, 0.2, 0.8)):
    """(sim_thr, real_thr, references) with every deciding cost at its margin, some environment that overrides (with
    `need_over`) and some that never does, or None.  The simulator threshold lies between neighbouring unscreened
    ensemble costs; the path does not depend on the real threshold, taken between neighbouring real costs."""
    for q in quantiles:
        s = _midpoint(sc, q)
        refs = _refs_at(O, ro, sims, pols, starts, H, A, b, s, np.inf, Wb, u0, K, clip)
        if refs is None:
            continue
        ov = np.array([r[5] for r in refs])
        if (need_over and not (ov > 0).any()) or not (ov == 0).any():
            continue
        taken = np.concatenate([r[7] for r in refs])
        if taken.size < 2:
            continue
        for rq in (0.8, 0.9, 0.7, 0.95, 0.6):
            r_thr = _midpoint(taken, rq)
            if all(_ok(r[7], r_thr) for r in refs):
                return s, r_thr, [x[:3] + (int((x[7] > r_thr).sum()),) + x[4:] for x in refs]
    return None


@functools.lru_cache(maxsize=None)
def _case(O, n, kind, backup, M, K, B=24, H=120, clip=False):
    """Explicit policies, starts, cost, backup, thresholds and references (oracle only): the first of a few seeded
    populations whose references override somewhere and hold every margin."""
    ro, sims = _ensemble(O, n)
    A, b = _rows(kind, n)
    Wb, u0 = _backup(backup, n)
    if clip:  # a damping gain that saturates at +-max_u inside the lookahead
        Wb = 40.0 * Wb
    for seed in range(6):
        W, init = _population(n, B, seed=700 + n + 1000 * seed)
        init[:, :2] *= 0.1
        sc, _ = _costs(O, n, W, init, H, A, b)
        found = _thresholds(O, ro, sims[:M], W, init, H, A, b, Wb, u0, K, np.max(sc[:M], axis=0), clip)
        if found is not None:
            return W, init, A, b, Wb, u0, found[0], found[1], found[2]
    raise AssertionError("no population for n=%d, %s, %s, M=%d, K=%d" % (n, kind, backup, M, K))


@functools.lru_cache(maxsize=None)
def _bending_case(O, n=3, M=2, K=10, B=16, H=150):
    """The claim of the feature on the oracle: with bending limits |th_i - th_{i+1}| <= thr, a swimmer that starts
    straight and slow, policies that bend it, and a damping backup of gain 10 on the relative joint velocities, the
    one-step shield never overrides; a K-step one overrides, and some rollout that freezes at K = 0 then freezes later
    or not at all.  -> (policies, starts, A, b, Wb, u0, thr, references at K = 0, references at K)."""
    ro, sims = _ensemble(O, n)
    A, b = cost_rows("bend", n)
    Wb, u0 = _backup("damping", n)
    Wb = 10.0 * Wb
    for seed in range(4):
        rng = np.random.default_rng(3 + seed)
        W = 5.0 * _population(n, B, seed=903 + seed)[0]
        init = np.zeros((B, 2 * n + 2))
        init[:, 2::2] = np.pi / 2 + 0.01 * rng.standard_normal((B, n))
        init[:, 3::2] = 0.1 * rng.standard_normal((B, n))
        for thr in (0.05, 0.15):
            r0 = _refs_at(O, ro, sims[:M], W, init, H, A, b, thr, np.inf, Wb, u0, 0)
            rk = _refs_at(O, ro, sims[:M], W, init, H, A, b, thr, np.inf, Wb, u0, K)
            if r0 is None or rk is None:
                continue
            if any(r0[e][4] < H and rk[e][4] > r0[e][4] for e in range(B)) and sum(r[5] for r in rk) > 0:
                return W, init, A, b, Wb, u0, thr, r0, rk
    raise AssertionError("no bending population shows the lookahead overriding")


def _oracle_env(S, O, p):
    """A simulator environment that steps through the oracle (for Safe_ARS.isSafe / isRecoverable on the host)."""
    class OracleEnv(S.SwimmerEnv):
        def next_observation(self, torque, G_dot, theta, theta_dot):
            s = O.step(p, O.GYM, self._pack(G_dot, theta, theta_dot), np.asarray(torque, dtype=np.float64))[0]
            return s[:2].copy(), s[2::2].copy(), s[3::2].copy()
    return OracleEnv("Simulator", n=p.n)


# ---- CPU tests -------------------------------------------------------------------------------------------------------
def test_rollout_lookahead_argument_checks(S):
    """Whatever swm_rollout_shielded refuses, with the same status; then a lookahead outside 0..SWM_MAX_LOOKAHEAD,
    also for an empty batch; no device needed."""
    L = S._lib.lib()
    n = 3
    real, sims = _ensemble(S, n)
    A, b = builtin_rows(n)
    F = np.ascontiguousarray(np.hstack([A, b[:, None]]))
    fp = F.ctypes.data_as(ctypes.c_void_p)
    Wb, u0 = _backup("linear", n)
    BK = np.ascontiguousarray(np.concatenate([Wb.reshape(-1), u0]))
    bp = BK.ctypes.data_as(ctypes.c_void_p)

    def cfg(**kw):
        c = S._lib.SwmRollout()
        c.variant, c.policy_mode, c.H, c.B, c.rollouts_per_policy = S.GYM, S.ops.POLICY_EXPLICIT, 10, 64, 1
        c.screen.enabled = 1
        for k, v in kw.items():
            if k == "enabled":
                c.screen.enabled = v
            else:
                setattr(c, k, v)
        return c

    def models(ps):
        return (S._lib.SwmParams * len(ps))(*ps)

    good = models(sims[:3])

    def call(c, ms=good, M=3, forms=fp, J=len(F), bk=bp, K=4):
        return L.swm_rollout_lookahead(ctypes.byref(real), ctypes.byref(c), ms, M, forms, J, bk, K, None, None)

    def shield(c, ms=good, M=3, forms=fp, J=len(F), bk=bp):
        return L.swm_rollout_shielded(ctypes.byref(real), ctypes.byref(c), ms, M, forms, J, bk, None, None)

    bad, unsup, kmax = -1, -2, S._lib.MAX_LOOKAHEAD
    dummy = (ctypes.c_double * 64)()
    zero_l = S.make_params(n=n)
    zero_l.l_i = 0.0
    nan_bk = BK.copy()
    nan_bk[0] = np.nan
    for forms in (fp, None):
        cases = [dict(c=cfg(enabled=0)), dict(c=cfg(), M=0), dict(c=cfg(), M=17), dict(c=cfg(), ms=None),
                 dict(c=cfg(), ms=models(sims[:2] + [S.make_params(n=4)])), dict(c=cfg(H=-1)),
                 dict(c=cfg(rollouts_per_policy=0)), dict(c=cfg(B=63, policy_mode=S.ops.POLICY_PHILOX)),
                 dict(c=cfg(), ms=models([sims[0], zero_l]), M=2), dict(c=cfg(), bk=None),
                 dict(c=cfg(B=0), bk=None), dict(c=cfg(), bk=nan_bk.ctypes.data_as(ctypes.c_void_p))]
        for kw in cases:
            for K in (0, 4, -1, kmax + 1):  # the shield's errors come first, whatever the lookahead
                assert call(forms=forms, K=K, **kw) == bad == shield(forms=forms, **kw)
        for c in [cfg(kernel=k) for k in (S.KERNEL_LANES, S.KERNEL_LANES2, S.KERNEL_LANES3)] + [
                cfg(variant=S.RLGLUE), cfg(normalize=1), cfg(stats_partial=ctypes.cast(dummy, ctypes.c_void_p)),
                cfg(policy_mode=S.ops.POLICY_FIXED_ACTION), cfg(schedule_sub=2, schedule_chunk=64)]:
            for K in (0, 1, kmax, -1):
                assert call(c, forms=forms, K=K) == unsup == shield(c, forms=forms)
        for K in (0, 1, 63, kmax):
            assert call(cfg(B=0), forms=forms, K=K) == 0
        for K in (-1, kmax + 1, -2 ** 31):
            assert call(cfg(B=0), forms=forms, K=K) == bad and call(cfg(), forms=forms, K=K) == bad
    assert call(cfg(), J=0) == bad == shield(cfg(), J=0)


def test_lookahead_value_errors(S):
    """ops.rollout and Safe_ARS refuse a lookahead that is negative, not an integer, too large, or without a backup,
    before they need a device; lookahead=0 leaves Safe_ARS's screen the shield's."""
    n = 3
    real = S.make_params(n=n)
    sims = [S.make_params(n=n, l_i=1.01)]
    bk = dict(policy=None, action=None)
    for K, with_backup in ((-1, True), (S._lib.MAX_LOOKAHEAD + 1, True), (2.0, True), ("3", True), (True, True),
                           (None, True), (1, False), (S._lib.MAX_LOOKAHEAD, False)):
        screen = dict(sim_params=sims, sim_thresh=1.0, real_thresh=1.0, lookahead=K)
        if with_backup:
            screen["backup"] = bk
        with pytest.raises(ValueError):
            S.ops.rollout(real, 10, actions=np.zeros((4, n - 1)), screen=screen)
    assert S.ops.check_lookahead(np.int64(7), True) == 7 and S.ops.check_lookahead(0, False) == 0
    env_r = S.SwimmerEnv("RealWorld", n=n)
    sim = S.SwimmerEnv("Simulator", n=n, l_i=1.01)
    Wb, u0 = _backup("damping", n)
    for kw in (dict(lookahead=1), dict(lookahead=-1, backup_policy=Wb), dict(lookahead=1.5, backup_policy=Wb),
               dict(lookahead=S._lib.MAX_LOOKAHEAD + 1, backup_action=u0)):
        with pytest.raises(ValueError):
            S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sim, **kw)
    shielded = S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sim, backup_policy=Wb, backup_action=u0)
    zero = S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sim, backup_policy=Wb, backup_action=u0, lookahead=0)
    assert zero.lookahead == 0 and set(zero._screen(env_r)) == set(shielded._screen(env_r))
    assert "lookahead" not in zero._screen(env_r)
    assert S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sim, lookahead=0).lookahead == 0
    la = S.Safe_ARS(S.builtin_cost, 1.0, 0.5, [sim, sim], backup_policy=Wb, lookahead=5)
    assert la._screen(env_r)["lookahead"] == 5 and "backup" in la._screen(env_r)


@pytest.mark.parametrize("n,kind,backup", [(2, "builtin", "zero"), (3, "gdot", "damping"), (6, "builtin", "linear"),
                                           (3, "bend", "damping")])
def test_reference_without_lookahead_is_shielded_reference(O, n, kind, backup):
    """K = 0: the reference is rollout_safe_step_shielded bit for bit."""
    ro, sims = _ensemble(O, n)
    A, b = _rows(kind, n)
    Wb, u0 = _backup(backup, n)
    W, init = _population(n, 12, seed=31 + n)
    init[:, :2] *= 0.1
    sc, rc = _costs(O, n, W, init, 80, A, b)
    thr, rthr = _midpoint(np.max(sc[:2], axis=0), 0.5), _midpoint(rc.reshape(-1), 0.8)
    kinds = set()
    for e in range(len(W)):
        got = rollout_safe_step_lookahead(O, ro, sims[:2], W[e], 80, A, b, thr, rthr, Wb, u0, 0, init[e], True)
        want = rollout_safe_step_shielded(O, ro, sims[:2], W[e], 80, A, b, thr, rthr, Wb, u0, init[e], True)
        assert got[3:6] == want[3:6] and got[8] == want[8] and _bits([got[0]]) == _bits([want[0]])
        assert np.array_equal(_bits(got[1]), _bits(want[1])) and np.array_equal(_bits(got[2]), _bits(want[2]))
        assert np.array_equal(_bits(got[7]), _bits(want[7]))
        kinds.add("over" if got[5] else "frozen" if got[4] < 80 else "never")
    assert len(kinds) >= 2


def test_lookahead_shield_acts_on_bending_limits(O):
    """The capability, on the oracle alone: with bending limits the one-step shield never overrides, while the K-step
    shield overrides and lets some rollout that froze at K = 0 run on longer."""
    H = 150
    W, init, A, b, Wb, u0, thr, r0, rk = _bending_case(O)
    assert all(r[5] == 0 for r in r0) and any(r[4] < H for r in r0)
    assert sum(r[5] for r in rk) > 0
    assert any(r0[e][4] < H and rk[e][4] > r0[e][4] for e in range(len(W)))


@pytest.mark.parametrize("n,kind,backup,M,K", [(3, "builtin", "zero", 2, 3), (3, "gdot", "damping", 3, 2),
                                               (4, "builtin", "linear", 2, 5)])
def test_shielded_action_with_lookahead_matches_reference_first_decision(S, O, n, kind, backup, M, K):
    """Safe_ARS.shielded_action with a lookahead (isRecoverable on each judgement, simulator environments stepping
    through the oracle) against the reference's first decision."""
    _, so = _ensemble(O, n)
    W, init, A, b, Wb, u0, thr, rthr, refs = _case(O, n, kind, backup, M, K)
    envs = [_oracle_env(S, O, p) for p in so[:M]]
    cost = S.builtin_cost if kind == "builtin" else S.MaxAffineCost(A, b)
    ag = S.Safe_ARS(cost, rthr, thr, envs, backup_policy=Wb, backup_action=u0, lookahead=K)
    kinds = set()
    for e in range(len(W)):
        a = W[e] @ init[e]
        got = ag.shielded_action(cost, thr, envs, list(init[e]), a)
        first = refs[e][9][:1]
        if first == "f":
            assert got is None, e
        elif first == "b":
            assert got is not a and np.array_equal(got, Wb @ init[e] + u0), e
        else:
            assert got is a, e
        kinds.add(first)
    assert "p" in kinds and len(kinds) >= 2, kinds


# ---- GPU tests -------------------------------------------------------------------------------------------------------
def _run(S, real, sims, H, kind, sim_thr, real_thr, Wb, u0, K, **kw):
    screen = dict(sim_params=list(sims), sim_thresh=sim_thr, real_thresh=real_thr, backup=dict(policy=Wb, action=u0),
                  lookahead=K)
    if kind != "builtin":
        screen["cost"] = S.MaxAffineCost(*_rows(kind, real.n))
    return S.ops.rollout(real, H, want_final=True, want_trajectory=True, screen=screen, **kw)


@gpu
@pytest.mark.parametrize("M,K", [(1, 8), (16, 1)])
@pytest.mark.parametrize("kind,backup", [("builtin", "zero"), ("gdot", "damping")])
@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 7, 8, 9, 10])
def test_lookahead_matches_oracle(S, O, n, kind, backup, M, K):
    """Explicit policies, B = 24, H = 120."""
    real, sims = _ensemble(S, n)
    W, init, A, b, Wb, u0, thr, rthr, refs = _case(O, n, kind, backup, M, K)
    res = _run(S, real, sims[:M], 120, kind, thr, rthr, Wb, u0, K, policies=_cuda(W), init_state=_cuda(init))
    errs = _compare(refs, res, 120)
    print("\n[lookahead] n=%d M=%d K=%d %s/%s: return %.2e, final %.2e, trajectory %.2e"
          % ((n, M, K, kind, backup) + errs))


@gpu
@pytest.mark.parametrize("M", [2, 7])
@pytest.mark.parametrize("n", [3, 5, 10])
def test_lookahead_linear_backup_matches_oracle(S, O, n, M):
    """A constant torque u_0 plus a linear term W_b, K = 4."""
    real, sims = _ensemble(S, n)
    W, init, A, b, Wb, u0, thr, rthr, refs = _case(O, n, "builtin", "linear", M, 4)
    res = _run(S, real, sims[:M], 120, "builtin", thr, rthr, Wb, u0, 4, policies=_cuda(W), init_state=_cuda(init))
    _compare(refs, res, 120)


@gpu
def test_lookahead_bending_population(S, O):
    """The kernel reproduces the oracle's bending-limit population: overrides and later freezes with K = 10, none at
    K = 0."""
    n, M, K, H = 3, 2, 10, 150
    real, sims = _ensemble(S, n)
    W, init, A, b, Wb, u0, thr, r0, rk = _bending_case(O)
    for k, refs in ((0, r0), (K, rk)):
        res = _run(S, real, sims[:M], H, "bend", thr, np.inf, Wb, u0, k, policies=_cuda(W), init_state=_cuda(init))
        _compare(refs, res, H)
    assert int(res.overrides.sum()) > 0


@gpu
@pytest.mark.parametrize("n,R,D", [(3, 1, 12), (3, 3, 4), (6, 32, 1)])
def test_lookahead_policy_sources_match_oracle(S, O, n, R, D):
    """In-kernel Philox perturbations against the oracle and the same read from memory (bit-identical), R = 1, 3 and
    32 (for n = 6 the warp-shared policy layout)."""
    H, nu, seed, it, dir0, M, K = 100, 0.3, 31 + n, 2, 5, 3, 3
    B, ws = 2 * D * R, (n - 1) * (2 * n + 2)
    (real, sims), (ro, so) = _ensemble(S, n), _ensemble(O, n)
    A, b = builtin_rows(n)
    Wb, u0 = _backup("zero", n)
    rng = np.random.default_rng(7 * n + R)
    Wbase = rng.uniform(-1, 1, ws) * 0.1
    count = B if R == 1 else R
    init = _starts(rng, n, count)
    pols = np.array([Wbase + (-nu if (e // R) & 1 else nu) * O.philox_delta(seed, it, dir0 + ((e // R) >> 1), ws)
                     for e in range(B)]).reshape(B, n - 1, 2 * n + 2)
    starts = np.array([init[e % count] for e in range(B)])
    sc, _ = _costs(O, n, pols, starts, H, A, b)
    found = _thresholds(O, ro, so[:M], pols, starts, H, A, b, Wb, u0, K, np.max(sc[:M], axis=0), need_over=False)
    assert found is not None
    thr, rthr, refs = found
    kw = dict(B=B, base_policy=_cuda(Wbase), nu=nu, seed=seed, iteration=it, dir0=dir0, rollouts_per_policy=R,
              init_state=_cuda(init))
    res = _run(S, real, sims[:M], H, "builtin", thr, rthr, Wb, u0, K, **kw)
    _compare(refs, res, H)
    mem = _run(S, real, sims[:M], H, "builtin", thr, rthr, Wb, u0, K, deltas=S.ops.philox_deltas(seed, it, dir0, D, ws),
               **kw)
    _same(mem, res, ("returns", "frozen_at", "violations", "overrides", "final_state", "trajectory"))


@gpu
@pytest.mark.parametrize("n", [3, 8])
def test_lookahead_dir_mask(S, n):
    D, R, H, M, K = 6, 2, 130, 4, 4
    B, ws = 2 * D * R, (n - 1) * (2 * n + 2)
    real, sims = _ensemble(S, n)
    rng = np.random.default_rng(40 + n)
    init = _starts(rng, n, R)
    Wb, u0 = _backup("zero", n)
    thr = float(np.median(np.max(np.abs(init[:, 3::2]), axis=1))) + 0.05
    kw = dict(B=B, base_policy=_cuda(rng.uniform(-1, 1, ws) * 0.3), nu=0.8, seed=3, iteration=1,
              rollouts_per_policy=R, init_state=_cuda(init))
    full = _run(S, real, sims[:M], H, "builtin", thr, 0.8 * thr, Wb, u0, K, **kw)
    mask = torch.tensor([1, 0, 1, 1, 0, 1], dtype=torch.int32, device="cuda")
    out = {k: torch.full((B,), -7, dtype=torch.int32, device="cuda") for k in ("frozen_at", "violations", "overrides")}
    m = _run(S, real, sims[:M], H, "builtin", thr, 0.8 * thr, Wb, u0, K, dir_mask=mask, out=out, **kw)
    live = np.repeat(mask.cpu().numpy().astype(bool), 2 * R)
    assert (m.frozen_at.cpu().numpy()[~live] == H).all() and (m.violations.cpu().numpy()[~live] == 0).all()
    assert (m.overrides.cpu().numpy()[~live] == 0).all() and np.isnan(m.returns.cpu().numpy()[~live]).all()
    lv = torch.as_tensor(live, device="cuda")
    for k in ("returns", "frozen_at", "violations", "overrides", "final_state"):
        assert torch.equal(getattr(m, k)[lv], getattr(full, k)[lv]), k


@gpu
@pytest.mark.parametrize("H", [0, 1, 63, 64, 201])
def test_lookahead_horizon_edges(S, O, H):
    """Short and odd horizons on the 201-step case's thresholds (their margins hold for every prefix), n = 3, K = 2."""
    n, M, K = 3, 2, 2
    ro, so = _ensemble(O, n)
    real, sims = _ensemble(S, n)
    W, init, A, b, Wb, u0, thr, rthr, _ = _case(O, n, "builtin", "zero", M, K, B=16, H=201)
    refs = _refs_at(O, ro, so[:M], W, init, H, A, b, thr, rthr, Wb, u0, K, check=False)
    res = _run(S, real, sims[:M], H, "builtin", thr, rthr, Wb, u0, K, policies=_cuda(W), init_state=_cuda(init))
    _compare(refs, res, H)
    if H == 0:
        assert (res.frozen_at.cpu().numpy() == 0).all() and (res.overrides.cpu().numpy() == 0).all()


@gpu
@pytest.mark.parametrize("K", [1, 63, 64, 65])
def test_lookahead_lengths(S, O, K):
    """Lookaheads around the 64-step exact re-evaluation of the simulated sines and cosines, n = 3 and n = 8."""
    for n in (3, 8):
        real, sims = _ensemble(S, n)
        W, init, A, b, Wb, u0, thr, rthr, refs = _case(O, n, "builtin", "damping", 1, K, B=12, H=60)
        res = _run(S, real, sims[:1], 60, "builtin", thr, rthr, Wb, u0, K, policies=_cuda(W), init_state=_cuda(init))
        _compare(refs, res, 60)


@gpu
def test_lookahead_longest(S, O):
    """K = SWM_MAX_LOOKAHEAD at a small batch and horizon: straight, slow starts under a damping backup, where some
    rollouts take the policy, some the backup and some freeze."""
    n, M, K, H, B, thr = 3, 1, S._lib.MAX_LOOKAHEAD, 6, 8, 0.15
    ro, so = _ensemble(O, n)
    real, sims = _ensemble(S, n)
    A, b = builtin_rows(n)
    Wb, u0 = _backup("damping", n)
    rng = np.random.default_rng(5)
    W = 20.0 * _population(n, B, seed=5)[0]
    init = np.zeros((B, 2 * n + 2))
    init[:, 2::2] = np.pi / 2 + 0.01 * rng.standard_normal((B, n))
    init[:, 3::2] = 0.1 * rng.standard_normal((B, n))
    refs = _refs_at(O, ro, so[:M], W, init, H, A, b, thr, np.inf, Wb, u0, K)
    assert refs is not None and {r[9][:1] for r in refs} == {"p", "b", "f"}
    res = _run(S, real, sims[:M], H, "builtin", thr, np.inf, Wb, u0, K, policies=_cuda(W), init_state=_cuda(init))
    _compare(refs, res, H)


@gpu
def test_lookahead_clipped_backup(S, O):
    """clip_actions with a damping backup of gain 20 that saturates at +-max_u inside the lookahead."""
    n, M, K = 3, 2, 4
    real, sims = _ensemble(S, n)
    W, init, A, b, Wb, u0, thr, rthr, refs = _case(O, n, "builtin", "damping", M, K, clip=True)
    res = _run(S, real, sims[:M], 120, "builtin", thr, rthr, Wb, u0, K, policies=_cuda(W), init_state=_cuda(init),
               clip_actions=True)
    _compare(refs, res, 120)


@gpu
@pytest.mark.parametrize("kind", ["builtin", "gdot"])
def test_lookahead_zero_is_shield(S, O, monkeypatch, kind):
    """swm_rollout_lookahead with K = 0 gives swm_rollout_shielded's outputs bit for bit, for every n."""
    L = S._lib.lib()
    shielded = L.swm_rollout_shielded
    for n in range(2, 11):
        real, sims = _ensemble(S, n)
        W, init = _population(n, 24, seed=60 + n)
        init[:, :2] *= 0.1
        Wb, u0 = _backup("damping", n)
        kw = dict(policies=_cuda(W), init_state=_cuda(init))
        want = _run(S, real, sims[:5], 150, kind, 1.0, 0.9, Wb, u0, 0, **kw)
        # the shield's own call, routed through swm_rollout_lookahead with K = 0
        monkeypatch.setattr(L, "swm_rollout_shielded", lambda *a: L.swm_rollout_lookahead(*a[:7], 0, *a[7:]))
        got = _run(S, real, sims[:5], 150, kind, 1.0, 0.9, Wb, u0, 0, **kw)
        monkeypatch.setattr(L, "swm_rollout_shielded", shielded)
        _same(got, want, ("returns", "frozen_at", "violations", "overrides", "final_state", "trajectory"))
        assert (want.frozen_at.cpu().numpy() < 150).any() or (want.overrides.cpu().numpy() > 0).any(), n


@gpu
@pytest.mark.parametrize("n", [3, 8])
def test_engine_lookahead_graph_equals_eager(S, n):
    """ArsEngine(step_screen=... lookahead ...): graph-replayed iterations equal eager ones bit for bit."""
    N, b, H, nu, alpha, seed, M, K = 8, 4, 150, 0.3, 0.02, 21, 3, 3
    real, sims = _ensemble(S, n)
    ws = (n - 1) * (2 * n + 2)
    W0 = np.random.default_rng(n).uniform(-1, 1, ws) * 0.3
    Wb, u0 = _backup("damping", n)
    screen = dict(sim_params=sims[:M], sim_thresh=0.5, real_thresh=0.4, backup=dict(policy=Wb, action=u0),
                  lookahead=K)
    engines = [S.ArsEngine(real, N=N, b=b, alpha=alpha, nu=nu, H=H, semantics=S.ARS_TOPB, seed=seed,
                           distributed=False, initial_policy=W0, step_screen=screen, use_graph=g) for g in (False, True)]
    total = 0
    for it in range(4):
        got = [e.run_iteration().clone() for e in engines]
        assert torch.equal(got[0], got[1]) and torch.equal(engines[0].W, engines[1].W), it
        for k in ("overrides", "frozen_at", "violations"):
            assert torch.equal(getattr(engines[0].last, k), getattr(engines[1].last, k)), (it, k)
        total += int(engines[0].last.overrides.sum())
    assert engines[1]._graph is not None and total > 0


@gpu
def test_safe_ars_train_with_lookahead(S, O):
    """Safe_ARS(..., lookahead=K).train with numpy deltas against a host ARS loop whose every step is
    Safe_ARS.shielded_action on oracle-stepped simulators (built-in cost, two models), the margins checked on the
    reference loop."""
    n, N, b, alpha, nu, H, n_iter, K = 3, 3, 2, 0.02, 0.3, 100, 2, 3
    consts = [dict(m_i=1.05, l_i=0.95, k=9.5), dict(m_i=0.97, l_i=1.02, k=10.4)]
    real = S.SwimmerEnv("RealWorld", n=n)
    sims = [S.SwimmerEnv("Simulator", n=n, **c) for c in consts]
    ro = O.make_params(n=n)
    so = [O.make_params(n=n, **c) for c in consts]
    A, bb = builtin_rows(n)
    Wb, u0 = _backup("damping", n)
    start = S.ops.reset_state(n).cpu().numpy()
    thr, rthr = 0.35, 0.3
    host = S.Safe_ARS(S.builtin_cost, rthr, thr, [_oracle_env(S, O, p) for p in so], backup_policy=Wb,
                      backup_action=u0, lookahead=K)

    def host_rollout(W):
        W = W.reshape(n - 1, 2 * n + 2)
        st, total, over = start.copy(), 0.0, 0
        for _ in range(H):
            a = W @ st
            act = host.shielded_action(S.builtin_cost, thr, host.sim_env, list(st), a)
            if act is None:
                break
            over += act is not a
            r, st, _ = O.rollout(ro, O.GYM, 1, action=np.ascontiguousarray(act), init_state=st)
            total += r
        return total, over

    np.random.seed(2)
    W, curve, over = np.zeros((n - 1) * (2 * n + 2)), [], 0
    for it in range(n_iter):
        d = np.stack([2 * np.random.rand(n - 1, 2 * n + 2) - 1 for _ in range(N)]).reshape(N, -1)
        rets = []
        for k in range(N):
            for s in (1, -1):
                p = W + s * nu * d[k]
                r = rollout_safe_step_lookahead(O, ro, so, p, H, A, bb, thr, rthr, Wb, u0, K, start)
                assert _ok(r[6], thr) and _ok(r[7], rthr)
                got, o = host_rollout(p)
                assert o == r[5] and abs(got - r[0]) <= 1e-9 * max(1.0, abs(r[0]))
                rets.append(got)
                over += o
        curve.append(np.mean(rets))
        W, _ = O.update_policy(W, d, np.array(rets), b=b, alpha=alpha, semantics=1)
    assert over > 0
    ag = S.Safe_ARS(S.builtin_cost, rthr, thr, sims, backup_policy=Wb, backup_action=u0, lookahead=K)
    np.random.seed(2)
    with contextlib.redirect_stdout(io.StringIO()):
        got_curve, _ = ag.train(n_iter, real, N, b, alpha, nu, H)
    np.testing.assert_allclose(got_curve, curve, rtol=1e-6, atol=1e-10)
    assert rel_err(ag.policy.reshape(-1), W) < 1e-6
