"""Per-step screening with a shield (swm_rollout_shielded; ops.rollout with screen["backup"]; Safe_ARS with a backup)
against a CPU reference: rollout_safe_step_ensemble's loop with a backup action, every simulator and real step taken
by the oracle's own one-step rollout.

When the models reject the policy's action a = W s, the backup b = W_b s + u_0 is judged by every model by the same
rule; if it is safe the real step takes b (one override), otherwise the environment freezes for good.  The shielded
path leaves the unscreened one at its first override, so every threshold is accepted only if every deciding cost along
the reference's own path -- the ensemble maximum of the proposal at every step, of the backup where it was judged, and
the real cost of every step taken -- is at least MARGIN * max(1, |thr|) away from it: the exact checks of freeze
steps, override and violation counts then cannot flip on rounding."""
import contextlib
import ctypes
import functools
import io

import numpy as np
import pytest
import torch

from conftest import rel_err
from test_costed_screening import _affine_cost, builtin_rows, cost_rows
from test_ensemble_screening import _costs, _ensemble, _same, rollout_safe_step_ensemble
from test_step_screening import MARGIN, RET_TOL, STATE_TOL, _bits, _cuda, _midpoint, _population, _ret_err, _starts

gpu = pytest.mark.gpu
NEED = dict(never=2, over_h=2, over_frozen=2, frozen_first=1, violated=2)


# ---- backups and reference --------------------------------------------------------------------------------------------
def _backup(kind, n):
    """(W_b [n-1, 2n+2], u_0 [n-1]): zero torque; a damping controller of the joint velocities; a constant torque plus
    a small linear term."""
    na, no = n - 1, 2 * n + 2
    W, u0 = np.zeros((na, no)), np.zeros(na)
    if kind == "damping":
        for k in range(na):
            W[k, 3 + 2 * k], W[k, 5 + 2 * k] = 0.5, -0.5
    elif kind == "linear":
        rng = np.random.default_rng(77 + n)
        W = rng.uniform(-1, 1, (na, no)) * 0.05
        u0 = rng.uniform(-0.2, 0.2, na)
    return W, u0


def rollout_safe_step_shielded(O, real_p, sims, policy, H, A, b, sim_thresh, real_thresh, Wb, u0, init_state=None,
                               want_traj=False):
    """rollout_safe_step_ensemble with a shield.  -> (return, final state, trajectory [H, 2n+2] or None, violations,
    freeze step, overrides, deciding simulator costs, real costs of the steps taken, first rejection's backup
    rejected)."""
    n = real_p.n
    W = np.ascontiguousarray(policy, dtype=np.float64).reshape(n - 1, 2 * n + 2)
    st = O.rollout(real_p, O.GYM, 0, policy=W)[1] if init_state is None else np.array(init_state, dtype=np.float64)
    traj = np.zeros((H, 2 * n + 2)) if want_traj else None
    total, viol, frozen, over = 0.0, 0, H, 0
    sim_costs, real_costs, first_rejected = [], [], None
    for t in range(H):
        c = [_affine_cost(A, b, O.rollout(s, O.GYM, 1, policy=W, init_state=st)[1]) for s in sims]
        sim_costs.append(np.max(c))
        if all(x <= sim_thresh for x in c):
            r, st, _ = O.rollout(real_p, O.GYM, 1, policy=W, init_state=st)
        else:
            bu = np.ascontiguousarray(Wb @ st + u0)
            c = [_affine_cost(A, b, O.rollout(s, O.GYM, 1, action=bu, init_state=st)[1]) for s in sims]
            sim_costs.append(np.max(c))
            safe = all(x <= sim_thresh for x in c)
            if first_rejected is None:
                first_rejected = not safe
            if not safe:
                frozen = t
                if want_traj:
                    traj[t:] = st
                break
            r, st, _ = O.rollout(real_p, O.GYM, 1, action=bu, init_state=st)
            over += 1
        total += r
        real_costs.append(_affine_cost(A, b, st))
        if real_costs[-1] > real_thresh:
            viol += 1
        if want_traj:
            traj[t] = st
    return (total, st, traj, viol, frozen, over, np.array(sim_costs), np.array(real_costs), bool(first_rejected))


def _rows(kind, n):
    return builtin_rows(n) if kind == "builtin" else cost_rows(kind, n)


def _ok(sim_costs, thr):
    return not np.isfinite(thr) or (np.abs(np.asarray(sim_costs) - thr) >= MARGIN * max(1.0, abs(thr))).all()


def _population_spread(refs, H, need):
    fz = np.array([r[4] for r in refs])
    ov = np.array([r[5] for r in refs])
    viol = np.array([r[3] for r in refs])
    first = np.array([r[8] for r in refs])
    return ((ov == 0) & (fz == H)).sum() >= need["never"] and ((ov > 0) & (fz == H)).sum() >= need["over_h"] and \
        ((ov > 0) & (fz < H)).sum() >= need["over_frozen"] and \
        ((ov == 0) & (fz < H) & first).sum() >= need["frozen_first"] and (viol > 0).sum() >= need["violated"]


def _shield_thresholds(O, ro, so, pols, starts, H, A, b, Wb, u0, sc, need, quantiles=(0.5, 0.3, 0.7, 0.2, 0.8, 0.4, 0.6)):
    """Thresholds whose shielded reference has the required spread with every deciding cost at its margin.  The
    simulator threshold is taken between neighbouring unscreened ensemble costs; the path does not depend on the
    real threshold, which is then taken between neighbouring real costs of the steps taken.  -> (sim_thr, real_thr,
    references) or None."""
    for q in quantiles:
        s = _midpoint(sc, q)
        refs = [rollout_safe_step_shielded(O, ro, so, pols[e], H, A, b, s, np.inf, Wb, u0, starts[e], True)
                for e in range(len(pols))]
        if not all(_ok(r[6], s) for r in refs):
            continue
        taken = np.concatenate([r[7] for r in refs])
        if taken.size < 2:
            continue
        for rq in (0.8, 0.9, 0.7, 0.95, 0.6):
            r_thr = _midpoint(taken, rq)
            if not all(_ok(r[7], r_thr) for r in refs):
                continue
            refs2 = [x[:3] + (int((x[7] > r_thr).sum()),) + x[4:] for x in refs]
            if _population_spread(refs2, H, need):
                return s, r_thr, refs2
    return None


@functools.lru_cache(maxsize=None)
def _case(O, n, kind, backup, M, B=37, H=201):
    """Explicit policies, starts, cost, backup, thresholds and the shielded references with the required spread
    (oracle only): the first of a few seeded populations that gives it."""
    _, sims = _ensemble(O, n)
    ro = _ensemble(O, n)[0]
    A, b = _rows(kind, n)
    Wb, u0 = _backup(backup, n)
    for seed in range(6):
        W, init = _population(n, B, seed=500 + n + 1000 * seed)
        init[:, :2] *= 0.1
        sc, _ = _costs(O, n, W, init, H, A, b)
        found = _shield_thresholds(O, ro, sims[:M], W, init, H, A, b, Wb, u0, np.max(sc[:M], axis=0), NEED)
        if found is not None:
            return W, init, A, b, Wb, u0, found[0], found[1], found[2]
    raise AssertionError("no population gives the required spread for n=%d, %s, %s, M=%d" % (n, kind, backup, M))


# ---- CPU tests -------------------------------------------------------------------------------------------------------
def test_rollout_shielded_argument_checks(S):
    """Everything swm_rollout_ensemble refuses, with the same status, and a bad backup; no device needed."""
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

    def call(c, ms=good, M=3, forms=fp, J=len(F), bk=bp):
        return L.swm_rollout_shielded(ctypes.byref(real), ctypes.byref(c), ms, M, forms, J, bk, None, None)

    def ens(c, ms=good, M=3, forms=fp, J=len(F)):
        return L.swm_rollout_ensemble(ctypes.byref(real), ctypes.byref(c), ms, M, forms, J, None)

    bad, unsup = -1, -2
    for forms in (fp, None):
        cases = [dict(c=cfg(enabled=0)), dict(c=cfg(), M=0), dict(c=cfg(), M=17), dict(c=cfg(), ms=None),
                 dict(c=cfg(), ms=models(sims[:2] + [S.make_params(n=4)])), dict(c=cfg(H=-1)),
                 dict(c=cfg(rollouts_per_policy=0)), dict(c=cfg(B=63, policy_mode=S.ops.POLICY_PHILOX))]
        zero_l = S.make_params(n=n)
        zero_l.l_i = 0.0
        cases.append(dict(c=cfg(), ms=models([sims[0], zero_l]), M=2))
        for kw in cases:
            assert call(forms=forms, **kw) == bad == ens(forms=forms, **kw)
        dummy = (ctypes.c_double * 64)()
        for c in [cfg(kernel=k) for k in (S.KERNEL_LANES, S.KERNEL_LANES2, S.KERNEL_LANES3)] + [
                cfg(variant=S.RLGLUE), cfg(normalize=1), cfg(stats_partial=ctypes.cast(dummy, ctypes.c_void_p)),
                cfg(policy_mode=S.ops.POLICY_FIXED_ACTION), cfg(schedule_sub=2, schedule_chunk=64)]:
            assert call(c, forms=forms) == unsup == ens(c, forms=forms)
        assert call(cfg(B=0), forms=forms) == 0
        assert call(cfg(B=0), ms=models(sims), M=16, forms=forms) == 0
        # the backup: NULL or non-finite, also for an empty batch; checked after the forms, before the other checks
        assert call(cfg(), forms=forms, bk=None) == bad and call(cfg(B=0), forms=forms, bk=None) == bad
        for i in (0, Wb.size - 1, Wb.size, BK.size - 1):
            for v in (np.nan, np.inf, -np.inf):
                G = BK.copy(); G[i] = v
                gp = G.ctypes.data_as(ctypes.c_void_p)
                assert call(cfg(), forms=forms, bk=gp) == bad and call(cfg(B=0), forms=forms, bk=gp) == bad
                assert call(cfg(kernel=S.KERNEL_LANES), forms=forms, bk=gp) == bad
    assert call(cfg(), J=0) == bad and call(cfg(), J=33) == bad
    assert call(cfg(B=0), J=0, forms=None) == 0
    for v in (np.nan, np.inf, -np.inf):
        G = F.copy(); G[2, 4] = v
        assert call(cfg(), forms=G.ctypes.data_as(ctypes.c_void_p), bk=None) == bad  # the forms' error first


def test_safe_ars_backup_construction(S):
    n = 3
    real = S.SwimmerEnv("RealWorld", n=n)
    sim = S.SwimmerEnv("Simulator", n=n, l_i=1.01)
    Wb, u0 = _backup("linear", n)
    ag = S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sim)
    assert ag.backup is None and "backup" not in ag._screen(real)
    ag = S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sim, backup_policy=Wb, backup_action=u0)
    scr = ag._screen(real)
    assert np.array_equal(scr["backup"]["policy"], Wb) and np.array_equal(scr["backup"]["action"], u0)
    ag = S.Safe_ARS(S.builtin_cost, 1.0, 0.5, [sim, sim], backup_action=u0)
    assert not ag.backup["policy"].any() and np.array_equal(ag.backup["action"], u0)
    ag = S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sim, backup_policy=Wb)
    assert not ag.backup["action"].any()
    for kw in (dict(backup_policy=Wb.T), dict(backup_policy=Wb.reshape(-1)), dict(backup_action=u0[:1]),
               dict(backup_policy=np.zeros((n, 2 * n + 4))), dict(backup_action=np.zeros(n))):
        with pytest.raises(ValueError):
            S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sim, **kw)
    for v in (np.nan, np.inf, -np.inf):
        W2 = Wb.copy(); W2[1, 3] = v
        with pytest.raises(ValueError):
            S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sim, backup_policy=W2)
        u2 = u0.copy(); u2[0] = v
        with pytest.raises(ValueError):
            S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sim, backup_action=u2)
    with pytest.raises(ValueError):  # n of the simulator: the backup of a 4-segment swimmer
        S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sim, backup_policy=_backup("linear", 4)[0])


@pytest.mark.parametrize("kind,backup", [("builtin", "zero"), ("gdot", "damping"), ("builtin", "linear")])
def test_shielded_action_matches_reference_first_decision(S, O, kind, backup):
    """Safe_ARS.shielded_action (isSafe on each judgement) against the reference loop's first step, with simulator
    environments that step through the oracle (no device)."""
    n, M = 3, 3
    _, so = _ensemble(O, n)
    W, init, A, b, Wb, u0, thr, rthr, refs = _case(O, n, kind, backup, M)

    class OracleEnv(S.SwimmerEnv):
        def __init__(self, p):
            super().__init__("Simulator", n=n)
            self.p = p

        def next_observation(self, torque, G_dot, theta, theta_dot):
            s = O.step(self.p, O.GYM, self._pack(G_dot, theta, theta_dot), np.asarray(torque, dtype=np.float64))[0]
            return s[:2].copy(), s[2::2].copy(), s[3::2].copy()

    envs = [OracleEnv(p) for p in so[:M]]
    cost = S.builtin_cost if kind == "builtin" else S.MaxAffineCost(A, b)
    ag = S.Safe_ARS(cost, rthr, thr, envs, backup_policy=Wb, backup_action=u0)
    kinds = set()
    for e in range(len(W)):
        a = W[e] @ init[e]
        got = ag.shielded_action(cost, thr, envs, list(init[e]), a)
        ref = refs[e]
        if ref[4] == 0:
            assert got is None, e
            kinds.add("freeze")
        elif ref[5] > 0 and np.array_equal(ref[2][0], O.rollout(_ensemble(O, n)[0], O.GYM, 1, action=Wb @ init[e] + u0,
                                                                init_state=init[e])[1]):
            assert got is not a and np.array_equal(got, Wb @ init[e] + u0), e
            kinds.add("backup")
        else:
            assert got is a, e
            kinds.add("policy")
    assert "freeze" in kinds and "policy" in kinds


@pytest.mark.parametrize("n", [2, 6, 10])
def test_reference_with_unused_backup_equals_ensemble_reference(O, n):
    """With thresholds no proposal exceeds, the shielded reference is rollout_safe_step_ensemble bit for bit; with a
    cost of the next angles only (bending), whose one-step prediction no action changes, every rejected proposal has
    its backup rejected too and the shielded reference is again the ensemble reference."""
    ro, sims = _ensemble(O, n)
    W, init, A, b, Wb, u0, thr, rthr, _ = _case(O, n, "builtin", "zero", 2)
    Ab, bb = cost_rows("bend", n)
    for e in range(0, len(W), 4):
        for (AA, bbb, s_thr) in ((A, b, np.inf), (Ab, bb, 0.05)):
            got = rollout_safe_step_shielded(O, ro, sims[:2], W[e], 201, AA, bbb, s_thr, rthr, Wb, u0, init[e], True)
            want = rollout_safe_step_ensemble(O, ro, sims[:2], W[e], 201, AA, bbb, s_thr, rthr, init[e], True)
            assert got[5] == 0 and got[3:5] == want[3:5] and _bits([got[0]]) == _bits([want[0]])
            assert np.array_equal(_bits(got[1]), _bits(want[1])) and np.array_equal(_bits(got[2]), _bits(want[2]))


# ---- GPU tests -------------------------------------------------------------------------------------------------------
def _run(S, real, sims, H, kind, sim_thr, real_thr, Wb=None, u0=None, backup=True, **kw):
    screen = dict(sim_params=list(sims), sim_thresh=sim_thr, real_thresh=real_thr)
    if kind != "builtin":
        screen["cost"] = S.MaxAffineCost(*_rows(kind, real.n))
    if backup:
        screen["backup"] = dict(policy=Wb, action=u0)
    return S.ops.rollout(real, H, want_final=True, want_trajectory=True, screen=screen, **kw)


def _host(res):
    return (res.returns.cpu().numpy(), res.final_state.cpu().numpy(), res.trajectory.cpu().numpy(),
            res.frozen_at.cpu().numpy(), res.violations.cpu().numpy(), res.overrides.cpu().numpy())


def _compare(refs, res, H):
    got_r, got_f, traj, fz, viol, ov = _host(res)
    er = ef = et = 0.0
    for e, ref in enumerate(refs):
        r, f, t, v, z, o = ref[:6]
        assert (fz[e], viol[e], ov[e]) == (z, v, o), (e, fz[e], z, viol[e], v, ov[e], o)
        er = max(er, _ret_err(got_r[e], r))
        ef = max(ef, rel_err(got_f[e], f))
        et = max(et, rel_err(traj[:H, e], t[:H]) if H else 0.0)
    assert er < RET_TOL and ef < STATE_TOL and et < STATE_TOL, (er, ef, et)
    return er, ef, et


def _prefix_refs(O, ro, so, pols, starts, H, A, b, thr, rthr, Wb, u0):
    return [rollout_safe_step_shielded(O, ro, so, pols[e], H, A, b, thr, rthr, Wb, u0, starts[e], True)
            for e in range(len(pols))]


@gpu
@pytest.mark.parametrize("kind,backup", [("builtin", "zero"), ("gdot", "damping")])
@pytest.mark.parametrize("M", [1, 16])
@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 7, 8, 9, 10])
def test_shield_matches_oracle(S, O, n, M, kind, backup):
    """Explicit policies, B = 37, H = 201."""
    H = 201
    real, sims = _ensemble(S, n)
    W, init, A, b, Wb, u0, thr, rthr, refs = _case(O, n, kind, backup, M)
    res = _run(S, real, sims[:M], H, kind, thr, rthr, Wb, u0, policies=_cuda(W), init_state=_cuda(init))
    errs = _compare(refs, res, H)
    print("\n[shield] n=%d M=%d %s/%s: return %.2e, final %.2e, trajectory %.2e" % ((n, M, kind, backup) + errs))


@gpu
@pytest.mark.parametrize("kind", ["builtin", "gdot"])
@pytest.mark.parametrize("M", [2, 7])
@pytest.mark.parametrize("n", [3, 5, 10])
def test_shield_linear_backup_matches_oracle(S, O, n, M, kind):
    """A constant torque u_0 plus a linear term W_b."""
    H = 201
    real, sims = _ensemble(S, n)
    W, init, A, b, Wb, u0, thr, rthr, refs = _case(O, n, kind, "linear", M)
    res = _run(S, real, sims[:M], H, kind, thr, rthr, Wb, u0, policies=_cuda(W), init_state=_cuda(init))
    _compare(refs, res, H)


@gpu
@pytest.mark.parametrize("n,R,D", [(3, 1, 16), (3, 3, 8), (6, 32, 2), (6, 3, 8)])
def test_shield_policy_sources_match_oracle(S, O, n, R, D):
    """In-kernel Philox perturbations and the same read from memory (bit-identical), R = 1, 3 and 32."""
    H, nu, seed, it, dir0, M = 201, 0.3, 31 + n, 2, 5, 4
    B, ws = 2 * D * R, (n - 1) * (2 * n + 2)
    (real, sims), (ro, so) = _ensemble(S, n), _ensemble(O, n)
    _, _, A, b, Wb, u0, thr, rthr, _ = _case(O, n, "builtin", "zero", M)
    rng = np.random.default_rng(7 * n + R)
    Wbase = rng.uniform(-1, 1, ws) * 0.1
    count = B if R == 1 else R
    init = _starts(rng, n, count)
    pols = np.array([Wbase + (-nu if (e // R) & 1 else nu) * O.philox_delta(seed, it, dir0 + ((e // R) >> 1), ws)
                     for e in range(B)]).reshape(B, n - 1, 2 * n + 2)
    starts = np.array([init[e % count] for e in range(B)])
    refs = _prefix_refs(O, ro, so[:M], pols, starts, H, A, b, thr, rthr, Wb, u0)
    for r in refs:
        assert _ok(r[6], thr) and _ok(r[7], rthr)
    kw = dict(B=B, base_policy=_cuda(Wbase), nu=nu, seed=seed, iteration=it, dir0=dir0, rollouts_per_policy=R,
              init_state=_cuda(init))
    res = _run(S, real, sims[:M], H, "builtin", thr, rthr, Wb, u0, **kw)
    _compare(refs, res, H)
    mem = _run(S, real, sims[:M], H, "builtin", thr, rthr, Wb, u0,
               deltas=S.ops.philox_deltas(seed, it, dir0, D, ws), **kw)
    _same(mem, res, ("returns", "frozen_at", "violations", "overrides", "final_state", "trajectory"))


@gpu
@pytest.mark.parametrize("n", [3, 8])
@pytest.mark.parametrize("H", [0, 1, 63, 64, 201])
def test_shield_horizon_edges(S, O, n, H):
    """Short horizons on the 201-step case's thresholds (their margins hold for every prefix)."""
    ro, so = _ensemble(O, n)
    real, sims = _ensemble(S, n)
    W, init, A, b, Wb, u0, thr, rthr, _ = _case(O, n, "builtin", "zero", 2)
    refs = _prefix_refs(O, ro, so[:2], W, init, H, A, b, thr, rthr, Wb, u0)
    res = _run(S, real, sims[:2], H, "builtin", thr, rthr, Wb, u0, policies=_cuda(W), init_state=_cuda(init))
    _compare(refs, res, H)
    if H == 0:
        assert (res.frozen_at.cpu().numpy() == 0).all() and (res.overrides.cpu().numpy() == 0).all()


@gpu
@pytest.mark.parametrize("n", [3, 8])
def test_shield_dir_mask(S, n):
    D, R, H, M = 6, 2, 130, 4
    B, ws = 2 * D * R, (n - 1) * (2 * n + 2)
    real, sims = _ensemble(S, n)
    rng = np.random.default_rng(40 + n)
    init = _starts(rng, n, R)
    Wb, u0 = _backup("zero", n)
    thr = float(np.median(np.max(np.abs(init[:, 3::2]), axis=1))) + 0.05
    kw = dict(B=B, base_policy=_cuda(rng.uniform(-1, 1, ws) * 0.3), nu=0.8, seed=3, iteration=1,
              rollouts_per_policy=R, init_state=_cuda(init))
    full = _run(S, real, sims[:M], H, "builtin", thr, 0.8 * thr, Wb, u0, **kw)
    mask = torch.tensor([1, 0, 1, 1, 0, 1], dtype=torch.int32, device="cuda")
    out = {k: torch.full((B,), -7, dtype=torch.int32, device="cuda") for k in ("frozen_at", "violations", "overrides")}
    m = _run(S, real, sims[:M], H, "builtin", thr, 0.8 * thr, Wb, u0, dir_mask=mask, out=out, **kw)
    live = np.repeat(mask.cpu().numpy().astype(bool), 2 * R)
    assert (m.frozen_at.cpu().numpy()[~live] == H).all() and (m.violations.cpu().numpy()[~live] == 0).all()
    assert (m.overrides.cpu().numpy()[~live] == 0).all() and np.isnan(m.returns.cpu().numpy()[~live]).all()
    lv = torch.as_tensor(live, device="cuda")
    for k in ("returns", "frozen_at", "violations", "overrides", "final_state"):
        assert torch.equal(getattr(m, k)[lv], getattr(full, k)[lv]), k


@gpu
@pytest.mark.parametrize("kind", ["builtin", "gdot"])
@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 7, 8, 9, 10])
def test_shield_exact_against_ensemble_path(S, O, n, kind):
    """No oracle: (1) a backup equal to the policy (one base policy, nu = 0) never overrides and every output is the
    ensemble path's bit for bit; (2) in a mixed batch every environment without overrides is the ensemble path's bit
    for bit, and one with overrides follows it bit for bit up to that path's freeze step, where it first overrides;
    (3) permuting the environments permutes the results."""
    H, M = 201, 7
    real, sims = _ensemble(S, n)
    W, init, A, b, Wb, u0, thr, rthr, _ = _case(O, n, kind, "damping" if kind == "gdot" else "zero", 1)
    kw = dict(policies=_cuda(W), init_state=_cuda(init))
    ens = _run(S, real, sims[:M], H, kind, thr, rthr, backup=False, **kw)
    # (1)
    B = len(W)
    big = W[int(np.argmax(np.abs(W).reshape(B, -1).sum(axis=1)))]  # the largest policy: some of its rollouts freeze
    pkw = dict(B=2 * B, base_policy=_cuda(big.reshape(-1)), nu=0.0, init_state=_cuda(np.repeat(init, 2, axis=0)))
    same = _run(S, real, sims[:M], H, kind, thr, rthr, big, None, **pkw)
    plain = _run(S, real, sims[:M], H, kind, thr, rthr, backup=False, **pkw)
    _same(same, plain)
    assert (same.overrides.cpu().numpy() == 0).all() and (same.frozen_at.cpu().numpy() < H).any()
    # (2)
    sh = _run(S, real, sims[:M], H, kind, thr, rthr, Wb, u0, **kw)
    ov, fz_e = sh.overrides.cpu().numpy(), ens.frozen_at.cpu().numpy()
    assert (ov == 0).any() and (ov > 0).any()
    t_sh, t_en = sh.trajectory.cpu().numpy(), ens.trajectory.cpu().numpy()
    for e in range(B):
        if ov[e] == 0:
            for k in ("returns", "frozen_at", "violations", "final_state"):
                assert torch.equal(getattr(sh, k)[e], getattr(ens, k)[e]), (e, k)
            assert np.array_equal(_bits(t_sh[:, e]), _bits(t_en[:, e])), e
        else:
            f = int(fz_e[e])
            assert f < H and np.array_equal(_bits(t_sh[:f, e]), _bits(t_en[:f, e])), e
            # the backup was taken at step f: the state after it differs from the held state of the ensemble path
            assert not np.array_equal(_bits(t_sh[f, e]), _bits(t_en[f, e])), e
    # (3)
    p = np.random.default_rng(n).permutation(B)
    perm = _run(S, real, sims[:M], H, kind, thr, rthr, Wb, u0, policies=_cuda(W[p]), init_state=_cuda(init[p]))
    pt = torch.as_tensor(p, device="cuda")
    for k in ("returns", "frozen_at", "violations", "overrides", "final_state"):
        assert torch.equal(getattr(perm, k), getattr(sh, k)[pt]), k
    assert torch.equal(perm.trajectory, sh.trajectory[:, pt])


@gpu
@pytest.mark.parametrize("n", [3, 8])
def test_engine_shield_graph_equals_eager(S, O, n):
    """ArsEngine(step_screen=... backup ...): graph-replayed iterations equal eager ones bit for bit, and
    eng.last.overrides counts the backup steps."""
    N, b, H, nu, alpha, seed, M = 8, 4, 150, 0.3, 0.02, 21, 3
    real, sims = _ensemble(S, n)
    ws = (n - 1) * (2 * n + 2)
    W0 = np.random.default_rng(n).uniform(-1, 1, ws) * 0.3
    Wb, u0 = _backup("zero", n)
    thr = 0.5
    screen = dict(sim_params=sims[:M], sim_thresh=thr, real_thresh=0.4, backup=dict(policy=Wb, action=u0))
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
def test_safe_ars_train_with_backup(S, O):
    """Safe_ARS(..., backup_policy, backup_action).train with numpy deltas against an oracle ARS loop on
    rollout_safe_step_shielded (built-in cost, two models)."""
    n, N, b, alpha, nu, H, n_iter = 3, 3, 2, 0.02, 0.3, 150, 2
    consts = [dict(m_i=1.05, l_i=0.95, k=9.5), dict(m_i=0.97, l_i=1.02, k=10.4)]
    real = S.SwimmerEnv("RealWorld", n=n)
    sims = [S.SwimmerEnv("Simulator", n=n, **c) for c in consts]
    ro = O.make_params(n=n)
    so = [O.make_params(n=n, **c) for c in consts]
    A, bb = builtin_rows(n)
    Wb, u0 = _backup("linear", n)
    start = S.ops.reset_state(n).cpu().numpy()

    def loop(thr, rthr, check):
        np.random.seed(2)
        W, curve, over = np.zeros((n - 1) * (2 * n + 2)), [], 0
        for it in range(n_iter):
            d = np.stack([2 * np.random.rand(n - 1, 2 * n + 2) - 1 for _ in range(N)]).reshape(N, -1)
            rets = []
            for k in range(N):
                for s in (1, -1):
                    r = rollout_safe_step_shielded(O, ro, so, W + s * nu * d[k], H, A, bb, thr, rthr, Wb, u0, start)
                    if check:
                        assert _ok(r[6], thr) and _ok(r[7], rthr)
                    rets.append(r[0])
                    over += r[5]
            curve.append(np.mean(rets))
            W, _ = O.update_policy(W, d, np.array(rets), b=b, alpha=alpha, semantics=1)
        return np.array(curve), W, over

    thr, rthr = 0.35, 0.3
    want, W, over = loop(thr, rthr, True)
    assert over > 0
    ag = S.Safe_ARS(S.builtin_cost, rthr, thr, sims, backup_policy=Wb, backup_action=u0)
    np.random.seed(2)
    with contextlib.redirect_stdout(io.StringIO()):
        curve, _ = ag.train(n_iter, real, N, b, alpha, nu, H)
    np.testing.assert_allclose(curve, want, rtol=1e-6, atol=1e-10)
    assert rel_err(ag.policy.reshape(-1), W) < 1e-6
