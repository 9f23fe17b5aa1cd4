"""Per-step screening by an ensemble of simulator models (swm_rollout_ensemble; ops.rollout with a list of
sim_params; Safe_ARS with a list of simulator environments) against a CPU reference: rollout_safe_step_affine's loop
restated with a list of models, every simulator and real step taken by the oracle's own one-step rollout.

Before every real step each model takes one simulator step from the same state with the same action; the real step
is taken only if the cost of every model's next observation is <= sim_thresh, otherwise the environment freezes for
good.  The built-in cost max_i |thd_i| is the max-of-affine cost with the rows +-e_{3+2i} (bit for bit, see
test_costed_screening.py).  As in the other screening tests, every threshold sits between neighbouring costs of the
oracle's own rollouts and every deciding cost is asserted to be at least MARGIN * max(1, |thr|) away from it, so the
exact checks of freeze steps and violation counts cannot flip on rounding.  The ensemble's decision depends on the
largest of its models' costs only, so the margins are taken on that maximum."""
import contextlib
import ctypes
import functools
import io

import numpy as np
import pytest
import torch

from conftest import rel_err
from test_costed_screening import (_affine_cost, _freeze_steps, _margins_ok, builtin_rows, cost_rows,
                                   rollout_safe_step_affine)
from test_step_screening import (MARGIN, RET_TOL, STATE_TOL, _bits, _cuda, _midpoint, _models, _population,
                                 _ret_err, _spread, _starts)

gpu = pytest.mark.gpu
KINDS = ["builtin", "bend", "gdot", "dense32"]
MS = [1, 2, 7, 16]
NEED = dict(zero=2, mid=4, mid_steps=3, never=2, violated=2)


# ---- models and reference ---------------------------------------------------------------------------------------
def _ensemble(mod, n):
    """The real model and 16 simulator models: the first is test_step_screening's simulator, the others spread
    around it by up to +-6 % in l, m, k and h.  An ensemble of M models is the first M, so that the sets nest."""
    real, sim = _models(mod, n)
    rng = np.random.default_rng(4242)
    sims = [sim]
    for _ in range(15):
        f = 1.0 + rng.uniform(-0.06, 0.06, 4)
        sims.append(mod.make_params(n=n, l_i=.93 * f[0], m_i=1.05 * f[1], k=9.9 * f[2], h=0.0012 * f[3],
                                    direction=(.6, .8)))
    return real, sims


def rollout_safe_step_ensemble(O, real_p, sims, policy, H, A, b, sim_thresh, real_thresh, init_state=None,
                               want_traj=False):
    """rollout_safe_step_affine with a list of simulator models: the real step is taken only if every model's one-step
    oracle rollout from the current state has cost <= sim_thresh.  Once frozen the state and the policy never change
    again, so the rest of the horizon is the held state (the loop would repeat the same decision H - t times).
    -> (return, final state, trajectory [H, 2n+2] or None, violations, freeze step)."""
    n = real_p.n
    W = np.ascontiguousarray(policy, dtype=np.float64).reshape(n - 1, 2 * n + 2)
    st = O.rollout(real_p, O.GYM, 0, policy=W)[1] if init_state is None else np.array(init_state, dtype=np.float64)
    traj = np.zeros((H, 2 * n + 2)) if want_traj else None
    total, viol, frozen = 0.0, 0, H
    for t in range(H):
        if all(_affine_cost(A, b, O.rollout(s, O.GYM, 1, policy=W, init_state=st)[1]) <= sim_thresh for s in sims):
            r, st, _ = O.rollout(real_p, O.GYM, 1, policy=W, init_state=st)
            total += r
            if _affine_cost(A, b, st) > real_thresh:
                viol += 1
        else:
            frozen = t
            if want_traj:
                traj[t:] = st
            break
        if want_traj:
            traj[t] = st
    return total, st, traj, viol, frozen


def _rows(kind, n):
    return builtin_rows(n) if kind == "builtin" else cost_rows(kind, n)


@functools.lru_cache(maxsize=None)
def _next_states(O, n, W_bytes, init_bytes, B, H):
    """Along the UNSCREENED oracle rollout of every environment: the state before every step, the real post-step
    state and every model's one-step prediction from the state before the step.  -> (real [B, H, no], sims
    [16, B, H, no]).  The screened rollout follows the unscreened one up to and including its freeze step."""
    ro, sims = _ensemble(O, n)
    no = 2 * n + 2
    W = np.frombuffer(W_bytes).reshape(B, n - 1, no)
    init = np.frombuffer(init_bytes).reshape(B, no)
    real = np.zeros((B, H, no))
    nxt = np.zeros((len(sims), B, H, no))
    for e in range(B):
        _, _, real[e] = O.rollout(ro, O.GYM, H, policy=W[e], init_state=init[e], want_traj=True)
        pre = np.vstack([init[e][None], real[e, :-1]])
        for m, so in enumerate(sims):
            nxt[m, e] = O.step_batch(so, O.GYM, pre, pre @ W[e].T)[0]
    return real, nxt


def _costs(O, n, W, init, H, A, b):
    """Simulator costs [16, B, H] of every model before every step and real costs [B, H] after it."""
    real, nxt = _next_states(O, n, np.ascontiguousarray(W).tobytes(), np.ascontiguousarray(init).tobytes(),
                             len(W), H)
    return np.max(nxt @ A.T + b, axis=-1), np.max(real @ A.T + b, axis=-1)


def _ens_thresholds(sc, rc, M, quantiles=np.linspace(0.05, 0.995, 200), other=False, **need):
    """Thresholds for the first M models (their cost maximum decides) with the required spread of freeze steps and,
    with `other`, at least one environment that freezes earlier than the first model alone would make it."""
    H = rc.shape[1]
    ens = np.max(sc[:M], axis=0)
    for q in quantiles:
        s = _midpoint(ens, q)
        fz = _freeze_steps(ens, s)
        if other and not (fz < _freeze_steps(sc[0], s)).any():
            continue
        taken = np.concatenate([rc[e, :fz[e]] for e in range(len(fz))])
        if taken.size < 2:
            continue
        for rq in (0.8, 0.9, 0.7, 0.95, 0.6, 0.5):
            r = _midpoint(taken, rq)
            viol = np.array([(rc[e, :fz[e]] > r).sum() for e in range(len(fz))])
            if _spread(fz, viol, H, **need):
                assert _margins_ok(ens, rc, s, r)
                return s, r
    raise AssertionError("this population does not give the required spread of freeze steps")


@functools.lru_cache(maxsize=None)
def _case(O, n, kind, M, B=37, H=201):
    """Explicit policies, starts, the cost and thresholds with the required spread (oracle only): the first of a
    few seeded populations that gives it, for M >= 2 preferably one where another model than the first stops an
    environment (two models can be ordered for a cost: the bending cost of the next angles only sees h)."""
    A, b = _rows(kind, n)
    for other in ((True, False) if M > 1 else (False,)):
        for seed in range(6):
            W, init = _population(n, B, seed=300 + n + 1000 * seed)
            init[:, :2] *= 0.1
            sc, rc = _costs(O, n, W, init, H, A, b)
            try:
                sim_thr, real_thr = _ens_thresholds(sc, rc, M, other=other, **NEED)
            except AssertionError:
                continue
            return W, init, A, b, sim_thr, real_thr
    raise AssertionError("no population gives the required spread for n=%d, %s, M=%d" % (n, kind, M))


# ---- CPU tests -------------------------------------------------------------------------------------------------------
def test_rollout_ensemble_argument_checks(S):
    """Rejected before anything is launched: no device needed."""
    L = S._lib.lib()
    n = 3
    real, sims = _ensemble(S, n)
    A, b = builtin_rows(n)
    F = np.ascontiguousarray(np.hstack([A, b[:, None]]))
    fp = F.ctypes.data_as(ctypes.c_void_p)

    def cfg(**kw):
        c = S._lib.SwmRollout()
        c.variant, c.policy_mode, c.H, c.B, c.rollouts_per_policy = S.GYM, S.ops.POLICY_EXPLICIT, 10, 64, 1
        c.screen.enabled = 1  # screen.sim stays zero: it is not read
        for k, v in kw.items():
            if k == "enabled":
                c.screen.enabled = v
            else:
                setattr(c, k, v)
        return c

    def models(ps):
        return (S._lib.SwmParams * len(ps))(*ps)

    good = models(sims[:3])

    def call(c, ms=good, M=3, forms=fp, J=len(F)):
        return L.swm_rollout_ensemble(ctypes.byref(real), ctypes.byref(c), ms, M, forms, J, None)

    bad, unsup = -1, -2
    for forms in (fp, None):
        assert call(cfg(enabled=0), forms=forms) == bad
        assert call(cfg(), M=0, forms=forms) == bad and call(cfg(), M=17, forms=forms) == bad
        assert call(cfg(), ms=None, forms=forms) == bad
        assert call(cfg(), ms=models(sims[:2] + [S.make_params(n=4)]), forms=forms) == bad
        zero_l = S.make_params(n=n)
        zero_l.l_i = 0.0
        assert call(cfg(), ms=models([sims[0], zero_l]), M=2, forms=forms) == bad
        assert call(cfg(H=-1), forms=forms) == bad and call(cfg(rollouts_per_policy=0), forms=forms) == bad
        assert call(cfg(B=63, policy_mode=S.ops.POLICY_PHILOX), forms=forms) == bad
        for k in (S.KERNEL_LANES, S.KERNEL_LANES2, S.KERNEL_LANES3):
            assert call(cfg(kernel=k), forms=forms) == unsup
        assert call(cfg(variant=S.RLGLUE), forms=forms) == unsup
        assert call(cfg(normalize=1), forms=forms) == unsup
        dummy = (ctypes.c_double * 64)()
        assert call(cfg(stats_partial=ctypes.cast(dummy, ctypes.c_void_p)), forms=forms) == unsup
        assert call(cfg(policy_mode=S.ops.POLICY_FIXED_ACTION), forms=forms) == unsup
        assert call(cfg(schedule_sub=2, schedule_chunk=64), forms=forms) == unsup
        # an empty batch is accepted without a device; cfg->screen.sim (all zero here) is not looked at
        assert call(cfg(B=0), forms=forms) == 0
        assert call(cfg(B=0), ms=models(sims), M=16, forms=forms) == 0
    assert call(cfg(), J=0) == bad and call(cfg(), J=33) == bad
    assert call(cfg(B=0), J=0, forms=None) == 0  # n_forms is ignored without forms
    for v in (np.nan, np.inf, -np.inf):
        G = F.copy(); G[2, 4] = v
        assert call(cfg(), forms=G.ctypes.data_as(ctypes.c_void_p)) == bad


def test_safe_ars_ensemble_construction(S):
    real = S.SwimmerEnv("RealWorld", n=3)
    sims = [S.SwimmerEnv("Simulator", n=3, l_i=1.0 + 0.01 * i) for i in range(3)]
    ag = S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sims)
    scr = ag._screen(real)
    assert isinstance(scr["sim_params"], list) and len(scr["sim_params"]) == 3 and "cost" not in scr
    assert [p.l_i for p in scr["sim_params"]] == [e.l_i for e in sims]
    A, b = cost_rows("bend", 3)
    ag = S.Safe_ARS(S.MaxAffineCost(A, b), 1.0, 0.5, tuple(sims))
    assert ag._screen(real)["cost"] is ag.cost
    with pytest.raises(ValueError):
        S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sims + [S.SwimmerEnv("Simulator", n=4)])
    with pytest.raises(ValueError):
        S.Safe_ARS(S.builtin_cost, 1.0, 0.5, [])
    with pytest.raises(ValueError):
        S.Safe_ARS(S.builtin_cost, 1.0, 0.5, [S.SwimmerEnv("Simulator", n=3)] * 17)
    with pytest.raises(ValueError):
        S.Safe_ARS(S.MaxAffineCost(*cost_rows("bend", 4)), 1.0, 0.5, sims)
    with pytest.raises(ValueError):
        S.Safe_ARS(S.builtin_cost, 1.0, 0.5, sims)._screen(S.SwimmerEnv("RealWorld", n=4))
    assert len(S.Safe_ARS(S.builtin_cost, 1.0, 0.5, [sims[0]] * 16).sim_env) == 16


@pytest.mark.parametrize("n", [2, 6, 10])
def test_reference_ensemble_of_one_equals_single_model_reference(O, n):
    """The ensemble reference with one model is rollout_safe_step_affine bit for bit."""
    ro, sims = _ensemble(O, n)
    W, init, A, b, sim_thr, real_thr = _case(O, n, "bend", 1)
    for e in range(0, len(W), 3):
        got = rollout_safe_step_ensemble(O, ro, sims[:1], W[e], 201, A, b, sim_thr, real_thr, init[e], True)
        want = rollout_safe_step_affine(O, ro, sims[0], W[e], 201, A, b, sim_thr, real_thr, init[e], True)
        assert got[3:] == want[3:] and _bits([got[0]]) == _bits([want[0]])
        assert np.array_equal(_bits(got[1]), _bits(want[1])) and np.array_equal(_bits(got[2]), _bits(want[2]))


# ---- GPU tests -------------------------------------------------------------------------------------------------------
def _run(S, real, sims, H, kind, sim_thr, real_thr, kernel=0, **kw):
    screen = dict(sim_params=list(sims), sim_thresh=sim_thr, real_thresh=real_thr)
    if kind != "builtin":
        screen["cost"] = S.MaxAffineCost(*_rows(kind, real.n))
    return S.ops.rollout(real, H, want_final=True, want_trajectory=True, kernel=kernel, screen=screen, **kw)


def _host(res):
    return (res.returns.cpu().numpy(), res.final_state.cpu().numpy(), res.trajectory.cpu().numpy(),
            res.frozen_at.cpu().numpy(), res.violations.cpu().numpy())


def _compare(O, ro, sims, pols, starts, H, A, b, sim_thr, real_thr, res):
    got_r, got_f, traj, fz, viol = _host(res)
    er = ef = et = 0.0
    for e in range(len(got_r)):
        r, f, t, v, z = rollout_safe_step_ensemble(O, ro, sims, pols[e], H, A, b, sim_thr, real_thr, starts[e], True)
        assert (fz[e], viol[e]) == (z, v), (e, fz[e], z, viol[e], v)
        er = max(er, _ret_err(got_r[e], r))
        ef = max(ef, rel_err(got_f[e], f))
        et = max(et, rel_err(traj[:, e], t) if H else 0.0)
    assert er < RET_TOL and ef < STATE_TOL and et < STATE_TOL, (er, ef, et)
    return er, ef, et


def _frozen_tail(res, starts, H):
    """From the freeze on every stored state is the state before it, bit for bit."""
    _, fin, traj, fz, _ = _host(res)
    for e in range(fin.shape[0]):
        f = int(fz[e])
        if f == H:
            continue
        held = starts[e] if f == 0 else traj[f - 1, e]
        assert np.array_equal(_bits(traj[f:, e]), np.broadcast_to(_bits(held), traj[f:, e].shape)), e
        assert np.array_equal(_bits(fin[e]), _bits(held)), e


def _same(a, c, keys=("returns", "frozen_at", "violations", "final_state", "trajectory")):
    for k in keys:
        assert torch.equal(getattr(a, k), getattr(c, k)), k


@gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("M", MS)
@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 7, 8, 9, 10])
def test_ensemble_screening_matches_oracle(S, O, n, M, kind):
    """Explicit policies, B = 37, H = 201 (odd; crosses the sine/cosine re-evaluations at steps 63, 127, 191)."""
    H = 201
    (real, sims), (ro, so) = _ensemble(S, n), _ensemble(O, n)
    W, init, A, b, sim_thr, real_thr = _case(O, n, kind, M)
    res = _run(S, real, sims[:M], H, kind, sim_thr, real_thr, policies=_cuda(W), init_state=_cuda(init))
    errs = _compare(O, ro, so[:M], W, init, H, A, b, sim_thr, real_thr, res)
    _frozen_tail(res, init, H)
    fz = res.frozen_at.cpu().numpy()
    assert _spread(fz, res.violations.cpu().numpy(), H, **NEED)
    if M >= 7:  # some environment is stopped by a model other than the first
        sc, _ = _costs(O, n, W, init, H, A, b)
        assert (fz < _freeze_steps(sc[0], sim_thr)).any()
    print("\n[ensemble screening] n=%d M=%d %s: return %.2e, final %.2e, trajectory %.2e" % ((n, M, kind) + errs))


@gpu
@pytest.mark.parametrize("kind", ["builtin", "bend"])
@pytest.mark.parametrize("n,R,D", [(3, 1, 16), (5, 3, 8), (5, 32, 2), (8, 3, 8), (10, 32, 2)])
def test_ensemble_policy_sources_match_oracle(S, O, n, R, D, kind):
    """In-kernel Philox perturbations and the same read from memory (bit-identical), R = 1, 3 and 32 (32: one policy
    copy per warp), seven models."""
    H, nu, seed, it, dir0, M = 201, 0.3, 31 + n, 2, 5, 7
    B, ws = 2 * D * R, (n - 1) * (2 * n + 2)
    (real, sims), (ro, so) = _ensemble(S, n), _ensemble(O, n)
    A, b = _rows(kind, n)
    rng = np.random.default_rng(7 * n + R)
    Wb = rng.uniform(-1, 1, ws) * 0.05
    count = B if R == 1 else R
    init = _starts(rng, n, count)
    pols = np.array([Wb + (-nu if (e // R) & 1 else nu) * O.philox_delta(seed, it, dir0 + ((e // R) >> 1), ws)
                     for e in range(B)]).reshape(B, n - 1, 2 * n + 2)
    starts = np.array([init[e % count] for e in range(B)])
    sc, rc = _costs(O, n, pols, starts, H, A, b)
    sim_thr, real_thr = _ens_thresholds(sc, rc, M, other=True, zero=0, mid=2, mid_steps=2, never=1, violated=1)
    kw = dict(B=B, base_policy=_cuda(Wb), nu=nu, seed=seed, iteration=it, dir0=dir0, rollouts_per_policy=R,
              init_state=_cuda(init))
    res = _run(S, real, sims[:M], H, kind, sim_thr, real_thr, **kw)
    _compare(O, ro, so[:M], pols, starts, H, A, b, sim_thr, real_thr, res)
    _frozen_tail(res, starts, H)
    mem = _run(S, real, sims[:M], H, kind, sim_thr, real_thr, deltas=S.ops.philox_deltas(seed, it, dir0, D, ws), **kw)
    _same(mem, res)


@gpu
@pytest.mark.parametrize("kind", ["builtin", "dense32"])
@pytest.mark.parametrize("n", [3, 8])
@pytest.mark.parametrize("H", [0, 1, 63, 64, 65])
def test_ensemble_horizon_edges(S, O, n, H, kind):
    """Short horizons around the unroll and the sine/cosine re-evaluation step, on the 201-step case's thresholds
    (their margins hold for every prefix)."""
    (real, sims), (ro, so) = _ensemble(S, n), _ensemble(O, n)
    W, init, A, b, sim_thr, real_thr = _case(O, n, kind, 7)
    res = _run(S, real, sims[:7], H, kind, sim_thr, real_thr, policies=_cuda(W), init_state=_cuda(init))
    _compare(O, ro, so[:7], W, init, H, A, b, sim_thr, real_thr, res)
    _frozen_tail(res, init, H)
    if H == 0:
        assert (res.frozen_at.cpu().numpy() == 0).all() and (res.returns.cpu().numpy() == 0.0).all()
        assert np.array_equal(_bits(res.final_state.cpu().numpy()), _bits(init))


@gpu
@pytest.mark.parametrize("kind", ["builtin", "bend"])
@pytest.mark.parametrize("n", [3, 8])
def test_ensemble_dir_mask(S, O, n, kind):
    D, R, H, M = 6, 2, 130, 4
    B, ws = 2 * D * R, (n - 1) * (2 * n + 2)
    real, sims = _ensemble(S, n)
    rng = np.random.default_rng(40 + n)
    init = _starts(rng, n, R)
    A, b = _rows(kind, n)
    thr = float(np.median([_affine_cost(A, b, x) for x in init])) + 0.05
    kw = dict(B=B, base_policy=_cuda(rng.uniform(-1, 1, ws) * 0.05), nu=0.8, seed=3, iteration=1,
              rollouts_per_policy=R, init_state=_cuda(init))
    full = _run(S, real, sims[:M], H, kind, thr, 0.8 * thr, **kw)
    mask = torch.tensor([1, 0, 1, 1, 0, 1], dtype=torch.int32, device="cuda")
    out = {"frozen_at": torch.full((B,), -7, dtype=torch.int32, device="cuda"),
           "violations": torch.full((B,), -9, dtype=torch.int32, device="cuda")}
    m = _run(S, real, sims[:M], H, kind, thr, 0.8 * thr, dir_mask=mask, out=out, **kw)
    live = np.repeat(mask.cpu().numpy().astype(bool), 2 * R)
    assert (m.frozen_at.cpu().numpy()[~live] == H).all() and (m.violations.cpu().numpy()[~live] == 0).all()
    assert np.isnan(m.returns.cpu().numpy()[~live]).all()
    lv = torch.as_tensor(live, device="cuda")
    for k in ("returns", "frozen_at", "violations", "final_state"):
        assert torch.equal(getattr(m, k)[lv], getattr(full, k)[lv]), k


@gpu
@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 7, 8, 9, 10])
def test_ensemble_of_one_is_the_single_model_path(S, O, n):
    """M = 1 is swm_rollout (THREAD) with the built-in cost and swm_rollout_costed with an affine cost, bit for bit."""
    H = 201
    real, sims = _ensemble(S, n)
    for kind in ("builtin", "bend", "dense32"):
        W, init, A, b, thr, rthr = _case(O, n, kind, 1)
        kw = dict(policies=_cuda(W), init_state=_cuda(init), want_final=True, want_trajectory=True)
        screen = dict(sim_params=sims[0], sim_thresh=thr, real_thresh=rthr)
        if kind != "builtin":
            screen["cost"] = S.MaxAffineCost(A, b)
        single = S.ops.rollout(real, H, kernel=S.KERNEL_THREAD, screen=screen, **kw)
        for kern in (S.KERNEL_THREAD, S.KERNEL_AUTO):
            _same(S.ops.rollout(real, H, kernel=kern, screen=dict(screen, sim_params=[sims[0]]), **kw), single)


@gpu
@pytest.mark.parametrize("kind", ["builtin", "gdot"])
@pytest.mark.parametrize("n", [3, 5, 9])
def test_ensemble_duplicates_order_and_nesting(S, O, n, kind):
    """[a, a] = [a]; any order of the models gives the same result; adding models never moves a freeze later, and up
    to the earlier freeze the trajectories agree bit for bit."""
    H = 201
    real, sims = _ensemble(S, n)
    W, init, A, b, thr, rthr = _case(O, n, kind, 7)
    kw = dict(policies=_cuda(W), init_state=_cuda(init))
    one = _run(S, real, sims[:1], H, kind, thr, rthr, **kw)
    _same(_run(S, real, [sims[0], sims[0]], H, kind, thr, rthr, **kw), one)
    _same(_run(S, real, [sims[3]] * 5, H, kind, thr, rthr, **kw), _run(S, real, [sims[3]], H, kind, thr, rthr, **kw))
    seven = _run(S, real, sims[:7], H, kind, thr, rthr, **kw)
    rng = np.random.default_rng(n)
    for p in (list(reversed(range(7))), list(rng.permutation(7)), [6, 0, 5, 1, 4, 2, 3]):
        _same(_run(S, real, [sims[i] for i in p], H, kind, thr, rthr, **kw), seven)
    runs = [(M, _run(S, real, sims[:M], H, kind, thr, rthr, **kw)) for M in (1, 2, 4, 7, 12, 16)]
    moved = False
    for (_, a), (_, c) in zip(runs, runs[1:]):
        fa, fc = a.frozen_at.cpu().numpy(), c.frozen_at.cpu().numpy()
        assert (fc <= fa).all()
        moved |= bool((fc < fa).any())
        ta, tc = a.trajectory.cpu().numpy(), c.trajectory.cpu().numpy()
        for e in range(len(fa)):
            f = int(min(fa[e], fc[e]))
            assert np.array_equal(_bits(ta[:f, e]), _bits(tc[:f, e])), e
    assert moved


@gpu
@pytest.mark.parametrize("n", [3, 8])
def test_engine_ensemble_screening_matches_oracle_loop(S, O, n):
    """ArsEngine(step_screen=dict(sim_params=[...], ...)) for three iterations against the oracle loop; eager and
    graph replay bit-identical."""
    N, b, H, nu, alpha, seed, M = 8, 4, 150, 0.3, 0.02, 21, 3
    (real, sims), (ro, so) = _ensemble(S, n), _ensemble(O, n)
    ws = (n - 1) * (2 * n + 2)
    A, bb = cost_rows("bend", n)
    W0 = np.random.default_rng(n).uniform(-1, 1, ws) * 0.3
    start = S.ops.reset_state(n).cpu().numpy()

    def directions(W, it):
        deltas = np.stack([O.philox_delta(seed, it, k, ws) for k in range(N)])
        return deltas, np.array([W + s * nu * deltas[k] for k in range(N) for s in (+1, -1)])

    def costs(pols):
        return _costs(O, n, pols.reshape(len(pols), n - 1, -1), np.tile(start, (len(pols), 1)), H, A, bb)

    _, pols = directions(W0, 0)
    sc, rc = costs(pols)
    sim_thr, real_thr = _ens_thresholds(sc, rc, M, zero=0, mid=2, mid_steps=2, never=1, violated=1)
    screen = dict(sim_params=sims[:M], sim_thresh=sim_thr, real_thresh=real_thr, cost=S.MaxAffineCost(A, bb))
    engines = [S.ArsEngine(real, N=N, b=b, alpha=alpha, nu=nu, H=H, semantics=S.ARS_TOPB, seed=seed,
                           distributed=False, initial_policy=W0, step_screen=screen, use_graph=g) for g in (False, True)]
    W, frozen = W0, []
    for it in range(3):
        got = [e.run_iteration().clone() for e in engines]
        fz, viol = engines[0].last.frozen_at.cpu().numpy(), engines[0].last.violations.cpu().numpy()
        deltas, pols = directions(W, it)
        sc, rc = costs(pols)
        assert _margins_ok(np.max(sc[:M], axis=0), rc, sim_thr, real_thr), it
        rets = []
        for e, p in enumerate(pols):
            r, _, _, v, z = rollout_safe_step_ensemble(O, ro, so[:M], p, H, A, bb, sim_thr, real_thr)
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
def test_safe_ars_train_with_ensemble(S, O):
    """Safe_ARS([sim_a, sim_b, sim_c]).train with numpy deltas against the same oracle loop (built-in cost)."""
    n, N, b, alpha, nu, H, n_iter = 3, 3, 2, 0.02, 0.3, 150, 2
    consts = [dict(m_i=1.05, l_i=0.95, k=9.5), dict(m_i=0.97, l_i=1.02, k=10.4), dict(m_i=1.01, l_i=0.9, k=9.8)]
    real = S.SwimmerEnv("RealWorld", n=n)
    sims = [S.SwimmerEnv("Simulator", n=n, **c) for c in consts]
    ro = O.make_params(n=n)
    so = [O.make_params(n=n, **c) for c in consts]
    A, bb = builtin_rows(n)
    start = S.ops.reset_state(n).cpu().numpy()

    def ens_costs(W):
        rcs, scs = None, []
        for s in so:
            W2 = np.asarray(W).reshape(n - 1, 2 * n + 2)
            _, _, traj = O.rollout(ro, O.GYM, H, policy=W2, init_state=start, want_traj=True)
            pre = np.vstack([start[None], traj[:-1]])
            nxt, _ = O.step_batch(s, O.GYM, pre, pre @ W2.T)
            scs.append(np.max(nxt @ A.T + bb, axis=-1))
            rcs = np.max(traj @ A.T + bb, axis=-1)
        return np.max(scs, axis=0), rcs

    np.random.seed(2)
    d0 = np.stack([2 * np.random.rand(n - 1, 2 * n + 2) - 1 for _ in range(N)]).reshape(N, -1)
    costs = [ens_costs(s * nu * d0[k]) for k in range(N) for s in (1, -1)]
    sc, rc = np.array([c[0] for c in costs]), np.array([c[1] for c in costs])
    sim_thr, real_thr = _ens_thresholds(sc[None], rc, 1, zero=0, mid=1, mid_steps=1, never=0, violated=1)
    ag = S.Safe_ARS(S.builtin_cost, real_thr, sim_thr, sims)
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
                esc, erc = ens_costs(W + s * nu * d[k])
                assert _margins_ok(esc[None], erc[None], sim_thr, real_thr)
                rets.append(rollout_safe_step_ensemble(O, ro, so, W + s * nu * d[k], H, A, bb, sim_thr, real_thr)[0])
        want.append(np.mean(rets))
        W, _ = O.update_policy(W, d, np.array(rets), b=b, alpha=alpha, semantics=1)
    np.testing.assert_allclose(curve, want, rtol=1e-6, atol=1e-10)
    assert rel_err(ag.policy.reshape(-1), W) < 1e-6


@gpu
@pytest.mark.parametrize("kind", ["builtin", "bend"])
def test_is_safe_with_ensemble_agrees_with_kernel(S, O, kind):
    """Safe_ARS.isSafe with a list of environments against the kernel's decision at step 0 from the same states (one
    explicit policy per state), thresholds between neighbouring ensemble costs; each env is left in its simulated
    state."""
    n, B, M = 4, 40, 5
    real, sims = _ensemble(S, n)
    _, so = _ensemble(O, n)
    envs = [S.SwimmerEnv("Simulator", n=n, l_i=p.l_i, m_i=p.m_i, k=p.k, h=p.h, direction=[.6, .8]) for p in sims[:M]]
    A, b = _rows(kind, n)
    cost = S.builtin_cost if kind == "builtin" else S.MaxAffineCost(A, b)
    rng = np.random.default_rng(11)
    states = _starts(rng, n, B)
    W = rng.uniform(-1, 1, (B, n - 1, 2 * n + 2)) * 0.5
    acts = np.einsum("bij,bj->bi", W, states)
    ens = np.array([max(_affine_cost(A, b, O.step(s, O.GYM, states[e], acts[e])[0]) for s in so[:M])
                    for e in range(B)])
    thr = _midpoint(ens, 0.5)
    assert (np.abs(ens - thr) >= MARGIN * max(1.0, abs(thr))).all()
    res = _run(S, real, sims[:M], 1, kind, thr, np.inf, policies=_cuda(W), init_state=_cuda(states))
    kernel_safe = res.frozen_at.cpu().numpy() == 1
    ag = S.Safe_ARS(cost, np.inf, thr, envs)
    got = np.array([bool(ag.isSafe(cost, thr, envs, list(states[e]), acts[e])) for e in range(B)])
    assert np.array_equal(got, kernel_safe) and got.any() and (~got).any()
    for env, s in zip(envs, so[:M]):  # left in the state simulated from the last sample
        assert rel_err(np.array(env.get_state()), O.step(s, O.GYM, states[-1], acts[-1])[0]) < 1e-12
