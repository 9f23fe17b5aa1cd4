"""Reward-constraint screening of ARS directions by an ensemble of simulator models (swm_rollout_models,
swm_screen_mask_models; ops.rollout_models, ops.screen_mask with [M, 2N] returns, ArsEngine(sim_params=[...]),
ARSAgent(sim_models=[...])).

A direction k reaches the real world only if both of its simulated returns exceed the simulator threshold under
EVERY model: mask[k] = AND_m (r+[m, k] > thr and r-[m, k] > thr), NaN screened out.  The CPU reference is one ARS
iteration restated from the oracle's own rollouts of every model (restated_iteration); with one model it reproduces
the reference's safe-mode fixture.  The model-set rollout kernels are held to a plain swm_rollout of each model on the
same kernel, bit for bit, and to the oracle's rollouts of that model.  Decisions are compared exactly, so every
simulated return a decision depends on is asserted to lie at least MARGIN * max(1, |thr|) from the threshold."""
import contextlib
import ctypes
import dataclasses
import io
import os
import tempfile

import numpy as np
import pytest
import torch

from conftest import golden, rel_err

gpu = pytest.mark.gpu
TOL = 1e-6                      # test_parity_ars: returns and policies against the reference fixtures
RET_TOL, STATE_TOL = 1e-6, 1e-8  # rollouts against the oracle (relative, floor 1e-3 / norm-relative, floor 1)
MARGIN = 1e-9
KERNELS = ["THREAD", "LANES", "LANES2", "LANES3"]
MS = [1, 2, 7, 16]


# ---- reference ---------------------------------------------------------------------------------------------------
def restated_iteration(O, real, sims, W, deltas, H, nu, thr, b, alpha, semantics, mean=None, inv_sigma=None):
    """One reward-constraint-screened ARS iteration (ars_agent.py:140-185) with a list of simulator models, built from
    the oracle's rollouts.  -> (sim returns [M, 2N], mask [N] bool, real returns [2N] (NaN where screened out),
    updated policy, real trajectories of the survivors)."""
    N = len(deltas)
    W = np.asarray(W, dtype=np.float64)
    pols = [W + s * nu * deltas[k].reshape(W.shape) for k in range(N) for s in (+1, -1)]
    sim = np.array([[O.rollout(p, O.GYM, H, policy=q, mean=mean, inv_sigma=inv_sigma)[0] for q in pols]
                    for p in sims])
    ok = np.all((sim[:, 0::2] > thr) & (sim[:, 1::2] > thr), axis=0)
    rets, trajs = np.full(2 * N, np.nan), []
    for j, q in enumerate(pols):
        if ok[j // 2]:
            r, _, tr = O.rollout(real, O.GYM, H, policy=q, mean=mean, inv_sigma=inv_sigma, want_traj=True)
            rets[j] = r
            trajs.append(tr)
    keep = np.nonzero(ok)[0]
    if len(keep):
        W, _ = O.update_policy(W, deltas[keep].reshape(len(keep), -1), rets.reshape(N, 2)[keep].ravel(), b=b,
                               alpha=alpha, semantics=semantics)
    return sim, ok, rets, W, trajs


def _margin_ok(sim, thr):
    return bool(np.all(np.abs(np.asarray(sim) - thr) >= MARGIN * max(1.0, abs(thr))))


def _ensemble(mod, n, count=16, spread=0.05, seed=7):
    """The real model of bench's config[3] and `count` simulators around it: model 0 is 1e-3 away in (l, m, k), the
    others up to +-spread (relative) in l, m and k, so that they disagree on some directions."""
    real = mod.make_params(n=n, l_i=.8, m_i=1.2, k=10.2)
    rng = np.random.default_rng(seed)
    sims = [mod.make_params(n=n, l_i=.8005, m_i=1.2005, k=10.2005)]
    for _ in range(count - 1):
        f = 1.0 + rng.uniform(-spread, spread, 3)
        sims.append(mod.make_params(n=n, l_i=.8 * f[0], m_i=1.2 * f[1], k=10.2 * f[2]))
    return real, sims


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_restated_iteration_of_one_model_reproduces_safe_fixture(O):
    """The restatement with one model is the reference's safe mode: the fixture's rand deltas, thresholds, screened
    iterations, returns and policies (the run of test_ars_agent_safe_mode_matches_reference_run)."""
    g = golden("ars_agent_safe.npz")
    l, m, k = g["sim_params"]
    real = O.make_params(n=3, l_i=.8, m_i=1.2, k=10.2)
    sim = O.make_params(n=3, l_i=l, m_i=m, k=k)
    thr = float(g["sim_threshold"])
    assert abs(float(g["threshold"]) + float(g["alpha_H"]) * 0.001 - thr) < 1e-12
    W = g["W0"]
    for it in range(len(g["rand"])):
        deltas = (2 * g["rand"][it] - 1)[None]  # N = 1
        sim_r, ok, rets, W, _ = restated_iteration(O, real, [sim], W, deltas, 300, 0.01, thr, 1, 0.0075, 0)
        assert _margin_ok(sim_r, thr), it
        want = g["returns"][it]
        assert ok[0] == (not np.isnan(want[0]))
        if ok[0]:
            np.testing.assert_allclose(rets, want, rtol=TOL)
        else:
            assert np.isnan(rets).all()
        assert rel_err(W, g["policies"][it]) < TOL
    assert np.isnan(g["returns"][:, 0]).any() and (~np.isnan(g["returns"][:, 0])).any()


def test_rollout_models_argument_checks(S):
    """Rejected before anything is launched: no device needed."""
    L = S._lib.lib()
    n = 3
    _, sims = _ensemble(S, n)

    def cfg(**kw):
        c = S._lib.SwmRollout()
        c.variant, c.policy_mode, c.H, c.B, c.rollouts_per_policy = S.GYM, S.ops.POLICY_PHILOX, 10, 64, 1
        for key, v in kw.items():
            setattr(c, key, v)
        return c

    def models(ps):
        return (S._lib.SwmParams * len(ps))(*ps)

    good = models(sims[:3])

    def call(c, ms=good, M=3):
        return L.swm_rollout_models(ms, M, ctypes.byref(c), None)

    bad, unsup = -1, -2
    assert call(cfg(), M=0) == bad and call(cfg(), ms=models(sims + sims[:1]), M=17) == bad
    assert call(cfg(), ms=None) == bad and L.swm_rollout_models(good, 3, None, None) == bad
    assert call(cfg(), ms=models(sims[:2] + [S.make_params(n=4)])) == bad
    zero_m = S.make_params(n=n)
    zero_m.m_i = 0.0
    assert call(cfg(), ms=models([sims[0], zero_m]), M=2) == bad
    assert call(cfg(H=-1)) == bad and call(cfg(rollouts_per_policy=0)) == bad
    assert call(cfg(B=63)) == bad  # +delta / -delta pairs
    assert call(cfg(kernel=7)) == bad
    assert call(cfg(variant=S.RLGLUE)) == unsup
    assert call(cfg(policy_mode=S.ops.POLICY_FIXED_ACTION)) == unsup
    dummy = (ctypes.c_double * 64)()
    ptr = ctypes.cast(dummy, ctypes.c_void_p)
    assert call(cfg(stats_partial=ptr, stats_pivot=ptr)) == unsup
    assert call(cfg(trajectory=ptr)) == unsup
    assert call(cfg(schedule_sub=2, schedule_chunk=64)) == unsup
    for k in (S.KERNEL_AUTO, S.KERNEL_THREAD, S.KERNEL_LANES, S.KERNEL_LANES2, S.KERNEL_LANES3):
        assert call(cfg(clip_actions=1, kernel=k)) == unsup
    c = cfg()
    c.screen.enabled = 1
    c.screen.sim = sims[0]
    assert call(c) == unsup
    # an empty batch is accepted without a device, with any model count in range
    assert call(cfg(B=0)) == 0 and call(cfg(B=0), ms=models(sims), M=16) == 0
    assert call(cfg(B=0), M=1) == 0
    # the mask over models
    M = L.swm_screen_mask_models
    p = ctypes.c_void_p(1)
    assert M(None, 2, 4, 0.0, p, None, None, None) == bad and M(p, 2, 4, 0.0, None, None, None, None) == bad
    assert M(p, 0, 4, 0.0, p, None, None, None) == bad and M(p, 17, 4, 0.0, p, None, None, None) == bad
    assert M(p, 2, 0, 0.0, p, None, None, None) == bad
    assert L.swm_screen_mask(p, 0, 0.0, p, None, None, None) == bad


# ---- GPU: the model-set rollout kernels --------------------------------------------------------------------------
def _cuda(a, dtype=np.float64):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=dtype)).cuda()


def _bits_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int64), b.contiguous().view(torch.int64))


# (policy source, R, directions / policies, V2, start): B = 2 D R or P R is never a multiple of 32 or of a lane
# group except for R = 32
CONFIGS = [("explicit", 1, 37, False, "state"), ("philox", 3, 7, True, "perturb"), ("deltas", 1, 11, False, "perturb"),
           ("philox", 32, 1, False, "state"), ("deltas", 3, 5, True, "state"), ("explicit", 3, 9, True, "perturb")]


def _case(S, n, source, R, D, v2, start, seed):
    """Keyword arguments of ops.rollout for one configuration (B environments per model)."""
    rng = np.random.default_rng(seed)
    no, ws = 2 * n + 2, (n - 1) * (2 * n + 2)
    kw = dict(rollouts_per_policy=R, want_final=True, seed=seed, iteration=3, dir0=2, nu=0.2)
    if source == "explicit":
        kw["policies"] = _cuda(rng.uniform(-1, 1, (D, n - 1, no)) * 0.4)
        B = D * R
    else:
        kw["base_policy"] = _cuda(rng.uniform(-1, 1, ws) * 0.3)
        B = 2 * D * R
        if source == "deltas":
            kw["deltas"] = _cuda(rng.uniform(-1, 1, (D, ws)))
    kw["B"] = B
    if v2:
        kw["mean"] = _cuda(rng.normal(size=no) * 0.1)
        kw["inv_sigma"] = _cuda(rng.uniform(0.5, 2.0, no))
    if start == "state":
        kw["init_state"] = _cuda(np.hstack([rng.normal(size=(R, 2)) * 0.1,
                                            np.stack([rng.uniform(-2, 2, (R, n)), rng.normal(size=(R, n))],
                                                     axis=2).reshape(R, 2 * n)]))
    else:
        kw["init_perturb"] = 0.05
    return kw


@gpu
@pytest.mark.parametrize("kern", KERNELS)
@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 7, 8, 9, 10])
def test_model_rows_equal_plain_rollouts_bit_for_bit(S, n, kern):
    """Row m of rollout_models is swm_rollout of model m forced to the same kernel, bit for bit (returns and final
    states), for M in {1, 2, 7, 16} over explicit / Philox / in-memory perturbations, R in {1, 3, 32}, V1 and V2,
    start states and init_perturb."""
    _, sims = _ensemble(S, n)
    K = getattr(S, "KERNEL_" + kern)
    H = 131
    for i, (source, R, D, v2, start) in enumerate(CONFIGS):
        kw = _case(S, n, source, R, D, v2, start, seed=100 * n + i)
        M = MS[i % len(MS)]
        got = S.ops.rollout_models(sims[:M], H, kernel=K, **kw)
        assert got.returns.shape == (M, kw["B"]) and got.final_state.shape == (M, kw["B"], 2 * n + 2)
        for m in range(M):
            want = S.ops.rollout(sims[m], H, kernel=K, schedule="plain", **kw)
            assert _bits_equal(got.returns[m], want.returns), (source, M, m)
            assert _bits_equal(got.final_state[m], want.final_state), (source, M, m)
        assert torch.isfinite(got.returns).all()


@gpu
@pytest.mark.parametrize("n,B,R", [(3, 512, 1), (3, 8192, 1), (5, 512, 1), (6, 512, 1), (6, 96, 3), (9, 256, 1)])
def test_auto_picks_the_kernel_of_the_whole_batch(S, n, B, R):
    """Under AUTO the model-set rollout runs the kernel swm_rollout_kernel_choice gives for M * B environments: its
    rows equal that kernel forced, bit for bit."""
    _, sims = _ensemble(S, n)
    W = _cuda(np.random.default_rng(n).uniform(-1, 1, (n - 1) * (2 * n + 2)) * 0.3)
    seen = set()
    for M in (1, 2, 4, 8, 16):
        name = S.ops.rollout_kernel_choice(sims[0], M * B, rollouts_per_policy=R)
        seen.add(name)
        kw = dict(B=B, base_policy=W, nu=0.1, seed=1, rollouts_per_policy=R, want_final=True, init_perturb=0.01)
        auto = S.ops.rollout_models(sims[:M], 70, **kw)
        forced = S.ops.rollout_models(sims[:M], 70, kernel=getattr(S, "KERNEL_" + name.upper()), **kw)
        assert _bits_equal(auto.returns, forced.returns) and _bits_equal(auto.final_state, forced.final_state), M
    if (n, B) == (3, 512):
        assert {"lanes2", "lanes"} <= seen


_ORACLE_ERR = {}


@gpu
@pytest.mark.parametrize("kern", KERNELS)
@pytest.mark.parametrize("n", [2, 3, 5, 7, 8, 10])
def test_model_rows_match_oracle(S, O, n, kern):
    """Every model's returns and final states against the oracle's rollouts of that model: returns 1e-6 relative,
    final states 1e-8 (explicit policies, V1 and V2, start states)."""
    _, sims = _ensemble(S, n)
    _, so = _ensemble(O, n)
    K = getattr(S, "KERNEL_" + kern)
    H, M, P = 300, 3, 13
    rng = np.random.default_rng(n)
    no = 2 * n + 2
    pols = rng.uniform(-1, 1, (P, n - 1, no)) * 0.4
    init = np.hstack([rng.normal(size=(P, 2)) * 0.1,
                      np.stack([rng.uniform(-2, 2, (P, n)), rng.normal(size=(P, n))], axis=2).reshape(P, 2 * n)])
    errs = []
    for v2 in (False, True):
        mean = rng.normal(size=no) * 0.1 if v2 else None
        inv_sigma = rng.uniform(0.5, 2.0, no) if v2 else None
        kw = dict(mean=_cuda(mean), inv_sigma=_cuda(inv_sigma)) if v2 else {}
        res = S.ops.rollout_models(sims[:M], H, policies=_cuda(pols), init_state=_cuda(init), want_final=True,
                                   kernel=K, **kw)
        r, f = res.returns.cpu().numpy(), res.final_state.cpu().numpy()
        for m in range(M):
            for e in range(P):
                wr, wf, _ = O.rollout(so[m], O.GYM, H, policy=pols[e], mean=mean, inv_sigma=inv_sigma,
                                      init_state=init[e])
                errs.append((abs(r[m, e] - wr) / max(1e-3, abs(wr)), rel_err(f[m, e], wf)))
    er, ef = np.max(errs, axis=0)
    prev = _ORACLE_ERR.get(kern, (0.0, 0.0))
    _ORACLE_ERR[kern] = (max(prev[0], er), max(prev[1], ef))
    print("model-set oracle parity %s n=%d: returns %.2e, final states %.2e (running max %.2e, %.2e)"
          % (kern, n, er, ef, *_ORACLE_ERR[kern]))
    assert er < RET_TOL and ef < STATE_TOL, (er, ef)


# ---- GPU: the mask ------------------------------------------------------------------------------------------------
@gpu
def test_screen_mask_over_models_matches_numpy(S):
    rng = np.random.default_rng(0)
    thr = 0.25
    total = torch.zeros(1, dtype=torch.int64, device="cuda")
    running = 0
    for M in range(1, 17):
        for N in (1, 7, 255, 256, 257, 3001):
            r = rng.normal(size=(M, 2 * N))
            special = rng.integers(0, 2 * N, size=(M, 6))
            for m in range(M):  # a NaN, +-inf and returns exactly at the threshold in single models
                r[m, special[m, 0]] = np.nan
                r[m, special[m, 1]] = np.inf
                r[m, special[m, 2]] = -np.inf
                r[m, special[m, 3:]] = thr
            want = np.all((r[:, 0::2] > thr) & (r[:, 1::2] > thr), axis=0)
            mask, n_pass = S.ops.screen_mask(_cuda(r), thr, n_pass_total=total)
            assert np.array_equal(mask.cpu().numpy() != 0, want), (M, N)
            assert int(n_pass.item()) == int(want.sum())
            running += int(want.sum())
            assert int(total.item()) == running
            if M == 1:
                single, sp = S.ops.screen_mask(_cuda(r[0]), thr)
                assert torch.equal(single, mask) and torch.equal(sp, n_pass)
    # a NaN or -inf in any one model screens a direction that every other model passes
    for bad in (np.nan, -np.inf, thr):
        r = np.ones((16, 8))
        r[rng.integers(0, 16), 5] = bad
        mask, _ = S.ops.screen_mask(_cuda(r), thr)
        assert mask.cpu().tolist() == [1, 1, 0, 1]


# ---- GPU: the engine ----------------------------------------------------------------------------------------------
def _pick_threshold(sim):
    """A threshold between two neighbouring direction keys of simulated returns sim [M, 2N] at which some direction
    survives every model and, for M > 1, some direction passes model 0 but is screened out by another model; of
    those the one that leaves closest to half of the directions."""
    ens = np.min(np.minimum(sim[:, 0::2], sim[:, 1::2]), axis=0)
    z = np.minimum(sim[0, 0::2], sim[0, 1::2])
    v = np.unique(np.concatenate([ens, z]))
    best = None
    for t in (v[1:] + v[:-1]) / 2:
        alive, other = int((ens > t).sum()), int(((z > t) & (ens <= t)).sum())
        if alive >= 1 and (other >= 1 or len(sim) == 1) and alive < len(z):
            if best is None or abs(alive - len(z) / 2) < abs(best[1] - len(z) / 2):
                best = (float(t), alive)
    assert best is not None, "these models do not disagree on any direction"
    return best[0]


def _first_sim_returns(S, sims, W0, N, H, nu, seed, R=1, v2=False, init_perturb=0.0, **_):
    """Simulated returns [M, 2N] of an engine's first iteration from W0 (per-direction means over R rollouts)."""
    n = sims[0].n
    kw = dict(mean=_cuda(np.zeros(2 * n + 2)), inv_sigma=_cuda(np.ones(2 * n + 2))) if v2 else {}
    r = S.ops.rollout_models(sims, H, B=2 * N * R, base_policy=_cuda(W0), nu=nu, seed=seed, rollouts_per_policy=R,
                             init_perturb=init_perturb, **kw).returns.cpu().numpy()
    return r.reshape(len(sims), 2 * N, R).mean(axis=2)


@gpu
@pytest.mark.parametrize("use_graph", [False, True])
def test_engine_list_of_one_is_the_single_model_path(S, use_graph):
    n, N, H = 3, 16, 160
    real, sims = _ensemble(S, n)
    W0 = np.random.default_rng(1).uniform(-1, 1, 16) * 0.3
    kw = dict(N=N, b=5, alpha=0.01, nu=0.05, H=H, seed=5, semantics=S.ARS_TOPB)
    thr = _pick_threshold(_first_sim_returns(S, sims[:1], W0, **kw))
    a = S.ArsEngine(real, initial_policy=W0, distributed=False, sim_params=sims[0], sim_threshold=thr,
                    use_graph=use_graph, **kw)
    b = S.ArsEngine(real, initial_policy=W0, distributed=False, sim_params=[sims[0]], sim_threshold=thr,
                    use_graph=use_graph, **kw)
    assert b.sim_returns.shape == (1, 2 * N)
    screened = 0
    for it in range(5):
        ra, rb = a.run_iteration().clone(), b.run_iteration().clone()
        assert torch.equal(torch.isnan(ra), torch.isnan(rb)) and _bits_equal(torch.nan_to_num(ra), torch.nan_to_num(rb))
        assert torch.equal(a.mask, b.mask) and torch.equal(a.n_pass_total, b.n_pass_total)
        assert _bits_equal(a.W, b.W) and _bits_equal(a.sim_returns, b.sim_returns[0])
        screened += int(torch.isnan(ra).sum())
    assert 0 < screened < 5 * 2 * N and (b._graph is not None) == use_graph


def _engine_vs_oracle(S, O, n, M, iters, v2=False, R=1, speculate=True):
    """ArsEngine with M simulator models against restated_iteration, iteration by iteration from the engine's own
    previous policy.  Returns how often a direction passed model 0 and was screened out by another model."""
    N, b, H, nu, alpha, seed = 12, 6, 150, 0.3, 0.02, 9
    (real, sims), (ro, so) = _ensemble(S, n), _ensemble(O, n)
    ws, no = (n - 1) * (2 * n + 2), 2 * n + 2
    W0 = np.random.default_rng(n + M).uniform(-1, 1, ws) * 0.3
    kw = dict(N=N, b=b, alpha=alpha, nu=nu, H=H, seed=seed, semantics=S.ARS_TOPB, v2=v2, rollouts_per_direction=R)
    init_perturb = 0.02 if R > 1 else 0.0
    # model 0 and the M - 1 models that are most pessimistic about the first iteration's directions, so that some
    # direction model 0 passes is screened out by another one
    first = _first_sim_returns(S, sims, W0, init_perturb=init_perturb, R=R, **kw)
    pick = [0] + [1 + int(i) for i in np.argsort(np.minimum(first[1:, 0::2], first[1:, 1::2]).mean(axis=1))[:M - 1]]
    sims, so = [sims[i] for i in pick], [so[i] for i in pick]
    thr = _pick_threshold(first[pick])
    eng = S.ArsEngine(real, initial_policy=W0, distributed=False, sim_params=sims, sim_threshold=thr,
                      speculate=speculate, init_perturb=init_perturb, **kw)
    starts = None
    if R > 1:  # the R perturbed start states of iteration it: a zero-step rollout returns them as final states
        def starts(it):
            return S.ops.rollout(real, 0, B=2 * R, base_policy=eng.W, seed=seed, iteration=it, rollouts_per_policy=R,
                                 init_perturb=init_perturb, want_final=True).final_state[:R].cpu().numpy()
    other, survivors, all_trajs = 0, 0, []
    mean, inv_sigma = (np.zeros(no), np.ones(no)) if v2 else (None, None)
    for it in range(iters):
        W = eng.W.cpu().numpy()
        got = eng.run_iteration().cpu().numpy()
        deltas = np.stack([O.philox_delta(seed, it, k, ws) for k in range(N)])
        pols = [W + s * nu * deltas[k] for k in range(N) for s in (+1, -1)]
        st = starts(it) if R > 1 else [None]
        sim = np.array([[np.mean([O.rollout(p, O.GYM, H, policy=x, mean=mean, inv_sigma=inv_sigma, init_state=s0)[0]
                                  for s0 in st]) for x in pols] for p in so])
        assert _margin_ok(sim, thr), it
        ok = np.all((sim[:, 0::2] > thr) & (sim[:, 1::2] > thr), axis=0)
        ok0 = (sim[0, 0::2] > thr) & (sim[0, 1::2] > thr)
        other += int((ok0 & ~ok).sum())
        survivors += int(ok.sum())
        assert np.array_equal(eng.mask.cpu().numpy() != 0, ok), it
        np.testing.assert_allclose(eng.sim_returns.cpu().numpy(), sim, rtol=RET_TOL, atol=1e-9)
        rets = np.full(2 * N, np.nan)
        for j, x in enumerate(pols):
            if ok[j // 2]:
                rr = []
                for s0 in st:
                    r, _, tr = O.rollout(ro, O.GYM, H, policy=x, mean=mean, inv_sigma=inv_sigma, init_state=s0,
                                         want_traj=True)
                    rr.append(r)
                    all_trajs.append(tr)
                rets[j] = np.mean(rr)
        assert np.array_equal(np.isnan(got), np.isnan(rets)), it
        live = ~np.isnan(rets)
        np.testing.assert_allclose(got[live], rets[live], rtol=RET_TOL, atol=1e-9)
        keep = np.nonzero(ok)[0]
        want_W = W
        if len(keep):
            want_W, _ = O.update_policy(W, deltas[keep], got.reshape(N, 2)[keep].ravel(), b=b, alpha=alpha,
                                        semantics=1)
        assert rel_err(eng.W.cpu().numpy(), want_W) < 1e-9, it
        if v2:  # statistics over the real states of the survivors only, cumulative
            if all_trajs:
                mean, var = O.mean_var(np.concatenate(all_trajs))
                inv_sigma = var ** -0.5
            np.testing.assert_allclose(eng.mean.cpu().numpy(), mean, rtol=TOL, atol=1e-9)
            np.testing.assert_allclose(eng.inv_sigma.cpu().numpy(), inv_sigma, rtol=TOL)
    assert 0 < survivors < iters * N
    return other


@gpu
@pytest.mark.parametrize("n,M", [(3, 2), (3, 7), (5, 16), (8, 3)])
def test_engine_ensemble_matches_oracle_loop(S, O, n, M):
    assert _engine_vs_oracle(S, O, n, M, iters=3) > 0


@gpu
def test_engine_ensemble_v2_counts_survivors_only(S, O):
    assert _engine_vs_oracle(S, O, 3, 4, iters=3, v2=True) > 0


@gpu
def test_engine_ensemble_rollouts_per_direction(S, O):
    assert _engine_vs_oracle(S, O, 3, 3, iters=2, R=3) > 0


@gpu
@pytest.mark.parametrize("use_graph", [False, True])
def test_engine_ensemble_speculative_equals_screen_first(S, use_graph):
    n, N, H, M = 3, 16, 130, 5
    real, sims = _ensemble(S, n)
    W0 = np.random.default_rng(2).uniform(-1, 1, 16) * 0.3
    kw = dict(N=N, b=5, alpha=0.01, nu=0.1, H=H, seed=5, semantics=S.ARS_TOPB)
    thr = _pick_threshold(_first_sim_returns(S, sims[:M], W0, **kw))
    spec, first = [S.ArsEngine(real, initial_policy=W0, distributed=False, sim_params=sims[:M], sim_threshold=thr,
                               use_graph=use_graph, speculate=s, **kw) for s in (True, False)]
    assert spec.speculate and not first.speculate
    screened = 0
    for it in range(4):
        a, b = spec.run_iteration().clone(), first.run_iteration().clone()
        assert torch.equal(torch.isnan(a), torch.isnan(b)) and _bits_equal(torch.nan_to_num(a), torch.nan_to_num(b))
        assert torch.equal(spec.mask, first.mask) and _bits_equal(spec.W, first.W)
        assert torch.equal(spec.n_pass_total, first.n_pass_total) and _bits_equal(spec.sim_returns, first.sim_returns)
        screened += int(torch.isnan(a).sum())
    assert 0 < screened < 4 * 2 * N and (spec._graph is not None) == use_graph


@gpu
def test_engine_model_order_duplicates_and_nesting(S):
    """Permuting the models permutes the rows of sim_returns and leaves mask and policy bit-identical; [a, a] is [a];
    a model added to the set never adds a survivor."""
    n, N, H = 3, 32, 150
    real, sims = _ensemble(S, n)
    W0 = np.random.default_rng(3).uniform(-1, 1, 16) * 0.3
    kw = dict(N=N, b=8, alpha=0.01, nu=0.1, H=H, seed=11, semantics=S.ARS_TOPB)
    thr = _pick_threshold(_first_sim_returns(S, sims, W0, **kw))

    def run(models, iters=3):
        e = S.ArsEngine(real, initial_policy=W0, distributed=False, sim_params=models, sim_threshold=thr, **kw)
        out = []
        for _ in range(iters):
            r = e.run_iteration().clone()
            out.append((r, e.mask.clone(), e.W.clone(), e.sim_returns.clone(), e.n_pass_total.clone()))
        return out

    base = run(sims[:5])
    perm = [3, 0, 4, 2, 1]
    for (r, m, W, sr, tot), (r2, m2, W2, sr2, tot2) in zip(base, run([sims[i] for i in perm])):
        assert torch.equal(m, m2) and _bits_equal(W, W2) and torch.equal(tot, tot2)
        assert _bits_equal(torch.nan_to_num(r), torch.nan_to_num(r2))
        assert _bits_equal(sr[perm], sr2)
    for x, y in zip(run([sims[0]]), run([sims[0], sims[0]])):
        assert torch.equal(x[1], y[1]) and _bits_equal(x[2], y[2]) and torch.equal(x[4], y[4])
        assert _bits_equal(torch.nan_to_num(x[0]), torch.nan_to_num(y[0]))
        assert _bits_equal(y[3][0], x[3][0]) and _bits_equal(y[3][1], x[3][0])
    prev, counts = None, []
    for M in range(1, 17):
        mask = run(sims[:M], iters=1)[0][1].cpu().numpy()
        if prev is not None:
            assert not (mask & ~prev).any(), M
        prev = mask
        counts.append(int(mask.sum()))
    assert counts[0] > counts[-1]


@gpu
def test_engine_rejects_bad_model_lists(S):
    real, sims = _ensemble(S, 3)
    kw = dict(N=4, b=2, alpha=0.01, nu=0.1, H=10, distributed=False, sim_threshold=0.0)
    for bad in ([], sims + sims[:1], [sims[0], S.make_params(n=4)]):
        with pytest.raises(ValueError):
            S.ArsEngine(real, sim_params=bad, **kw)
    with pytest.raises(ValueError):
        S.ArsEngine(real, sim_params=sims[:2], clip_actions=True, **kw)
    W = _cuda(np.zeros(16))
    for k in (S.KERNEL_LANES, S.KERNEL_LANES2, S.KERNEL_LANES3):
        with pytest.raises(S._lib.SwimmerLibError):
            S.ops.rollout_models(sims[:2], 10, B=8, base_policy=W, clip_actions=True, kernel=k)
    with pytest.raises(S._lib.SwimmerLibError):
        S.ops.rollout_models(sims[:2], 10, B=8, base_policy=W, want_trajectory=True)
    # per-step screening is refused whatever its models; an ensemble screen leaves cfg.screen.sim unset (bad argument)
    screen = dict(sim_thresh=1e9, real_thresh=1e9)
    with pytest.raises(S._lib.SwimmerLibError, match="unsupported configuration"):
        S.ops.rollout_models(sims[:4], 10, B=8, base_policy=W, screen=dict(screen, sim_params=sims[0]))
    for ens in (sims[:1], sims[:7]):
        with pytest.raises(S._lib.SwimmerLibError, match="bad argument"):
            S.ops.rollout_models(sims[:4], 10, B=8, base_policy=W, screen=dict(screen, sim_params=ens))
    with pytest.raises(ValueError):
        S.ops.rollout_models([], 10, B=8, base_policy=W)


# ---- GPU: the agent -----------------------------------------------------------------------------------------------
def _agent_setup(S, td, threshold, H=200, N=4):
    wpath = os.path.join(td, "w0.npy")
    np.save(wpath, np.random.default_rng(5).uniform(-1, 1, (2, 8)) * 0.2)
    dpath = os.path.join(td, "db.npz")
    np.savez(dpath, policies=[np.zeros((2, 8))], trajectories=[np.zeros((50, 8))])
    ep = S.EnvParam("real", n=3, H=H, l_i=.8, m_i=1.2, h=1e-3, k=10.2, epsilon=0.001)
    ap = S.ARSParam("x", V1=True, n_iter=3, H=H, N=N, b=2, alpha=0.0075, nu=0.3, safe=True, threshold=threshold,
                    initial_w=wpath)
    return ep, ap, dpath, np.load(wpath)


@gpu
def test_agent_with_sim_models_matches_oracle_loop(S, O):
    """ARSAgent(sim_models=[...]) with numpy deltas against restated_iteration; sim_models=[estimated_param] is the
    default safe agent bit for bit."""
    H, N, seed = 200, 4, 4
    th = S.Threshold(K=1, A=0.1, B=0.001)
    alpha_eps = th.compute_alpha(H) * 0.001
    with tempfile.TemporaryDirectory() as td:
        ep, ap, dpath, W0 = _agent_setup(S, td, 0.0, H, N)
        sims = [dataclasses.replace(ep, name="sim%d" % i, l_i=ep.l_i * f[0], m_i=ep.m_i * f[1], k=ep.k * f[2])
                for i, f in enumerate([(1.0005, 1.0005, 1.0005), (1.04, .97, 1.02), (.96, 1.03, .98)])]
        so = [O.make_params(n=3, l_i=p.l_i, m_i=p.m_i, k=p.k) for p in sims]
        real = O.make_params(n=3, l_i=.8, m_i=1.2, k=10.2)
        rs = np.random.RandomState(seed)
        d0 = np.stack([2 * rs.rand(2, 8) - 1 for _ in range(N)])
        sim0 = np.array([[O.rollout(p, O.GYM, H, policy=W0 + s * ap.nu * d0[k])[0] for k in range(N) for s in (1, -1)]
                         for p in so])
        ap = dataclasses.replace(ap, threshold=_pick_threshold(sim0) - alpha_eps)
        iters = 4

        def run(**kw):
            """A fresh agent (each constructor reseeds numpy's global stream) and its iterations."""
            np.random.seed(77)
            with contextlib.redirect_stdout(io.StringIO()):
                a = S.ARSAgent(ep, ap, data_path=dpath, seed=seed, approx_error=0.001, sim_thresh=th, **kw)
                out = []
                for _ in range(iters):
                    r = a.runOneIteration()
                    out.append((r, a.engine.mask.clone(), a.engine.W.clone()))
            return a, out

        default, plain = run()
        single, one = run(sim_models=[default.estimated_param])
        assert single.estimated_param == default.estimated_param
        for (r, m, W), (r1, m1, W1) in zip(plain, one):
            assert r == r1 and torch.equal(m, m1) and _bits_equal(W, W1)
        ag, ens = run(sim_models=sims)
        assert ag.estimated_param == default.estimated_param
        thr = ag.sim_threshold
        rs = np.random.RandomState(seed)
        W, other = W0, 0
        for it in range(iters):
            deltas = np.stack([2 * rs.rand(2, 8) - 1 for _ in range(N)])
            got, mask, Wg = ens[it]
            sim, ok, rets, W, _ = restated_iteration(O, real, so, W, deltas, H, ap.nu, thr, ap.b, ap.alpha, 0)
            assert _margin_ok(sim, thr), it
            other += int((((sim[0, 0::2] > thr) & (sim[0, 1::2] > thr)) & ~ok).sum())
            assert np.array_equal(mask.cpu().numpy() != 0, ok), it
            np.testing.assert_allclose(got, rets[~np.isnan(rets)], rtol=TOL)
            assert rel_err(Wg.cpu().numpy(), W.reshape(-1)) < TOL
        assert other > 0 and len(ag.screened_fraction) == iters
    with pytest.raises(ValueError):
        S.ARSAgent(ep, dataclasses.replace(ap, safe=False), sim_models=sims)
