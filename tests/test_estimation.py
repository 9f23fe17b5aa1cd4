"""Simulator-model estimation on the device: the fused prediction-error objective (swm_prediction_error) against
the CPU oracle, and CMA-ES (swm_cmaes_*) against a numpy restatement of Hansen's tutorial (2016), recovery of
noise-free models, determinism, and the ARSAgent "computed estimation" path without the `cma` package.
The numpy restatement of CMA-ES below is the reference these tests compare against; the product has none."""
import contextlib
import ctypes
import io
import math
import sys

import numpy as np
import pytest
import torch

from conftest import rel_err

REAL = dict(m_i=1.2, l_i=0.8, k=10.2)  # config[4] real model


def _cuda(a):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _record(O, n, H, K, seed, model=REAL, scale=0.5):
    """K trajectories [K, H, 2n+2] and their V1 policies [K, n-1, 2n+2], recorded by the oracle."""
    po = O.make_params(n=n, **model)
    rng = np.random.default_rng(seed)
    pols = rng.uniform(-1, 1, (K, n - 1, 2 * n + 2)) * scale
    trajs = np.stack([O.rollout(po, 0, H, policy=W, want_traj=True)[2] for W in pols])
    return trajs, pols


def _oracle_error(O, n, trajs, pols, m, l, k):
    p = O.make_params(n=n, m_i=m, l_i=l, k=k)
    total = 0.0
    for traj, W in zip(trajs, pols):
        nxt, _ = O.step_batch(p, 0, traj[:-1], traj[:-1] @ W.T)
        total += np.linalg.norm(nxt - traj[1:], axis=1).sum()
    return total


# ---- numpy restatement of the tutorial's CMA-ES (positive weights, no active update) ----------------------
def _strategy(d, lam):
    mu = lam // 2
    w = np.log((lam + 1) / 2.0) - np.log(np.arange(1, mu + 1))
    w = w / w.sum()
    mueff = 1.0 / np.sum(w ** 2)
    cs = (mueff + 2) / (d + mueff + 5)
    ds = 1 + 2 * max(0.0, math.sqrt((mueff - 1) / (d + 1)) - 1) + cs
    cc = (4 + mueff / d) / (d + 4 + 2 * mueff / d)
    c1 = 2 / ((d + 1.3) ** 2 + mueff)
    cmu = min(1 - c1, 2 * (mueff - 2 + 1 / mueff) / ((d + 2) ** 2 + mueff))
    chiN = math.sqrt(d) * (1 - 1 / (4 * d) + 1 / (21 * d * d))
    return w, mueff, cs, ds, cc, c1, cmu, chiN


def _np_update(prev, z, fit, d, lam):
    w, mueff, cs, ds, cc, c1, cmu, chiN = _strategy(d, lam)
    mu = len(w)
    order = sorted(range(lam), key=lambda c: (not np.isfinite(fit[c]), fit[c] if np.isfinite(fit[c]) else 0.0, c))
    B, D, C, sigma = prev["B"], prev["D"], prev["C"], float(prev["sigma"])
    y = (B @ (D[:, None] * z.T)).T
    ysel = y[order[:mu]]
    yw = w @ ysel
    gen = float(prev["generation"]) + 1
    mean = prev["mean"] + sigma * yw
    ps = (1 - cs) * prev["p_sigma"] + math.sqrt(cs * (2 - cs) * mueff) * (B @ np.diag(1 / D) @ B.T @ yw)
    psn = np.linalg.norm(ps)
    hsig = psn / math.sqrt(1 - (1 - cs) ** (2 * gen)) < (1.4 + 2 / (d + 1)) * chiN
    pc = (1 - cc) * prev["p_c"] + (math.sqrt(cc * (2 - cc) * mueff) * yw if hsig else 0.0)
    dh = 0.0 if hsig else cc * (2 - cc)
    rmu = sum(wi * np.outer(yi, yi) for wi, yi in zip(w, ysel))
    C = (1 + c1 * dh - c1 - cmu * w.sum()) * C + c1 * np.outer(pc, pc) + cmu * rmu
    sigma = sigma * math.exp(cs / ds * (psn / chiN - 1))
    return dict(mean=mean, sigma=sigma, C=C, p_sigma=ps, p_c=pc)


def _view(S, state, d, lam):
    return {k: v.cpu().numpy() for k, v in S.ops.cmaes_view(state, d, lam).items()}


# ---- CPU -----------------------------------------------------------------------------------------------------
def test_estimation_abi_rejects_bad_arguments_without_a_device(S):
    L = S._lib.lib()
    assert L.swm_cmaes_state_doubles(3, 7) == S.ops.cmaes_state_doubles(3, 7) > 0
    for d, lam in ((0, 7), (4, 7), (3, 1), (3, S._lib.MAX_CANDIDATES + 1)):
        assert L.swm_cmaes_state_doubles(d, lam) == 0
    assert L.swm_prediction_error_workspace_doubles(3, 200, 40) == ((3 * 199 + 127) // 128) * 40
    assert L.swm_prediction_error_workspace_doubles(3, 1, 40) == 0
    BAD = -1
    fake = ctypes.c_void_p(16)  # never dereferenced: every call below fails its argument checks first
    x0 = (ctypes.c_double * 3)(1.0, 1.0, 10.0)
    assert L.swm_cmaes_init(fake, 4, 7, x0, 1.0, 1e-11, 1e-11, 0, None) == BAD
    assert L.swm_cmaes_init(fake, 3, 1, x0, 1.0, 1e-11, 1e-11, 0, None) == BAD
    assert L.swm_cmaes_init(fake, 3, 7, x0, 0.0, 1e-11, 1e-11, 0, None) == BAD
    assert L.swm_cmaes_init(fake, 3, 7, None, 1.0, 1e-11, 1e-11, 0, None) == BAD
    assert L.swm_cmaes_sample(fake, 3, 2000, 0, fake, None) == BAD
    assert L.swm_cmaes_update(fake, 0, 7, fake, fake, None) == BAD

    def data(d=3, fields=(0, 1, 2), K=1, H=10):
        e = S._lib.SwmEstimateData()
        e.trajectories = e.policies = e.workspace = 16
        e.K, e.H, e.d = K, H, d
        for i, f in enumerate(fields):
            e.fields[i] = f
        return e

    base = S.make_params(n=3)
    for dd in (data(d=0), data(d=4), data(fields=(0, 0, 1)), data(fields=(0, 1, 3)), data(K=0), data(H=1)):
        assert L.swm_prediction_error(ctypes.byref(base), ctypes.byref(dd), fake, 7, fake, None) == BAD
    good = data()
    for M in (0, S._lib.MAX_CANDIDATES + 1):
        assert L.swm_prediction_error(ctypes.byref(base), ctypes.byref(good), fake, M, fake, None) == BAD
    for n in (1, 11):
        bp = S._lib.SwmParams(); bp.n = n
        assert L.swm_prediction_error(ctypes.byref(bp), ctypes.byref(good), fake, 7, fake, None) == BAD
        assert L.swm_cmaes_generation(fake, 3, 7, 0, ctypes.byref(bp), ctypes.byref(good), fake, fake, None) == BAD
    # d of the state and of the data must agree; lambda in range
    assert L.swm_cmaes_generation(fake, 2, 7, 0, ctypes.byref(base), ctypes.byref(good), fake, fake, None) == BAD
    assert L.swm_cmaes_generation(fake, 3, 1, 0, ctypes.byref(base), ctypes.byref(good), fake, fake, None) == BAD


def test_cmaes_layout_and_defaults(S):
    assert [S.ops.cmaes_default_popsize(d) for d in (1, 2, 3)] == [4, 6, 7]
    for d, lam in ((1, 2), (2, 6), (3, 7), (3, 1024)):
        total = S.ops.cmaes_state_doubles(d, lam)
        v = S.ops.cmaes_view(torch.zeros(total, dtype=torch.float64), d, lam)
        assert sum(t.numel() for t in v.values()) == total
        assert v["z"].shape == (lam, d) and v["history"].numel() == 10 + math.ceil(30 * d / lam)


# ---- objective -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 5, 10])
def test_prediction_error_matches_oracle(S, O, n):
    H, K, M = 200, 3, 40
    trajs, pols = _record(O, n, H, K, seed=n, scale=0.3)
    rng = np.random.default_rng(100 + n)
    truth = np.array([REAL["m_i"], REAL["l_i"], REAL["k"]])
    cand = truth * (1 + rng.uniform(-0.1, 0.1, (M, 3)))
    cand[0] = truth
    cand[5, 0] = 0.0     # m_i <= 0
    cand[6, 0] = -1.0
    cand[7, 1] = 0.0     # l_i = 0
    cand[8, 1] = -0.3
    bad = {5, 6, 7, 8}
    data = S.ops.EstimateData(_cuda(trajs), _cuda(pols), ("m_i", "l_i", "k"), max_candidates=M)
    base = S.make_params(n=n)
    err = S.ops.prediction_error(base, data, _cuda(cand)).cpu().numpy()
    assert err[0] < 1e-12
    for c in range(M):
        if c in bad:
            assert err[c] == np.inf
        elif c > 0:
            want = _oracle_error(O, n, trajs, pols, *cand[c])
            assert abs(err[c] - want) <= 1e-10 * want, (c, err[c], want)
    perm = rng.permutation(M)
    err_p = S.ops.prediction_error(base, data, _cuda(cand[perm])).cpu().numpy()
    assert np.array_equal(err_p, err[perm])  # bit for bit, +inf included
    # the estimator's population objective is this kernel
    db = S.Database()
    for t, W in zip(trajs, pols):
        db.add_trajectory(t, W)
    est = S.Estimator(db, S.EnvParam("sim", n=n, H=H, m_i=1.0, l_i=1.0, h=0.001, k=10.0, epsilon=0.01), capacity=K)
    est.subset = np.arange(K)
    pop = np.array(est.I_population(cand.tolist()))
    ok = np.isfinite(err)
    assert np.array_equal(np.isfinite(pop), ok)
    assert np.all(np.abs(pop[ok] - err[ok]) <= 1e-12 * np.maximum(1.0, err[ok]))


@pytest.mark.gpu
def test_prediction_error_large_population_and_subsets(S, O):
    """M above 256 and d < 3 in any field order: each candidate's sum does not depend on M or its position."""
    n, H, K = 3, 150, 2
    trajs, pols = _record(O, n, H, K, seed=3)
    rng = np.random.default_rng(4)
    M = 1000
    cand = np.array([REAL["k"], REAL["l_i"]]) * (1 + rng.uniform(-0.2, 0.2, (M, 2)))
    data = S.ops.EstimateData(_cuda(trajs), _cuda(pols), ("k", "l_i"), max_candidates=M)
    base = S.make_params(n=n, m_i=REAL["m_i"])
    err = S.ops.prediction_error(base, data, _cuda(cand)).cpu().numpy()
    head = S.ops.prediction_error(base, data, _cuda(cand[:7])).cpu().numpy()
    assert np.array_equal(err[:7], head)
    again = S.ops.prediction_error(base, data, _cuda(cand)).cpu().numpy()
    assert np.array_equal(err, again)
    for c in (0, 999):
        want = _oracle_error(O, n, trajs, pols, REAL["m_i"], cand[c, 1], cand[c, 0])
        assert abs(err[c] - want) <= 1e-10 * want
    exact = S.ops.prediction_error(base, data, _cuda([[REAL["k"], REAL["l_i"]]])).cpu().numpy()
    assert exact[0] < 1e-12


# ---- CMA-ES --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cmaes_sampling(S, O):
    d, lam, seed = 3, 64, 12345
    state = torch.zeros(S.ops.cmaes_state_doubles(d, lam), dtype=torch.float64, device="cuda")
    S.ops.cmaes_init(state, [1.0, 2.0, 3.0], lam, sigma0=0.7)
    v = S.ops.cmaes_view(state, d, lam)
    rng = np.random.default_rng(0)
    A = rng.normal(size=(d, d))
    C = A @ A.T + 0.1 * np.eye(d)
    ev, B = np.linalg.eigh(C)
    v["C"].copy_(_cuda(C)); v["B"].copy_(_cuda(B)); v["D"].copy_(_cuda(np.sqrt(ev)))
    v["generation"].fill_(5.0)
    x = torch.empty(lam, d, dtype=torch.float64, device="cuda")
    S.ops.cmaes_sample(state, d, lam, seed, x)
    z = v["z"].cpu().numpy()
    want = np.array([1.0, 2.0, 3.0]) + 0.7 * (B @ (np.sqrt(ev)[:, None] * z.T)).T
    assert rel_err(x.cpu().numpy(), want) < 1e-14
    # the Philox addressing: counter (pair j, candidate c, generation, stream 2), key = seed
    for c in (0, 1, 63):
        for j in (0, 1):
            o = O.philox([j, c, 5, 2], [seed & 0xffffffff, seed >> 32])
            u0 = ((o[0] >> 5) * 67108864.0 + (o[1] >> 6)) / 9007199254740992.0
            u1 = ((o[2] >> 5) * 67108864.0 + (o[3] >> 6)) / 9007199254740992.0
            r = math.sqrt(-2.0 * math.log(1.0 - u0))
            assert abs(z[c, 2 * j] - r * math.cos(2 * math.pi * u1)) < 1e-14 * max(1.0, r)
            if 2 * j + 1 < d:
                assert abs(z[c, 2 * j + 1] - r * math.sin(2 * math.pi * u1)) < 1e-14 * max(1.0, r)
    z0 = v["z"].clone()
    S.ops.cmaes_sample(state, d, lam, seed, x)
    assert torch.equal(v["z"], z0)
    # 10^5 draws against N(0, 1)
    from scipy import stats
    lam2 = 1000
    st2 = torch.zeros(S.ops.cmaes_state_doubles(2, lam2), dtype=torch.float64, device="cuda")
    S.ops.cmaes_init(st2, [0.0, 0.0], lam2)
    x2 = torch.empty(lam2, 2, dtype=torch.float64, device="cuda")
    draws = []
    for s in range(50):
        S.ops.cmaes_sample(st2, 2, lam2, s, x2)
        draws.append(S.ops.cmaes_view(st2, 2, lam2)["z"].cpu().numpy().ravel())
    draws = np.concatenate(draws)
    assert draws.size == 100000
    assert stats.kstest(draws, "norm").pvalue > 1e-3


@pytest.mark.gpu
def test_cmaes_update_matches_tutorial_equations(S, O):
    n, H = 3, 300
    trajs, pols = _record(O, n, H, 1, seed=21)
    d, lam, seed = 3, 7, 9
    data = S.ops.EstimateData(_cuda(trajs), _cuda(pols), ("m_i", "l_i", "k"), max_candidates=lam)
    base = S.make_params(n=n)
    state = torch.empty(S.ops.cmaes_state_doubles(d, lam), dtype=torch.float64, device="cuda")
    S.ops.cmaes_init(state, [1.0, 1.0, 10.0], lam)
    x = torch.empty(lam, d, dtype=torch.float64, device="cuda")
    f = torch.empty(lam, dtype=torch.float64, device="cuda")
    best = np.inf
    for g in range(30):
        S.ops.cmaes_sample(state, d, lam, seed, x)
        S.ops.prediction_error(base, data, x, out=f)
        prev = _view(S, state, d, lam)
        S.ops.cmaes_update(state, d, lam, x, f)
        now = _view(S, state, d, lam)
        fit, xs = f.cpu().numpy(), x.cpu().numpy()
        assert now["status"] == 0 and now["generation"] == g + 1
        assert rel_err(xs, prev["mean"] + prev["sigma"] * (prev["B"] @ (prev["D"][:, None] * now["z"].T)).T) < 1e-13
        want = _np_update(prev, now["z"], fit, d, lam)
        for key in ("mean", "C", "p_sigma", "p_c"):
            scale = max(np.max(np.abs(want[key])), 1e-300)
            assert np.max(np.abs(now[key] - want[key])) <= 1e-12 * scale, (g, key)
        assert abs(now["sigma"] - want["sigma"]) <= 1e-12 * want["sigma"]
        BD = now["B"] @ np.diag(now["D"] ** 2) @ now["B"].T
        assert np.max(np.abs(BD - now["C"])) <= 1e-12 * np.max(np.abs(now["C"]))
        assert np.max(np.abs(now["B"].T @ now["B"] - np.eye(d))) < 1e-13
        if fit.min() < best:
            best = fit.min()
            assert np.array_equal(now["best_x"], xs[np.argmin(fit)])
        assert now["best_f"] == best


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 5])
@pytest.mark.parametrize("K", [1, 4])
def test_cmaes_recovers_the_real_model(S, O, n, K):
    H = 1000
    trajs, pols = _record(O, n, H, K, seed=10 * n + K)
    db = S.Database()
    for t, W in zip(trajs, pols):
        db.add_trajectory(t, W)
    guess = S.EnvParam("sim", n=n, H=H, m_i=1.0, l_i=1.0, h=0.001, k=10.0, epsilon=0.01)
    est = S.Estimator(db, guess, capacity=K)
    est.subset = np.arange(K)
    p, info = est.estimate_on_device(seed=1)
    for name in ("m_i", "l_i", "k"):
        assert abs(getattr(p, name) - REAL[name]) <= 1e-6 * REAL[name], (name, getattr(p, name), info)
    assert info["stop"] in ("tolfun", "tolx"), info
    assert info["evaluations"] == info["generations"] * info["popsize"] == info["generations"] * 7
    assert info["f"] < 1e-8 and list(info["x"]) == [p.m_i, p.l_i, p.k]
    if n == 3 and K == 1:  # d = 2: the mass is known
        guess2 = S.EnvParam("sim", n=n, H=H, m_i=REAL["m_i"], l_i=1.0, h=0.001, k=10.0, epsilon=0.01)
        est2 = S.Estimator(db, guess2, capacity=1, unknowns=("l_i", "k"))
        est2.subset = np.arange(1)
        p2, info2 = est2.estimate_on_device(seed=2)
        assert abs(p2.l_i - REAL["l_i"]) <= 1e-6 * REAL["l_i"] and abs(p2.k - REAL["k"]) <= 1e-6 * REAL["k"]
        assert p2.m_i == REAL["m_i"] and info2["popsize"] == 6 and info2["stop"] in ("tolfun", "tolx")


@pytest.mark.gpu
def test_cmaes_run_is_deterministic_and_stops_for_good(S, O):
    n, H = 3, 400
    trajs, pols = _record(O, n, H, 1, seed=5)
    db = S.Database()
    db.add_trajectory(trajs[0], pols[0])
    guess = S.EnvParam("sim", n=n, H=H, m_i=1.0, l_i=1.0, h=0.001, k=10.0, epsilon=0.01)
    est = S.Estimator(db, guess, capacity=1)
    p1, i1 = est.estimate_on_device(seed=7, generations_per_poll=1)
    s1 = est.cmaes_state.clone()
    p16, i16 = est.estimate_on_device(seed=7, generations_per_poll=16)
    s16 = est.cmaes_state
    assert torch.equal(s1, s16) and p1 == p16 and i1["generations"] == i16["generations"]
    assert i1["stop"] != "running"
    # replaying generations past the stop changes nothing
    data, lam = est._device_data(7), 7
    x = torch.zeros(lam, 3, dtype=torch.float64, device="cuda")
    f = torch.zeros(lam, dtype=torch.float64, device="cuda")
    for _ in range(3):
        S.ops.cmaes_generation(s16, lam, 7, est._base_params(), data, x, f)
    assert torch.equal(s16, s1)
    assert not x.any() and not f.any()  # no kernel of a stopped generation writes anything
    _, i3 = est.estimate_on_device(seed=8, generations_per_poll=16)
    assert not torch.equal(est.cmaes_state, s1)  # another seed is another run


@pytest.mark.gpu
def test_ars_agent_computed_estimation_without_cma(S, tmp_path, monkeypatch):
    H = 300
    real = S.EnvParam("real", n=3, H=H, l_i=REAL["l_i"], m_i=REAL["m_i"], h=1e-3, k=REAL["k"], epsilon=0.001)
    path = str(tmp_path / "db.npz")
    unsafe = S.ARSParam("unsafe", V1=True, n_iter=10, H=H, N=2, b=2, alpha=0.02, nu=0.05, safe=False,
                        threshold=0.0, initial_w="Zero")
    np.random.seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        S.ARSAgent(real, unsafe, seed=1).runTraining(save_data_path=path)
    monkeypatch.setitem(sys.modules, "cma", None)
    with pytest.raises(ImportError):
        import cma  # noqa: F401
    guess = S.EnvParam("sim", n=3, H=H, l_i=1.0, m_i=1.0, h=1e-3, k=10.0, epsilon=0.001)
    safe = S.ARSParam("safe", V1=True, n_iter=1, H=H, N=2, b=2, alpha=0.02, nu=0.05, safe=True,
                      threshold=-1e9, initial_w="Zero")
    out = io.StringIO()
    with contextlib.redirect_stdout(out):
        ag = S.ARSAgent(real, safe, data_path=path, seed=3, guess_param=guess,
                        sim_thresh=S.Threshold(K=1, A=0.1, B=0.001))
    assert "Using computed estimation..." in out.getvalue()
    for name in ("m_i", "l_i", "k"):
        assert abs(getattr(ag.estimated_param, name) - REAL[name]) <= 1e-6 * REAL[name]
    with contextlib.redirect_stdout(io.StringIO()):
        rets = ag.runOneIteration()
    assert len(rets) in (0, 2, 4)
