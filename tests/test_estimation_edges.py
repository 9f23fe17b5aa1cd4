"""Edges of the simulator-model estimation path (csrc/estimate.cu, the ops.prediction_error / ops.cmaes_* wrappers
and Estimator): the fused prediction-error objective against a high-precision oracle reference at every n, at
transition counts and population sizes on warp, CTA and grid edges, for every field map and for non-finite
candidates and data; CMA-ES sampling against Philox; the CMA-ES update, ranking, eigendecomposition and stop
tests against a numpy restatement of Hansen's tutorial (2016); the composition of the three kernels; guard zones
around every buffer; and the host-side checks of the wrappers and of the Estimator's device data.  The references
are restated here: the product has none."""
import itertools
import math

import numpy as np
import pytest
import torch

from conftest import rel_err

EPS = float(np.finfo(np.float64).eps)
# The recorded ("real") model: every field and h differ from make_params' defaults (1, 1, 10, 0.001), so that a
# wrong field map or a hard-coded h shows.
REAL = dict(m_i=1.2, l_i=0.8, k=10.2, h=0.002)
OFF = dict(m_i=1.5, l_i=0.6, k=9.0)  # the base model's value of a field a candidate replaces
FIELDS = ("m_i", "l_i", "k")
RUNNING, MAXITER, TOLFUN, TOLX, CONDITIONCOV = 0, 1, 2, 3, 4  # swm_cmaes_status

# Tolerance of the objective: |err - ref| <= 1e-12 ref + C_FLOOR eps sum_t ||s_{t+1}||.
# Near the truth each residual r_t = step(s_t) - s_{t+1} is a difference of nearly equal vectors, so what the
# kernel and the reference can disagree by is set by the rounding of the next state, not by |r_t|.  With
# |  ||r_K|| - ||r_O||  | <= ||x'_K - x'_O|| <= ||x'_K - x'|| + ||x'_O - x'|| (x' the exact next state):
#   - each side rounds its final x + h v once: <= eps/2 |x'_i| per component, eps/2 ||x'|| per vector;
#   - the oracle rounds the product h v before the sum, the kernel fuses it: <= eps/2 h |v_i| <= eps/2 |x'_i|
#     for the small steps here (h |v| well below |x|);
#   - the accelerations of the two solves differ by a few units of rounding of |a|, scaled by h = 0.002: below
#     eps/2 ||x'|| as long as h |a| < ||x'|| / (a few), which holds for these bounded recordings.
# That is 4 half-ulps on the kernel's side and on the oracle's, c = 4, with ||x'|| = ||s_{t+1}|| + O(|r_t|).  The
# norms, the kernel's fixed-order sum and math.fsum are relative errors, covered by the 1e-12 ref term.
C_FLOOR = 4.0


def _cuda(a):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _record(O, n, K, H, seed, scale=0.3):
    """K trajectories [K, H, 2n+2] of the real model, recorded by the oracle under V1 policies [K, n-1, 2n+2]."""
    po = O.make_params(n=n, **REAL)
    rng = np.random.default_rng(seed)
    pols = rng.uniform(-1, 1, (K, n - 1, 2 * n + 2)) * scale
    trajs = np.stack([O.rollout(po, 0, H, policy=W, want_traj=True)[2] for W in pols])
    return trajs, pols


class _Reference:
    """The objective restated: every transition stepped by the oracle (O.step_batch) with the action s_t W_k^T,
    each residual's norm in float64, all norms summed exactly (math.fsum)."""

    def __init__(self, O, n, trajs, pols):
        self.O, self.n = O, n
        self.s0 = np.concatenate([t[:-1] for t in trajs])
        self.a = np.concatenate([t[:-1] @ W.T for t, W in zip(trajs, pols)])
        self.s1 = np.concatenate([t[1:] for t in trajs])
        self.floor = C_FLOOR * EPS * math.fsum(np.linalg.norm(self.s1, axis=1))

    def err(self, unknowns, x, base=REAL):
        p = dict(base)
        p.update(zip(unknowns, (float(v) for v in x)))
        nxt, _ = self.O.step_batch(self.O.make_params(n=self.n, **p), 0, self.s0, self.a)
        return math.fsum(np.linalg.norm(nxt - self.s1, axis=1))

    def check(self, got, unknowns, x, what):
        want = self.err(unknowns, x)
        assert abs(got - want) <= 1e-12 * want + self.floor, (what, got, want, self.floor)


def _base(S, n, unknowns):
    """Base model: the real value of every fixed field and h, a wrong value in every field a candidate replaces."""
    p = dict(REAL)
    p.update({f: OFF[f] for f in unknowns})
    return S.make_params(n=n, **p)


def _near_truth(rng, unknowns, M, rel=1e-8):
    """M candidates: the exact truth first, then the truth moved by up to `rel` (relative) in every unknown."""
    truth = np.array([REAL[f] for f in unknowns])
    cand = truth * (1 + rng.uniform(-rel, rel, (M, len(unknowns))))
    cand[0] = truth
    return cand


def _data(S, trajs, pols, unknowns, M):
    return S.ops.EstimateData(_cuda(trajs), _cuda(pols), unknowns, max_candidates=M)


# ---- A. objective ------------------------------------------------------------------------------------------------
# (K, H): T = K (H - 1) transitions = 1, 127, 128 (one full CTA), 129 with H - 1 = 43 (CTAs span trajectory
# boundaries), 257 in one trajectory, and 257 trajectories of H = 2 (every lane of a warp has its own policy).
SHAPES = [(1, 2), (1, 128), (1, 129), (3, 44), (1, 258), (257, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("K,H", SHAPES, ids=["T%d_K%d" % (k * (h - 1), k) for k, h in SHAPES])
@pytest.mark.parametrize("n", range(2, 11))
def test_objective_matches_reference_every_n_and_transition_count(S, O, n, K, H):
    trajs, pols = _record(O, n, K, H, seed=100 * n + K + H)
    ref = _Reference(O, n, trajs, pols)
    rng = np.random.default_rng(n * H)
    M = 33
    cand = _near_truth(rng, FIELDS, M)
    cand[1] = (REAL["m_i"] * (1 + 1e-8), REAL["l_i"], REAL["k"])
    data = _data(S, trajs, pols, FIELDS, M)
    base = _base(S, n, FIELDS)
    err = S.ops.prediction_error(base, data, _cuda(cand)).cpu().numpy()
    assert 0.0 <= err[0] <= ref.floor, (err[0], ref.floor)  # the exact truth: rounding only
    for c in range(1, M):
        ref.check(err[c], FIELDS, cand[c], c)
    # The tolerance resolves the candidate to ~1e-12: candidate 1 is m_i (1 + 1e-8); the reference at
    # m_i (1 + 1.0001e-8), 1.2e-12 (about 5000 ulps of m_i) further, disagrees with the kernel.
    want = ref.err(FIELDS, (REAL["m_i"] * (1 + 1.0001e-8), REAL["l_i"], REAL["k"]))
    assert abs(err[1] - want) > 1e-12 * want + ref.floor, (err[1], want, ref.floor)
    perm = rng.permutation(M)
    assert np.array_equal(S.ops.prediction_error(base, data, _cuda(cand[perm])).cpu().numpy(), err[perm])
    assert np.array_equal(S.ops.prediction_error(base, data, _cuda(cand)).cpu().numpy(), err)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 8, 10])
def test_objective_population_sizes_and_prefix_bit_identity(S, O, n):
    """M on warp (32), CTA (128) and reduce-grid (129) edges up to SWM_MAX_CANDIDATES; n = 10 with M = 1024 is the
    largest shared-memory size (candidate constants, warp partials and factorisation rows, ~194 KiB)."""
    K, H = 3, 44  # T = 129: a ragged second CTA, CTAs across trajectory boundaries
    trajs, pols = _record(O, n, K, H, seed=n)
    ref = _Reference(O, n, trajs, pols)
    rng = np.random.default_rng(7 * n)
    cand = _near_truth(rng, FIELDS, 1024)
    data = _data(S, trajs, pols, FIELDS, 1024)
    base = _base(S, n, FIELDS)
    full = S.ops.prediction_error(base, data, _cuda(cand)).cpu().numpy()
    assert 0.0 <= full[0] <= ref.floor
    for M in (1, 31, 32, 33, 127, 128, 129, 1024):
        head = S.ops.prediction_error(base, _data(S, trajs, pols, FIELDS, M), _cuda(cand[:M])).cpu().numpy()
        assert np.array_equal(head, full[:M]), M  # a candidate's sum depends on neither M nor the workspace
    sample = {1, 31, 32, 33, 127, 128, 129, 255, 256, 1022, 1023} | set(rng.integers(1, 1024, 16).tolist())
    for c in sorted(sample):
        ref.check(full[c], FIELDS, cand[c], c)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4, 9])
def test_objective_every_field_map(S, O, n):
    """d = 1 for each field, every ordered pair, every order of the three: candidate coordinate i replaces
    fields[i] of a base model whose replaced fields are wrong and whose fixed fields and h are the real ones."""
    trajs, pols = _record(O, n, 2, 80, seed=n)
    ref = _Reference(O, n, trajs, pols)
    rng = np.random.default_rng(n)
    maps = [m for d in (1, 2, 3) for m in itertools.permutations(FIELDS, d)]
    assert len(maps) == 3 + 6 + 6
    for unknowns in maps:
        cand = _near_truth(rng, unknowns, 9)
        err = S.ops.prediction_error(_base(S, n, unknowns), _data(S, trajs, pols, unknowns, 9),
                                     _cuda(cand)).cpu().numpy()
        assert err[0] <= ref.floor, (unknowns, err[0])
        for c in range(1, 9):
            ref.check(err[c], unknowns, cand[c], (unknowns, c))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 10])
def test_objective_non_physical_candidates(S, O, n):
    trajs, pols = _record(O, n, 2, 60, seed=n)
    ref = _Reference(O, n, trajs, pols)
    inf, nan = math.inf, math.nan
    m, l, k = REAL["m_i"], REAL["l_i"], REAL["k"]
    bad = [(0.0, l, k), (-0.0, l, k), (-1.0, l, k), (-inf, l, k), (m, 0.0, k), (m, -0.0, k), (m, -0.5, k),
           (nan, l, k), (m, nan, k), (m, l, nan), (inf, l, k), (m, inf, k), (inf, inf, k)]
    good = [(m, l, 0.0), (m, l, -0.0), (m, l, -3.5), (m, l, k)]  # k <= 0 is physical
    cand = np.array(bad + good)
    err = S.ops.prediction_error(_base(S, n, FIELDS), _data(S, trajs, pols, FIELDS, len(cand)),
                                 _cuda(cand)).cpu().numpy()
    for c, x in enumerate(bad):
        assert err[c] == math.inf, (x, err[c])
    for c, x in enumerate(good, len(bad)):
        assert np.isfinite(err[c]), (x, err[c])
        ref.check(err[c], FIELDS, x, x)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 8])
@pytest.mark.parametrize("where", ["state", "last_state", "policy"])
@pytest.mark.parametrize("value", [math.nan, math.inf, -math.inf], ids=["nan", "inf", "-inf"])
def test_objective_non_finite_data_makes_every_candidate_inf(S, O, n, where, value):
    K, H = 3, 44
    trajs, pols = _record(O, n, K, H, seed=n)
    if where == "state":
        trajs[1, 20, 3] = value
    elif where == "last_state":
        trajs[2, H - 1, 2 * n + 1] = value
    else:
        pols[1, n - 2, 2] = value
    cand = _near_truth(np.random.default_rng(0), FIELDS, 40)
    cand[5] = (0.0, REAL["l_i"], REAL["k"])
    err = S.ops.prediction_error(_base(S, n, FIELDS), _data(S, trajs, pols, FIELDS, 40), _cuda(cand)).cpu().numpy()
    assert np.all(err == math.inf), err


# ---- B. CMA-ES sampling ------------------------------------------------------------------------------------------
def _u53(a, b):
    return ((a >> 5) * 67108864.0 + (b >> 6)) / 9007199254740992.0


@pytest.mark.gpu
@pytest.mark.parametrize("lam", [2, 3, 129, 1024])
@pytest.mark.parametrize("d", [1, 2, 3])
def test_cmaes_sampling_against_philox(S, O, d, lam):
    seed, gen = 0xC0FFEE0012345678, 70001  # high key word set; the generation counter above 2^16
    state = torch.zeros(S.ops.cmaes_state_doubles(d, lam), dtype=torch.float64, device="cuda")
    S.ops.cmaes_init(state, [1.0, -2.0, 3.0][:d], lam, sigma0=0.37)
    v = S.ops.cmaes_view(state, d, lam)
    rng = np.random.default_rng(d * lam)
    B, _ = np.linalg.qr(rng.normal(size=(d, d)))
    D = rng.uniform(0.5, 2.0, d)
    v["B"].copy_(_cuda(B)); v["D"].copy_(_cuda(D)); v["generation"].fill_(float(gen))
    before = state.cpu().numpy()
    x = torch.full((lam, d), -777.25, dtype=torch.float64, device="cuda")
    S.ops.cmaes_sample(state, d, lam, seed, x)
    after = state.cpu().numpy()
    z0 = S.ops.cmaes_view(torch.as_tensor(before), d, lam)["z"].numel()
    assert np.array_equal(after[:-z0], before[:-z0])  # sampling writes z only
    z, xs = v["z"].cpu().numpy(), x.cpu().numpy()
    for c in range(lam):
        for j in range((d + 1) // 2):
            o = O.philox([j, c, gen, 2], [seed & 0xffffffff, seed >> 32])
            r = math.sqrt(-2.0 * math.log(1.0 - _u53(o[0], o[1])))
            ang = 2.0 * math.pi * _u53(o[2], o[3])
            assert abs(z[c, 2 * j] - r * math.cos(ang)) <= 1e-14 * max(1.0, r), (c, j)
            if 2 * j + 1 < d:
                assert abs(z[c, 2 * j + 1] - r * math.sin(ang)) <= 1e-14 * max(1.0, r), (c, j)
    want = np.array([1.0, -2.0, 3.0][:d]) + 0.37 * (B @ (D[:, None] * z.T)).T
    assert rel_err(xs, want) <= 1e-14


# ---- C. CMA-ES update against the tutorial, restated ---------------------------------------------------------------
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


def _rank(fit):
    """Ascending; +inf and NaN last; -inf an ordinary value (first); ties by the lower index."""
    bad = [not (f < math.inf) for f in fit]
    return sorted(range(len(fit)), key=lambda c: (bad[c], 0.0 if bad[c] else fit[c], c))


def _ref_stop(gen, L, fbest, fworst, hist, sigma, C, pc, tolfun, tolx, max_gen):
    """Stop tests in the header's order: tolfun, tolx, condition, max generations."""
    if gen >= L:
        lo, hi = np.fmin.reduce(np.append(hist, fbest)), np.fmax.reduce(np.append(hist, fworst))
        if hi - lo < tolfun:
            return TOLFUN
    d = len(pc)
    if all(sigma * math.sqrt(C[i, i]) < tolx and sigma * abs(pc[i]) < tolx for i in range(d)):
        return TOLX
    ev = np.linalg.eigvalsh(C)
    if not (ev.min() > 0 and ev.max() / ev.min() <= 1e14):
        return CONDITIONCOV
    if gen >= max_gen:
        return MAXITER
    return RUNNING


def _ref_update(prev, cand, fit, d, lam):
    """One generation of the tutorial's CMA-ES from the state before the update -> (state after, h_sigma)."""
    w, mueff, cs, ds, cc, c1, cmu, chiN = _strategy(d, lam)
    order = _rank(fit)
    sel = order[:len(w)]
    B, D, C, sigma, z = prev["B"], prev["D"], prev["C"], float(prev["sigma"]), prev["z"]
    y = (B @ (D[:, None] * z.T)).T
    yw, zw = w @ y[sel], w @ z[sel]
    gen = float(prev["generation"]) + 1
    out = {k: np.array(v, copy=True) for k, v in prev.items()}
    out["mean"] = prev["mean"] + sigma * yw
    # C^{-1/2} <y>_w = B D^{-1} B^T B D <z>_w = B <z>_w (also for a singular D)
    ps = (1 - cs) * prev["p_sigma"] + math.sqrt(cs * (2 - cs) * mueff) * (B @ zw)
    psn = float(np.linalg.norm(ps))
    hsig = psn / math.sqrt(1 - (1 - cs) ** (2 * gen)) < (1.4 + 2 / (d + 1)) * chiN
    pc = (1 - cc) * prev["p_c"] + (math.sqrt(cc * (2 - cc) * mueff) * yw if hsig else 0.0)
    dh = 0.0 if hsig else cc * (2 - cc)
    rmu = sum(wi * np.outer(yi, yi) for wi, yi in zip(w, y[sel]))
    C = (1 + c1 * dh - c1 - cmu * w.sum()) * C + c1 * np.outer(pc, pc) + cmu * rmu
    sigma_new = sigma * math.exp(cs / ds * (psn / chiN - 1))
    out.update(p_sigma=ps, p_c=pc, C=C, sigma=np.float64(sigma_new), generation=np.float64(gen))
    fbest = fit[order[0]]
    if fbest < prev["best_f"]:
        out["best_f"], out["best_x"] = np.float64(fbest), cand[order[0]].copy()
    L = len(out["history"])
    out["history"][int(prev["generation"]) % L] = fbest
    out["status"] = np.float64(_ref_stop(gen, L, fbest, fit[order[-1]], out["history"], sigma_new, C, pc,
                                         float(prev["tolfun"]), float(prev["tolx"]), float(prev["max_generations"])))
    return out, hsig


def _view(S, state, d, lam):
    return {k: v.cpu().numpy().copy() for k, v in S.ops.cmaes_view(state, d, lam).items()}


def _assert_state(now, want, d, what):
    for key in ("generation", "status", "max_generations", "tolfun", "tolx"):
        assert now[key] == want[key], (what, key, now[key], want[key])
    assert np.array_equal(now["best_x"], want["best_x"]) and now["best_f"] == want["best_f"], what
    assert np.array_equal(now["history"], want["history"], equal_nan=True), what
    assert np.array_equal(now["z"], want["z"]), what
    for key in ("mean", "p_sigma", "p_c", "C"):
        scale = max(float(np.max(np.abs(want[key]))), 1e-300)
        assert np.max(np.abs(now[key] - want[key])) <= 1e-12 * scale, (what, key, now[key], want[key])
    assert abs(now["sigma"] - want["sigma"]) <= 1e-12 * want["sigma"], (what, now["sigma"], want["sigma"])
    # B and D: the eigenpairs of the new C, in whatever order and sign the Jacobi sweeps leave them
    C, B, D = now["C"], now["B"], now["D"]
    ev = np.linalg.eigvalsh(C)
    scale = float(np.max(np.abs(C)))
    assert np.max(np.abs(np.sort(D ** 2) - np.maximum(ev, 0.0))) <= 1e-12 * scale, (what, D ** 2, ev)
    assert np.max(np.abs(B.T @ B - np.eye(d))) <= 1e-13, what
    assert np.max(np.abs(B @ np.diag(D ** 2) @ B.T - C)) <= 1e-12 * scale, what


def _generation(S, state, d, lam, seed, fitness_of, before_update=None):
    """sample on the device, fitness in numpy, update on the device; the whole state after it against the
    restatement applied to the state before it -> (state after, the restatement's h_sigma, fitness)."""
    x = torch.empty(lam, d, dtype=torch.float64, device="cuda")
    S.ops.cmaes_sample(state, d, lam, seed, x)
    if before_update is not None:
        before_update(S.ops.cmaes_view(state, d, lam))
    prev = _view(S, state, d, lam)
    xs = x.cpu().numpy()
    fit = np.asarray(fitness_of(xs), dtype=np.float64)
    S.ops.cmaes_update(state, d, lam, x, _cuda(fit))
    now = _view(S, state, d, lam)
    want, hsig = _ref_update(prev, xs, fit, d, lam)
    _assert_state(now, want, d, int(prev["generation"]))
    return now, hsig, fit


def _quadratic(d, seed=0):
    """A rotated quadratic with condition 1e4 around x* = (0.3, -0.2, 0.5)[:d]."""
    Q, _ = np.linalg.qr(np.random.default_rng(seed).normal(size=(d, d)))
    A = Q @ np.diag([1.0, 1e2, 1e4][:d]) @ Q.T
    xs = np.array([0.3, -0.2, 0.5][:d])
    return lambda x: np.einsum("ci,ij,cj->c", x - xs, A, x - xs)


def _init(S, d, lam, x0=(1.0, 1.0, 1.0), **kw):
    state = torch.empty(S.ops.cmaes_state_doubles(d, lam), dtype=torch.float64, device="cuda")
    S.ops.cmaes_init(state, list(x0[:d]), lam, **kw)
    return state


LAMBDAS = [2, 3, 4, 6, 7, 32, 33, 64, 1000, 1024]


@pytest.mark.gpu
@pytest.mark.parametrize("lam", LAMBDAS)
@pytest.mark.parametrize("d", [1, 2, 3])
def test_cmaes_update_matches_restatement(S, d, lam):
    """20 generations; every generation's whole state against the restatement.  Ties (gen 3), NaN and +inf
    (gen 5), an all-+inf generation (gen 9), a forced h_sigma = false (gen 11), -inf (gen 17)."""
    state = _init(S, d, lam, sigma0=0.5)
    v0 = _view(S, state, d, lam)
    assert v0["max_generations"] == 100 + math.floor(150 * (d + 3) ** 2 / math.sqrt(lam))
    f = _quadratic(d, seed=lam)
    cs = _strategy(d, lam)[2]  # p_sigma of 20 / (1 - c_sigma) decays to norm ~20 in the update: h_sigma = false

    def fitness(g):
        def fit(x):
            v = f(x)
            if g == 3:
                v = np.round(v, 0)  # many ties: ranked by the lower index
            elif g == 5:
                v[0], v[-1] = math.nan, math.inf
            elif g == 9:
                v[:] = math.inf
            elif g == 17:
                v[lam // 2] = -math.inf
            return v
        return fit

    for g in range(20):
        best_before = _view(S, state, d, lam)["best_f"]
        force = (lambda v: v["p_sigma"].fill_(20.0 / ((1 - cs) * math.sqrt(d)))) if g == 11 else None
        now, hsig, fit = _generation(S, state, d, lam, seed=lam + 1, fitness_of=fitness(g), before_update=force)
        if g == 9:
            assert now["best_f"] == best_before  # no finite fitness: best-ever unchanged
        if g == 11:
            assert not hsig
        if g == 17:
            assert now["best_f"] == -math.inf
        if now["status"] != RUNNING:
            break


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["ties", "-inf", "nan_inf"])
def test_cmaes_ranking_ties_and_non_finite(S, case):
    """Fitness with a tie at the minimum, -inf, or NaN and +inf at chosen indices: the ranking shows in best-ever
    and, through the recombination weights, in the mean the restatement checks."""
    d, lam = 2, 33
    v = np.arange(lam, 0, -1, dtype=np.float64)  # without edits the last index is the best
    if case == "ties":
        v[[9, 4, 30]] = 0.5  # a tie at the minimum: index 4 ranks first
    elif case == "-inf":
        v[20] = -math.inf  # an ordinary value, and the least
    else:
        v[[0, 32]] = math.nan  # the two smallest indices and the best value become NaN / +inf: ranked last
        v[[1, 31]] = math.inf
    best = {"ties": 4, "-inf": 20, "nan_inf": 30}[case]
    state = _init(S, d, lam)
    x = torch.empty(lam, d, dtype=torch.float64, device="cuda")
    S.ops.cmaes_sample(state, d, lam, 3, x)
    xs = x.cpu().numpy()
    S.ops.cmaes_update(state, d, lam, x, _cuda(v))
    now = _view(S, state, d, lam)
    assert now["best_f"] == v[best] and np.array_equal(now["best_x"], xs[best])
    state = _init(S, d, lam)
    _generation(S, state, d, lam, seed=3, fitness_of=lambda _: v)


# ---- C. Jacobi eigendecomposition and stop tests -----------------------------------------------------------------
def _rot(d, angle):
    if d == 2:
        c, s = math.cos(angle), math.sin(angle)
        return np.array([[c, -s], [s, c]])
    Q, _ = np.linalg.qr(np.random.default_rng(int(angle * 1000)).normal(size=(d, d)))
    return Q


EIGEN_CASES = {
    "repeated": (3, _rot(3, 0.4) @ np.diag([2.0, 2.0, 5.0]) @ _rot(3, 0.4).T, RUNNING),
    "scalar": (3, 3.0 * np.eye(3), RUNNING),
    "diagonal": (3, np.diag([1.0, 4.0, 9.0]), RUNNING),
    "tiny_offdiagonal": (2, np.array([[1.0, 1e-160], [1e-160, 2.0]]), RUNNING),  # |theta| > 1e150
    "tiny_offdiagonal_3": (3, np.array([[1.0, 1e-160, 0.0], [1e-160, 2.0, 3e-170], [0.0, 3e-170, 4.0]]), RUNNING),
    "condition_below": (2, _rot(2, 0.3) @ np.diag([1.0, 1.0 / 0.8e14]) @ _rot(2, 0.3).T, RUNNING),
    "condition_above": (2, _rot(2, 0.3) @ np.diag([1.0, 1.0 / 1.25e14]) @ _rot(2, 0.3).T, CONDITIONCOV),
    "condition_above_3": (3, _rot(3, 0.7) @ np.diag([1.0, 0.5, 1.0 / 1.25e14]) @ _rot(3, 0.7).T, CONDITIONCOV),
}


def _freeze_to(C):
    """State edit before an update so that the new C is exactly keep * C: D = 0 (every y = 0, so the rank-mu
    and rank-one terms vanish with p_c = 0); tolfun and tolx are 0 from the init."""
    def edit(v):
        v["C"].copy_(_cuda(C)); v["D"].zero_(); v["p_c"].zero_()
    return edit


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(EIGEN_CASES))
def test_cmaes_jacobi_eigendecomposition(S, case):
    d, C, status = EIGEN_CASES[case]
    lam = 2
    state = _init(S, d, lam, tolfun=0.0, tolx=0.0)
    now, _, _ = _generation(S, state, d, lam, seed=1, fitness_of=lambda x: np.array([1.0, 2.0]),
                            before_update=_freeze_to(C))
    assert now["status"] == status
    ev = np.sort(now["D"] ** 2)
    want = np.linalg.eigvalsh(now["C"])
    assert np.max(np.abs(ev - want)) <= 1e-14 * np.max(want), (ev, want)
    if case in ("diagonal", "scalar"):  # apq == 0: no rotation at all
        assert np.array_equal(now["B"], np.eye(d)) and np.array_equal(now["D"], np.sqrt(np.diag(now["C"])))


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 2, 3])
def test_cmaes_stop_tests_and_precedence(S, d):
    lam = 6
    L = 10 + -(-30 * d // lam)
    f = _quadratic(d)
    rng = np.random.default_rng(d)

    def run(state, fitness_of=f, edit=None, gens=1):
        for _ in range(gens):
            now, _, _ = _generation(S, state, d, lam, seed=5, fitness_of=fitness_of, before_update=edit)
            if now["status"] != RUNNING:
                return now
        return now

    # tolx alone fires in the first generation; tolfun alone when the history first fills (generation L)
    assert run(_init(S, d, lam, tolfun=0.0, tolx=1e300))["status"] == TOLX
    now = run(_init(S, d, lam, tolfun=1e300, tolx=0.0), gens=L + 1)
    assert now["status"] == TOLFUN and now["generation"] == L
    # tolfun after the ring has wrapped: varied fitness up to generation L + 3, constant afterwards
    state = _init(S, d, lam, tolx=0.0)
    count = [0]

    def plateau(x):
        count[0] += 1
        return rng.uniform(0, 1, lam) if count[0] <= L + 3 else np.ones(lam)

    now = run(state, fitness_of=plateau, gens=3 * L)
    assert now["status"] == TOLFUN and now["generation"] == 2 * L + 3 > L
    # maxiter, given and default
    now = run(_init(S, d, lam, tolfun=0.0, tolx=0.0, max_generations=3), gens=5)
    assert now["status"] == MAXITER and now["generation"] == 3
    state = _init(S, d, lam, tolfun=0.0, tolx=0.0)
    default = 100 + math.floor(150 * (d + 3) ** 2 / math.sqrt(lam))
    S.ops.cmaes_view(state, d, lam)["generation"].fill_(default - 1)
    now = run(state)
    assert now["status"] == MAXITER and now["generation"] == default == now["max_generations"]

    # two or more in the same generation: tolfun > tolx > condition > max generations
    def at_last(state):
        S.ops.cmaes_view(state, d, lam)["generation"].fill_(L - 1)
        return state

    assert run(at_last(_init(S, d, lam, tolfun=1e300, tolx=1e300, max_generations=L)))["status"] == TOLFUN
    assert run(_init(S, d, lam, tolfun=0.0, tolx=1e300, max_generations=1))["status"] == TOLX
    if d >= 2:
        ill = EIGEN_CASES["condition_above" if d == 2 else "condition_above_3"][1]
        now = run(_init(S, d, lam, tolfun=0.0, tolx=0.0, max_generations=1), edit=_freeze_to(ill))
        assert now["status"] == CONDITIONCOV
        now = run(_init(S, d, lam, tolfun=0.0, tolx=1e300), edit=_freeze_to(ill))
        assert now["status"] == TOLX

    # after a stop, every kernel is a no-op: the state, the candidates and the fitness keep their bits
    state = _init(S, d, lam, tolfun=0.0, tolx=1e300)
    assert run(state)["status"] == TOLX
    trajs = torch.zeros(1, 2, 8, dtype=torch.float64, device="cuda")
    data = S.ops.EstimateData(trajs, torch.zeros(1, 2, 8, dtype=torch.float64, device="cuda"), FIELDS[:d], lam)
    s0 = state.clone()
    x = torch.full((lam, d), -777.25, dtype=torch.float64, device="cuda")
    fit = torch.full((lam,), -555.5, dtype=torch.float64, device="cuda")
    S.ops.cmaes_sample(state, d, lam, 9, x)
    S.ops.cmaes_update(state, d, lam, x, fit)
    S.ops.cmaes_generation(state, lam, 9, S.make_params(n=3), data, x, fit)
    assert torch.equal(state, s0) and bool((x == -777.25).all()) and bool((fit == -555.5).all())


# ---- D. composition --------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("lam", [2, 33])
def test_generation_equals_sample_objective_update(S, O, lam):
    n, d = 3, 3
    trajs, pols = _record(O, n, 2, 60, seed=lam)
    data = _data(S, trajs, pols, FIELDS, lam)
    base = _base(S, n, FIELDS)
    a, b = _init(S, d, lam, x0=(1.0, 1.0, 10.0)), _init(S, d, lam, x0=(1.0, 1.0, 10.0))
    xa, xb = (torch.empty(lam, d, dtype=torch.float64, device="cuda") for _ in range(2))
    fa, fb = (torch.empty(lam, dtype=torch.float64, device="cuda") for _ in range(2))
    for _ in range(12):
        S.ops.cmaes_generation(a, lam, 11, base, data, xa, fa)
        S.ops.cmaes_sample(b, d, lam, 11, xb)
        S.ops.prediction_error(base, data, xb, out=fb)
        S.ops.cmaes_update(b, d, lam, xb, fb)
        assert torch.equal(a, b) and torch.equal(xa, xb) and torch.equal(fa, fb)


@pytest.mark.gpu
def test_graph_replay_equals_eager_generations(S, O):
    n, d, lam, G = 4, 2, 6, 4
    trajs, pols = _record(O, n, 2, 50, seed=4)
    unknowns = ("k", "m_i")
    data = _data(S, trajs, pols, unknowns, lam)
    base = _base(S, n, unknowns)
    eager, graphed = _init(S, d, lam, x0=(10.0, 1.0)), _init(S, d, lam, x0=(10.0, 1.0))
    xe, xg = (torch.empty(lam, d, dtype=torch.float64, device="cuda") for _ in range(2))
    fe, fg = (torch.empty(lam, dtype=torch.float64, device="cuda") for _ in range(2))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(G):
            S.ops.cmaes_generation(graphed, lam, 5, base, data, xg, fg)
    for rep in range(3):
        graph.replay()
        for _ in range(G):
            S.ops.cmaes_generation(eager, lam, 5, base, data, xe, fe)
        torch.cuda.synchronize()
        assert torch.equal(eager, graphed) and torch.equal(xe, xg) and torch.equal(fe, fg), rep


def _estimator(S, O, n, K, H, unknowns, seed):
    trajs, pols = _record(O, n, K, H, seed=seed)
    db = S.Database()
    for t, W in zip(trajs, pols):
        db.add_trajectory(t, W)
    g = dict(REAL)
    g.update({f: OFF[f] for f in unknowns})
    guess = S.EnvParam("sim", n=n, H=H, epsilon=0.01, **g)
    est = S.Estimator(db, guess, capacity=K, unknowns=unknowns)
    est.subset = np.arange(K)
    return est


@pytest.mark.gpu
@pytest.mark.parametrize("unknowns", [("k",), ("l_i",), ("m_i", "k"), ("k", "l_i")], ids="_".join)
@pytest.mark.parametrize("n", [2, 8])
def test_estimate_on_device_recovers_the_real_model(S, O, n, unknowns):
    est = _estimator(S, O, n, 1, 400, unknowns, seed=n)
    p, info = est.estimate_on_device(seed=3)
    for name in FIELDS:
        want = REAL[name]
        assert abs(getattr(p, name) - want) <= 1e-6 * want, (name, getattr(p, name), info)
    assert p.h == REAL["h"] and info["stop"] in ("tolfun", "tolx"), info
    assert info["popsize"] == S.ops.cmaes_default_popsize(len(unknowns))


@pytest.mark.gpu
def test_population_objective_follows_the_subset(S, O):
    est = _estimator(S, O, 5, 4, 70, FIELDS, seed=9)
    xs = _near_truth(np.random.default_rng(1), FIELDS, 6, rel=1e-3).tolist()
    est.subset = np.array([0, 1])
    first = est.I_population(xs)
    est.subset = np.array([3, 2])
    pop = est.I_population(xs)
    one = [est.I(x) for x in xs]
    s1 = [np.asarray(est.database.trajectories[k])[1:] for k in est.subset]
    floor = 2 * C_FLOOR * EPS * math.fsum(np.linalg.norm(np.concatenate(s1), axis=1))  # two kernels, each near the oracle
    for p, q, r in zip(pop, one, first):
        assert abs(p - q) <= 1e-12 * q + floor, (p, q)
        assert p != r
    est.subset[1] = 0  # an in-place edit is a new subset too
    assert est.I_population(xs[:2]) == pytest.approx([est.I(x) for x in xs[:2]], rel=1e-12)


# ---- E. guard zones ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("lam", [2, 33, 1024])
def test_no_out_of_bounds_writes_estimation(S, O, lam):
    """The objective's workspace and output, the candidates, the fitness and the CMA-ES state, each inside a
    larger allocation filled with a sentinel: after the objective, sampling, update and whole generations at a
    ragged transition count, the guard zones are untouched and every output was written."""
    n, d, K, H = 8, 3, 3, 44  # T = 129: two CTAs, the second with one transition
    SENT, PAD = -777.25, 4096
    trajs, pols = _record(O, n, K, H, seed=lam)
    data = _data(S, trajs, pols, FIELDS, lam)

    def guarded(numel):
        big = torch.full((numel + 2 * PAD,), SENT, dtype=torch.float64, device="cuda")
        return big, big[PAD:PAD + numel]

    ws_big, ws = guarded(data.workspace.numel())
    data.workspace = ws
    data.c.workspace = ws.data_ptr()
    err_big, err = guarded(lam)
    x_big, x = guarded(lam * d)
    f_big, f = guarded(lam)
    s_big, state = guarded(S.ops.cmaes_state_doubles(d, lam))
    x = x.view(lam, d)
    base = _base(S, n, FIELDS)
    S.ops.cmaes_init(state, [REAL["m_i"], REAL["l_i"], REAL["k"]], lam, sigma0=0.01)
    S.ops.cmaes_sample(state, d, lam, 1, x)
    S.ops.prediction_error(base, data, x, out=err)
    S.ops.cmaes_update(state, d, lam, x, err)
    for _ in range(2):
        S.ops.cmaes_generation(state, lam, 1, base, data, x, f)
    torch.cuda.synchronize()
    for name, (big, view) in dict(workspace=(ws_big, ws), err=(err_big, err), candidates=(x_big, x),
                                  fitness=(f_big, f), state=(s_big, state)).items():
        assert bool((big[:PAD] == SENT).all()) and bool((big[-PAD:] == SENT).all()), (lam, name)
        assert not bool((view == SENT).any()), (lam, name)
    assert int(S.ops.cmaes_view(state, d, lam)["generation"]) == 3


# ---- host-side checks (no device needed) -------------------------------------------------------------------------
def _cpu_data(S, n=3, K=2, H=10, unknowns=FIELDS, max_candidates=7):
    no = 2 * n + 2
    return S.ops.EstimateData(torch.zeros(K, H, no, dtype=torch.float64), torch.zeros(K, n - 1, no, dtype=torch.float64),
                              unknowns, max_candidates=max_candidates)


def test_generation_refuses_a_population_larger_than_the_workspace(S):
    data = _cpu_data(S, max_candidates=7)
    state = torch.zeros(S.ops.cmaes_state_doubles(3, 64), dtype=torch.float64)
    x, f = torch.zeros(64, 3, dtype=torch.float64), torch.zeros(64, dtype=torch.float64)
    with pytest.raises(ValueError, match="popsize 64 exceeds the 7 candidates"):
        S.ops.cmaes_generation(state, 64, 0, S.make_params(n=3), data, x, f)


def test_objective_refuses_a_model_of_another_n(S):
    data = _cpu_data(S, n=3)
    x, f = torch.zeros(7, 3, dtype=torch.float64), torch.zeros(7, dtype=torch.float64)
    state = torch.zeros(S.ops.cmaes_state_doubles(3, 7), dtype=torch.float64)
    for n in (2, 4, 10):
        with pytest.raises(ValueError, match="n=%d segments, the recorded data n=3" % n):
            S.ops.prediction_error(S.make_params(n=n), data, x)
        with pytest.raises(ValueError, match="n=%d segments, the recorded data n=3" % n):
            S.ops.cmaes_generation(state, 7, 0, S.make_params(n=n), data, x, f)


def test_estimation_wrappers_validate_their_tensors(S):
    d, lam = 3, 7
    need = S.ops.cmaes_state_doubles(d, lam)
    f64 = dict(dtype=torch.float64)
    state, x, f = torch.zeros(need, **f64), torch.zeros(lam, d, **f64), torch.zeros(lam, **f64)
    data, base = _cpu_data(S, max_candidates=lam), S.make_params(n=3)
    bad_state = [(torch.zeros(need - 1, **f64), "state must hold at least %d doubles" % need),
                 (torch.zeros(need, dtype=torch.float32), "state must be a float64 tensor"),
                 (torch.zeros(2 * need, **f64)[::2], "state must be contiguous"),
                 (state, "must be a CUDA tensor")]
    bad_x = [(torch.zeros(lam, d + 1, **f64), r"candidates must have shape \(7, 3\)"),
             (torch.zeros(lam * d, **f64), r"candidates must have shape \(7, 3\)"),
             (torch.zeros(lam, d, dtype=torch.float32), "candidates must be a float64 tensor"),
             (torch.zeros(d, lam, **f64).t(), "candidates must be contiguous")]
    bad_f = [(torch.zeros(lam + 1, **f64), r"fitness must have shape \(7,\)"),
             (torch.zeros(lam, 1, **f64), r"fitness must have shape \(7,\)"),
             (torch.zeros(lam, dtype=torch.int64), "fitness must be a float64 tensor"),
             (torch.zeros(2 * lam, **f64)[::2], "fitness must be contiguous")]
    for s, msg in bad_state:
        with pytest.raises(ValueError, match=msg):
            S.ops.cmaes_sample(s, d, lam, 0, x)
        with pytest.raises(ValueError, match=msg):
            S.ops.cmaes_update(s, d, lam, x, f)
        with pytest.raises(ValueError, match=msg):
            S.ops.cmaes_generation(s, lam, 0, base, data, x, f)
    for c, msg in bad_x:
        with pytest.raises(ValueError, match=msg):
            S.ops.cmaes_sample(torch.zeros(need, **f64), d, lam, 0, c)
        with pytest.raises(ValueError, match=msg):
            S.ops.cmaes_update(torch.zeros(need, **f64), d, lam, c, f)
        with pytest.raises(ValueError, match=msg):
            S.ops.cmaes_generation(torch.zeros(need, **f64), lam, 0, base, data, c, f)
    for g, msg in bad_f:
        with pytest.raises(ValueError, match=msg):
            S.ops.cmaes_update(torch.zeros(need, **f64), d, lam, x, g)
        with pytest.raises(ValueError, match=msg):
            S.ops.cmaes_generation(torch.zeros(need, **f64), lam, 0, base, data, x, g)
    for out, msg in ((torch.zeros(lam + 1, **f64), r"out must have shape \(7,\)"),
                     (torch.zeros(lam, dtype=torch.float32), "out must be a float64 tensor"),
                     (torch.zeros(2 * lam, **f64)[::2], "out must be contiguous"),
                     (torch.zeros(lam, **f64), "must be a CUDA tensor")):
        with pytest.raises(ValueError, match=msg):
            S.ops.prediction_error(base, data, x, out=out)
    with pytest.raises(ValueError, match="candidates must be a CUDA tensor"):
        S.ops.prediction_error(base, data, x)


def test_device_data_follows_the_subset(S, monkeypatch):
    """The Estimator's uploaded data is keyed on the subset: reassigning or editing it rebuilds the data that the
    population objective and the device CMA-ES read.  Run on the CPU: the cache logic needs no device."""
    monkeypatch.setattr(S._lib, "require_cuda", lambda: None)
    n, H = 3, 6
    db = S.Database()
    rng = np.random.default_rng(0)
    trajs = rng.normal(size=(4, H, 2 * n + 2))
    pols = rng.normal(size=(4, n - 1, 2 * n + 2))
    for t, W in zip(trajs, pols):
        db.add_trajectory(t, W)
    est = S.Estimator(db, S.EnvParam("sim", n=n, H=H, m_i=1.0, l_i=1.0, h=0.001, k=10.0, epsilon=0.01),
                      capacity=2, device="cpu")

    def uploaded(M):
        data = est._device_data(M)
        return data.trajectories.numpy(), data.policies.numpy().reshape(-1, n - 1, 2 * n + 2)

    for subset in ([0, 1], [3, 2], [3, 3]):
        est.subset = np.array(subset)
        t, p = uploaded(7)
        assert np.array_equal(t, trajs[subset]) and np.array_equal(p, pols[subset]), subset
    est.subset[0] = 1
    t, _ = uploaded(7)
    assert np.array_equal(t, trajs[[1, 3]])
    data = est._device_data(7)
    assert est._device_data(5) is data  # same subset, enough workspace: no new upload
    assert est._device_data(9) is not data and est._device_data(9).max_candidates == 9
