"""The ARS bookkeeping kernels (csrc/ars_kernels.cu and the one-process paths of csrc/exchange.cu) against references
that are independent of them: the oracle where it has the operation (sort_directions, update_policy, philox_delta,
step), otherwise a restatement here in exact (fractions.Fraction) or extended (np.longdouble, 64-bit mantissa or
more) arithmetic.

Exact operations (orders, masks, counts, Philox words, copies, clip decisions) are compared bit for bit.  Rounded
ones are held to |kernel - exact| <= c * eps * sum|terms|, with c derived from the kernel's own summation order:
block_sum (256 threads) makes every term pass through at most ceil(m / 256) additions in its thread, 5 butterfly
levels and 8 sequential warp partials, so a sum of m terms has depth d = ceil(m / 256) + 13 and error
<= d * eps * sum|terms| (first order; every bar below adds a factor 2 for the second-order terms).  The largest
measured error / bar ratios are printed with -s and recorded in DESIGN.md section 6.
"""
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

from conftest import rand_states, rel_err

EPS = np.finfo(np.float64).eps / 2  # unit roundoff 2^-53
LD = np.longdouble
QNAN = 0x7FF8000000000000
ERR_BAD_ARG, ERR_UNSUPPORTED = -1, -2

gpu = pytest.mark.gpu


def _cuda(a, dtype=np.float64):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=dtype)).cuda()


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _i32(v):
    return torch.tensor([v], dtype=torch.int32, device="cuda")


def _report(name, ratio):
    print("%s: largest error / bar = %.3g" % (name, ratio))


def _depth(m):
    return math.ceil(m / 256) + 13


# ---- ranking -----------------------------------------------------------------------------------------------------

def rank_ref(returns, mask=None):
    """sort_directions restated in plain Python: key = max(r+, r-) with Python's max (max(NaN, x) = NaN,
    max(x, NaN) = x), descending, NaN keys first, ties to the higher index first; screened-out directions last,
    ordered among themselves by the same rule."""
    N = len(returns) // 2
    keys = [max(float(returns[2 * i]), float(returns[2 * i + 1])) for i in range(N)]
    valid = [True] * N if mask is None else [int(m) != 0 for m in mask]

    def sort_key(i):
        k = keys[i]
        nan = k != k
        return (not valid[i], not nan, 0.0 if nan else -k, -i)
    return np.array(sorted(range(N), key=sort_key), dtype=np.int32)


def _rank_keys(rng, N, kind):
    if kind == "random":
        return rng.normal(size=2 * N)
    if kind == "equal":
        return np.full(2 * N, 2.5)
    # few distinct values: ties everywhere, NaN in either slot, +-inf, -0.0 against +0.0
    pool = np.array([np.nan, np.inf, -np.inf, 0.0, -0.0, 1.0, -1.0, 3.5, 3.5, -2.0])
    r = rng.choice(pool, size=2 * N)
    sel = rng.random(2 * N) < 0.3
    r[sel] = np.round(rng.normal(size=int(sel.sum())) * 2)
    return r


def test_rank_reference_matches_oracle(O):
    """The Python restatement equals orc_sort_directions on tie-free keys, and on ties, NaN, +-inf and +-0 too
    (the oracle implements the same total order)."""
    rng = np.random.default_rng(1)
    for N in (1, 2, 7, 64, 333):
        r = rng.normal(size=2 * N)
        np.testing.assert_array_equal(rank_ref(r), O.sort_directions(r))
        r = _rank_keys(rng, N, "special")
        np.testing.assert_array_equal(rank_ref(r), O.sort_directions(r))
    # the rules spelled out on a hand-made case
    r = np.array([1.0, np.nan, np.nan, 1.0, 2.0, 2.0, -0.0, 0.0, 0.0, -0.0, np.inf, -np.inf])
    # keys: 1 (max(1, NaN) = 1), NaN, 2, -0.0, 0.0 (a tie with -0.0: higher index first), inf
    np.testing.assert_array_equal(rank_ref(r), [1, 5, 2, 0, 4, 3])
    np.testing.assert_array_equal(rank_ref(r), O.sort_directions(r))


@gpu
@pytest.mark.parametrize("N", [1, 7, 8, 9, 255, 256, 257, 4095, 4096, 4097, 17066])
def test_topb_matches_python_ranking(S, N):
    """ars_rank_kernel bit for bit, across the warp and block edges, the 48 KB dynamic shared-memory opt-in
    (N = 4096 -> 4097) and the largest supported N (200 KB)."""
    rng = np.random.default_rng(N)
    for kind in ("random", "special", "equal"):
        r = _rank_keys(rng, N, kind)
        masks = [None, np.zeros(N), np.ones(N), (rng.random(N) < 0.5)]
        for m in masks:
            mask = None if m is None else _cuda(m, np.int32)
            got = S.ops.ars_topb(_cuda(r), mask).cpu().numpy()
            np.testing.assert_array_equal(np.sort(got), np.arange(N, dtype=np.int32))
            np.testing.assert_array_equal(got, rank_ref(r, m), err_msg="N=%d %s mask=%s" % (
                N, kind, None if m is None else int(np.sum(m))))


@gpu
def test_topb_rejects_n_beyond_shared_memory(S):
    L = S._lib
    N = 17067
    r = torch.zeros(2 * N, dtype=torch.float64, device="cuda")
    order = torch.full((N,), -7, dtype=torch.int32, device="cuda")
    assert L.lib().swm_ars_topb(L.ptr(r), None, N, L.ptr(order), L.stream_ptr()) == ERR_UNSUPPORTED
    assert int(order.min()) == -7 and int(order.max()) == -7


# ---- update ------------------------------------------------------------------------------------------------------

def update_ref(W0, rets, deltas, sel, divisor, ddof, alpha):
    """W0 + alpha * sum_{k in sel} (r+_k - r-_k) delta_k / (divisor * sigma_R) in long double, plus the bar
    per element.  sigma_R over the 2 |sel| returns (ddof 0 or 1)."""
    sel = np.asarray(sel, dtype=np.int64)
    u = len(sel)
    rp, rm = rets[0::2][sel].astype(LD), rets[1::2][sel].astype(LD)
    allr = np.concatenate([rp, rm])
    mean = allr.sum() / LD(2 * u)
    V = ((allr - mean) ** 2).sum()
    sigma = np.sqrt(V / LD(2 * u - ddof))
    D = deltas[sel].astype(LD)
    g = ((rp - rm)[:, None] * D).sum(axis=0)
    scale = LD(divisor) * sigma
    step = LD(alpha) * g / scale
    W = W0.astype(LD) + step
    # bar: the kernel's mean has error <= (d+1) eps sum|r| / 2u; the two-pass V then carries the rounding of its
    # own sum, (d+3) eps V, plus the exact shift 2u (mean_err)^2; sigma half of V's relative error plus 2 roundings.
    # g: c_k = r+ - r- rounded once, then a chain of d fmas, so (d+2) eps sum(|r+|+|r-|) |delta|.  The last four
    # roundings (scale, quotient, alpha *, +=) give 4 eps |step| and eps |W|.
    d = 2 * math.ceil(u / 256) + 13
    absr = np.abs(rp) + np.abs(rm)
    mean_err = (d + 1) * EPS * absr.sum() / (2 * u)
    sig_rel = ((d + 3) * EPS + 2 * u * mean_err ** 2 / V) / 2 + 2 * EPS if V > 0 else np.inf
    g_err = (d + 2) * EPS * (absr[:, None] * np.abs(D)).sum(axis=0)
    bar = EPS * np.abs(W) + abs(alpha) / abs(scale) * g_err + np.abs(step) * (sig_rel + 4 * EPS)
    return W, sigma, 2 * bar


def _deltas_oracle(O, seed, it, dir0, N, ws, dist):
    return np.stack([O.philox_delta(seed, it, (dir0 + k) % 2 ** 32, ws, dist=dist) for k in range(N)])


def _b_cases(N):
    return sorted({max(1, N // 3), N, N + 5}) if N > 1 else [1, 2]


def test_oracle_topb_divisor_is_len_order_b(O):
    """safe_ars/ars.py:96 passes order[:b] and :64 divides by len(order): min(b, N) once b > N (the oracle used to
    divide by b).  ARSAgent (semantics 0) and the RL-Glue agent (2) keep the divisor b."""
    rng = np.random.default_rng(5)
    N, ws, alpha = 6, 8, 0.5
    W0, rets = rng.normal(size=ws), rng.normal(size=2 * N) * 10
    deltas = rng.uniform(-1, 1, (N, ws))
    for b in (2, N, N + 1, 3 * N):
        order = O.sort_directions(rets)
        for sem, sel, div, ddof in ((0, order, b, 0), (1, order[:b], min(b, N), 0), (2, np.arange(min(b, N)), b, 1)):
            want, want_sigma, bar = update_ref(W0, rets, deltas, sel, div, ddof, alpha)
            got, sigma = O.update_policy(W0, deltas, rets, b=b, alpha=alpha, semantics=sem)
            assert np.all(np.abs(got - want) <= bar), (sem, b)
            assert abs(sigma - want_sigma) <= 1e-14 * want_sigma


@gpu
@pytest.mark.parametrize("N", [1, 255, 256, 257, 1024, 4097])
@pytest.mark.parametrize("semantics", [0, 1, 2])
def test_update_matches_extended_reference(S, O, N, semantics):
    """ars_update_kernel for b < N, b = N, b > N; odd and real wsize; Philox U(-1,1) and U[0,1), dir0 != 0 and a
    device iteration: in-kernel Philox equals explicit deltas bit for bit, and both sit within the bar of the
    long-double reference.  The unmasked cases also match the oracle's update_policy."""
    rng = np.random.default_rng(100 * N + semantics)
    wss = {1: [1, 3, 199, 16], 255: [1, 3, 199], 256: [3, 16], 257: [1, 199], 1024: [3, 198], 4097: [1, 16]}[N]
    worst = 0.0
    for ci, b in enumerate(_b_cases(N)):
        for wi, ws in enumerate(wss):
            dist = (ci + wi + semantics) % 2
            dir0 = [0, 1000003, 2 ** 32 - N - 1][(ci + wi) % 3]
            host_it, dev_it = 11, (None if (ci + wi) % 2 == 0 else 29)
            it = host_it + (dev_it or 0)
            seed = 0x9E3779B97F4A7C15 + ws
            alpha = 0.0075 * (1 + wi)
            W0, rets = rng.normal(size=ws), rng.normal(size=2 * N) * 30 + 5
            deltas = _deltas_oracle(O, seed, it, dir0, N, ws, dist)
            use_order, n_order, divisor, ddof = S.ops.update_args(semantics, N, b)
            order_ref = rank_ref(rets) if use_order else np.arange(N)
            sel = order_ref[:min(n_order, N)]
            want, want_sigma, bar = update_ref(W0, rets, deltas, sel, divisor if divisor > 0 else len(sel),
                                               ddof, alpha)
            r = _cuda(rets)
            order = S.ops.ars_topb(r) if use_order else None
            outs = []
            for explicit in (False, True):
                W, sig = _cuda(W0), torch.full((1,), -1.0, dtype=torch.float64, device="cuda")
                kw = dict(order=order, n_order=n_order, divisor=divisor, ddof=ddof, alpha=alpha, seed=seed,
                          iteration=host_it, dir0=dir0, delta_dist=dist, sigma_out=sig,
                          iteration_dev=None if dev_it is None else _i32(dev_it))
                if explicit:
                    kw["deltas"] = S.ops.philox_deltas(seed, it, dir0, N, ws, dist=dist)
                S.ops.ars_update(W, r, N, **kw)
                outs.append((W.cpu().numpy(), float(sig.cpu()[0])))
            np.testing.assert_array_equal(_bits(outs[0][0]), _bits(outs[1][0]))
            assert outs[0][1] == outs[1][1]
            err = np.abs(outs[0][0] - want.astype(np.float64))
            assert np.all(err <= bar), "b=%d ws=%d: err %.3g, bar %.3g" % (b, ws, err.max(), bar.min())
            assert abs(outs[0][1] - float(want_sigma)) <= 1e-13 * float(want_sigma)
            worst = max(worst, float(np.max(err / bar)))
            o_W, o_sigma = O.update_policy(W0, deltas, rets, b=b, alpha=alpha, semantics=semantics)
            assert np.all(np.abs(o_W - want.astype(np.float64)) <= bar)
            assert np.all(np.abs(outs[0][0] - o_W) <= 2 * bar)
    _report("update N=%d semantics %d" % (N, semantics), worst)


@gpu
@pytest.mark.parametrize("N", [255, 256, 257, 1024, 4097])
@pytest.mark.parametrize("semantics", [0, 1])
def test_update_with_mask_covers_exactly_the_survivors(S, O, N, semantics):
    """Fewer survivors than n_order: the screened-out directions (NaN returns, as the engine leaves them) sort last,
    and sigma_R, the sum and (ARS_TOPB) the divisor cover exactly the survivors.  Zero survivors: W and sigma_out
    are left bit-unchanged."""
    rng = np.random.default_rng(7 * N + semantics)
    ws, seed, it, alpha = 16, 21, 3, 0.02
    for b, surv in ((N, N // 3), (N // 2 + 1, N // 4), (N + 3, N - 1), (N, 0)):
        m = np.zeros(N, dtype=np.int32)
        m[rng.permutation(N)[:surv]] = 1
        rets = rng.normal(size=2 * N) * 30
        rets[np.repeat(m == 0, 2)] = np.nan
        # ties among the survivors
        rets[0:2 * min(N, 40):4] = 3.0
        use_order, n_order, divisor, ddof = S.ops.update_args(semantics, N, b)
        W0 = rng.normal(size=ws)
        r, mask = _cuda(rets), _cuda(m, np.int32)
        order = S.ops.ars_topb(r, mask)
        np.testing.assert_array_equal(order.cpu().numpy(), rank_ref(rets, m))
        W, sig = _cuda(W0), torch.full((1,), -1.0, dtype=torch.float64, device="cuda")
        S.ops.ars_update(W, r, N, order=order, n_order=n_order, divisor=divisor, ddof=ddof, alpha=alpha,
                         seed=seed, iteration=it, mask=mask, sigma_out=sig)
        got = W.cpu().numpy()
        if surv == 0:
            np.testing.assert_array_equal(_bits(got), _bits(W0))
            assert float(sig.cpu()[0]) == -1.0
            continue
        sel = rank_ref(rets, m)[:min(n_order, surv)]
        assert np.all(m[sel] == 1)
        deltas = _deltas_oracle(O, seed, it, 0, N, ws, 0)
        want, want_sigma, bar = update_ref(W0, rets, deltas, sel, divisor if divisor > 0 else len(sel), ddof, alpha)
        assert np.all(np.abs(got - want.astype(np.float64)) <= bar), (b, surv)
        assert abs(float(sig.cpu()[0]) - float(want_sigma)) <= 1e-13 * float(want_sigma)


@gpu
@pytest.mark.parametrize("semantics", [0, 1, 2])
def test_update_with_all_equal_returns_follows_numpy(S, semantics):
    """sigma_R = 0: the reference's numpy arithmetic (np.std = 0, grad = 0 / 0) makes W NaN; the kernel must give
    the same, and sigma_out = 0.  Values chosen so every summation order is exact."""
    N, b, ws, alpha = 300, 40, 16, 0.02
    rets = np.full(2 * N, -12.25)
    deltas = np.stack([np.linspace(-1, 1, ws)] * N)
    use_order, n_order, divisor, ddof = S.ops.update_args(semantics, N, b)
    sel = np.arange(n_order)
    with np.errstate(invalid="ignore", divide="ignore"):
        rr = np.concatenate([rets[0::2][sel], rets[1::2][sel]])
        sigma = np.std(rr, ddof=ddof)
        grad = ((rets[0::2][sel] - rets[1::2][sel])[:, None] * deltas[sel]).sum(0)
        want = np.zeros(ws) + alpha * (grad / ((divisor if divisor > 0 else n_order) * sigma))
    r = _cuda(rets)
    W, sig = torch.zeros(ws, dtype=torch.float64, device="cuda"), torch.full((1,), -1.0, dtype=torch.float64,
                                                                           device="cuda")
    S.ops.ars_update(W, r, N, order=S.ops.ars_topb(r) if use_order else None, n_order=n_order, divisor=divisor,
                     ddof=ddof, alpha=alpha, deltas=_cuda(deltas), sigma_out=sig)
    assert sigma == 0.0 and float(sig.cpu()[0]) == 0.0
    np.testing.assert_array_equal(W.cpu().numpy(), want)
    assert np.all(np.isnan(want))


# ---- Philox table ------------------------------------------------------------------------------------------------

@gpu
def test_philox_table_matches_oracle_at_odd_sizes_and_counter_edges(S, O):
    """philox_deltas_kernel bit for bit against orc_philox_delta: odd wsize (the unpaired last element), dir0 near
    2^32 - count (and wrapping past it, mod 2^32 like the kernel's uint32 counter), both distributions, and a device
    iteration equal to the same host iteration."""
    seed = 0xDEADBEEFCAFEF00D
    for ws in (1, 3, 17, 199, 198):
        for count in (1, 5, 300):
            for dir0 in (0, 2 ** 32 - count, 2 ** 32 - 1 - count // 2):
                for dist in (0, 1):
                    want = _deltas_oracle(O, seed, 77, dir0, count, ws, dist)
                    got = S.ops.philox_deltas(seed, 77, dir0, count, ws, dist=dist).cpu().numpy()
                    np.testing.assert_array_equal(_bits(got), _bits(want))
                    dev = S.ops.philox_deltas(seed, 70, dir0, count, ws, dist=dist, iteration_dev=_i32(7))
                    np.testing.assert_array_equal(_bits(dev.cpu().numpy()), _bits(want))


# ---- select_action -----------------------------------------------------------------------------------------------

def _exact_actions(pols, obs, R, mean=None, inv_sigma=None):
    """Fraction dot products W . o or (W o sigma^-1) . (o - mean), exactly."""
    B, no = obs.shape
    na = pols.shape[1]
    out = np.empty((B, na), dtype=object)
    Fo = [[Fraction(float(v)) for v in row] for row in obs]
    Fm = None if mean is None else [Fraction(float(v)) for v in mean]
    Fs = None if inv_sigma is None else [Fraction(float(v)) for v in inv_sigma]
    for e in range(B):
        W = pols[e // R]
        x = Fo[e] if Fm is None else [Fo[e][j] - Fm[j] for j in range(no)]
        for a in range(na):
            w = [Fraction(float(v)) for v in W[a]]
            if Fs is not None:
                w = [w[j] * Fs[j] for j in range(no)]
            out[e, a] = sum(w[j] * x[j] for j in range(no))
    return out


def _clip_exact(v, max_u):
    m = Fraction(max_u)
    return float(min(max(v, -m), m))


@gpu
@pytest.mark.parametrize("n", list(range(2, 11)))
def test_policy_actions_match_exact_dot_product(S, n):
    """policy_actions_kernel against exact dot products, R = 1, 3, 32 (B not a multiple of 128 (n-1)), with and
    without normalisation.  Bar: (no + 2) eps sum|terms| -- a chain of `no` fmas, and in the normalised form the
    two rounded factors W sigma^-1 and o - mean of each term.  clip = clip of the unclipped output, bit for bit."""
    no, na = 2 * n + 2, n - 1
    ps = S.make_params(n=n, max_u=5.0)
    rng = np.random.default_rng(n)
    worst = 0.0
    for R, P in ((1, 37), (3, 43), (32, 5)):
        B = P * R
        assert (B * na) % (128 * na) != 0
        pols = rng.normal(size=(P, na, no)) * 2
        obs = rand_states(rng, n, B)
        for norm in (False, True):
            mean = rng.normal(size=no) if norm else None
            inv = rng.uniform(0.2, 3.0, no) if norm else None
            exact = _exact_actions(pols, obs, R, mean, inv)
            kw = dict(mean=_cuda(mean), inv_sigma=_cuda(inv)) if norm else {}
            got = S.ops.policy_actions(ps, _cuda(obs), _cuda(pols), R, **kw).cpu().numpy()
            clipped = S.ops.policy_actions(ps, _cuda(obs), _cuda(pols), R, clip=True, **kw).cpu().numpy()
            x = obs - mean if norm else obs
            w = pols * inv if norm else pols
            terms = np.abs(w[np.arange(B) // R] * x[:, None, :]).sum(-1)
            bar = 2 * (no + 2) * EPS * terms
            err = np.abs(got - exact.astype(np.float64))
            assert np.all(err <= bar), (R, norm)
            worst = max(worst, float(np.max(err / np.maximum(bar, 1e-300))))
            np.testing.assert_array_equal(_bits(clipped), _bits(np.clip(got, -5.0, 5.0)))
            assert np.mean(np.abs(got) > 5.0) > 0.05 and np.mean(np.abs(got) < 5.0) > 0.05
    _report("policy_actions n=%d" % n, worst)


@gpu
def test_policy_actions_clip_decision_at_max_u_is_exact(S):
    """Products that sum exactly to +-max_u and one ulp either side: the clip keeps what is inside, including the
    bounds themselves, and maps everything beyond to exactly +-max_u; without clip the value is returned as is."""
    for n, max_u in ((2, 5.0), (3, 0.7), (10, 1e-3)):
        no, na = 2 * n + 2, n - 1
        targets = [max_u, np.nextafter(max_u, np.inf), np.nextafter(max_u, 0.0),
                   -max_u, np.nextafter(-max_u, -np.inf), np.nextafter(-max_u, 0.0)]
        pols, obs = [], []
        for t in targets:
            for pattern in range(3):
                W = np.zeros((na, no))
                o = np.zeros(no)
                if pattern == 0:      # one product t * 1
                    W[:, 0], o[0] = t, 1.0
                elif pattern == 1:    # t/2 + t/4 + t/4, exact
                    W[:, :3], o[:3] = [t, t / 2, t], [0.5, 0.5, 0.25]
                else:                 # a cancelling pair, then 4t * 0.25
                    W[:, no - 3:], o[no - 3:] = [3.0, -3.0, 4 * t], [1.5, 1.5, 0.25]
                pols.append(W)
                obs.append(o)
        pols, obs = np.array(pols), np.array(obs)
        ps = S.make_params(n=n, max_u=max_u)
        one = np.ones(no)
        for kw in ({}, dict(mean=_cuda(np.zeros(no)), inv_sigma=_cuda(one))):
            raw = S.ops.policy_actions(ps, _cuda(obs), _cuda(pols), **kw).cpu().numpy()
            clp = S.ops.policy_actions(ps, _cuda(obs), _cuda(pols), clip=True, **kw).cpu().numpy()
            want_raw = np.repeat(np.repeat(targets, 3)[:, None], na, axis=1)
            np.testing.assert_array_equal(_bits(raw), _bits(want_raw))
            want_clp = np.vectorize(lambda v: _clip_exact(Fraction(v), max_u))(want_raw)
            np.testing.assert_array_equal(_bits(clp), _bits(want_clp))
            assert np.sum(clp == max_u) == 3 * 2 * na and np.sum(clp == -max_u) == 3 * 2 * na


@gpu
@pytest.mark.parametrize("n", [2, 5, 10])
def test_policy_actions_equal_rlglue_rollout_first_action(S, O, n):
    """The RL-Glue rollout kernel's first step from a state, stepped by the oracle with policy_actions' clipped
    action from the same state, is the kernel's own first state (RL-Glue bar 1e-11)."""
    no, na = 2 * n + 2, n - 1
    rng = np.random.default_rng(40 + n)
    ps, po = S.make_params(n=n, max_u=5.0), O.make_params(n=n, max_u=5.0)
    P = 40
    pols = rng.normal(size=(P, na, no)) * 3
    starts = rand_states(rng, n, P, scale=1.0)
    acts = S.ops.policy_actions(ps, _cuda(starts), _cuda(pols), clip=True).cpu().numpy()
    assert np.mean(np.abs(acts) == 5.0) > 0.1 and np.mean(np.abs(acts) < 5.0) > 0.1
    res = S.ops.rollout(ps, 1, policies=_cuda(pols), variant=S.RLGLUE, clip_actions=True,
                        init_state=_cuda(starts), want_trajectory=True)
    traj = res.trajectory.cpu().numpy()[0]
    for e in range(P):
        want, _ = O.step(po, O.RLGLUE, starts[e], acts[e])
        assert rel_err(traj[e], want) < 1e-11, e


# ---- statistics --------------------------------------------------------------------------------------------------

def _exact_record(S1, S2, count, pivot):
    """(mean, M2) from exact column sums: pivot + S1/n and max(S2 - S1^2/n, 0), as Fractions."""
    n = Fraction(count)
    mean = [Fraction(float(p)) + Fraction(s1) / n for p, s1 in zip(pivot, S1)]
    m2 = [max(Fraction(s2) - Fraction(s1) ** 2 / n, Fraction(0)) for s1, s2 in zip(S1, S2)]
    return mean, m2


def _check_record(rec, S1, S2, count, pivot, d):
    """rec = [count, mean[F], M2[F]] against exact sums; the column sums of depth d contribute d eps sum|terms|
    (zero when the rows are exactly summable), the conversion 3 roundings."""
    F = len(pivot)
    assert rec[0] == count
    if count == 0:
        np.testing.assert_array_equal(rec[1:], np.zeros(2 * F))
        return 0.0
    mean, m2 = _exact_record(S1, S2, count, pivot)
    a1, a2 = np.abs(np.asarray(S1, float)), np.abs(np.asarray(S2, float))
    bar_m = 2 * (2 * EPS * (np.abs(pivot) + a1 / count) + d * EPS * a1 / count)
    bar_M = 2 * (3 + 2 * d) * EPS * (a2 + a1 ** 2 / count)
    em = np.abs(rec[1:1 + F] - np.array([float(v) for v in mean]))
    eM = np.abs(rec[1 + F:] - np.array([float(v) for v in m2]))
    assert np.all(em <= bar_m) and np.all(eM <= bar_M)
    return float(max(np.max(em / np.maximum(bar_m, 1e-300)), np.max(eM / np.maximum(bar_M, 1e-300))))


def _exact_rows(rng, nb, F, scale=2 ** 20):
    """partial rows of multiples of 2^-10 below 2^20: every column sum is exact in double for nb <= 2^22, so any
    summation order gives the same sums."""
    s1 = rng.integers(-scale, scale, (nb, F)) / 1024.0
    s2 = rng.integers(0, scale, (nb, F)) / 1024.0 * 64
    return np.stack([s1, s2], axis=1)


@gpu
@pytest.mark.parametrize("nb,F", [(1, 1), (255, 8), (256, 22), (257, 33), (100000, 8), (300, 512)])
def test_stats_finalize_against_exact_sums(S, nb, F):
    """stats_colsum + stats_convert: rows with exact sums across the block edges and F past one warp; samples = 0
    and a device unit count of 0 give an empty record; units = 7 scales the count."""
    rng = np.random.default_rng(nb + F)
    part = _exact_rows(rng, nb, F)
    S1, S2 = part[:, 0].sum(0), part[:, 1].sum(0)
    pivot = rng.normal(size=F) * 100
    worst = 0.0
    for samples, units in ((float(nb * 3), None), (float(nb * 3), 7), (float(nb), 0), (0.0, None)):
        rec = S.ops.stats_finalize(_cuda(part), samples, _cuda(pivot),
                                   units=None if units is None else _i32(units)).cpu().numpy()
        count = samples * (1 if units is None else units)
        worst = max(worst, _check_record(rec, S1, S2, count, pivot, 0))
    _report("stats_finalize nb=%d F=%d" % (nb, F), worst)


@gpu
def test_stats_rejects_more_than_512_features(S):
    L = S._lib
    part = torch.zeros(2, 2, 513, dtype=torch.float64, device="cuda")
    rec = torch.zeros(1 + 2 * 513, dtype=torch.float64, device="cuda")
    piv = torch.zeros(513, dtype=torch.float64, device="cuda")
    assert L.lib().swm_stats_finalize(L.ptr(part), 2, 513, 4.0, None, L.ptr(piv), L.ptr(rec),
                                      L.stream_ptr()) == ERR_BAD_ARG
    assert L.lib().swm_stats_merge(L.ptr(rec), L.ptr(rec), 1, 513, None, None, L.stream_ptr()) == ERR_BAD_ARG


def m2_cancellation_bar(S1, S2, count, nb):
    """Bar on M2 = S2 - S1^2/n from per-sample rows (x - p, (x - p)^2) summed by block_sum over nb = count rows:
    each shifted sample is rounded once and squared once (3 eps on S2, 1 on S1), the sums have depth d, and the
    conversion rounds 3 times.  With all x - p of one sign (data far from the pivot) sum|x - p| = |S1|, so
    |M2^ - M2| <= (2d + 6) eps (S2 + S1^2/n).  Relative to M2 = n sigma^2 this is (2d + 6) eps (2 D^2/sigma^2 + 1)
    for data whose mean sits D away from the pivot."""
    d = _depth(nb)
    return (2 * d + 6) * EPS * (np.abs(S2) + S1 ** 2 / count)


@gpu
@pytest.mark.parametrize("pivot_kind", ["zero", "reset"])
def test_stats_m2_cancellation_far_from_pivot(S, pivot_kind):
    """Samples whose mean sits 1e4 sigma from the pivot (the shifted sums then cancel in M2 by a factor ~2e8): the
    error of M2 against the exact M2 of the samples stays within m2_cancellation_bar.  "reset": the engine's pivot,
    the reset state (theta = pi/2, everything else 0), for n = 3."""
    rng = np.random.default_rng(8)
    F = 8
    pivot = np.zeros(F) if pivot_kind == "zero" else S.ops.reset_state(3).cpu().numpy()
    sigma = rng.uniform(0.01, 2.0, F)
    D = 1e4 * sigma * rng.choice([-1.0, 1.0], F)
    for count in (1000, 10000, 65537):
        x = pivot + D + rng.normal(size=(count, F)) * sigma
        sh = x - pivot
        part = np.stack([sh, sh * sh], axis=1)
        rec = S.ops.stats_finalize(_cuda(part), float(count), _cuda(pivot)).cpu().numpy()
        worst_rel, worst = 0.0, 0.0
        for f in range(F):
            mu, M2 = exact_mean_m2(x[:, f])
            S1 = float(sh[:, f].sum())
            S2 = float((sh[:, f] ** 2).sum())
            bar = 2 * m2_cancellation_bar(S1, S2, count, count)
            err = abs(Fraction(float(rec[1 + F + f])) - M2)
            assert err <= bar, (count, f, float(err), bar)
            worst = max(worst, float(err) / bar)
            worst_rel = max(worst_rel, float(err / M2))
            assert abs(Fraction(float(rec[1 + f])) - mu) <= 4 * _depth(count) * EPS * (abs(mu) + abs(pivot[f]))
        _report("M2 far from pivot (%s) n=%d: largest relative M2 error %.3g" % (pivot_kind, count, worst_rel), worst)


def exact_mean_m2(col):
    """Exact mean and M2 = sum (x - mean)^2 of doubles, as Fractions: every double is an integer times a power of
    two, so with the common denominator D, mean = S / (n D) and M2 = (n Q - S^2) / (n D^2) in integers."""
    ratios = [float(v).as_integer_ratio() for v in col]
    den = max(d for _, d in ratios)
    ints = [p * (den // d) for p, d in ratios]
    n, s = len(ints), sum(ints)
    q = sum(i * i for i in ints)
    return Fraction(s, n * den), Fraction(n * q - s * s, n * den * den)


def _record_of(x):
    """(count, mean, M2) of samples x[count, F], each rounded once from the exact value."""
    count = len(x)
    F = x.shape[1]
    if count == 0:
        return np.concatenate([[0.0], np.full(F, np.nan), np.full(F, np.nan)])  # garbage: must be skipped
    mm = [exact_mean_m2(x[:, f]) for f in range(F)]
    return np.concatenate([[float(count)], [float(m) for m, _ in mm], [float(v) for _, v in mm]])


def _merge_bar(xs, R):
    """Bars on (M2, mean) after R merges.  Every mean and every d = m_b - m_a is bounded by 2 max|x|, and each merge
    rounds 3 times in the mean, so the mean error is <= c eps max|x|.  In M2 every term (M2_a, M2_b,
    d^2 n_a n_b / n) and the propagated mean errors times 2 |d| min(n_a, n_b) are bounded by n max|x|^2, each merge
    rounding 5 times; the inputs are rounded once.  c = 8 (R + 2) covers both with room for second-order terms."""
    mx = np.abs(xs).max(0)
    c = 8 * (R + 2)
    return c * EPS * len(xs) * mx ** 2, c * EPS * mx


def test_exact_moments_match_oracle_mean_var(O):
    """The Fraction moments used below agree with orc_mean_var (two-pass, long double) to rounding."""
    rng = np.random.default_rng(3)
    x = rng.normal(size=(500, 5)) * 3 + 7
    rec = _record_of(x)
    mean, var = O.mean_var(x)
    np.testing.assert_allclose(rec[1:6], mean, rtol=4 * EPS, atol=0)
    np.testing.assert_allclose(rec[6:] / 499, var, rtol=16 * EPS, atol=0)


@gpu
@pytest.mark.parametrize("F", [3, 33, 100, 512])
def test_stats_merge_against_concatenated_samples(S, F):
    """stats_merge_kernel: running <- merge(running, records...) equals the exact mean and M2 of the concatenated
    samples; empty records (count 0, NaN moments) are skipped; mean / inv_sigma are written from count 2 on."""
    rng = np.random.default_rng(F)
    worst = 0.0
    sizes_cases = [(0, [0, 5, 0, 17, 1, 0, 40]), (3, [0, 0, 9]), (1, [6, 0, 1000])]
    for run_n, sizes in sizes_cases:
        xs = [rng.normal(size=(s, F)) * rng.uniform(0.1, 5, F) + rng.normal(size=F) * 20 for s in [run_n] + sizes]
        running = _cuda(_record_of(xs[0]) if run_n else np.zeros(1 + 2 * F))
        recs = _cuda(np.stack([_record_of(x) for x in xs[1:]]))
        mean_out = torch.full((F,), 0.5, dtype=torch.float64, device="cuda")
        inv_out = torch.full((F,), 1.0, dtype=torch.float64, device="cuda")
        S.ops.stats_merge(running, recs, mean_out, inv_out)
        allx = np.concatenate(xs)
        want = _record_of(allx)
        got = running.cpu().numpy()
        assert got[0] == len(allx)
        barM, barm = _merge_bar(allx, len(sizes))
        eM = np.abs(got[1 + F:] - want[1 + F:])
        em = np.abs(got[1:1 + F] - want[1:1 + F])
        assert np.all(eM <= barM) and np.all(em <= barm)
        worst = max(worst, float(np.max(eM / barM)), float(np.max(em / barm)))
        np.testing.assert_array_equal(_bits(mean_out.cpu().numpy()), _bits(got[1:1 + F]))
        want_inv = 1.0 / np.sqrt(got[1 + F:] / (got[0] - 1.0))
        np.testing.assert_array_equal(_bits(inv_out.cpu().numpy()), _bits(want_inv))
    # count below 2: the record is merged, mean and inv_sigma stay untouched
    for run_n, sizes in ((0, [0, 0]), (0, [1, 0]), (1, [0]), (0, [0, 1])):
        xs = [rng.normal(size=(s, F)) for s in [run_n] + sizes]
        running = _cuda(_record_of(xs[0]) if run_n else np.zeros(1 + 2 * F))
        mean_out = torch.full((F,), 0.5, dtype=torch.float64, device="cuda")
        inv_out = torch.full((F,), 1.0, dtype=torch.float64, device="cuda")
        S.ops.stats_merge(running, _cuda(np.stack([_record_of(x) for x in xs[1:]])), mean_out, inv_out)
        got = running.cpu().numpy()
        allx = np.concatenate(xs)
        assert got[0] == len(allx)
        if len(allx) == 1:
            np.testing.assert_array_equal(got[1:1 + F], allx[0])
            np.testing.assert_array_equal(got[1 + F:], np.zeros(F))
        assert np.all(mean_out.cpu().numpy() == 0.5) and np.all(inv_out.cpu().numpy() == 1.0)
    _report("stats_merge F=%d" % F, worst)


# ---- record pack / unpack, one process --------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("R", [1, 3, 128])
def test_pack_records_and_unpack_gathered_world(S, world, R):
    """pack_exchange_kernel, pack-only (record_out, gathered_world > 1) for every rank of a world, then one unpack
    of the stacked records (gathered_in).  Each packed record against exact references (mean over R rollouts:
    R - 1 additions and a division, bar 2 R eps sum|r| / R; screened directions the canonical NaN even when their
    rollouts ran; mask 1.0 / 0.0; stats from exactly summable rows); the unpacked returns_all, mask_all and records
    equal the concatenation bit for bit."""
    rng = np.random.default_rng(world * 1000 + R)
    n_local = {1: 1000, 3: 1500, 128: 37}[R]
    F, nb = 8, 70
    pivot = rng.normal(size=F)
    recs, masks = [], []
    worst = 0.0
    for rank in range(world):
        rl = rng.normal(size=(2 * n_local, R)) * 40
        if R == 1:
            rl = np.round(rl * 64) / 64
        m = (rng.random(n_local) < 0.7).astype(np.int32)
        m[rank % n_local] = 0
        part = _exact_rows(rng, nb, F)
        units = rank % 3 * 7  # 0, 7, 14 units: rank 0 packs an empty stats record
        rec = torch.full((2 * n_local + n_local + 1 + 2 * F,), -1.0, dtype=torch.float64, device="cuda")
        S.ops.pack_exchange(None, returns_local=_cuda(rl), n_local=n_local, R=R, mask_local=_cuda(m, np.int32),
                            stats_partial=_cuda(part), samples=float(nb * 2), units=_i32(units), pivot=_cuda(pivot),
                            n_features=F, record_out=rec, gathered_world=world)
        got = rec.cpu().numpy()
        ret = got[:2 * n_local]
        live = np.repeat(m != 0, 2)
        assert np.all(_bits(ret[~live]) == QNAN)
        want = np.array([float(sum(Fraction(float(v)) for v in row) / R) for row in rl[live]])
        bar = 2 * R * EPS * np.abs(rl[live]).sum(1) / R
        err = np.abs(ret[live] - want)
        assert np.all(err <= bar)
        worst = max(worst, float(np.max(err / np.maximum(bar, 1e-300))))
        if R == 1:
            np.testing.assert_array_equal(ret[live], rl[live, 0])
        np.testing.assert_array_equal(got[2 * n_local:3 * n_local], m.astype(np.float64))
        _check_record(got[3 * n_local:], part[:, 0].sum(0), part[:, 1].sum(0), nb * 2.0 * units, pivot, 0)
        recs.append(got)
        masks.append(m)
    gathered = _cuda(np.stack(recs))
    N = world * n_local
    ret_all = torch.full((2 * N,), -2.0, dtype=torch.float64, device="cuda")
    mask_all = torch.full((N,), -2, dtype=torch.int32, device="cuda")
    records = torch.full((world, 1 + 2 * F), -2.0, dtype=torch.float64, device="cuda")
    S.ops.pack_exchange(None, n_local=n_local, R=R, mask_local=_cuda(masks[0], np.int32), n_features=F,
                        returns_all=ret_all, mask_all=mask_all, records=records, gathered_in=gathered,
                        gathered_world=world)
    stacked = np.stack(recs)
    np.testing.assert_array_equal(_bits(ret_all.cpu().numpy()), _bits(stacked[:, :2 * n_local].reshape(-1)))
    np.testing.assert_array_equal(mask_all.cpu().numpy(), np.concatenate(masks))
    np.testing.assert_array_equal(_bits(records.cpu().numpy()), _bits(stacked[:, 3 * n_local:]))
    _report("pack world=%d R=%d" % (world, R), worst)


# ---- small kernels -----------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("N", [1, 257, 5000])
def test_screen_mask_edges(S, N):
    """mask = r+ > thr and r- > thr: a return equal to the threshold is screened out, NaN returns and a NaN
    threshold screen out, +inf screens out everything, -inf keeps every non-NaN pair above it; n_pass_total
    accumulates over three calls."""
    rng = np.random.default_rng(N)
    total = torch.tensor([5], dtype=torch.int64, device="cuda")
    expect_total = 5
    for thr in (0.25, np.inf, -np.inf, np.nan):
        r = np.round(rng.normal(size=2 * N) * 4) / 4
        r[rng.random(2 * N) < 0.1] = np.nan
        r[rng.random(2 * N) < 0.05] = np.inf
        r[rng.random(2 * N) < 0.05] = -np.inf
        r[rng.random(2 * N) < 0.2] = thr if not np.isnan(thr) else 1.0
        if N == 1:
            r[:] = [0.5, 0.25] if thr == 0.25 else r
        want = np.array([1 if (r[2 * k] > thr and r[2 * k + 1] > thr) else 0 for k in range(N)], dtype=np.int32)
        if thr == 0.25 and N > 1:
            assert want.sum() > 0 and (want == 0).sum() > 0
        for _ in range(3 if thr == 0.25 else 1):
            mask, n_pass = S.ops.screen_mask(_cuda(r), thr, n_pass_total=total)
            expect_total += int(want.sum())
        np.testing.assert_array_equal(mask.cpu().numpy(), want)
        assert int(n_pass.cpu()[0]) == int(want.sum())
    assert int(total.cpu()[0]) == expect_total


@gpu
def test_record_nanmean(S):
    """curve[min(index, capacity - 1)] = mean of the non-NaN entries (NaN if there are none), index NULL -> 0; the
    other entries are untouched.  Bar: (d + 1) eps sum|x| / count."""
    rng = np.random.default_rng(2)
    for n in (1, 255, 257, 5000):
        x = rng.normal(size=n) * 100
        x[rng.random(n) < 0.3] = np.nan
        if n == 1:
            x[0] = 3.0
        live = x[~np.isnan(x)]
        exact = sum(Fraction(float(v)) for v in live) / len(live)
        for index, cap, at in ((None, 4, 0), (2, 4, 2), (4, 4, 3), (1000, 3, 2)):
            curve = torch.full((cap,), -9.0, dtype=torch.float64, device="cuda")
            S.ops.record_nanmean(_cuda(x), curve, None if index is None else _i32(index))
            got = curve.cpu().numpy()
            bar = 2 * (_depth(n) + 1) * EPS * np.abs(live).sum() / len(live)
            assert abs(Fraction(float(got[at])) - exact) <= bar
            assert np.all(np.delete(got, at) == -9.0)
    curve = torch.zeros(2, dtype=torch.float64, device="cuda")
    S.ops.record_nanmean(_cuda(np.full(300, np.nan)), curve, _i32(1))
    assert curve.cpu().numpy()[0] == 0.0 and _bits(curve.cpu().numpy())[1] == QNAN


@gpu
@pytest.mark.parametrize("R", [1, 3, 128])
def test_reduce_returns_ragged_groups(S, R):
    """reduce_returns_kernel: group means over R rollouts for group counts that are not multiples of the 128-thread
    block; bar 2 R eps sum|r| / R (R - 1 additions and a division); bit-identical to the pack kernel's returns."""
    rng = np.random.default_rng(R)
    for G in (1, 129, 1000):
        r = rng.normal(size=(G, R)) * 50
        got = S.ops.reduce_returns(_cuda(r), R).cpu().numpy()
        want = np.array([float(sum(Fraction(float(v)) for v in row) / R) for row in r])
        assert np.all(np.abs(got - want) <= 2 * R * EPS * np.abs(r).sum(1) / R)
        if G % 2 == 0:
            rec = torch.empty(G, dtype=torch.float64, device="cuda")
            S.ops.pack_exchange(None, returns_local=_cuda(r), n_local=G // 2, R=R, record_out=rec, gathered_world=2)
            np.testing.assert_array_equal(_bits(rec.cpu().numpy()), _bits(got))


# ---- step_batched_models -----------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("M", [1, 24, 25, 49])
@pytest.mark.parametrize("n", [3, 7])
def test_step_batched_models_per_model(S, O, M, n):
    """swm_step_batched_models across the 24-model chunking of ops.step_batched_models: every model (its own l, m,
    k, h and direction) against O.step at 1e-12 norm-relative, and bit-identical to step_batched on that model
    alone; T = 37 (ragged)."""
    rng = np.random.default_rng(M * 10 + n)
    T = 37
    specs = []
    for _ in range(M):
        ang = rng.uniform(0, 2 * np.pi)
        specs.append(dict(n=n, l_i=rng.uniform(0.5, 2), m_i=rng.uniform(0.5, 2), k=rng.uniform(5, 15),
                          h=float(rng.choice([5e-4, 1e-3, 2e-3])), direction=(np.cos(ang), np.sin(ang))))
    ps = [S.make_params(**s) for s in specs]
    states = np.stack([rand_states(rng, n, T) for _ in range(M)])
    actions = rng.uniform(-5, 5, (M, T, n - 1))
    nxt, rew = S.ops.step_batched_models(ps, _cuda(states), _cuda(actions), want_reward=True)
    nxt, rew = nxt.cpu().numpy(), rew.cpu().numpy()
    for m in range(M):
        w_nxt, w_rew = O.step_batch(O.make_params(**specs[m]), O.GYM, states[m], actions[m])
        assert rel_err(nxt[m], w_nxt) < 1e-12, m
        assert rel_err(rew[m], w_rew) < 1e-12, m
        one, one_r = S.ops.step_batched(ps[m], _cuda(states[m]), _cuda(actions[m]))
        np.testing.assert_array_equal(_bits(nxt[m]), _bits(one.cpu().numpy()))
        np.testing.assert_array_equal(_bits(rew[m]), _bits(one_r.cpu().numpy()))
