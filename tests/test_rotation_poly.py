"""The one-tier rotation polynomial of the per-thread rollout step (csrc/dynamics.cuh, small_sincos).

CPU: the coefficients in dynamics.cuh are the ones csrc/rotation_poly.py derives, and the polynomials with those
double coefficients, evaluated exactly, stay within the truncation bound against an exact rational sine and cosine
on a dense grid of |d| <= 1/8.  GPU: the thread kernel, stepped once by the oracle from every state it visited, with
increments placed on, just below and just above 1/32 and 1/8, on every segment count that takes the joint-angle form:
for n <= 3 these are the edges of the two tiers the one polynomial replaced, for n = 4, 5 the tier edges it still has."""
import importlib.util
import os
import re
import struct
from fractions import Fraction

import numpy as np
import pytest

import test_trig_tiers as tt

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "safe-exploration-with-simulator-in-rl-algorithms_b200", "csrc")


def _script():
    spec = importlib.util.spec_from_file_location("rotation_poly", os.path.join(CSRC, "rotation_poly.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _header_coefficients(kind):
    src = open(os.path.join(CSRC, "dynamics.cuh")).read()
    m = re.search(r"constexpr double kRotate%s\[4\] = \{([^}]*)\};" % kind, src)
    assert m, kind
    return [float(x) for x in m.group(1).split(",")]


def _sin_cos_m1(d, terms=14):
    """Exact rational sin d and cos d - 1 (Taylor series; the remainder is below 1e-40 for |d| <= 1/8)."""
    s, c, t = Fraction(0), Fraction(0), Fraction(d)  # t = d^k / k!
    for k in range(1, 2 * terms + 2):
        if k % 2:
            s += t if k % 4 == 1 else -t
        else:
            c += t if k % 4 == 0 else -t
        t = t * d / (k + 1)
    return s, c


def _poly(coef, z):
    acc = Fraction(0)
    for x in reversed(coef):
        acc = acc * z + Fraction(x)
    return acc


@pytest.mark.parametrize("kind", ["P", "Q"])
def test_header_coefficients_are_derived(kind):
    mod = _script()
    dbl, err = mod.coefficients(kind)
    assert _header_coefficients(kind) == dbl
    assert len(dbl) == mod.DEGREE[kind] + 1 == 4
    assert err <= mod.BOUND
    assert mod.least_degree(kind) == mod.DEGREE[kind]  # one degree less does not meet the bound


def test_truncation_bound_on_dense_grid():
    """|d| <= 1/8 in steps of 2^-14, plus the old tier edges and the largest increment the kernel's high-word test
    admits; the error of sin d and cos d - 1 with the shipped coefficients, evaluated exactly."""
    mod = _script()
    P, Q = _header_coefficients("P"), _header_coefficients("Q")
    _, bound_s = mod.coefficients("P")
    _, bound_c = mod.coefficients("Q")
    grid = [Fraction(k, 2 ** 14) for k in range(0, 2 ** 11 + 1)]
    top = struct.unpack("<d", struct.pack("<II", 0xFFFFFFFF, 0x3FC00000))[0]  # hi word of 1/8, largest low word
    grid += [Fraction(x) for x in (1 / 32, np.nextafter(1 / 32, 1), np.nextafter(1 / 32, 0), 1 / 8,
                                   np.nextafter(1 / 8, 0), top)]
    worst_s = worst_c = Fraction(0)
    for d in grid:
        z = d * d
        s, cm1 = _sin_cos_m1(d)
        es = abs(d + d ** 3 * _poly(P, z) - s)
        ec = abs(z * _poly(Q, z) - cm1)
        if d <= mod.D_MAX:
            assert es <= bound_s and ec <= bound_c, (float(d), float(es), float(ec))
        assert es <= mod.BOUND and ec <= mod.BOUND, (float(d), float(es), float(ec))
        # the sine's error scales with d^3: at most bound_s (1/8)^-3 d^3
        assert es * mod.D_MAX ** 3 <= bound_s * d ** 3
        worst_s, worst_c = max(worst_s, es), max(worst_c, ec)
    print("\n[rotation poly] max truncation over %d increments: sin %.2e, cos - 1 %.2e"
          % (len(grid), float(worst_s), float(worst_c)))


def _edge_increments_dense():
    """Increments on, and one and two ulps / high words either side of, 1/32 and 1/8, both signs."""
    out = []
    for edge in (tt.SHORT, tt.LONG):
        hi = struct.unpack("<II", struct.pack("<d", edge))[1]
        out += [tt._from_words(hi - 2, 0), tt._from_words(hi - 1, 0), np.nextafter(edge, 0), edge,
                np.nextafter(edge, 1), tt._from_words(hi, 0xFFFFFFFF), tt._from_words(hi + 1, 0),
                tt._from_words(hi + 2, 0)]
    out = np.array(out)
    return np.concatenate([out, -out])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 3, 4, 5])
def test_thread_kernel_at_old_tier_edges_matches_oracle(S, O, n):
    """h = 2^-10 so that d = h thd is exact; every other environment starts with one segment on an edge increment,
    and the calm ones stay far below 1/32.  Every visited state is stepped by the oracle (STEP_TOL of
    test_trig_tiers), and the spun environments are checked past the step where the edge increment set the angles."""
    h = 2.0 ** -10
    rng = np.random.default_rng(500 + n)
    dd = _edge_increments_dense()
    B, H = 2 * len(dd), 130
    init = tt._calm(rng, n, B)
    spun = np.arange(1, B, 2)
    for j, e in enumerate(spun):
        init[e, 3 + 2 * (j % n)] = dd[j] / h
    assert np.array_equal(h * init[spun, 3 + 2 * (np.arange(len(spun)) % n)], dd)
    ac = rng.uniform(-5, 5, (B, n - 1))
    ps, po = tt._params(S, n, h), tt._params(O, n, h)
    res = tt._launch(S, "THREAD", ps, H, S.ops.POLICY_FIXED_ACTION, B, actions=tt._cuda(ac), init_state=tt._cuda(init))
    traj = res.trajectory.cpu().numpy()
    worst, seen = tt._per_step(init, traj, lambda e, x: O.step(po, O.GYM, x, ac[e])[0])
    assert all(len(seen[e]) >= 3 for e in spun)
    tt._returns_consistent(res, traj, ps)
    print("\n[rotation poly] THREAD n=%d: %d edge increments, max per-step err %.2e" % (n, len(dd), worst))
