"""Coefficients of the one-tier rotation polynomial of gym_step_tracked (dynamics.cuh), in exact rational arithmetic.

For an angle increment |d| <= 1/8 and z = d^2 in [0, 1/64]:

    sin d     = d + d^3 P(z)      P(z) = sum_k (-1)^(k+1) z^k / (2k+3)!
    cos d - 1 = z Q(z)            Q(z) = sum_k (-1)^(k+1) z^k / (2k+2)!

P and Q themselves (not sin d and cos d - 1) are approximated in z, so that the error of the sine scales with d^3
and that of cos d - 1 with d^2: each Taylor series is cut at degree TAYLOR_DEGREE and then Chebyshev-economised
down to degree `DEGREE` on [0, Z_MAX].  The bounds below are rigorous for the rounded (double) coefficients
evaluated exactly: Taylor tail + economisation + coefficient rounding, each scaled by the largest |d|^3 or z.

  python rotation_poly.py     prints the coefficients as they appear in dynamics.cuh, the bounds, and the least
                              degrees that meet BOUND
"""
from fractions import Fraction
from math import factorial

D_MAX = Fraction(1, 8)
Z_MAX = D_MAX * D_MAX
BOUND = Fraction(3, 10 ** 17)  # absolute truncation error allowed for sin d and cos d - 1 over |d| <= D_MAX
DEGREE = {"P": 3, "Q": 3}
TAYLOR_DEGREE = 8


def taylor(kind, k):
    """Coefficient of z^k in P (kind 'P') or Q (kind 'Q')."""
    return Fraction((-1) ** (k + 1), factorial(2 * k + (3 if kind == "P" else 2)))


def shifted_chebyshev(k, a):
    """Coefficients (ascending powers of z) of T_k(2 z / a - 1)."""
    x = [Fraction(-1), Fraction(2) / a]  # 2 z / a - 1
    t0, t1 = [Fraction(1)], x
    if k == 0:
        return t0
    for _ in range(k - 1):
        t2 = [Fraction(0)] * (len(t1) + 1)
        for i, ci in enumerate(t1):
            for j, xj in enumerate(x):
                t2[i + j] += 2 * ci * xj
        for i, ci in enumerate(t0):
            t2[i] -= ci
        t0, t1 = t1, t2
    return t1


def economise(kind, degree, taylor_degree=TAYLOR_DEGREE, a=Z_MAX):
    """Exact coefficients of degree `degree` and a bound on |approximation - P or Q| over [0, a].

    The Taylor series is alternating with decreasing terms on [0, a], so its tail after taylor_degree is bounded by
    the first omitted term; each economisation step removes c_k z^k by subtracting c_k / lead(T_k*) T_k*, whose
    magnitude on [0, a] is |c_k / lead(T_k*)|."""
    c = [taylor(kind, k) for k in range(taylor_degree + 1)]
    err = abs(taylor(kind, taylor_degree + 1)) * a ** (taylor_degree + 1)
    for k in range(taylor_degree, degree, -1):
        t = shifted_chebyshev(k, a)
        f = c[k] / t[k]
        for i in range(k + 1):
            c[i] -= f * t[i]
        assert c[k] == 0
        err += abs(f)
    return c[:degree + 1], err


def coefficients(kind, degree=None):
    """The double coefficients (ascending powers of z) and a rigorous bound on the absolute error of sin d
    (kind 'P') or cos d - 1 (kind 'Q') over |d| <= D_MAX when the polynomial is evaluated exactly."""
    degree = DEGREE[kind] if degree is None else degree
    exact, err = economise(kind, degree)
    dbl = [float(x) for x in exact]  # int / int division in Python rounds correctly
    err += sum(abs(Fraction(x) - e) * Z_MAX ** k for k, (x, e) in enumerate(zip(dbl, exact)))
    scale = D_MAX ** 3 if kind == "P" else Z_MAX
    return dbl, err * scale


def least_degree(kind):
    return next(k for k in range(1, TAYLOR_DEGREE) if coefficients(kind, k)[1] <= BOUND)


def main():
    for kind, what in (("P", "sin d = d + d^3 P(z)"), ("Q", "cos d - 1 = z Q(z)")):
        dbl, err = coefficients(kind)
        print("// %s, degree %d: |error| <= %.3e over |d| <= 1/8 (least degree meeting %.0e: %d)"
              % (what, DEGREE[kind], float(err), float(BOUND), least_degree(kind)))
        print("constexpr double kRotate%s[%d] = {%s};" % (kind, len(dbl), ", ".join(repr(x) for x in dbl)))


if __name__ == "__main__":
    main()
