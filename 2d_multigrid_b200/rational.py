"""Rational approximations r(x) ~ x^p on [a, b] for the one-flavour RHMC (host only, mpmath).

r(x) = alpha0 + sum_k alpha_k / (x + beta_k),  beta_k > 0 and distinct,

the best approximation of type (n, n) in the relative error max |r(x) / x^p - 1|, found by a Remez exchange in mpmath.  x^p is
homogeneous, so the approximation is computed once on [a/b, 1] and scaled: x^p = b^p (x/b)^p.  The coefficients are returned in
float64 with the error the float64 coefficients achieve.

Two accuracy classes are used by HMC(flavours=1): PRECISE (1e-12) for the heat bath (p = +1/4) and the accept step (p = -1/2),
MD (1e-6, p = -1/2) for the force, where an error only costs acceptance.
"""
from __future__ import annotations

import functools
import math

import mpmath as mp

PRECISE_TOL = 1e-12
MD_TOL = 1e-6


class RationalApprox:
    """r(x) = alpha0 + sum_k alpha[k] / (x + beta[k]) ~ x^p on [a, b] with max relative error `error` (beta ascending)."""

    def __init__(self, p, a, b, alpha0, alpha, beta, error):
        self.p, self.a, self.b = p, a, b
        self.alpha0, self.alpha, self.beta, self.error = alpha0, list(alpha), list(beta), error

    @property
    def n(self) -> int:
        return len(self.beta)

    def __call__(self, x):
        """r(x) for a float or a numpy array (evaluated in the array's dtype)."""
        s = self.alpha0 + 0 * x
        for al, be in zip(self.alpha, self.beta):
            s = s + al / (x + be)
        return s

    def __repr__(self):
        return f"RationalApprox(p={self.p}, [{self.a:.3g}, {self.b:.3g}], n={self.n}, error={self.error:.3g})"


def rational_approx(p: float, a: float, b: float, tol: float) -> RationalApprox:
    """Best relative (n, n) approximation of x^p on [a, b] with the smallest n whose max relative error is <= tol.
    p in {-1/2, +1/4}; 0 < a < b."""
    if p not in (-0.5, 0.25):
        raise ValueError("p must be -1/2 or +1/4")
    if not (math.isfinite(a) and math.isfinite(b) and 0.0 < a < b):
        raise ValueError(f"need 0 < a < b, got [{a}, {b}]")
    if not 1e-15 <= tol < 0.1:
        raise ValueError("tol must be in [1e-15, 0.1)")
    eps = a / b
    n = _estimate_n(eps, tol)
    r = _scaled(p, n, a, b)
    if r.error <= tol:
        while n > 1:
            r1 = _scaled(p, n - 1, a, b)
            if r1.error > tol:
                break
            n, r = n - 1, r1
    else:
        while r.error > tol:
            n += 1
            if n > 64:
                raise ValueError(f"no approximation of x^{p} on [{a}, {b}] to {tol} with at most 64 poles")
            r = _scaled(p, n, a, b)
    return r


def _scaled(p, n, a, b):
    """The approximation of [a/b, 1] scaled to [a, b] in float64, x^p = b^p (x/b)^p, with the max relative error of the float64
    coefficients at the extrema of the exchange and on a log grid."""
    alpha0, alpha, beta, X = _remez(p, n, a / b)
    s = b ** p
    r = RationalApprox(p, a, b, alpha0 * s, [al * s * b for al in alpha], [be * b for be in beta], None)
    with mp.workdps(30):
        lo, hi = mp.log(a), mp.log(b)
        pts = [mp.mpf(x) * b for x in X] + [mp.exp(lo + (hi - lo) * i / (40 * n)) for i in range(40 * n + 1)]
        e = max(abs((mp.mpf(r.alpha0) + mp.fsum(mp.mpf(al) / (x + mp.mpf(be)) for al, be in zip(r.alpha, r.beta)))
                    / x ** mp.mpf(p) - 1) for x in pts)
    r.error = float(e * (1 + mp.mpf("1e-4")))          # the sup between the sampled points: within the levelling tolerance
    return r


def _estimate_n(eps, tol):
    """Degree from Zolotarev's asymptotic error 4 exp(-(2n+1) pi^2 / (2 ln(4/sqrt(eps)))) of the sign function."""
    n = (2.0 * math.log(4.0 / math.sqrt(eps)) * math.log(4.0 / tol) / math.pi ** 2 - 1.0) / 2.0
    return max(1, int(math.ceil(n)))


@functools.lru_cache(maxsize=None)
def _remez(p, n, eps):
    """(alpha0, alpha, beta, extrema of the relative error) of the best relative (n, n) approximation of x^p on [eps, 1], in
    float64."""
    dps = 30 + int(math.ceil(n * math.log10(1.0 / eps)))     # the monomial basis needs ~n log10(1/eps) digits
    with mp.workdps(dps):
        return _remez_mp(mp.mpf(p), n, mp.mpf(eps))


def _remez_mp(p, n, eps):
    # start from Zolotarev's optimal approximation of x^(-1/2): its reference points (the extrema of its relative error) and
    # its denominator.  x^(+1/4) is reached by continuation in p to x^(-1/4) (an exchange from a poor start can settle on a
    # degenerate solution with a cancelling pole-zero pair), and 1 / r(x) ~ x^(+1/4) when r(x) ~ x^(-1/4): the numerator of
    # the one is the denominator of the other.
    X, Q = _zolotarev_start(n, eps)
    X, P, Q = _exchange(mp.mpf(-0.5), n, eps, X, Q)
    if p > 0:
        for q in (-0.4375, -0.375, -0.3125, -0.25):
            X, P, Q = _exchange(mp.mpf(q), n, eps, X, Q)
        X, P, Q = _exchange(p, n, eps, X, [c / P[n] for c in P])
    # partial fractions r = P / Q = p_n + sum_k alpha_k / (x + beta_k), beta_k = -roots of Q (monic)
    roots = mp.polyroots(list(reversed(Q)), maxsteps=400, extraprec=4 * mp.mp.prec)
    beta = sorted(-mp.re(z) for z in roots)
    if any(abs(mp.im(z)) > mp.mpf(10) ** (-mp.mp.dps // 3) * abs(z) for z in roots) or min(beta) <= 0:
        raise ValueError(f"Remez for x^{p} of degree {n}: the poles are not all on the negative axis")
    dQ = [j * Q[j] for j in range(1, n + 1)]
    alpha = [_peval(P, -be) / _peval(dQ, -be) for be in beta]
    alpha0 = P[n]
    return float(alpha0), [float(v) for v in alpha], [float(v) for v in beta], [float(x) for x in X]


def _exchange(p, n, eps, X, Q):
    """Remez exchange from the reference X and denominator Q until the relative error of P / Q levels: (X, P, Q)."""
    m = 2 * n + 2
    E = mp.mpf(0)
    for outer in range(60):
        P, Q, E = _solve_levelled(p, n, X, Q, E)
        err = lambda x: _peval(P, x) / (_peval(Q, x) * x ** p) - 1
        # zeros of err between consecutive reference points, then the extremum of |err| between consecutive zeros
        Z = [mp.log(eps)] + [_bisect(err, mp.log(X[i]), mp.log(X[i + 1])) for i in range(m - 1)] + [mp.mpf(0)]
        X, vals = [], []
        for i in range(m):
            t, v = _golden_max(err, Z[i], Z[i + 1])
            X.append(mp.exp(t))
            vals.append(v)
        big, small = max(abs(v) for v in vals), min(abs(v) for v in vals)
        if big - small <= 1e-6 * big:
            return X, P, Q
    raise ValueError(f"Remez for x^{p} of degree {n} on [{eps}, 1] did not level")


def _zolotarev_coeffs(n, eps):
    """c_j = eps sn^2 / cn^2 (j K / (2n+1); k'), k'^2 = 1 - eps, j = 1 .. 2n: Zolotarev's optimal relative approximation of
    x^(-1/2) on [eps, 1] is proportional to prod_m (x + c_2m) / (x + c_2m-1)."""
    m = 1 - eps
    K = mp.ellipk(m)
    return [None] + [eps * (mp.ellipfun("sn", j * K / (2 * n + 1), m=m) / mp.ellipfun("cn", j * K / (2 * n + 1), m=m)) ** 2
                     for j in range(1, 2 * n + 1)]


def _zolotarev_start(n, eps):
    """(the 2n+2 extrema of Zolotarev's relative error on [eps, 1], its monic denominator)"""
    c = _zolotarev_coeffs(n, eps)
    lng = lambda t: t / 2 + mp.fsum(mp.log((mp.exp(t) + c[2 * j]) / (mp.exp(t) + c[2 * j - 1])) for j in range(1, n + 1))
    lo = mp.log(eps)
    T = [lo * (1 - mp.mpf(i) / (200 * n)) for i in range(200 * n + 1)]
    V = [lng(t) for t in T]
    ext = [T[0]] + [T[i] for i in range(1, len(T) - 1) if (V[i] - V[i - 1]) * (V[i + 1] - V[i]) <= 0] + [T[-1]]
    if len(ext) != 2 * n + 2:
        ext = [lo + (0 - lo) * (1 - mp.cos(mp.pi * i / (2 * n + 1))) / 2 for i in range(2 * n + 2)]
    Q = [mp.mpf(1)]
    for j in range(1, n + 1):
        Q = _polymul_linear(Q, c[2 * j - 1])
    return [mp.exp(t) for t in ext], Q


def _polymul_linear(c, r):
    """coefficients (ascending) of c(x) (x + r)"""
    out = [mp.mpf(0)] * (len(c) + 1)
    for j, v in enumerate(c):
        out[j] += v * r
        out[j + 1] += v
    return out


def _peval(c, x):
    s = mp.mpf(0)
    for v in reversed(c):
        s = s * x + v
    return s


def _solve_levelled(p, n, X, Q, E):
    """Newton on P(x_i) - x_i^p (1 + (-1)^i E) Q(x_i) = 0, i < 2n+2, for P (degree n), monic Q (degree n) and E."""
    m = 2 * n + 2
    q = list(Q[:n])
    P = [mp.mpf(0)] * (n + 1)
    for it in range(50):
        A = mp.matrix(m, m)
        F = mp.matrix(m, 1)
        Qc = q + [mp.mpf(1)]
        for i, x in enumerate(X):
            f = x ** p
            s = 1 if i % 2 == 0 else -1
            w = f * (1 + s * E)
            xp = mp.mpf(1)
            for j in range(n + 1):
                A[i, j] = xp
                if j < n:
                    A[i, n + 1 + j] = -w * xp
                xp *= x
            qv = _peval(Qc, x)
            A[i, m - 1] = -f * s * qv
            F[i] = -(_peval(P, x) - w * qv)
            # row scaling by 1 / (f Q(x_i)): every row of order one
            sc = 1 / (f * abs(qv))
            for j in range(m):
                A[i, j] *= sc
            F[i] *= sc
        d = mp.lu_solve(A, F)
        P = [P[j] + d[j] for j in range(n + 1)]
        q = [q[j] + d[n + 1 + j] for j in range(n)]
        E = E + d[m - 1]
        if abs(d[m - 1]) <= mp.mpf("1e-20") * abs(E) and it > 0:
            break
    return P, q + [mp.mpf(1)], E


def _bisect(err, t0, t1):
    """zero of err(e^t) in [t0, t1] (a sign change)"""
    f0 = err(mp.exp(t0))
    for _ in range(48):
        tm = (t0 + t1) / 2
        fm = err(mp.exp(tm))
        if (fm < 0) == (f0 < 0):
            t0, f0 = tm, fm
        else:
            t1 = tm
    return (t0 + t1) / 2


def _golden_max(err, t0, t1):
    """(t, err(e^t)) at the maximum of |err(e^t)| on [t0, t1], endpoints included"""
    g = (mp.sqrt(5) - 1) / 2
    a, b = t0, t1
    c, d = b - g * (b - a), a + g * (b - a)
    fc, fd = abs(err(mp.exp(c))), abs(err(mp.exp(d)))
    for _ in range(40):
        if fc > fd:
            b, d, fd = d, c, fc
            c = b - g * (b - a)
            fc = abs(err(mp.exp(c)))
        else:
            a, c, fc = c, d, fd
            d = a + g * (b - a)
            fd = abs(err(mp.exp(d)))
    best = [(t, err(mp.exp(t))) for t in ((a + b) / 2, t0, t1)]
    return max(best, key=lambda tv: abs(tv[1]))


def zolotarev_error(n: int, eps: float) -> float:
    """Zolotarev's optimal max relative error of a type (n, n) approximation of x^(-1/2) on [eps, 1], from the closed form
    r(x) ~ prod_m (x + c_2m) / (x + c_2m-1), c_j = eps sn^2 / cn^2 (j K / (2n+1); k'), k'^2 = 1 - eps: the relative error
    equioscillates with extrema at both ends of the interval, so delta = |g(1) - g(eps)| / (g(1) + g(eps)) with
    g = sqrt(x) prod (x + c_2m) / (x + c_2m-1)."""
    with mp.workdps(50):
        e = mp.mpf(eps)
        c = _zolotarev_coeffs(n, e)
        g = lambda x: mp.sqrt(x) * mp.fprod((x + c[2 * j]) / (x + c[2 * j - 1]) for j in range(1, n + 1))
        g0, g1 = g(e), g(mp.mpf(1))
        return float(abs(g1 - g0) / (g1 + g0))
