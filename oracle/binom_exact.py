"""TEST INFRASTRUCTURE ONLY -- exact reference for the binomial statistics of K6 (yacht_b200/csrc/binom_stats.cuh).

scipy (Boost.Math) is the reference the product is compared with, but scipy is itself an fp64 evaluation: it loses
p-values below ~1e-250 to underflow, settles exact ties of cdf(k) == q by rounding, and cannot resolve a 1e-15 tail next
to 1.  This module computes the same quantities with mpmath at DPS decimal digits, so a disagreement between the kernel
and scipy can be settled against the true value:

  * pmf from loggamma;
  * each tail as a direct sum of exact pmf ratios, started at the boundary term and running away from it until a term is
    below 2^-100 (8e-31) of the sum, in exact integer fixed point (mpmath.betainc does not converge for n >~ 1e5);
  * ppf(q) as the smallest k whose exact cdf is >= the exact value of the double q;
  * betaincinv(n - k, k + 1, y) as the root w of P[Bin(n, w) <= k] = y (x = 1 - w), bracketed and refined on the exact tail;
  * the alternative mutation rate 1 - w ** (1 / ksize) from that root;
  * ``cdf_fraction``: the cdf as a Fraction for dyadic p (exact ties, small n);
  * ``ambiguity_band``: the k whose exact cdf lies within what an fp64 evaluation can resolve from q.

Arguments p, q, y are the doubles the kernel receives; their exact binary values are used.  Only tests/ may import this.
"""
from __future__ import annotations

from fractions import Fraction
from typing import Iterable, List, Tuple

import mpmath

DPS = 50
EPS53 = 2.0 ** -53


def _mp(x) -> mpmath.mpf:
    return mpmath.mpf(x)   # exact for a double at DPS >= 16


def pmf(k: int, n: int, p: float) -> mpmath.mpf:
    """P[Bin(n, p) = k], 0 <= k <= n, 0 < p < 1."""
    with mpmath.workdps(DPS):
        p = _mp(p)
        return mpmath.exp(mpmath.loggamma(n + 1) - mpmath.loggamma(k + 1) - mpmath.loggamma(n - k + 1)
                          + k * mpmath.log(p) + (n - k) * mpmath.log1p(-p))


def _odds(p) -> Tuple[int, int]:
    """(a, b) with p = a / (a + b) exactly, for a double or an mpf p in (0, 1)."""
    man, exp = mpmath.mpf(p).man_exp
    den = 1 << -exp if exp < 0 else 1
    num = man << exp if exp > 0 else man
    return num, den - num


FIX = 192   # fixed-point bits of the ratio sums: each step truncates below 2^-192 of the boundary term


def _ratio_sum(k: int, n: int, p, down: bool) -> mpmath.mpf:
    """1 + r + r r' + ... with the exact ratios pmf(i -+ 1) / pmf(i), from k away from it, in integer fixed point."""
    a, b = _odds(p)
    one = 1 << FIX
    t = s = one
    if down:            # r_i = pmf(i-1) / pmf(i) = i b / ((n - i + 1) a)
        i = k
        while i >= 1 and t:
            num, den = i * b, (n - i + 1) * a
            t = t * num // den
            s += t
            i -= 1
            if num < den and t < (s >> 100):
                break
    else:               # u_i = pmf(i+1) / pmf(i) = (n - i) a / ((i + 1) b)
        i = k
        while i < n and t:
            num, den = (n - i) * a, (i + 1) * b
            t = t * num // den
            s += t
            i += 1
            if num < den and t < (s >> 100):
                break
    with mpmath.workdps(DPS):
        return mpmath.mpf(s) / one


def lower_tail(k: int, n: int, p) -> mpmath.mpf:
    """P[X <= k]: pmf(k) times 1 + r_k + r_k r_{k-1} + ..., r_i = pmf(i-1) / pmf(i), summed away from k until a term is
    below 2^-100 of the sum."""
    if k < 0:
        return mpmath.mpf(0)
    if k >= n:
        return mpmath.mpf(1)
    with mpmath.workdps(DPS):
        return pmf(k, n, p) * _ratio_sum(k, n, p, True)


def upper_tail(k: int, n: int, p) -> mpmath.mpf:
    """P[X >= k], summed away from k like lower_tail."""
    if k <= 0:
        return mpmath.mpf(1)
    if k > n:
        return mpmath.mpf(0)
    with mpmath.workdps(DPS):
        return pmf(k, n, p) * _ratio_sum(k, n, p, False)


def cdf_sf(k: int, n: int, p: float) -> Tuple[mpmath.mpf, mpmath.mpf]:
    """(P[X <= k], P[X > k]); the tail on k's side of the mode is summed, the other is its complement."""
    with mpmath.workdps(DPS):
        if k < 0:
            return mpmath.mpf(0), mpmath.mpf(1)
        if k >= n or p <= 0.0:
            return mpmath.mpf(1), mpmath.mpf(0)
        if p >= 1.0:
            return mpmath.mpf(0), mpmath.mpf(1)
        if p == 0.5 and 2 * k + 1 == n:     # symmetry: P[X <= (n-1)/2] = P[X >= (n+1)/2] = 1/2
            return mpmath.mpf(0.5), mpmath.mpf(0.5)
        if k + 1 <= (n + 1) * _mp(p):
            c = lower_tail(k, n, p)
            return c, 1 - c
        s = upper_tail(k + 1, n, p)
        return 1 - s, s


def cdf(k: int, n: int, p: float) -> mpmath.mpf:
    return cdf_sf(k, n, p)[0]


def ppf(q: float, n: int, p: float, guess: int = None) -> int:
    """Smallest k in [0, n] with the exact P[Bin(n, p) <= k] >= q (the double q taken exactly); -1 for q == 0.
    `guess` (e.g. scipy's answer) starts the search; the result does not depend on it."""
    if q == 0.0:
        return -1
    if q == 1.0 or p == 1.0:
        return n
    if n <= 0 or p == 0.0:
        return 0
    qe = _mp(q)
    ge = lambda k: cdf(k, n, p) >= qe   # noqa: E731
    k = min(max(int(guess) if guess is not None else int(n * p), 0), n)
    step = 1
    if ge(k):                  # gallop down to an lo with cdf(lo) < q (or lo = -1)
        hi = k
        while True:
            lo = hi - step
            if lo < 0:
                lo = -1
                break
            if not ge(lo):
                break
            hi, step = lo, step * 2
    else:                      # gallop up to an hi with cdf(hi) >= q (cdf(n) = 1 >= q)
        lo = k
        while True:
            hi = lo + step
            if hi >= n:
                hi = n
                break
            if ge(hi):
                break
            lo, step = hi, step * 2
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if ge(mid):
            hi = mid
        else:
            lo = mid
    return hi


def tau(q: float, c: mpmath.mpf) -> mpmath.mpf:
    """What an fp64 evaluation of cdf(k) = c can resolve from q: 4 ulp of max(q, 1 - q) plus 1e-13 of the small side."""
    with mpmath.workdps(DPS):
        qe = _mp(q)
        return 4 * EPS53 * max(qe, 1 - qe) + mpmath.mpf("1e-13") * min(c, 1 - c)


def ambiguity_band(q: float, n: int, p: float, ks: Iterable[int]) -> List[int]:
    """Those k of `ks` whose exact cdf(k) lies within tau of q: for them `cdf(k) >= q` is not decidable in fp64."""
    qe = _mp(q)
    out = []
    for k in ks:
        c = cdf(int(k), n, p)
        with mpmath.workdps(DPS):
            if abs(c - qe) <= tau(q, c):
                out.append(int(k))
    return out


def ppf_acceptable(got: int, q: float, n: int, p: float, exact: int = None) -> bool:
    """`got` is the exact ppf, or every k between it and the exact ppf lies in the ambiguity band, i.e. the two answers
    differ only in comparisons fp64 cannot settle."""
    exact = ppf(q, n, p, got) if exact is None else exact
    if got == exact:
        return True
    lo, hi = min(got, exact), max(got, exact)
    ks = range(lo, hi)   # the cdf(k) >= q decisions that differ: k in [lo, hi)
    return len(ks) <= 64 and ambiguity_band(q, n, p, ks) == list(ks)


def betaincinv_int(n: int, k: int, y: float) -> mpmath.mpf:
    """x with I_x(n - k, k + 1) = y, i.e. 1 - w for the root w of P[Bin(n, w) <= k] = y (0 <= k < n, 0 < y < 1)."""
    with mpmath.workdps(DPS):
        ye = _mp(y)
        if k == 0:
            return ye ** (mpmath.mpf(1) / n)          # I_x(n, 1) = x ** n
        if k == n - 1:
            return 1 - (1 - ye) ** (mpmath.mpf(1) / n)   # P[Bin(n, w) <= n - 1] = 1 - w ** n
        # residual g(w) = cdf(k; n, w) - y, decreasing in w, formed on the smaller side of y
        def g(w):
            c, sf = cdf_sf(k, n, w)
            return c - ye if ye <= 0.5 else (1 - ye) - sf
        lo, hi = mpmath.mpf(0), mpmath.mpf(1)
        w = mpmath.mpf(k) / n
        for _ in range(400):
            gw = g(w)
            if gw > 0:
                lo = w
            else:
                hi = w
            # Newton: d cdf / dw = -(n - k) pmf(k; n, w) / (1 - w)
            d = (n - k) * pmf(k, n, w) / (1 - w)
            wn = w + gw / d if d > 0 else (lo + hi) / 2
            if not (lo < wn < hi):
                wn = (lo + hi) / 2
            if abs(wn - w) <= w * mpmath.mpf(10) ** -(DPS - 15) or hi - lo <= w * mpmath.mpf(10) ** -(DPS - 15):
                return 1 - wn
            w = wn
        raise RuntimeError(f"betaincinv_int({n}, {k}, {y}) did not converge")


def alt_mut_rate(nu: int, thresh: int, ksize: int, significance: float) -> float:
    """get_alt_mut_rate(nu, thresh, ksize, significance), exactly, as a double; -1.0 where scipy's betaincinv is NaN
    (a = nu - thresh <= 0, b = 1 + thresh <= 0).  Edge values follow betaincinv: y = 0 -> x = 0, y = 1 -> x = 1."""
    if nu - thresh <= 0 or thresh + 1 <= 0:
        return -1.0
    if significance == 0.0:
        return 0.0
    if significance == 1.0:
        return 1.0
    with mpmath.workdps(DPS):
        x = betaincinv_int(nu, thresh, significance)
        return float(1 - (1 - x) ** (mpmath.mpf(1) / ksize))


def cdf_fraction(k: int, n: int, p: float) -> Fraction:
    """P[Bin(n, p) <= k] exactly, for any double p (its exact binary value); meant for small n."""
    pf = Fraction(p)
    qf = 1 - pf
    s = Fraction(0)
    for i in range(0, min(k, n) + 1):
        s += _binom(n, i) * pf ** i * qf ** (n - i)
    return s


def _binom(n: int, i: int) -> int:
    from math import comb
    return comb(n, i)
