"""Reference values of the rolling z-score (Feature.normalise, rl4mm/features/Features.py:67-74) for the z-score tests.

The reference keeps the clamped feature values in a deque(maxlen=max_norm_len) and returns
scipy.stats.zscore(np.asarray(history))[-1]; the history starts as [x0 + 1e-06, x0] at the first update.  Three views of
one window:

* ``scipy_z``: the reference's own operation, numpy's pairwise sums and rounding included (scipy 1.18.1, the version
  DESIGN.md and the oracle follow);
* ``exact_z``: mean and variance of the double inputs in exact rational arithmetic, square root and quotient in 60 digits;
* ``regime``: which of the device's three paths (csrc/env.cuh feature_normalise) the window falls in, and so how a device
  value has to be compared: bit for bit where the reference's answer is decided by its rounding (NaN, constant and
  noise-dominated windows), within ``NORMAL_C * EPS * kappa`` of the exact value elsewhere.
"""
from __future__ import annotations

import math
import warnings
from collections import Counter
from decimal import Decimal, localcontext
from fractions import Fraction

import numpy as np
import scipy.stats

EPS = float(np.finfo(np.float64).eps)
NORMAL_C = 256          # normal-regime tolerance in units of EPS * kappa


def scipy_z(window) -> float:
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return float(scipy.stats.zscore(np.array(window, dtype=np.float64))[-1])


def _dec(q: Fraction) -> Decimal:
    return Decimal(q.numerator) / Decimal(q.denominator)


def exact_z(window):
    """(z, sd, mean) of the window in exact arithmetic (z NaN when the variance is 0); sd and mean rounded to double."""
    return exact_z_counts(Counter(float(x) for x in window).items(), float(window[-1]))


def exact_z_counts(items, last: float):
    """exact_z of a window given as (value, count) pairs whose last entry is ``last``."""
    items = [(Fraction(v), k) for v, k in items]
    n = sum(k for _, k in items)
    mean = sum(v * k for v, k in items) / n
    var = sum(k * (v - mean) ** 2 for v, k in items) / n
    if var == 0:
        return float("nan"), 0.0, float(mean)
    with localcontext() as ctx:
        ctx.prec = 60
        sd = _dec(var).sqrt()
        z = (_dec(Fraction(last)) - _dec(mean)) / sd
    return float(z), float(sd), float(mean)


def kappa(x: float, z: float, sd: float, mean: float) -> float:
    """Condition number of z = (x - mean) / sd with respect to relative perturbations of the window's entries."""
    return 1.0 + abs(z) + (abs(x) + abs(mean)) / sd


def numpy_moments(window):
    """scipy's mean and standard deviation of the window (numpy's pairwise sums, ddof 0)."""
    a = np.array(window, dtype=np.float64)
    mean = np.mean(a)
    return float(mean), float(np.sqrt(np.mean((a - mean) * (a - mean))))


def regime(window) -> str:
    """'nan' (a non-finite entry), 'constant' (all entries equal), 'noise' (sd <= 0.5e-8 |mean|: a factor 2 inside the
    device's 1e-8 switch, so that a device whose running sums put the window on the other side of 1e-8 still replays it
    exactly) or 'normal'."""
    a = np.array(window, dtype=np.float64)
    if not np.all(np.isfinite(a)):
        return "nan"
    if np.all(a == a[0]):
        return "constant"
    mean, sd = numpy_moments(a)
    return "noise" if sd <= 0.5e-8 * abs(mean) else "normal"


def same_bits(a: float, b: float) -> bool:
    return (math.isnan(a) and math.isnan(b)) or np.float64(a).tobytes() == np.float64(b).tobytes()


def np_pairwise_sum(a, lo: int = 0, n: int | None = None) -> float:
    """numpy's pairwise_sum_DOUBLE (contiguous input): eight accumulators over blocks of <= 128 entries, split in two
    (the first half a multiple of 8) above that."""
    n = len(a) if n is None else n
    if n < 8:
        r = -0.0
        for i in range(n):
            r += float(a[lo + i])
        return r
    if n <= 128:
        r = [float(a[lo + j]) for j in range(8)]
        body = n - n % 8
        for i in range(8, body, 8):
            for j in range(8):
                r[j] += float(a[lo + i + j])
        res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
        for i in range(body, n):
            res += float(a[lo + i])
        return res
    n2 = pairwise_split(n)
    return np_pairwise_sum(a, lo, n2) + np_pairwise_sum(a, lo + n2, n - n2)


def pairwise_split(n: int) -> int:
    """Length of the first half when numpy's pairwise sum splits n > 128 entries."""
    n2 = n // 2
    return n2 - n2 % 8
