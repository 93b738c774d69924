"""Integer-valued time series and exact references for the time-correlation kernels (host only).

When every term and every partial sum of a correlation is an integer below 2^53, every fp64 add and FMA on it is exact,
in any order.  So on such inputs

* the direct correlation k_xcorr returns fl(X(tau) / (T - tau)) with X(tau) the exact integer lag sum: bit for bit the
  host's int64 sum divided in fp64;
* the windowed MSD k_msd_window (ops.msd_all_origins, scale 1) returns the exact sum of (x(t + tau) - x(t))^2: it takes
  the difference before squaring, so large offsets cost nothing;
* the cumulative trapezoid k_cumtrapz with integer y, dx = 2^-k and a power-of-two scale returns the host's int64
  cumulative sum, scaled, bit for bit.

The ``assert_exact_*`` functions check that condition on the actual data, so a test cannot silently leave the exact
regime.  The references are int64 sums at sampled lags (``sample_lags``): at long T a full host reference is O(T^2).
"""
from __future__ import annotations

import math

import numpy as np
from scipy.signal import lfilter

EXACT = 2 ** 53


# ----------------------------------------------------------------------------------------------------------------------
# generators
# ----------------------------------------------------------------------------------------------------------------------
def ou_series(rng, C, T, tau=40.0, sigma=300.0, offset=0):
    """[C, T] int64: an Ornstein-Uhlenbeck-like process (AR(1) with correlation time ``tau`` steps and stationary
    standard deviation ``sigma``) rounded to integers, plus ``offset``.  Pressure- or velocity-like."""
    phi = math.exp(-1.0 / tau)
    noise = rng.normal(0.0, sigma * math.sqrt(1.0 - phi * phi), (C, T))
    noise[:, 0] = rng.normal(0.0, sigma, C)              # start in the stationary distribution
    return np.rint(lfilter([1.0], [1.0, -phi], noise, axis=1)).astype(np.int64) + int(offset)


def walk_series(rng, C, T, max_step=2, max_offset=10 ** 6):
    """[C, T] int64 random walks with steps in [-max_step, max_step] and a per-channel offset in
    [-max_offset, max_offset]: unwrapped coordinates far from the origin."""
    steps = rng.integers(-max_step, max_step + 1, (C, T), dtype=np.int64)
    steps[:, 0] = 0
    return np.cumsum(steps, axis=1) + rng.integers(-max_offset, max_offset + 1, (C, 1), dtype=np.int64)


def complex_rho(rng, nchan, nk, T, sigma=200.0):
    """[nchan, nk, T] complex128 density modes with integer real and imaginary parts (OU-like)."""
    re = ou_series(rng, nchan * nk, T, tau=25.0, sigma=sigma).reshape(nchan, nk, T)
    im = ou_series(rng, nchan * nk, T, tau=25.0, sigma=sigma).reshape(nchan, nk, T)
    return re.astype(np.float64) + 1j * im.astype(np.float64)


def sample_lags(T, nlags, rng, n=64):
    """sorted distinct lags < nlags: the first n, the last n (where T - tau is smallest when nlags = T) and n at random"""
    lags = np.concatenate((np.arange(min(n, nlags)), np.arange(max(0, nlags - n), nlags),
                           rng.integers(0, nlags, n)))
    return np.unique(lags).astype(np.int64)


# ----------------------------------------------------------------------------------------------------------------------
# exactness conditions
# ----------------------------------------------------------------------------------------------------------------------
def _int_valued(x):
    x = np.asarray(x)
    if x.dtype.kind in "iu":
        return x.astype(np.int64)
    if not np.array_equal(x, np.rint(x)):
        raise AssertionError("series is not integer-valued")
    return x.astype(np.int64)


def assert_exact_xcorr(a, b, terms=1):
    """Every partial sum of ``terms`` lag sums of a[t + tau] * b[t] (a, b [.., T]) stays below 2^53: max|a| max|b| T terms."""
    a, b = _int_valued(a), _int_valued(b)
    bound = int(np.abs(a).max()) * int(np.abs(b).max()) * a.shape[-1] * int(terms)
    assert bound < EXACT, f"xcorr sums may reach {bound} >= 2^53: not exact in fp64"
    return bound


def assert_exact_msd(x, channels=None):
    """Every partial sum of (x(t + tau) - x(t))^2 over the origins and ``channels`` channels (default: all of x [C, T])
    stays below 2^53: the largest squared range times T times the channel count."""
    x = _int_valued(x).reshape(-1, np.shape(x)[-1])
    rng2 = int((x.max(axis=1) - x.min(axis=1)).max()) ** 2
    bound = rng2 * x.shape[1] * int(x.shape[0] if channels is None else channels)
    assert bound < EXACT, f"MSD sums may reach {bound} >= 2^53: not exact in fp64"
    return bound


def _pow2(v):
    m, _ = math.frexp(float(v))
    return abs(m) == 0.5


def assert_exact_cumtrapz(y, dx, scale):
    """dx and scale are powers of two and the running sum of (y[k + 1] + y[k]) stays below 2^53."""
    y = _int_valued(y)
    assert _pow2(dx) and _pow2(scale), "dx and scale must be powers of two"
    bound = 2 * int(np.abs(y).sum(axis=-1).max())
    assert bound < EXACT, f"trapezoid sums may reach {bound} >= 2^53: not exact in fp64"
    return bound


# ----------------------------------------------------------------------------------------------------------------------
# int64 references
# ----------------------------------------------------------------------------------------------------------------------
def xcorr_sums(a, b, lags):
    """exact int64 X(tau) = sum_{t < T - tau} a[t + tau] * b[t] for 1-D integer series, at ``lags``"""
    a, b = _int_valued(a), _int_valued(b)
    T = a.shape[0]
    return np.array([int(np.dot(a[tau:], b[:T - tau])) for tau in lags], dtype=np.int64)


def xcorr_lags(a, b, lags):
    """what k_xcorr returns at ``lags`` on exact inputs: fl(X(tau) / (T - tau))"""
    assert_exact_xcorr(a, b)
    T = np.shape(a)[-1]
    lags = np.asarray(lags, dtype=np.int64)
    return xcorr_sums(a, b, lags).astype(np.float64) / (T - lags).astype(np.float64)


def msd_sums(x, lags):
    """exact int64 sum over the channels of x [C, T] and the origins of (x(t + tau) - x(t))^2, at ``lags``"""
    x = _int_valued(x).reshape(-1, np.shape(x)[-1])
    assert_exact_msd(x)
    T = x.shape[1]
    out = np.empty(len(lags), dtype=np.int64)
    for i, tau in enumerate(lags):
        d = x[:, tau:] - x[:, :T - tau]
        out[i] = int(np.einsum("ij,ij->", d, d))
    return out


def cumtrapz_exact(y, dx, scale=1.0, leading_zero=True):
    """scale * cumulative trapezoid of integer y [.., T] with step dx, from the int64 running sum of y[k + 1] + y[k]"""
    y = _int_valued(y)
    assert_exact_cumtrapz(y, dx, scale)
    run = np.cumsum(y[..., 1:] + y[..., :-1], axis=-1)
    if leading_zero:
        run = np.concatenate((np.zeros(y.shape[:-1] + (1,), dtype=np.int64), run), axis=-1)
    return run.astype(np.float64) * (0.5 * float(dx) * float(scale))
