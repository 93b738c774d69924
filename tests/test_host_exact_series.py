"""The integer-series references of tests/exact_series.py against the oracle's direct sums on short series.

The oracle accumulates in long double and rounds its normalised result to double, so it may differ from the exact
fp64 quotient by one rounding: the comparisons allow one ulp and require most lags to agree bit for bit.
"""
import numpy as np
import pytest

from oracle import oracle as O
from tests import exact_series as ES


def _within_one_ulp(got, ref):
    ulp = np.spacing(np.maximum(np.abs(got), np.abs(ref)))
    assert np.all(np.abs(got - ref) <= ulp)
    return np.mean(got == ref)


@pytest.mark.parametrize("T", [1, 2, 7, 300, 2049])
def test_xcorr_lags_match_oracle(T):
    rng = np.random.default_rng(T)
    a = ES.ou_series(rng, 1, T)[0]
    b = ES.ou_series(rng, 1, T, offset=-50)[0]
    for x, y in [(a, b), (b, a), (a, a)]:
        ref = O.xcorr_direct(x.astype(np.float64), y.astype(np.float64))
        got = ES.xcorr_lags(x, y, np.arange(T))
        assert _within_one_ulp(got, ref) >= 0.9
    lags = ES.sample_lags(T, T, rng)
    assert np.array_equal(ES.xcorr_lags(a, b, lags), ES.xcorr_lags(a, b, np.arange(T))[lags])


@pytest.mark.parametrize("T,N", [(2, 1), (40, 3), (600, 5)])
def test_msd_sums_match_oracle(T, N):
    """walks offset by up to 10^6 as traj [T, 3, N]: the oracle's per-axis mean over atoms and origins"""
    rng = np.random.default_rng(T + N)
    chans = ES.walk_series(rng, 3 * N, T)                      # channel 3 i + c is axis c of atom i
    traj = chans.reshape(N, 3, T).transpose(2, 1, 0).astype(np.float64)
    ref = O.msd_all_origins(traj, T)
    lags = np.arange(T)
    for c in range(3):
        got = ES.msd_sums(chans[c::3], lags) / (N * (T - lags)).astype(np.float64)
        assert _within_one_ulp(got, ref[:, c]) >= 0.9
    got = ES.msd_sums(chans, lags) / (N * (T - lags)).astype(np.float64)
    assert _within_one_ulp(got, ref[:, 3]) >= 0.9


@pytest.mark.parametrize("T", [2, 3, 1025, 5001])
@pytest.mark.parametrize("lead", [True, False])
def test_cumtrapz_exact_matches_oracle(T, lead):
    """dyadic steps and integer y: the oracle's fp64 cumsum is exact too, so the match is bit for bit"""
    rng = np.random.default_rng(T)
    y = ES.ou_series(rng, 3, T)
    for dx, scale in [(1.0, 1.0), (2.0 ** -4, 0.5), (0.25, 8.0)]:
        got = ES.cumtrapz_exact(y, dx, scale, lead)
        ref = np.stack([scale * O.cumtrapz(r.astype(np.float64), dx, lead) for r in y])
        assert np.array_equal(got, ref), (dx, scale)


def test_sample_lags_cover_both_ends():
    rng = np.random.default_rng(0)
    lags = ES.sample_lags(10 ** 6, 10 ** 6, rng)
    assert lags[0] == 0 and lags[-1] == 10 ** 6 - 1
    assert set(range(64)) <= set(lags) and set(range(10 ** 6 - 64, 10 ** 6)) <= set(lags)
    assert np.all(np.diff(lags) > 0) and len(lags) <= 192
    assert np.array_equal(ES.sample_lags(5, 3, rng), [0, 1, 2])


def test_generators_are_integer_valued_and_in_range():
    rng = np.random.default_rng(1)
    w = ES.walk_series(rng, 4, 1000)
    assert w.dtype == np.int64 and np.abs(w).max() <= 10 ** 6 + 2 * 1000
    assert np.abs(np.diff(w, axis=1)).max() <= 2
    o = ES.ou_series(rng, 2, 10 ** 5, sigma=300.0, offset=1000)
    assert o.dtype == np.int64 and abs(o.mean() - 1000) < 30 and 250 < o.std() < 350
    r = ES.complex_rho(rng, 2, 3, 100)
    assert r.shape == (2, 3, 100) and np.array_equal(r.real, np.rint(r.real)) and np.array_equal(r.imag, np.rint(r.imag))


def test_bound_assertions_fire():
    """inputs that break the 2^53 condition, or are not integers, or have non-dyadic steps, are refused"""
    big = np.full(8, 2 ** 26, dtype=np.int64)                  # 2^52 per product, 8 terms: 2^55
    with pytest.raises(AssertionError, match="2\\^53"):
        ES.xcorr_lags(big, big, [0])
    ES.assert_exact_xcorr(big[:1], big[:1])                    # one term of 2^52 is still exact
    with pytest.raises(AssertionError, match="2\\^53"):
        ES.assert_exact_xcorr(np.ones((1, 4)), np.ones((1, 4)), terms=2 ** 52)
    walk = np.array([[0, 2 ** 25, 0, 2 ** 25]])                # range^2 = 2^50, 4 origins x 2 channels: 2^53
    with pytest.raises(AssertionError, match="2\\^53"):
        ES.assert_exact_msd(walk, channels=2)
    ES.assert_exact_msd(walk)
    with pytest.raises(AssertionError, match="2\\^53"):
        ES.msd_sums(np.concatenate([walk] * 2), [1])
    with pytest.raises(AssertionError, match="integer"):
        ES.xcorr_lags(np.array([0.5, 1.0]), np.array([1.0, 1.0]), [0])
    with pytest.raises(AssertionError, match="powers of two"):
        ES.cumtrapz_exact(np.arange(4), 0.1)
    with pytest.raises(AssertionError, match="2\\^53"):
        ES.cumtrapz_exact(np.full(3, 2 ** 51, dtype=np.int64), 1.0)
