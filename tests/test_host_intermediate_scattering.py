"""Host checks of the coherent intermediate scattering function: the shared bodies of the binned FFT correlation
(csrc/isf_fft.h, run by tests/native/isf_fft_host.cpp) against the oracle's long-double direct sum, the oracle against the
closed form of a rigidly translating configuration, the bin sharding, the lag-time axis and the table's empty bins."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from mdproptools_b200.common import constants as K
from mdproptools_b200.dynamical.intermediate_scattering import isf_table, lag_times, shard_bins
from tests import isf_oracle as IO
from tests import sk_oracle as SO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONTRACT = 1e-10


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = tmp_path_factory.mktemp("isf_fft") / "isf_fft_host.so"
    src = os.path.join(ROOT, "tests", "native", "isf_fft_host.cpp")
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-o", str(so), src], check=True)
    fn = ctypes.CDLL(str(so)).emulate_isf_fft
    fn.restype = ctypes.c_int

    def run(re, im, pairs, bin_off, nlags):
        nchan, nk, T = re.shape
        z = np.ascontiguousarray(np.stack([re, im], axis=-1), dtype=np.float64)
        pr = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        bo = np.ascontiguousarray(bin_off, dtype=np.int64)
        out = np.empty((len(pr), len(bo) - 1, nlags))
        fn(z.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), ctypes.c_int(nchan), ctypes.c_longlong(nk), ctypes.c_longlong(T),
           pr.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), ctypes.c_int(len(pr)), bo.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)),
           ctypes.c_int(len(bo) - 1), ctypes.c_longlong(nlags), out.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
        return out
    return run


def contract_error(got, want):
    """worst |got - want| over max_tau |want| per (pair, bin); a (pair, bin) whose direct sum is zero must be zero."""
    worst = 0.0
    for q in range(want.shape[0]):
        for b in range(want.shape[1]):
            scale = float(np.abs(want[q, b]).max())
            if scale == 0.0:
                assert not np.any(got[q, b]), (q, b)
                continue
            worst = max(worst, float(np.abs(got[q, b] - want[q, b]).max()) / scale)
    return worst


def _series(rng, nchan, nk, T):
    """complex series with a nonzero mean (a Bragg-like constant part) plus a slowly varying and a noisy part"""
    t = np.arange(T)
    base = rng.normal(0, 3, (nchan, nk, 1)) + 1j * rng.normal(0, 3, (nchan, nk, 1))
    wave = np.exp(1j * rng.uniform(0, 0.3, (nchan, nk, 1)) * t)
    z = base + wave + 0.5 * (rng.normal(0, 1, (nchan, nk, T)) + 1j * rng.normal(0, 1, (nchan, nk, T)))
    return z.real.copy(), z.imag.copy()


PAIRS = [(3, 3), (0, 1), (2, 2), (1, 0), (0, 2)]              # self and cross pairs, one swapped, an odd count


@pytest.mark.parametrize("p", [4, 7, 9])
@pytest.mark.parametrize("which", ["one", "half", "all"])
def test_isf_fft_bodies_match_direct_sum(emu, p, which):
    """T around 2^p - nlags (the smallest transform that holds the lags, and one step past it), nlags in {1, T/2, T},
    self and cross pairs, an odd number of pairs, bins of 0, 1 and several k-vectors: within 1e-10 of max_tau of the
    long-double direct sum per (pair, bin); an empty bin is exactly zero."""
    rng = np.random.default_rng(100 * p + len(which))
    bin_off = np.array([0, 3, 3, 4, 9])
    for T0 in ((1 << p) // 2, (1 << p) // 2 + 1, (1 << p) - 1):
        T = max(T0, 2)
        nlags = {"one": 1, "half": max(1, T // 2), "all": T}[which]
        re, im = _series(rng, 4, int(bin_off[-1]), T)
        want = IO.direct_corr(re, im, PAIRS, bin_off, nlags)
        got = emu(re, im, PAIRS, bin_off, nlags)
        assert not np.any(got[:, 1]), T
        assert contract_error(got, want.astype(np.float64)) < CONTRACT, (T, nlags)


def test_isf_fft_bodies_symmetric_in_the_pair(emu):
    """(a, b) and (b, a) give the same bits; the cross correlation is not the unsymmetrised one."""
    rng = np.random.default_rng(5)
    re, im = _series(rng, 2, 5, 300)
    bo = [0, 2, 5]
    a = emu(re, im, [(0, 1), (1, 1), (0, 0)], bo, 150)
    b = emu(re, im, [(1, 0), (1, 1), (0, 0)], bo, 150)
    assert np.array_equal(a, b)
    z = re + 1j * im
    one_sided = np.array([[np.mean((z[0, k, tau:] * np.conj(z[1, k, :300 - tau])).real) for tau in range(150)] for k in range(5)])
    assert np.abs(a[0, 0] - one_sided[:2].sum(axis=0)).max() > 1e-3 * np.abs(a[0, 0]).max()


def test_oracle_matches_rigid_translation_closed_form():
    """Positions r_j(t) = r_j(0) + v t in a triclinic cell: the oracle's rho series and direct sum give
    C_ab(k, tau) = Re(rho_a(k,0) rho_b(k,0)*) cos(k.v tau) for every pair, the total included."""
    rng = np.random.default_rng(6)
    cell = (17.0, 15.0, 16.0, 2.0, -1.5, 1.0)
    H = SO.cell_matrix(cell)
    n, T, L = 60, 24, 12
    pos0 = rng.uniform(0, 1, (n, 3)) @ H.T
    cls = rng.integers(0, 3, n)
    v = np.array([0.37, -0.21, 0.12])
    miller, bin_off, _ = SO.kset_brute(cell, 1.6, 0.2)
    frames = [pos0 + v * t for t in range(T)]
    re, im = IO.series(cell, frames, cls, 3, miller)
    re = np.concatenate([re, re.sum(axis=0, keepdims=True)])
    im = np.concatenate([im, im.sum(axis=0, keepdims=True)])
    pairs = [(3, 3), (0, 1), (2, 2), (1, 2)]
    got = IO.direct_corr(re, im, pairs, bin_off, L).astype(np.float64)
    want = IO.rigid_translation(cell, pos0, cls, 3, miller, v, pairs, bin_off, L)
    scale = np.abs(want).max(axis=2, keepdims=True) + 1e-300
    assert np.all(np.abs(got - want) <= 1e-9 * scale + 1e-9)
    assert np.abs(want[:, :, 1:] - want[:, :, :1]).max() > 1e-2 * np.abs(want).max()     # the cosines do turn


@pytest.mark.parametrize("w", [1, 2, 3, 4, 7])
def test_shard_bins_contiguous_covering_balanced(w):
    rng = np.random.default_rng(w)
    for _ in range(20):
        counts = rng.integers(0, 40, rng.integers(1, 30))
        counts[rng.random(len(counts)) < 0.2] = 0
        bo = np.concatenate(([0], np.cumsum(counts)))
        nk = int(bo[-1])
        cuts = [shard_bins(bo, r, w) for r in range(w)]
        assert cuts[0][0] == 0 and cuts[-1][1] == len(counts)
        assert all(cuts[r][1] == cuts[r + 1][0] for r in range(w - 1))
        assert all(lo <= hi for lo, hi in cuts)
        for lo, hi in cuts:
            assert bo[hi] - bo[lo] <= nk / w + counts.max()
        assert cuts == [shard_bins(bo.copy(), r, w) for r in range(w)]
        assert cuts == [shard_bins(list(bo), r, w) for r in range(w)]


def test_lag_times_and_even_spacing():
    t = lag_times([100, 150, 200, 250], 3, 2.0, "real", "'x'")
    assert np.array_equal(t, np.arange(3) * (50.0 * 2.0 * K.TIME_CONVERSION["real"]))
    with pytest.raises(ValueError, match="intermediate scattering function needs evenly spaced frames"):
        lag_times([0, 10, 30], 2, 1, "real", "'x'")
    with pytest.raises(ValueError, match="intermediate scattering function needs evenly spaced frames"):
        lag_times([0, 10, 10], 2, 1, "real", "'x'")
    with pytest.raises(ValueError, match="no dump frames found for 'x'"):
        lag_times([], 1, 1, "real", "'x'")


def test_conductivity_keeps_its_even_spacing_message(tmp_path):
    from mdproptools_b200.dynamical.conductivity import Conductivity
    c = Conductivity("dump.*", [1], [1], 1000.0, working_dir=str(tmp_path))
    with pytest.raises(ValueError, match="the Einstein and Nernst-Einstein conductivity need evenly spaced frames"):
        c._set_even_time([0, 1, 3])
    c._set_even_time([0, 5, 10])
    assert c.time == [0.0, 5 * K.TIME_CONVERSION["real"], 10 * K.TIME_CONVERSION["real"]]


def test_table_layout_and_empty_bins():
    rng = np.random.default_rng(9)
    bo = np.array([0, 0, 4, 4, 9])
    L = 3
    sums = rng.normal(size=(3, 4, L))
    rel = np.array([[1, 2], [2, 2]])
    t = np.arange(L) * 1e-12
    df = isf_table(sums, bo, 50, {1: 20, 2: 30}, rel, 0.5, t)
    assert list(df.columns) == ["k ($\\AA^{-1}$)", "t (s)", "F(k,t)", "F_1-2", "F_2-2", "n_k"]
    a = df.to_numpy().reshape(4, L, -1)
    assert np.array_equal(a[:, :, 0], np.repeat([[0.25], [0.75], [1.25], [1.75]], L, axis=1))
    assert np.array_equal(a[:, :, 1], np.tile(t, (4, 1)))
    assert np.all(np.isnan(a[[0, 2], :, 2:5])) and not np.any(np.isnan(a[[1, 3], :, 2:5]))
    assert np.allclose(a[3, :, 2], sums[0, 3] / (5 * 50)) and np.allclose(a[1, :, 3], sums[1, 1] / (4 * np.sqrt(600.0)))
    assert np.allclose(a[1, :, 4], sums[2, 1] / (4 * 30.0))
