"""Host checks of the velocity autocorrelation route: the shared bodies of the grouped FFT autocorrelation (csrc/msd_fft.h,
run by tests/native/acf_fft_host.cpp) against the long-double direct sum, the oracle's restatements against a brute force
on a tiny trajectory, and the VDOS transform (``vdos_transform``, on CPU tensors) against its identities and the oracle's
explicit cosine sum."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from tests import vacf_oracle as VO
from tests.test_host_einstein import GROUPINGS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONTRACT = 1e-10


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = tmp_path_factory.mktemp("acf_fft") / "acf_fft_host.so"
    src = os.path.join(ROOT, "tests", "native", "acf_fft_host.cpp")
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-o", str(so), src], check=True)
    fn = ctypes.CDLL(str(so)).emulate_group_acf
    fn.restype = ctypes.c_int
    dp = ctypes.POINTER(ctypes.c_double)

    def run(a, group_off, nlags):
        a = np.ascontiguousarray(a, dtype=np.float64)
        go = np.ascontiguousarray(group_off, dtype=np.int64)
        out = np.empty((len(go) - 1, nlags))
        fn(a.ctypes.data_as(dp), ctypes.c_longlong(a.shape[1]), go.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)),
           ctypes.c_int(len(go) - 1), ctypes.c_longlong(nlags), out.ctypes.data_as(dp))
        return out
    return run


def velocity_series(rng, C, T, offset=1e3):
    """Ornstein-Uhlenbeck channels (memory of 20 steps) plus a constant offset, which a centred correlation would lose"""
    phi = np.exp(-1 / 20)
    x = np.empty((C, T))
    x[:, 0] = rng.normal(0, 1, C)
    noise = rng.normal(0, np.sqrt(1 - phi * phi), (C, T))
    for t in range(1, T):
        x[:, t] = phi * x[:, t - 1] + noise[:, t]
    return x + offset


def acf_error(got, want, counts):
    """worst |got - want| over max_tau |want[g]| (out[g][0] up to the noise of the last lags' few origins); empty groups
    must be exactly zero"""
    worst = 0.0
    for g, n in enumerate(counts):
        if n == 0:
            assert not np.any(got[g]), g
            continue
        worst = max(worst, np.abs(got[g] - want[g]).max() / np.abs(want[g]).max())
    return worst


@pytest.mark.parametrize("T", [1, 2, 3, 7, 2047, 2048, 2049, 4097])
def test_acf_fft_bodies_match_direct_sum(emu, T):
    """nlags = T and T // 3, odd channel counts (the last channel of a group is paired with zero), empty groups, series
    offset by 10^3: within 1e-10 of max_tau |out[g]| of the long-double direct sum; empty groups exactly zero."""
    rng = np.random.default_rng(2000 + T)
    for name, counts in GROUPINGS.items():
        off = np.concatenate(([0], np.cumsum(counts))).astype(np.int64)
        a = velocity_series(rng, int(off[-1]), T)
        for nlags in sorted({T, max(1, T // 3)}):
            want = VO.acf_direct(a, off, nlags)
            got = emu(a, off, nlags)
            err = acf_error(got, want, counts)
            assert err < CONTRACT, (name, nlags, err)


def test_acf_fft_bodies_are_deterministic_and_uncentred(emu):
    """the same bits twice; a constant series gives its square at every lag (no centring)"""
    rng = np.random.default_rng(5)
    a = velocity_series(rng, 5, 999)
    off = [0, 2, 5]
    assert np.array_equal(emu(a, off, 500), emu(a, off, 500))
    c = np.full((3, 400), 2.5)
    got = emu(c, [0, 3], 400)[0]
    assert np.abs(got - 3 * 6.25).max() < 1e-12 * 18.75


# ---------------------------------------------------------------------------------------------------------------------
# oracle restatements against a brute force
# ---------------------------------------------------------------------------------------------------------------------
def write_vel_dump(path, steps, vel, types, mass, pos=None, L=20.0):
    """One LAMMPS dump of every frame: velocities vel [T, 3, N] (and, when given, unwrapped positions pos [T, 3, N]),
    full-precision numbers, rows in reverse id order (the readers sort by id)."""
    def r(v):
        return repr(float(v))
    N = vel.shape[2]
    with open(path, "w") as f:
        for k, s in enumerate(steps):
            f.write(f"ITEM: TIMESTEP\n{int(s)}\nITEM: NUMBER OF ATOMS\n{N}\nITEM: BOX BOUNDS pp pp pp\n")
            for _ in range(3):
                f.write(f"0.0 {r(L)}\n")
            f.write("ITEM: ATOMS id type mass vx vy vz" + (" xu yu zu\n" if pos is not None else "\n"))
            for i in reversed(range(N)):
                row = f"{i + 1} {int(types[k][i] if np.ndim(types) == 2 else types[i])} {r(mass[i])} " + \
                      " ".join(r(v) for v in vel[k, :, i])
                if pos is not None:
                    row += " " + " ".join(r(v) for v in pos[k, :, i])
                f.write(row + "\n")


def tiny_velocities(rng, T=12):
    num_mols, num_atoms = [2, 3], [2, 1]
    types = np.array([1, 3, 1, 3, 2, 2, 2])
    mass = np.array([12.0, 1.0, 12.0, 1.0, 23.0, 23.0, 23.0])
    vel = rng.normal(0, 0.01, (T, 3, 7)) + 0.003
    return num_mols, num_atoms, types, mass, vel, np.arange(T) * 20


def test_oracle_vacf_matches_bruteforce(tmp_path):
    from mdproptools_b200.common import constants as K
    rng = np.random.default_rng(41)
    num_mols, num_atoms, types, mass, vel, steps = tiny_velocities(rng)
    write_vel_dump(tmp_path / "dump.v.lammpstrj", steps, vel, types, mass)
    vc, dts = K.VELOCITY_CONVERSION["real"], K.TIME_CONVERSION["real"]
    T, L = len(steps), 5
    v = vel * vc

    def corr(series, lag):                          # series [T, 3, n] -> mean over origins and members, per axis
        return np.array([np.mean([series[t + lag, k] * series[t, k] for t in range(T - lag)], axis=0).sum()
                         for k in range(3)])
    got = VO.get_vacf(str(tmp_path / "dump.v.lammpstrj"), dts, vc, max_lag=L)
    assert list(got) == ["Time (s)"] + [f"{n}{t}" for t in (1, 2, 3) for n in ("vxvx", "vyvy", "vzvz", "vacf")] + ["vacf"]
    np.testing.assert_allclose(got["Time (s)"], np.arange(L) * 20 * dts, rtol=1e-15)
    for t in (1, 2, 3):
        idx = np.nonzero(types == t)[0]
        want = np.array([corr(v[:, :, idx], l) for l in range(L)]) / len(idx)          # [L, 3]
        for k, n in enumerate(("vxvx", "vyvy", "vzvz")):
            np.testing.assert_allclose(got[f"{n}{t}"], want[:, k], rtol=1e-13)
        np.testing.assert_allclose(got[f"vacf{t}"], want.sum(axis=1), rtol=1e-13)
    allv = np.array([corr(v, l) for l in range(L)]).sum(axis=1) / 7
    np.testing.assert_allclose(got["vacf"], allv, rtol=1e-13)
    # centre-of-mass velocities by explicit loops
    com = np.zeros((T, 3, 5))
    m, a = 0, 0
    for nm, na in zip(num_mols, num_atoms):
        for _ in range(nm):
            w = mass[a:a + na]
            com[:, :, m] = (v[:, :, a:a + na] * w).sum(axis=2) / w.sum()
            m, a = m + 1, a + na
    got = VO.get_vacf(str(tmp_path / "dump.v.lammpstrj"), dts, vc, max_lag=L, vacf_type="com", num_mols=num_mols,
                      num_atoms_per_mol=num_atoms, mass=None)
    assert list(got) == ["Time (s)"] + [f"{n}{t}" for t in (1, 2) for n in ("vxvx", "vyvy", "vzvz", "vacf")]
    for g, sl in ((1, slice(0, 2)), (2, slice(2, 5))):
        want = np.array([corr(com[:, :, sl], l) for l in range(L)]) / (sl.stop - sl.start)
        np.testing.assert_allclose(got[f"vacf{g}"], want.sum(axis=1), rtol=1e-13)
    # Green-Kubo: the running trapezoid and the window statistics
    t = np.arange(L) * 2.0
    c = np.array([3.0, 1.0, -0.5, 0.25, 0.0])
    D, std, run = VO.green_kubo(t, c, dimension=3)
    want_run = [0.0, 4.0, 4.5, 4.25, 4.5]
    np.testing.assert_allclose(run, want_run, rtol=1e-15)
    assert D == pytest.approx(np.mean(want_run[1:]) / 3, rel=1e-15) and std == pytest.approx(np.std(want_run[1:]) / 3, rel=1e-15)


# ---------------------------------------------------------------------------------------------------------------------
# the VDOS transform
# ---------------------------------------------------------------------------------------------------------------------
def _vdos(c, dt, window):
    from mdproptools_b200.dynamical.diffusion import vdos_transform
    nu, S = vdos_transform(torch.from_numpy(np.asarray(c, dtype=np.float64)), dt, window)
    return nu.numpy(), S.numpy()


@pytest.mark.parametrize("window", ["hann", "none"])
@pytest.mark.parametrize("L", [2, 3, 50, 513])
def test_vdos_identities_and_cosine_sum(window, L):
    """unit trapezoid area over nu; S(0) C_0 / 4 = trapezoid integral of w C; equal to the oracle's explicit cosine sum"""
    rng = np.random.default_rng(L)
    dt = 2e-15
    lag = np.arange(L)
    c = np.exp(-lag / 7.0) * np.cos(0.3 * lag) + 0.05 * rng.normal(size=L)
    c[0] = 1.7
    nu, S = _vdos(c, dt, window)
    assert abs(np.trapezoid(S, nu) - 1.0) < 1e-12
    w = 0.5 * (1 + np.cos(np.pi * lag / (L - 1))) if window == "hann" else np.ones(L)
    wc = w * c
    assert abs(S[0] * c[0] / 4 - np.trapezoid(wc, dx=dt)) < 1e-12 * np.abs(wc).sum() * dt
    onu, oS = VO.vdos(c, dt, window)
    np.testing.assert_allclose(nu, onu, rtol=1e-15)
    assert np.abs(S - oS).max() < 1e-12 * np.abs(oS).max()


def test_vdos_of_cosine_peaks_at_its_frequency():
    L, dt, k0 = 401, 1e-15, 37
    nu0 = k0 / (2 * (L - 1) * dt)
    c = np.cos(2 * np.pi * nu0 * np.arange(L) * dt)
    for window in ("hann", "none"):
        nu, S = _vdos(c, dt, window)
        assert np.argmax(S) == k0 and nu[k0] == pytest.approx(nu0, rel=1e-14)


def test_vdos_rejects_unknown_window():
    with pytest.raises(ValueError):
        _vdos(np.ones(4), 1.0, "hamming")
