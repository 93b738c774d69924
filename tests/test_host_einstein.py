"""Host checks of the Einstein / Nernst-Einstein conductivity: the shared bodies of the FFT all-origins MSD (csrc/msd_fft.h,
run by tests/native/msd_fft_host.cpp) against the oracle's long-double direct sum, and the oracle's numpy restatements
of ``Conductivity.einstein`` / ``Conductivity.nernst`` against an independent brute force on a tiny trajectory."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
from tests import einstein_oracle as EO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONTRACT = 1e-10


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = tmp_path_factory.mktemp("msd_fft") / "msd_fft_host.so"
    src = os.path.join(ROOT, "tests", "native", "msd_fft_host.cpp")
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-o", str(so), src], check=True)
    lib = ctypes.CDLL(str(so))
    fn = lib.emulate_cross_msd
    fn.restype = ctypes.c_int
    dp = ctypes.POINTER(ctypes.c_double)

    def run(a, b, group_off, nlags, centre=True):
        a = np.ascontiguousarray(a, dtype=np.float64)
        bb = None if b is None else np.ascontiguousarray(b, dtype=np.float64)
        go = np.ascontiguousarray(group_off, dtype=np.int64)
        out = np.empty((len(go) - 1, nlags))
        fn(a.ctypes.data_as(dp), None if bb is None else bb.ctypes.data_as(dp), ctypes.c_longlong(a.shape[1]),
           go.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)), ctypes.c_int(len(go) - 1), ctypes.c_longlong(nlags),
           ctypes.c_int(1 if centre else 0), out.ctypes.data_as(dp))
        return out
    return run


def _series(rng, C, T, step=0.1):
    """diffusive channels (random walks) plus noise"""
    return np.cumsum(rng.normal(0, step, (C, T)), axis=1) + rng.normal(0, 1, (C, T))


def contract_error(got, want, floor=0.0):
    """worst |got - want| over max_tau |want| per group.  A group whose direct sum is zero at every lag (an empty group,
    or nlags = 1) is measured against ``floor`` instead, the summed variance of its inputs; an empty group must come out
    exactly zero (floor 0)."""
    worst = 0.0
    for g in range(want.shape[0]):
        scale = np.abs(want[g]).max()
        if scale == 0.0:
            assert np.abs(got[g]).max() <= CONTRACT * floor, g
            continue
        worst = max(worst, np.abs(got[g] - want[g]).max() / scale)
    return worst


GROUPINGS = {                   # channel counts per group: odd counts, an empty group first, middle and last
    "one": [1],
    "odd": [3, 5, 1],
    "empty": [0, 2, 0, 3, 0],
    "pairs": [2, 4],
}


@pytest.mark.parametrize("T", [1, 2, 3, 7, 2047, 2048, 2049, 4097])
@pytest.mark.parametrize("case", ["self", "cross"])
def test_msd_fft_bodies_match_direct_sum(emu, T, case):
    """Self and cross cases, nlags < T and nlags = T, odd channel counts (the last channel of a self group is paired with
    zero), empty groups: within 1e-10 of max_tau |out[g]| of the long-double direct sum."""
    rng = np.random.default_rng(1000 + T)
    for name, counts in GROUPINGS.items():
        off = np.concatenate(([0], np.cumsum(counts))).astype(np.int64)
        C = int(off[-1])
        a = _series(rng, C, T)
        b = None if case == "self" else _series(rng, C, T) + 3.0
        for nlags in sorted({T, max(1, T // 3)}):
            want = EO.cross_msd_direct(a, b, off, nlags)
            got = emu(a, b, off, nlags)
            for g in range(len(counts)):
                if counts[g] == 0:
                    assert not np.any(got[g]), (name, nlags, g)
            floor = np.var(a, axis=1).sum() + (0.0 if b is None else np.var(b, axis=1).sum())
            assert contract_error(got, want, floor) < CONTRACT, (name, nlags)


def test_msd_fft_bodies_large_offset(emu):
    """A series offset by 1e8 times its step size (unwrapped coordinates far from the origin): the mean centring keeps it
    within the contract; without it the same arithmetic is far outside."""
    rng = np.random.default_rng(7)
    T, step = 4097, 0.05
    a = np.cumsum(rng.normal(0, step, (3, T)), axis=1) + 1e8 * step
    b = a[::-1].copy() - 2e8 * step
    off = np.array([0, 3])
    for bb in (None, b):
        want = EO.cross_msd_direct(a, bb, off, T)
        assert contract_error(emu(a, bb, off, T), want) < CONTRACT
        assert contract_error(emu(a, bb, off, T, centre=False), want) > 1e3 * CONTRACT


def test_msd_fft_bodies_single_channel_equals_msd_definition(emu):
    """A cross MSD of (x, x) is the self MSD of x, and a group of the three axes is the MSD of the oracle's all-origins
    kernel restatement (orc_msd_all_origins, [T, 3, N] layout)."""
    rng = np.random.default_rng(8)
    T, N = 300, 4
    traj = np.cumsum(rng.normal(0, 0.3, (T, 3, N)), axis=0)
    chans = traj.transpose(2, 1, 0).reshape(-1, T)              # [N * 3, T]
    got = emu(chans, None, [0, 3 * N], T)[0] / N
    want = O.msd_all_origins(traj, T)[:, 3]
    assert np.abs(got - want).max() < CONTRACT * np.abs(want).max()
    assert np.array_equal(emu(chans, None, [0, 3 * N], T), emu(chans, None, [0, 3 * N], T))
    cross = emu(chans, chans, [0, 3 * N], T)
    assert np.abs(cross - emu(chans, None, [0, 3 * N], T)).max() < CONTRACT * np.abs(cross).max()


# ---------------------------------------------------------------------------------------------------------------------
# oracle restatements of einstein() / nernst() against a brute force
# ---------------------------------------------------------------------------------------------------------------------
def write_dump(path, steps, pos, image, q, mass, types, L, columns="xu"):
    """One LAMMPS dump file with every frame: pos [T, 3, N] unwrapped (with ``columns="image"``: wrapped x y z plus
    ix iy iz = image [T, 3, N]), full-precision numbers."""
    def r(v):
        return repr(float(v))
    with open(path, "w") as f:
        for k, s in enumerate(steps):
            f.write(f"ITEM: TIMESTEP\n{s}\nITEM: NUMBER OF ATOMS\n{pos.shape[2]}\nITEM: BOX BOUNDS pp pp pp\n")
            for _ in range(3):
                f.write(f"0.0 {r(L)}\n")
            if columns == "xu":
                f.write("ITEM: ATOMS id type mass q xu yu zu\n")
                for i in range(pos.shape[2]):
                    f.write(f"{i + 1} {types[i]} {r(mass[i])} {r(q[i])} {r(pos[k, 0, i])} {r(pos[k, 1, i])} {r(pos[k, 2, i])}\n")
            else:
                f.write("ITEM: ATOMS id type mass q x y z ix iy iz\n")
                for i in range(pos.shape[2]):
                    w = pos[k, :, i] - image[k, :, i] * L
                    f.write(f"{i + 1} {types[i]} {r(mass[i])} {r(q[i])} {r(w[0])} {r(w[1])} {r(w[2])} "
                            f"{int(image[k, 0, i])} {int(image[k, 1, i])} {int(image[k, 2, i])}\n")


def tiny_system(rng, T=14):
    num_mols, num_atoms = [2, 3], [2, 1]
    N = 2 * 2 + 3
    types = np.array([1, 2, 1, 2, 3, 3, 3])
    mass = np.array([12.0, 1.0, 12.0, 1.0, 23.0, 23.0, 23.0])
    q = np.array([0.7, -0.2, 0.7, -0.2, -0.4, -0.2, -0.2])
    pos = np.cumsum(rng.normal(0, 0.4, (T, 3, N)), axis=0) + rng.uniform(0, 10, (1, 3, N))
    steps = np.arange(T) * 50
    return num_mols, num_atoms, types, mass, q, pos, steps


def brute_force(num_mols, num_atoms, mass, q, pos, dt, kb, temp, vol, dconv, qconv, max_lag):
    """sigma_E and sigma_NE by explicit loops (lstsq fit with intercept over the default window)."""
    T = pos.shape[0]
    mols, a = [], 0
    for g, (nm, na) in enumerate(zip(num_mols, num_atoms)):
        for _ in range(nm):
            mols.append((g, list(range(a, a + na))))
            a += na
    com = np.zeros((T, len(mols), 3))
    qm = np.zeros(len(mols))
    for m, (g, idx) in enumerate(mols):
        w = mass[idx]
        for t in range(T):
            com[t, m] = (pos[t][:, idx] * w).sum(axis=1) / w.sum() * dconv
        qm[m] = q[idx].sum() * qconv
    G = len(num_mols)
    M = np.zeros((T, G + 1, 3))
    for m, (g, _) in enumerate(mols):
        M[:, g] += qm[m] * com[:, m]
    M[:, G] = M[:, :G].sum(axis=1)
    lags = np.arange(max_lag)
    i0 = max(1, max_lag // 10)
    sel = lags[i0:max_lag]
    X = np.stack([sel * dt, np.ones(len(sel))], axis=1)

    def slope(y):
        return np.linalg.lstsq(X, y[i0:max_lag], rcond=None)[0][0]
    sig_e = []
    for i in range(G + 1):
        y = np.array([np.mean([np.dot(M[t + l, i] - M[t, i], M[t + l, G] - M[t, G]) for t in range(T - l)]) for l in lags])
        sig_e.append(slope(y) / (6 * kb * temp * vol))
    sig_ne = []
    for g in range(G):
        ms = [m for m, (gg, _) in enumerate(mols) if gg == g]
        y = np.array([np.mean([np.sum((com[t + l, m] - com[t, m]) ** 2) for t in range(T - l) for m in ms]) for l in lags])
        sig_ne.append(slope(y) / 6 * np.sum(qm[ms] ** 2) / (vol * kb * temp))
    return np.array(sig_e), np.append(sig_ne, sum(sig_ne))


@pytest.mark.parametrize("columns", ["xu", "image"])
def test_oracle_einstein_and_nernst_restatements_match_bruteforce(tmp_path, columns):
    from mdproptools_b200.common import constants as K
    rng = np.random.default_rng(21)
    num_mols, num_atoms, types, mass, q, pos, steps = tiny_system(rng)
    L = 10.0
    image = np.floor(pos / L)
    write_dump(tmp_path / "dump.tiny.lammpstrj", steps, pos, image, q, mass, types, L, columns)
    if columns == "image":
        pos = (pos - image * L) + image * L                     # the unwrapping arithmetic the restatement does
    dt = 50 * K.TIME_CONVERSION["real"]
    vol = (L * K.DISTANCE_CONVERSION["real"]) ** 3
    args = (str(tmp_path / "dump.tiny.lammpstrj"), num_mols, num_atoms, vol, 300.0, dt, None, K.DISTANCE_CONVERSION["real"],
            K.CHARGE_CONVERSION["real"], K.BOLTZMANN)
    sig_e, msd = EO.einstein_conductivity(*args, unwrap=columns)
    sig_ne, D = EO.nernst_einstein(*args, unwrap=columns)
    assert msd.shape == (3, len(steps) // 2) and D.shape == (2,)
    want_e, want_ne = brute_force(num_mols, num_atoms, mass, q, pos, dt, K.BOLTZMANN, 300.0, vol,
                                  K.DISTANCE_CONVERSION["real"], K.CHARGE_CONVERSION["real"], len(steps) // 2)
    np.testing.assert_allclose(sig_e, want_e, rtol=1e-9, atol=1e-12 * np.abs(want_e).max())
    np.testing.assert_allclose(sig_ne, want_ne, rtol=1e-9)
