"""Host checks of the reorientation route: the kernel body (csrc/orient.h, run by tests/native/orient_host.cpp) against the
oracle's vectors and channels on triclinic cells, the channel identities P1 = u.u' and P2 = 1.5 q.q', the oracle's direct
Legendre sums against a brute force, the t_end rule, and the checks of the vector definitions (raised without a GPU)."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from mdproptools_b200.dynamical import reorientation as R
from tests import reorient_oracle as RO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KIND = {"bond": 0, "bisector": 1, "normal": 2}


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = tmp_path_factory.mktemp("orient") / "orient_host.so"
    src = os.path.join(ROOT, "tests", "native", "orient_host.cpp")
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-o", str(so), src], check=True)
    fn = ctypes.CDLL(str(so)).emulate_orient_series
    vp, ll = ctypes.c_void_p, ctypes.c_longlong

    def run(xyz, cells, kind, atoms, out=None, frame0=0):
        """xyz [F, 3, n], cells [F, 6], atoms [nvec, 3] -> out [8, nvec, T] (a new [8, nvec, F] series when None)"""
        xyz = np.ascontiguousarray(xyz, dtype=np.float64)
        cells = np.ascontiguousarray(cells, dtype=np.float64)
        atoms = np.ascontiguousarray(atoms, dtype=np.int32).reshape(-1, 3)
        F, _, n = xyz.shape
        if out is None:
            out = np.zeros((8, len(atoms), F))
        fn(ctypes.c_int(F), ll(n), vp(xyz.ctypes.data), vp(cells.ctypes.data), ctypes.c_int(KIND[kind]), ll(len(atoms)),
           vp(atoms.ctypes.data), vp(out.ctypes.data), ll(out.shape[2]), ll(frame0))
        return out
    return run


def random_cell(rng):
    """(lx, ly, lz, xy, xz, yz) of a restricted triclinic cell with tilts up to 0.4 of the length they shear"""
    lx, ly, lz = rng.uniform(18, 30, 3)
    return np.array([lx, ly, lz, rng.uniform(-0.4, 0.4) * lx, rng.uniform(-0.4, 0.4) * lx, rng.uniform(-0.4, 0.4) * ly])


def cell_matrix(cell):
    lx, ly, lz, xy, xz, yz = cell
    return np.array([[lx, xy, xz], [0.0, ly, yz], [0.0, 0.0, lz]])          # columns a, b, c


def wrap(pos, cell):
    """positions [..., 3] folded into the cell (fractional coordinates in [0, 1))"""
    H = cell_matrix(cell)
    s = np.linalg.solve(H, pos.reshape(-1, 3).T)
    return (H @ (s - np.floor(s))).T.reshape(pos.shape)


def three_site_molecules(rng, cell, M):
    """[M, 3, 3] (molecule, site, xyz) of bent three-site molecules (bonds of 1-1.5 A at 90-120 degrees, so that no vector
    kind is ill-conditioned), half of them centred within 0.5 A of a cell face (every face), the rest anywhere; not
    wrapped"""
    H = cell_matrix(cell)
    s = rng.uniform(0, 1, (M, 3))
    for m in range(M // 2):
        s[m, m % 3] = (m // 3) % 2 + rng.uniform(-0.5, 0.5) / cell[m % 3]
    centre = s @ H.T
    e1 = rng.normal(size=(M, 3))
    e1 /= np.linalg.norm(e1, axis=1)[:, None]
    e2 = np.cross(e1, rng.normal(size=(M, 3)))
    e2 /= np.linalg.norm(e2, axis=1)[:, None]
    ang = np.radians(rng.uniform(90, 120, M))[:, None]
    d1 = e1 * rng.uniform(1.0, 1.5, (M, 1))
    d2 = (np.cos(ang) * e1 + np.sin(ang) * e2) * rng.uniform(1.0, 1.5, (M, 1))
    return np.stack([centre, centre + d1, centre + d2], axis=1)


def write_pos_dump(path, steps, pos, cells, cols=("x", "y", "z"), mode="w"):
    """A triclinic LAMMPS dump of every frame: positions pos [T, 3, N], cells [T, 6] or [6], full-precision numbers, rows in
    reverse id order (the readers sort by id)."""
    def r(v):
        return repr(float(v))
    cells = np.broadcast_to(np.asarray(cells, dtype=np.float64), (len(steps), 6))
    N = pos.shape[2]
    with open(path, mode) as f:
        for k, s in enumerate(steps):
            lx, ly, lz, xy, xz, yz = cells[k]
            xs = (0.0, xy, xz, xy + xz)
            f.write(f"ITEM: TIMESTEP\n{int(s)}\nITEM: NUMBER OF ATOMS\n{N}\nITEM: BOX BOUNDS xy xz yz pp pp pp\n")
            f.write(f"{r(min(xs))} {r(lx + max(xs))} {r(xy)}\n{r(min(0.0, yz))} {r(ly + max(0.0, yz))} {r(xz)}\n"
                    f"0.0 {r(lz)} {r(yz)}\n")
            f.write("ITEM: ATOMS id type " + " ".join(cols) + "\n")
            for i in reversed(range(N)):
                f.write(f"{i + 1} 1 " + " ".join(r(v) for v in pos[k, :, i]) + "\n")


# ---------------------------------------------------------------------------------------------------------------------
# the kernel body against the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["bond", "bisector", "normal"])
@pytest.mark.parametrize("placement", ["wrapped", "unwrapped", "scattered"])
def test_orient_body_matches_oracle(emu, kind, placement):
    """Random triclinic cells, three-site molecules straddling every face: u and the 8 channels against the oracle's
    long-double values.  Wrapped positions, and unwrapped ones (whole molecules moved by a lattice vector of up to 3 cells),
    within 1e-14.  Scattered: every atom moved by its own lattice vector of up to 3 cells, so that r_j - r_i is tens of
    Angstrom before the image shift; the positions then carry the rounding of their magnitude into u, and the bound is
    16 ulp of the largest coordinate over the shortest w (0.5 A here)."""
    rng = np.random.default_rng(100 + 10 * KIND[kind] + (placement == "unwrapped"))
    F, M = 5, 120
    cells = np.stack([random_cell(rng) for _ in range(F)])
    xyz = np.empty((F, 3, 3 * M))
    for f in range(F):
        mol = three_site_molecules(rng, cells[f], M).reshape(-1, 3)
        if placement == "wrapped":
            mol = wrap(mol, cells[f])
        elif placement == "unwrapped":
            mol = mol + np.repeat(rng.integers(-3, 4, (M, 3)), 3, axis=0) @ cell_matrix(cells[f]).T
        else:
            mol = mol + rng.integers(-3, 4, mol.shape) @ cell_matrix(cells[f]).T
        xyz[f] = mol.T
    rows = 3 * np.arange(M)[:, None] + np.array([0, 1, 2])[None, :]
    got = emu(xyz, cells, kind, rows)
    u = RO.unit_vectors(xyz, cells, rows if kind != "bond" else rows[:, :2], kind)        # [F, M, 3]
    want = np.asarray(RO.channels(u), dtype=np.float64).transpose(0, 2, 1)               # [8, M, F]
    tol = 1e-14 if placement != "scattered" else 16 * 2.0 ** -52 * np.abs(xyz).max() / 0.5
    assert np.abs(got - want).max() <= tol
    assert np.abs(got[:3] - np.asarray(u, dtype=np.float64).transpose(2, 1, 0)).max() <= tol


def test_orient_body_fills_only_its_columns(emu):
    """frames go to columns frame0 + f of a longer series; the other columns keep their values"""
    rng = np.random.default_rng(7)
    cell = random_cell(rng)
    xyz = wrap(three_site_molecules(rng, cell, 10).reshape(-1, 3), cell).T[None].repeat(4, axis=0)
    rows = 3 * np.arange(10)[:, None] + np.array([0, 1, 2])[None, :]
    out = np.full((8, 10, 11), -7.0)
    emu(xyz, np.tile(cell, (4, 1)), "normal", rows, out=out, frame0=5)
    assert np.all(out[:, :, :5] == -7.0) and np.all(out[:, :, 9:] == -7.0)
    assert np.array_equal(out[:, :, 5:9], emu(xyz, np.tile(cell, (4, 1)), "normal", rows))


def test_degenerate_vector_gives_nan(emu):
    """two coincident atoms: NaN channels (0/0), and only for that vector"""
    xyz = np.array([[[0.0, 0.0, 1.0, 2.0], [0.0, 0.0, 1.0, 0.0], [0.0, 0.0, 0.0, 3.0]]])
    out = emu(xyz, [[10.0, 10.0, 10.0, 0.0, 0.0, 0.0]], "bond", [[0, 1, 0], [2, 3, 2]])
    assert np.all(np.isnan(out[:, 0])) and np.all(np.isfinite(out[:, 1]))


def test_channel_identities(emu):
    """10^4 random pairs of directions: u.u' = P1 and 1.5 q.q' = P2(u.u'), to 1e-15, from the emulated channels"""
    rng = np.random.default_rng(8)
    P = 10_000
    d = rng.normal(size=(2, P, 3)) * rng.uniform(0.5, 3.0, (2, P, 1))
    xyz = np.zeros((2, 3, 2 * P))
    xyz[:, :, 1::2] = d.transpose(0, 2, 1)
    rows = 2 * np.arange(P)[:, None] + np.array([0, 1, 0])[None, :]
    ch = emu(xyz, np.tile([100.0, 100.0, 100.0, 0.0, 0.0, 0.0], (2, 1)), "bond", rows)     # [8, P, 2]
    u = d.astype(np.longdouble) / np.sqrt((d.astype(np.longdouble) ** 2).sum(axis=2))[:, :, None]
    x = (u[0] * u[1]).sum(axis=1)
    p2 = (1.5 * x * x - 0.5).astype(np.float64)
    assert np.abs((ch[:3, :, 0] * ch[:3, :, 1]).sum(axis=0) - x.astype(np.float64)).max() <= 1e-15
    assert np.abs(1.5 * (ch[3:, :, 0] * ch[3:, :, 1]).sum(axis=0) - p2).max() <= 1e-15
    assert np.abs(1.5 * (ch[3:, :, 0] ** 2).sum(axis=0) - 1.0).max() <= 4e-15                # C2(0) = 1, to a few ulp


# ---------------------------------------------------------------------------------------------------------------------
# the oracle against a brute force, and the t_end rule
# ---------------------------------------------------------------------------------------------------------------------
def test_oracle_legendre_sums_match_brute_force():
    rng = np.random.default_rng(9)
    T, M = 7, 3
    u = rng.normal(size=(T, M, 3))
    u /= np.linalg.norm(u, axis=2)[:, :, None]
    c1, c2 = RO.legendre_corr(u, 5)
    for tau in range(5):
        s1 = s2 = 0.0
        for m in range(M):
            for t in range(T - tau):
                x = sum(u[t, m, a] * u[t + tau, m, a] for a in range(3))
                s1 += x / (T - tau)
                s2 += (3 * x * x - 1) / 2 / (T - tau)
        assert math.isclose(c1[tau], s1 / M, rel_tol=0, abs_tol=1e-15)
        assert math.isclose(c2[tau], s2 / M, rel_tol=0, abs_tol=1e-15)
    assert c1[0] == pytest.approx(1.0, abs=1e-15) and c2[0] == pytest.approx(1.0, abs=1e-15)


def test_oracle_mic_is_the_nearest_image():
    """the oracle's fractional-form minimum image of short vectors moved by lattice vectors is the short vector"""
    rng = np.random.default_rng(10)
    for _ in range(20):
        cell = random_cell(rng)
        d = rng.normal(size=(50, 3))
        moved = d + rng.integers(-4, 5, (50, 3)) @ cell_matrix(cell).T
        assert np.abs(np.asarray(RO.mic(moved, cell), dtype=np.float64) - d).max() < 1e-12


@pytest.mark.parametrize("curve, end", [([1.0, 0.6, 0.2, -0.1, -0.3, 0.1], 3),      # first crossing
                                        ([1.0, 0.8, 0.6, 0.5, 0.45], 4),            # never reaches 0: last lag
                                        ([1.0, 0.0, 0.3, 0.2], 1),                  # exactly 0 at lag 1
                                        ([1.0, -0.2, 0.5], 1)])                     # below 0 at lag 1
def test_t_end_rule(curve, end):
    """library and oracle read the integral at the same lag; the oracle's tau is the trapezoid area up to it"""
    assert R.t_end_index(curve) == end == RO.t_end_index(curve)
    t = np.arange(len(curve)) * 0.5
    tau, t_end = RO.correlation_time(t, curve)
    assert t_end == t[end]
    assert tau == pytest.approx(np.trapezoid(curve[:end + 1], t[:end + 1]), abs=1e-15)


# ---------------------------------------------------------------------------------------------------------------------
# vector definitions
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("spec, match", [((1, "dipole", (1, 2)), "unknown kind"),
                                         ((1, "bond", (1, 2, 3)), "takes 2 atoms"),
                                         ((1, "normal", (1, 2)), "takes 3 atoms"),
                                         ((1, "bond", (1, 4)), "outside 1..3"),
                                         ((1, "bisector", (0, 1, 2)), "outside 1..3"),
                                         ((1, "bisector", (1, 2, 1)), "repeated"),
                                         ((3, "bond", (1, 2)), "molecule type 3"),
                                         ((0, "bond", (1, 2)), "molecule type 0"),
                                         ((1, "bond"), "expected")])
def test_vector_definitions_are_checked_before_reading(spec, match):
    """ValueError before any frame is parsed (the dump named here does not exist, and no device is needed)"""
    with pytest.raises(ValueError, match=match):
        R.calc_reorientation("/nonexistent/dump.*.lammpstrj", {"v": spec}, [4, 2], [3, 5])


def test_max_lag_checked_before_reading():
    with pytest.raises(ValueError, match="max_lag"):
        R.calc_reorientation("/nonexistent/dump.*.lammpstrj", {"v": (1, "bond", (1, 2))}, [4, 2], [3, 5], max_lag=0)


def test_vector_rows_layout():
    """rows of every molecule of the type, 0-based, in atom-id order; a bond's third row repeats its first; the oracle's
    rows agree"""
    defs = R.vector_rows({"a": (2, "bond", (3, 1)), "b": (1, "normal", (2, 3, 1))}, [4, 2], [3, 5])
    assert [d[:2] for d in defs] == [("a", 0), ("b", 2)]
    assert defs[0][2].tolist() == [[14, 12, 14], [19, 17, 19]]
    assert np.array_equal(defs[1][2], RO.mol_rows([4, 2], [3, 5], 1, (2, 3, 1)))
    assert np.array_equal(defs[0][2][:, :2], RO.mol_rows([4, 2], [3, 5], 2, (3, 1)))
