"""Reorientation on the device: mdp_orient_series (csrc/orient.cu) against the host build of its body bit for bit, and the
arguments it rejects; calc_reorientation / calc_reorientation_times end to end against exact references (rigid rotors,
static molecules), the oracle on the mini trajectory, the law of a random rotational walk, the errors they raise, and N
ranks against one."""
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from tests import reorient_oracle as RO  # noqa: E402
from tests.conftest import NUM_ATOMS  # noqa: E402
from tests.test_host_reorientation import (cell_matrix, emu, random_cell, three_site_molecules, wrap,  # noqa: E402,F401
                                           write_pos_dump)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KIND = {"bond": 0, "bisector": 1, "normal": 2}
DT = 1e-14                                      # seconds per frame: 10 steps of 1 fs ("real" units)
CELL = np.array([31.0, 29.0, 27.0, 4.0, -3.0, 2.5])


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mdproptools_b200 import ops as _ops
    return _ops


def _calc(path, vectors, num_mols, num_atoms_per_mol, **kw):
    from mdproptools_b200.dynamical.reorientation import calc_reorientation
    return calc_reorientation(str(path), vectors, num_mols, num_atoms_per_mol, save_mode=False, **kw)


def _times(corr):
    from mdproptools_b200.dynamical.reorientation import calc_reorientation_times
    return calc_reorientation_times(corr)


def rodrigues(axis, ang):
    """rotation matrices [..., 3, 3] by ``ang`` about ``axis`` [..., 3]"""
    axis = axis / np.linalg.norm(axis, axis=-1)[..., None]
    K = np.zeros(axis.shape[:-1] + (3, 3))
    K[..., 0, 1], K[..., 0, 2], K[..., 1, 2] = -axis[..., 2], axis[..., 1], -axis[..., 0]
    K = K - np.swapaxes(K, -1, -2)
    ang = np.asarray(ang, dtype=np.float64)[..., None, None]
    return np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * K @ K


def _body_vectors(b):
    """the bond, bisector and normal of body sites b [M, 3, 3] (site 0 the origin atom)"""
    d1, d2 = b[:, 1] - b[:, 0], b[:, 2] - b[:, 0]
    return {"bond": d1, "bisector": (d1 + d2) / 2, "normal": np.cross(d1, d2)}


VECTORS = {"bond": (1, "bond", (1, 2)), "bisector": (1, "bisector", (1, 2, 3)), "normal": (1, "normal", (1, 2, 3))}


# ------------------------------------------------------------------------------------------------
# the kernel
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["bond", "bisector", "normal"])
def test_orient_series_matches_host_build_bit_for_bit(ops, emu, kind):
    """Three batches of frames (one of them beyond one 16-frame tile, NPT-like cells that change per frame) written through
    frame0 into one series of 77 vectors (beyond two 32-vector tiles): the host build's bits; the columns no batch covers
    keep their values."""
    rng = np.random.default_rng(300 + KIND[kind])
    M, F = 77, 45
    cells = np.stack([random_cell(rng) for _ in range(F)])
    xyz = np.stack([wrap(three_site_molecules(rng, cells[f], M).reshape(-1, 3), cells[f]).T for f in range(F)])
    for f in range(0, F, 7):                                            # some frames unwrapped by a lattice vector
        xyz[f] += 3 * cell_matrix(cells[f])[:, 0][:, None]
    rows = rng.permuted(np.tile(3 * np.arange(M)[:, None] + np.array([0, 1, 2]), 1), axis=1)
    stride, frame0 = 60, 6
    want = np.full((8, M, stride), -3.0)
    got = torch.full((8, M, stride), -3.0, dtype=torch.float64, device="cuda")
    for a, b in ((0, 5), (5, 39), (39, 45)):
        emu(xyz[a:b], cells[a:b], kind, rows, out=want, frame0=frame0 + a)
        ops.orient_series(torch.from_numpy(xyz[a:b]).cuda(), cells[a:b], KIND[kind], rows, got, frame0=frame0 + a)
    got = got.cpu().numpy()
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
    assert np.all(got[:, :, :frame0] == -3.0) and np.all(got[:, :, frame0 + F:] == -3.0)


def test_orient_series_bad_arguments(ops):
    from mdproptools_b200._lib import MdpropError
    xyz = torch.zeros((2, 3, 6), dtype=torch.float64, device="cuda")
    xyz[:, 0, 1::2] = 1.0
    cells = np.tile([10.0, 10.0, 10.0, 0.0, 0.0, 0.0], (2, 1))
    out = torch.zeros((8, 1, 4), dtype=torch.float64, device="cuda")
    ok = [[0, 1, 2]]
    ops.orient_series(xyz, cells, 1, ok, out)
    before = out.clone()
    bad = [(dict(atoms=[[0, 6, 2]]), "outside"), (dict(atoms=[[-1, 1, 2]]), "outside"), (dict(atoms=[[0, 1, 1]]), "repeats"),
           (dict(atoms=[[3, 3, 2]], kind=0), "repeats"), (dict(kind=3), "kind"), (dict(kind=-1), "kind"),
           (dict(cells=np.tile([10.0, 0.0, 10.0, 0.0, 0.0, 0.0], (2, 1))), "length"),
           (dict(cells=np.tile([10.0, 10.0, np.inf, 0.0, 0.0, 0.0], (2, 1))), "length"),
           (dict(cells=np.tile([10.0, 10.0, 10.0, np.nan, 0.0, 0.0], (2, 1))), "tilt"),
           (dict(frame0=3), "do not fit"), (dict(frame0=-1), "do not fit")]
    for kw, msg in bad:
        args = dict(cells=cells, kind=1, atoms=ok, frame0=0) | kw
        with pytest.raises(MdpropError, match=f"rc=-2.*{msg}"):
            ops.orient_series(xyz, args["cells"], args["kind"], args["atoms"], out, frame0=args["frame0"])
    assert torch.equal(out, before)                                     # the rejected calls wrote nothing


# ------------------------------------------------------------------------------------------------
# exact references
# ------------------------------------------------------------------------------------------------
def rotor_trajectory(seed, M, T, omega, perpendicular=False):
    """Rigid three-site molecules spinning about one axis n at omega rad per frame while their centres drift across the
    periodic faces of CELL (wrapped positions [T, 3, 3 M]); also n and the body sites [M, 3, 3] at t = 0 (relative to the
    centre).  ``perpendicular``: the bond lies in the plane normal to n (a pure spin of the bond)."""
    rng = np.random.default_rng(seed)
    n = rng.normal(size=3)
    n /= np.linalg.norm(n)
    b = three_site_molecules(rng, CELL, M)
    b = b - b[:, :1]
    if perpendicular:
        d1 = b[:, 1] - (b[:, 1] @ n)[:, None] * n
        b[:, 1] = d1 * (1.2 / np.linalg.norm(d1, axis=1))[:, None]
    centre = rng.uniform(0, 1, (M, 3)) @ cell_matrix(CELL).T
    drift = rng.normal(0, 0.4, (M, 3))
    pos = np.empty((T, 3, 3 * M))
    for t in range(T):
        R = rodrigues(n, omega * t)
        sites = np.einsum("ij,msj->msi", R, b) + (centre + drift * t)[:, None, :]
        pos[t] = wrap(sites.reshape(-1, 3), CELL).T
    return pos, n, b


@pytest.mark.parametrize("omega", [2 * np.pi / 97, 0.0])
def test_rigid_rotors_closed_form(ops, tmp_path, omega):
    """u(t).u(t+tau) = cos^2 theta + sin^2 theta cos(omega tau) for every origin, theta the angle of the vector to the axis:
    C1 and C2 = P2 of it, averaged over the molecules, for bond, bisector and normal alike, within 1e-10 at every lag (the
    FFT correlator's contract).  omega = 0: static molecules (drifting only), C1 = C2 = 1."""
    M, T = 40, 300
    pos, n, b = rotor_trajectory(11, M, T, omega)
    write_pos_dump(tmp_path / "dump.rot.lammpstrj", np.arange(T) * 10, pos, CELL)
    got = _calc(tmp_path / "dump.rot.lammpstrj", VECTORS, [M], [3], max_lag=150)
    tau = np.arange(150)
    assert np.allclose(got["Time (s)"], tau * DT, rtol=1e-14, atol=0)
    for name, w in _body_vectors(b).items():
        c = (w @ n) / np.linalg.norm(w, axis=1)
        x = c[:, None] ** 2 + (1 - c[:, None] ** 2) * np.cos(omega * tau)[None, :]
        assert np.abs(got[f"C1_{name}"] - x.mean(axis=0)).max() <= 1e-10, name
        assert np.abs(got[f"C2_{name}"] - (1.5 * x * x - 0.5).mean(axis=0)).max() <= 1e-10, name
        if omega == 0.0:
            assert np.abs(got[f"C1_{name}"] - 1).max() <= 1e-12 and np.abs(got[f"C2_{name}"] - 1).max() <= 1e-12


def test_pure_spin_correlation_time(ops, tmp_path):
    """a bond normal to the spin axis: C1 = cos(omega tau), whose integral to its first zero is 1/omega; tau_1 within the
    trapezoid error (the step past the zero and the rule's curvature, both under 0.3 % at 0.05 rad per frame)"""
    M, T, omega = 30, 400, 0.05
    pos, _, _ = rotor_trajectory(12, M, T, omega, perpendicular=True)
    write_pos_dump(tmp_path / "dump.spin.lammpstrj", np.arange(T) * 10, pos, CELL)
    corr = _calc(tmp_path / "dump.spin.lammpstrj", {"oh": (1, "bond", (1, 2))}, [M], [3])
    tab = _times(corr)
    assert list(tab.columns) == ["tau (s)", "t_end (s)"] and list(tab.index) == ["C1_oh", "C2_oh"]
    assert tab.loc["C1_oh", "tau (s)"] == pytest.approx(DT / omega, rel=3e-3)
    k = int(np.ceil(np.pi / 2 / omega))                                    # the first lag with cos(omega tau) <= 0
    assert tab.loc["C1_oh", "t_end (s)"] == pytest.approx(k * DT, rel=1e-12)
    t = corr["Time (s)"].to_numpy()
    for col in ("C1_oh", "C2_oh"):
        want, t_end = RO.correlation_time(t, corr[col].to_numpy())
        assert tab.loc[col, "tau (s)"] == pytest.approx(want, rel=1e-12) and tab.loc[col, "t_end (s)"] == t_end


def random_walk_trajectory(seed, M, T, alpha):
    """Three-site molecules at fixed centres, each turned every frame by alpha about its own uniformly random axis"""
    rng = np.random.default_rng(seed)
    b = three_site_molecules(rng, CELL, M)
    centre = b[:, 0].copy()
    b = b - b[:, :1]
    pos = np.empty((T, 3, 3 * M))
    for t in range(T):
        if t:
            b = np.einsum("mij,msj->msi", rodrigues(rng.normal(size=(M, 3)), np.full(M, alpha)), b)
        pos[t] = wrap((b + centre[:, None, :]).reshape(-1, 3), CELL).T
    return pos


def test_random_rotational_walk(ops, tmp_path):
    """Rotations by a fixed angle alpha = 0.5 about uniformly random axes: E[C_l(n)] = lambda_l^n with lambda_1 =
    (1 + 2 cos a)/3 and lambda_2 = (1 + 2 cos a + 2 cos 2a)/5.  500 molecules, 200 frames, 100 lags.  Host runs of the
    oracle's law on six seeds gave max_n |C_l(n) - lambda_l^n| of 0.006-0.022 (C1) and 0.006-0.011 (C2), and tau_1/tau_2
    of 3.07-3.29 (3.10 from the lambdas; 3 in the small-angle limit); the tolerances are 0.04 and [2.7, 3.5]."""
    M, T, alpha = 500, 200, 0.5
    write_pos_dump(tmp_path / "dump.walk.lammpstrj", np.arange(T) * 10, random_walk_trajectory(13, M, T, alpha), CELL)
    corr = _calc(tmp_path / "dump.walk.lammpstrj", {"b": (1, "bond", (1, 2)), "n": (1, "normal", (1, 2, 3))}, [M], [3],
                 max_lag=100)
    n = np.arange(100)
    l1 = (1 + 2 * np.cos(alpha)) / 3
    l2 = (1 + 2 * np.cos(alpha) + 2 * np.cos(2 * alpha)) / 5
    for v in ("b", "n"):
        assert np.abs(corr[f"C1_{v}"] - l1 ** n).max() < 0.04, v
        assert np.abs(corr[f"C2_{v}"] - l2 ** n).max() < 0.04, v
    tab = _times(corr)
    ratio = tab.loc["C1_b", "tau (s)"] / tab.loc["C2_b", "tau (s)"]
    assert 2.7 < ratio < 3.5, ratio


# ------------------------------------------------------------------------------------------------
# the mini trajectory against the oracle
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mini_mols():
    from tests.conftest import GOLDEN
    return np.load(os.path.join(GOLDEN, "ref_dynamical.npz"))["mini_num_mols"].tolist()


MINI_VECTORS = {"dme_bond": (1, "bond", (1, 2)), "dme_bis": (1, "bisector", (1, 3, 5)), "dme_norm": (1, "normal", (2, 7, 11)),
                "tfsi_bond": (2, "bond", (1, 4)), "tfsi_bis": (2, "bisector", (5, 1, 2)), "tfsi_norm": (2, "normal", (1, 3, 9))}


def _unwrapped_copy(src, dst):
    """the mini dumps with the wrapped columns removed: id type xu yu zu, xu = x + ix (xhi - xlo) at full precision, so that
    the two dumps hold the same trajectory"""
    import glob
    os.makedirs(dst, exist_ok=True)
    for f in glob.glob(os.path.join(src, "dump.mini.*.dump")):
        lines = open(f).read().splitlines()
        cols = lines[8].split()[2:]
        lo_hi = [[float(v) for v in lines[k].split()[:2]] for k in (5, 6, 7)]
        out = lines[:8] + ["ITEM: ATOMS id type xu yu zu"]
        for row in lines[9:]:
            if not row.strip():
                continue
            v = row.split()
            val = {c: v[k] for k, c in enumerate(cols)}
            u = [float(val[a]) + float(val["i" + a]) * (hi - lo) for a, (lo, hi) in zip("xyz", lo_hi)]
            out.append(f"{val['id']} {val['type']} " + " ".join(repr(x) for x in u))
        with open(os.path.join(dst, os.path.basename(f)), "w") as fh:
            fh.write("\n".join(out) + "\n")


def test_mini_traj_against_oracle(ops, mini_dir, mini_mols, tmp_path):
    """bonds, bisectors and normals of DME and TFSI on the 26 frames: every column within 1e-10 of the oracle's direct
    long-double sums; the same trajectory as unwrapped positions only (xu yu zu) within 1e-12; the saved CSV"""
    from mdproptools_b200.common import constants as K
    pattern = os.path.join(mini_dir, "dump.mini.*.dump")
    csv = tmp_path / "reorientation.csv"
    from mdproptools_b200.dynamical.reorientation import calc_reorientation
    got = calc_reorientation(pattern, MINI_VECTORS, mini_mols, NUM_ATOMS, path_or_buff=str(csv))
    want = RO.calc_reorientation(pattern, MINI_VECTORS, mini_mols, NUM_ATOMS, K.TIME_CONVERSION["real"])
    assert list(got.columns) == list(want) and len(got) == 13
    for col, w in want.items():
        assert np.abs(got[col].to_numpy() - w).max() <= 1e-10 * max(np.abs(w).max(), 1e-300), col
    assert np.allclose(np.loadtxt(csv, delimiter=",", skiprows=1), got.to_numpy(), rtol=1e-15, atol=0)
    _unwrapped_copy(mini_dir, str(tmp_path / "u"))
    unw = _calc(os.path.join(str(tmp_path / "u"), "dump.mini.*.dump"), MINI_VECTORS, mini_mols, NUM_ATOMS)
    for col in got.columns:
        assert np.abs(unw[col].to_numpy() - got[col].to_numpy()).max() <= 1e-12 * np.abs(got[col].to_numpy()).max(), col


# ------------------------------------------------------------------------------------------------
# errors
# ------------------------------------------------------------------------------------------------
def test_reorientation_errors(ops, tmp_path, monkeypatch):
    """ValueError for a dump without positions, a molecule layout that does not hold the atoms, a changing atom count,
    uneven frames, fewer than 2 frames, max_lag < 1, channels above the device's free memory, and a degenerate vector
    (two coincident atoms in one frame), named in the message"""
    rng = np.random.default_rng(14)
    M, T = 6, 8
    pos = np.stack([wrap(three_site_molecules(rng, CELL, M).reshape(-1, 3), CELL).T for _ in range(T)])
    v = {"w": (1, "bisector", (1, 2, 3))}

    def dump(name, steps=np.arange(T) * 10, p=pos, cols=("x", "y", "z")):
        d = tmp_path / name
        d.mkdir()
        write_pos_dump(d / "dump.lammpstrj", steps, p, CELL, cols=cols)
        return d / "dump.lammpstrj"

    ok = dump("ok")
    assert np.isfinite(_calc(ok, v, [M], [3]).to_numpy()).all()
    assert np.isfinite(_calc(dump("xu", cols=("xu", "yu", "zu")), v, [M], [3]).to_numpy()).all()
    cases = [(dump("nopos", cols=("vx", "vy", "vz")), {}, "x y z or xu yu zu"),
             (ok, dict(num_mols=[M + 1]), "does not match length"),
             (ok, dict(num_mols=[M - 1]), "does not match length"),
             (dump("uneven", steps=np.r_[np.arange(T - 1) * 10, 10 * T + 3]), {}, "evenly spaced"),
             (dump("one", steps=[0], p=pos[:1]), {}, "at least 2 frames"),
             (ok, dict(max_lag=0), "max_lag")]
    d = tmp_path / "natoms"
    d.mkdir()
    write_pos_dump(d / "dump.lammpstrj", np.arange(4) * 10, pos[:4], CELL)
    write_pos_dump(d / "dump.lammpstrj", np.arange(4, 8) * 10, pos[4:, :, :-3], CELL, mode="a")
    cases.append((d / "dump.lammpstrj", dict(num_mols=[M]), "does not match length|fixed atom count"))
    for path, kw, msg in cases:
        args = dict(num_mols=[M], num_atoms_per_mol=[3]) | kw
        with pytest.raises(ValueError, match=msg):
            _calc(path, v, args["num_mols"], args["num_atoms_per_mol"], **{k: w for k, w in kw.items() if k == "max_lag"})
    bad = pos.copy()
    bad[5, :, 3 * 2 + 1] = bad[5, :, 3 * 2]                                 # molecule 2: atoms 1 and 2 coincide in frame 5
    with pytest.raises(ValueError, match="'oh'.*degenerate"):
        _calc(dump("degenerate", p=bad), {"w": (1, "bond", (1, 3)), "oh": (1, "bond", (1, 2))}, [M], [3])
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda *a: (1024, 1 << 40))
    with pytest.raises(ValueError, match="free memory.*fewer vectors or more GPUs"):
        _calc(ok, v, [M], [3])


# ------------------------------------------------------------------------------------------------
# N ranks against one
# ------------------------------------------------------------------------------------------------
WORKER = '''
import os, sys
import numpy as np
sys.path.insert(0, sys.argv[3])
import torch
import torch.distributed as dist
from tests.conftest import NUM_ATOMS
from tests.test_gpu_reorientation import MINI_VECTORS
from mdproptools_b200.dynamical.reorientation import calc_reorientation, calc_reorientation_times
world = int(os.environ.get("WORLD_SIZE", "1"))
torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
if world > 1:
    dist.init_process_group("nccl")
num_mols = [int(v) for v in sys.argv[4].split(",")]
corr = calc_reorientation(os.path.join(sys.argv[2], "dump.mini.*.dump"), MINI_VECTORS, num_mols, NUM_ATOMS, save_mode=False)
res = {"corr": corr.to_numpy(), "times": calc_reorientation_times(corr).to_numpy()}
if int(os.environ.get("RANK", "0")) == 0:
    np.savez(sys.argv[1], **res)
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
'''


def test_reorientation_nrank_equals_1rank(ops, mini_dir, mini_mols, tmp_path):
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs at least 2 GPUs")
    worker = tmp_path / "reorient_worker.py"
    worker.write_text(WORKER)
    res = {}
    for n in sorted({1, 2, min(ngpu, 4)}):
        out = tmp_path / f"n{n}.npz"
        cmd = ([sys.executable] if n == 1 else
               [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
                "127.0.0.1", "--master-port", str(29771 + n)])
        r = subprocess.run(cmd + [str(worker), str(out), mini_dir, ROOT, ",".join(map(str, mini_mols))], cwd=ROOT,
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        res[n] = np.load(out)
    for n in res:
        for k in res[1].files:
            a, b = res[1][k], res[n][k]
            assert a.shape == b.shape, (n, k)
            assert np.abs(a - b).max() <= 1e-12 * np.abs(a).max(), (n, k)
