"""Static structure factor on the device: mdp_structure_factor (csrc/sk.cu) against the oracle (tests/sk_oracle.py) within
the accuracy contract, its determinism, scratch-limited sub-batches and argument errors; calc_structure_factor end to end
against the oracle on the sample frames, the water box, a triclinic dump and a trajectory whose cell changes; N ranks
against one."""
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from tests import sk_oracle as SO  # noqa: E402
from tests.conftest import NUM_ATOMS, NUM_MOLS  # noqa: E402
from tests.test_gpu_einstein import fresh_ctx  # noqa: E402,F401

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = 1e-5


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mdproptools_b200 import ops as _ops
    return _ops


def _dev(a, dtype=torch.float64):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dtype).cuda()


def _bound(re, im, counts, bin_off):
    """per (row, bin): sum over the bin's k of eps (N_a |rho_b| + N_b |rho_a|) + eps^2 N_a N_b -- the contract carried
    through Re(rho_a conj(rho_b)) -- plus the fp64 round-off of the sums."""
    ncls = re.shape[0]
    amp = np.hypot(re, im)
    out = []
    for a in range(ncls):
        for b in range(a, ncls):
            t = EPS * (counts[a] * amp[b] + counts[b] * amp[a]) + EPS * EPS * counts[a] * counts[b] + 1e-12 * (counts[a] * counts[b] + 1)
            out.append([t[bin_off[q]:bin_off[q + 1]].sum() for q in range(len(bin_off) - 1)])
    return np.asarray(out).reshape(-1, len(bin_off) - 1)


def _check_kernel(ops, cell, pos, cls, ncls, miller, bin_off):
    """pos [F, N, 3], cls [N] or [F, N]: device sums against the oracle's fp64 sums within the contract."""
    F = pos.shape[0]
    xyz = _dev(pos.transpose(0, 2, 1))
    cls_d = None if cls is None else _dev(cls, torch.int32)
    got = ops.structure_factor(xyz, cls_d, ncls, cell, miller, bin_off, len(bin_off) - 1).cpu().numpy()
    for f in range(F):
        c = np.zeros(pos.shape[1], dtype=np.int64) if cls is None else np.asarray(cls if np.ndim(cls) == 1 else cls[f])
        re, im = SO.class_rho(cell, pos[f], c, ncls, miller)
        want = SO.pair_sums(re, im, bin_off)
        bound = _bound(re, im, np.bincount(c, minlength=ncls), bin_off)
        assert np.all(np.abs(got[f] - want) <= bound), (f, np.max(np.abs(got[f] - want) / np.maximum(bound, 1e-300)))
    return got


CELLS = {"ortho": (23.0, 17.5, 31.25, 0.0, 0.0, 0.0), "triclinic": (25.0, 21.0, 18.0, 5.0, -2.5, 3.15)}


@pytest.mark.parametrize("name", list(CELLS))
@pytest.mark.parametrize("n,ncls,per_frame", [(1, 1, False), (1000, 1, False), (1537, 4, False), (777, 3, True)])
def test_kernel_matches_oracle(ops, name, n, ncls, per_frame):
    """n around the tile (512) and chunk (32) sizes, nk = a k-set that is no multiple of the k-block (512), one and several
    classes with an empty one (class 1 of 3 or more), per-frame classes, unwrapped positions up to two cells out."""
    cell = CELLS[name]
    rng = np.random.default_rng(n + ncls)
    F = 3
    pos = rng.uniform(-1, 2, (F, n, 3)) @ SO.cell_matrix(cell).T
    choices = [c for c in range(ncls) if ncls < 3 or c != 1]
    cls = rng.choice(choices, (F, n) if per_frame else n).astype(np.int32) if ncls > 1 else None
    miller, bin_off, _ = SO.kset_brute(cell, 2.0, 0.1)
    assert len(miller) % 512 != 0 and len(miller) > 512
    got = _check_kernel(ops, cell, pos, cls, ncls, miller, bin_off)
    if ncls >= 3:
        assert not np.any(got[:, ops.sym_row(1, 1, ncls)]) and not np.any(got[:, ops.sym_row(0, 1, ncls)])


def test_miller_components_at_the_bound_and_empty_sets(ops):
    from mdproptools_b200._lib import SK_NLIM
    rng = np.random.default_rng(11)
    cell = CELLS["triclinic"]
    m = np.concatenate([np.array([[SK_NLIM, SK_NLIM, SK_NLIM], [SK_NLIM, -SK_NLIM, SK_NLIM], [0, 0, SK_NLIM], [SK_NLIM, 0, -SK_NLIM],
                                  [1, -SK_NLIM, 0], [-SK_NLIM, SK_NLIM, -SK_NLIM]]),
                        rng.integers(-SK_NLIM, SK_NLIM + 1, (700, 3))])
    bin_off = np.array([0, 6, 6, 300, len(m)])
    pos = rng.uniform(0, 1, (2, 600, 3)) @ SO.cell_matrix(cell).T
    cls = rng.integers(0, 2, 600).astype(np.int32)
    _check_kernel(ops, cell, pos, cls, 2, m, bin_off)
    # nk = 0: zeros; no atoms: zeros
    z = ops.structure_factor(_dev(pos.transpose(0, 2, 1)), _dev(cls, torch.int32), 2, cell, np.zeros((0, 3)), [0, 0, 0], 2)
    assert z.shape == (2, 3, 2) and not torch.any(z)
    e = ops.structure_factor(torch.zeros((2, 3, 0), dtype=torch.float64, device="cuda"), None, 1, cell, m, bin_off, 4)
    assert not torch.any(e)


def test_wrapped_and_unwrapped_positions_agree(ops):
    rng = np.random.default_rng(12)
    cell = CELLS["triclinic"]
    H = SO.cell_matrix(cell)
    s = rng.uniform(0, 1, (1, 900, 3))
    shift = rng.integers(-3, 4, (1, 900, 3))
    miller, bin_off, _ = SO.kset_brute(cell, 1.5, 0.1)
    a = ops.structure_factor(_dev((s @ H.T).transpose(0, 2, 1)), None, 1, cell, miller, bin_off, len(bin_off) - 1)
    b = ops.structure_factor(_dev(((s + shift) @ H.T).transpose(0, 2, 1)), None, 1, cell, miller, bin_off, len(bin_off) - 1)
    re, im = SO.rho(cell, s[0] @ H.T, miller)
    bound = _bound(re[None], im[None], [900], bin_off)
    assert np.all(np.abs((a - b).cpu().numpy()) <= 2 * bound)


def test_kernel_is_deterministic(ops):
    rng = np.random.default_rng(13)
    cell = CELLS["ortho"]
    xyz = _dev((rng.uniform(0, 1, (4, 3000, 3)) @ SO.cell_matrix(cell).T).transpose(0, 2, 1))
    cls = _dev(rng.integers(0, 3, 3000), torch.int32)
    miller, bin_off, _ = SO.kset_brute(cell, 2.0, 0.05)
    r1 = ops.structure_factor(xyz, cls, 3, cell, miller, bin_off, len(bin_off) - 1)
    r2 = ops.structure_factor(xyz, cls, 3, cell, miller, bin_off, len(bin_off) - 1)
    assert torch.equal(r1, r2)


def test_subbatches_under_scratch_limits(ops, fresh_ctx):  # noqa: F811
    """12 frames swept over scratch limits from below the smallest that holds one frame to all frames in one sub-batch:
    every working limit gives the bits of the unlimited call, calls never fail above the smallest working limit, and the
    number of launches falls from one sub-batch per frame to one."""
    from mdproptools_b200._lib import MdpropError
    rng = np.random.default_rng(14)
    cell = CELLS["triclinic"]
    F, n, ncls = 12, 2000, 3
    xyz = _dev((rng.uniform(0, 1, (F, n, 3)) @ SO.cell_matrix(cell).T).transpose(0, 2, 1))
    cls = _dev(rng.integers(0, ncls, n), torch.int32)
    miller, bin_off, _ = SO.kset_brute(cell, 2.0, 0.1)
    nk = len(miller)
    nb = len(bin_off) - 1
    ref = ops.structure_factor(xyz, cls, ncls, cell, miller, bin_off, nb)
    per_frame = 16 * n + 4 * (ncls + 1) + 16 * ncls * nk
    fixed = 16 * nk + 8 * (nb + 1)
    seen = {}
    for lim in sorted({fixed + per_frame * m + d for m in (1, 2, 3, 5, 8, 12, 20) for d in (-8192, 0, 4096, 8192, 16384)}):
        ctx = fresh_ctx(lim)
        try:
            seen[lim] = (ops.structure_factor(xyz, cls, ncls, cell, miller, bin_off, nb), ctx.launch_count())
        except MdpropError as e:
            seen[lim] = str(e)
    ok = sorted(l for l, v in seen.items() if not isinstance(v, str))
    bad = sorted(l for l, v in seen.items() if isinstance(v, str))
    assert ok and bad, (ok, bad)
    for l in bad:
        assert "exceeds the context limit" in seen[l], seen[l]
        assert l < ok[0]
    launches = [seen[l][1] for l in ok]
    assert all(x >= y for x, y in zip(launches, launches[1:]))
    assert launches[0] == 3 * F and launches[-1] == 3, launches
    for l in ok:
        assert torch.equal(seen[l][0], ref), l


def test_bad_arguments(ops):
    from mdproptools_b200 import _lib
    from mdproptools_b200._lib import MdpropError
    xyz = _dev(np.ones((1, 3, 10)))
    m = np.array([[1, 0, 0], [0, 1, 0]])
    cell = (10.0, 10.0, 10.0, 0.0, 0.0, 0.0)
    cases = [dict(cell=(0.0, 10.0, 10.0, 0, 0, 0)), dict(cell=(10.0, -1.0, 10.0, 0, 0, 0)), dict(cell=(10, 10, np.inf, 0, 0, 0)),
             dict(ncls=0), dict(ncls=_lib.SK_MAX_CLASSES + 1), dict(miller=np.array([[1, 0, 0], [0, _lib.SK_NLIM + 1, 0]])),
             dict(miller=np.array([[1, 0, 0], [0, 0, -_lib.SK_NLIM - 1]])), dict(bin_off=[1, 2]), dict(bin_off=[0, 1]),
             dict(bin_off=[0, 2, 1, 2], nbins=3)]
    for c in cases:
        a = dict(cell=cell, ncls=1, miller=m, bin_off=[0, 2], nbins=1)
        a.update(c)
        with pytest.raises(MdpropError, match="rc=-2"):
            ops.structure_factor(xyz, None, a["ncls"], a["cell"], a["miller"], a["bin_off"], a["nbins"])
    ctx = _lib.Context.get()
    cl = np.array(cell)
    mm = np.ascontiguousarray(m, dtype=np.int32)
    bo = np.array([0, 2], dtype=np.int64)
    out = torch.empty((1, 1, 1), dtype=torch.float64, device="cuda")
    for F, n, nk, nb in ((-1, 10, 2, 1), (1, -10, 2, 1), (1, 10, -2, 1), (1, 10, 2, -1)):
        rc = _lib.lib().mdp_structure_factor(ctx.handle, F, n, _lib.ptr(xyz), None, 0, 1, _lib.dptr(cl), nk,
                                             mm.ctypes.data_as(_lib.POINTER(_lib.c_int32)), nb,
                                             bo.ctypes.data_as(_lib.POINTER(_lib.c_int64)), _lib.ptr(out), _lib.stream_ptr())
        assert rc == -2, (F, n, nk, nb)


# ------------------------------------------------------------------------------------------------
# calc_structure_factor end to end
# ------------------------------------------------------------------------------------------------
def _oracle_e2e(frames, k_max, bin_size, relations, k_min=None, max_k=None, seed=0):
    """frames [(cell, pos [N,3], types)] -> (S, S_ab, n_k mean, bound on S, bound on S_ab): the oracle with the contract's
    bound carried through each frame's normalisation and the average."""
    named = sorted(set(int(t) for pair in relations for t in pair))
    ncls = len(named) + 1
    w = np.array([1.0 if a == b else 2.0 for a in range(ncls) for b in range(a, ncls)])
    rel = [(named.index(int(a)), named.index(int(b))) for a, b in relations]
    tot_f, part_f, btot_f, bpart_f, nk_f = [], [], [], [], []
    for cell, pos, types in frames:
        t = np.asarray(types).astype(np.int64)
        cls = np.array([named.index(v) if v in named else len(named) for v in t])
        miller, bin_off, _ = SO.kset_brute(cell, k_max, bin_size, k_min, max_k, seed)
        re, im = SO.class_rho(cell, pos, cls, ncls, miller)
        P = SO.pair_sums(re, im, bin_off)
        counts = np.bincount(cls, minlength=ncls)
        nk = np.diff(bin_off)
        tot, part = SO.normalise(P, nk, counts, rel)
        B = _bound(re, im, counts, bin_off)
        bt, bp = SO.normalise(B, nk, counts, rel)
        for acc, v in ((tot_f, tot), (part_f, part), (btot_f, bt), (bpart_f, bp), (nk_f, nk)):
            acc.append(v)
    return (SO.average(tot_f), SO.average(part_f), np.mean(nk_f, axis=0), SO.average(btot_f), SO.average(bpart_f))


def _read(pattern, altered=False):
    from mdproptools_b200.io.dump import read_dumps
    from mdproptools_b200.structural.rdf_cn import calc_atom_type_ids
    out = []
    for fr in read_dumps(pattern, ["id", "type", "x", "y", "z"]):
        b = fr.box
        cell = tuple(b.bound_lengths()) + (tuple(b.tilt) if b.tilt is not None else (0.0, 0.0, 0.0))
        typ = calc_atom_type_ids(fr.data["id"], NUM_MOLS, NUM_ATOMS) if altered else fr.data["type"]
        out.append((cell, np.stack([fr.data[c] for c in "xyz"], axis=1), typ))
    return out


def _compare(df, want, relations):
    S, Sab, nk, bS, bSab = want
    got = df.to_numpy()
    assert list(df.columns) == ["k ($\\AA^{-1}$)", "S(k)"] + [f"S_{a}-{b}" for a, b in np.asarray(relations).T] + ["n_k"]
    assert np.array_equal(np.isnan(got[:, 1]), np.isnan(S)) and np.array_equal(got[:, -1], nk)
    ok = ~np.isnan(S)
    assert ok.sum() > 3
    assert np.all(np.abs(got[ok, 1] - S[ok]) <= bS[ok] + 1e-12), np.max(np.abs(got[ok, 1] - S[ok]) - bS[ok])
    for r in range(Sab.shape[0]):
        assert np.all(np.abs(got[ok, 2 + r] - Sab[r, ok]) <= bSab[r, ok] + 1e-12), r


@pytest.mark.parametrize("altered", [False, True])
def test_calc_structure_factor_on_sample_frames(ops, sample_dir, tmp_path, altered):
    from mdproptools_b200.structural.structure_factor import calc_structure_factor
    rel = [[32, 1], [1, 5]] if altered else [[9, 1], [1, 5]]
    kw = dict(num_mols=NUM_MOLS, num_atoms_per_mol=NUM_ATOMS) if altered else {}
    pat = os.path.join(sample_dir, "dump.nvt.*.dump")
    out = tmp_path / "sk.csv"
    df = calc_structure_factor(1.6, 0.05, rel, pat, max_k_per_bin=24, seed=3, path_or_buff=str(out), **kw)
    _compare(df, _oracle_e2e(_read(pat, altered), 1.6, 0.05, list(zip(*rel)), max_k=24, seed=3), rel)
    assert out.stat().st_size > 0 and np.isnan(df["S(k)"].iloc[0])          # no k-vector below 2 pi / 49.2 A


def test_calc_structure_factor_on_water_box(ops, water_dir):
    from mdproptools_b200.structural.structure_factor import calc_structure_factor
    pat = os.path.join(water_dir, "dump.water.*.dump")
    frames = _read(pat)
    types = sorted(set(int(t) for t in frames[0][2]))
    rel = [[types[0], types[0]], [types[-1], types[0]]]
    df = calc_structure_factor(4.0, 0.1, rel, pat, save_mode=False)
    _compare(df, _oracle_e2e(frames, 4.0, 0.1, list(zip(*rel))), rel)


def _write_dump(path, frames):
    """frames [(timestep, cell, pos [N,3], types [N])] -> one LAMMPS dump file (triclinic header when a tilt is nonzero)."""
    with open(path, "w") as f:
        for ts, cell, pos, types in frames:
            lx, ly, lz, xy, xz, yz = (float(v) for v in cell)
            f.write(f"ITEM: TIMESTEP\n{ts}\nITEM: NUMBER OF ATOMS\n{len(pos)}\n")
            if xy or xz or yz:
                xlo_b, xhi_b = min(0.0, xy, xz, xy + xz), lx + max(0.0, xy, xz, xy + xz)
                ylo_b, yhi_b = min(0.0, yz), ly + max(0.0, yz)
                f.write(f"ITEM: BOX BOUNDS xy xz yz pp pp pp\n{xlo_b!r} {xhi_b!r} {xy!r}\n{ylo_b!r} {yhi_b!r} {xz!r}\n0.0 {lz!r} {yz!r}\n")
            else:
                f.write(f"ITEM: BOX BOUNDS pp pp pp\n0.0 {lx!r}\n0.0 {ly!r}\n0.0 {lz!r}\n")
            f.write("ITEM: ATOMS id type x y z\n")
            for i in range(len(pos)):
                f.write(f"{i + 1} {int(types[i])} {float(pos[i, 0])!r} {float(pos[i, 1])!r} {float(pos[i, 2])!r}\n")


@pytest.fixture
def triclinic_dump(tmp_path):
    rng = np.random.default_rng(21)
    cell = (26.0, 22.0, 19.0, 4.0, -2.0, 3.0)
    n = 1500
    types = rng.integers(1, 4, n)
    frames = [(ts, cell, rng.uniform(0, 1, (n, 3)) @ SO.cell_matrix(cell).T, types) for ts in (0, 100)]
    path = tmp_path / "dump.tri.lammpstrj"
    _write_dump(path, frames)
    return str(path), [(c, p, t) for _, c, p, t in frames]


def test_calc_structure_factor_on_a_triclinic_dump(ops, triclinic_dump):
    from mdproptools_b200.structural.structure_factor import calc_structure_factor
    path, frames = triclinic_dump
    got = _read(path)
    assert all(np.allclose(g[0], f[0], rtol=0, atol=1e-12) for g, f in zip(got, frames))
    rel = [[1, 1, 2], [1, 2, 3]]
    df = calc_structure_factor(2.5, 0.1, rel, path, save_mode=False)
    _compare(df, _oracle_e2e(got, 2.5, 0.1, list(zip(*rel))), rel)


def test_calc_structure_factor_with_a_changing_cell(ops, tmp_path):
    """NPT-like: three frames, two cells (one call per run of frames that share a cell), so the k-sets and n_k differ per
    frame and bins empty in one cell enter only the other's average."""
    from mdproptools_b200.structural.structure_factor import calc_structure_factor
    rng = np.random.default_rng(22)
    n = 800
    types = rng.integers(1, 3, n)
    cells = [(18.0, 18.0, 18.0, 0.0, 0.0, 0.0), (18.0, 18.0, 18.0, 0.0, 0.0, 0.0), (21.0, 19.0, 20.0, 1.0, 0.5, -0.7)]
    frames = [(10 * k, c, rng.uniform(0, 1, (n, 3)) @ SO.cell_matrix(c).T, types) for k, c in enumerate(cells)]
    path = tmp_path / "dump.npt.lammpstrj"
    _write_dump(path, frames)
    got = _read(str(path))
    rel = [[1, 2], [2, 2]]
    df = calc_structure_factor(2.0, 0.04, rel, str(path), save_mode=False)
    want = _oracle_e2e(got, 2.0, 0.04, list(zip(*rel)))
    _compare(df, want, rel)
    nk = df["n_k"].to_numpy()
    assert np.any((nk > 0) & (nk != np.round(nk)))                  # bins whose count differs between the cells


# ------------------------------------------------------------------------------------------------
# N ranks against one
# ------------------------------------------------------------------------------------------------
WORKER = '''
import os, sys
import numpy as np
sys.path.insert(0, sys.argv[3])
import torch
import torch.distributed as dist
world = int(os.environ.get("WORLD_SIZE", "1"))
torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
if world > 1:
    dist.init_process_group("nccl")
from mdproptools_b200.structural.structure_factor import calc_structure_factor
df = calc_structure_factor(3.0, 0.05, [[1, 3], [3, 3]], sys.argv[2], max_k_per_bin=64, save_mode=False)
if int(os.environ.get("RANK", "0")) == 0:
    np.save(sys.argv[1], df.to_numpy())
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
'''


def test_structure_factor_nrank_equals_1rank(ops, water_dir, tmp_path):
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs at least 2 GPUs")
    worker = tmp_path / "sk_worker.py"
    worker.write_text(WORKER)
    res = {}
    for n in sorted({1, 2, min(ngpu, 4)}):
        out = tmp_path / f"n{n}.npy"
        cmd = ([sys.executable] if n == 1 else
               [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
                "127.0.0.1", "--master-port", str(29761 + n)])
        r = subprocess.run(cmd + [str(worker), str(out), os.path.join(water_dir, "dump.water.*.dump"), ROOT], cwd=ROOT,
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        res[n] = np.load(out)
    for n in res:
        assert np.array_equal(res[1], res[n], equal_nan=True), n
