"""Parity of the CUDA path (through the C ABI / the reference-facing Python API) against
  (1) golden outputs of the unmodified reference (tests/golden/, see oracle/gen_golden.py), and
  (2) the CPU oracle on seeded synthetic inputs (ragged sizes, several classes, triclinic-length boxes, ...).
Integer results must be bit-exact; floating-point results carry the tolerance stated at the assert.
"""
import json
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import oracle as O  # noqa: E402
from tests.conftest import ELEMENTS, GOLDEN, MASS, NUM_ATOMS, NUM_MOLS  # noqa: E402

REL = [[9, 9, 9, 9], [1, 4, 6, 9]]


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mdproptools_b200 import ops as _ops
    return _ops


def _dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


def _rand_box(rng, n, L, ntypes):
    pos = rng.uniform(0, 1, (3, n)) * np.asarray(L)[:, None]
    typ = rng.integers(1, ntypes + 1, n).astype(np.float64)
    return pos, typ


# ------------------------------------------------------------------------------------------------
# pair histogram kernel vs oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,L,rc,ddr,flags", [
    (1000, (21.0, 22.5, 24.0), 7.0, 0.05, 0),
    (777, (15.0, 15.0, 15.0), 7.4, 0.1, 0),          # r_cut close to L/2: general minimum-image path everywhere
    (3000, (60.0, 40.0, 35.0), 6.0, 0.05, 0),        # culling active
    (3000, (60.0, 40.0, 35.0), 6.0, 0.05, 1),        # MDP_PAIR_NO_CULL
    (3000, (60.0, 40.0, 35.0), 6.0, 0.05, 3),        # no cull, no sort (brute force in caller order)
    (257, (9.0, 9.0, 9.0), 12.0, 0.25, 0),           # r_cut > L/2 (single-shift semantics, not true MIC)
    (31, (9.0, 9.0, 9.0), 4.0, 0.25, 0),             # less than one group
    (1, (9.0, 9.0, 9.0), 4.0, 0.25, 0),              # a single atom: no pairs
])
def test_pair_hist_symmetric_vs_oracle(ops, n, L, rc, ddr, flags):
    from mdproptools_b200._lib import bin_edges
    rng = np.random.default_rng(n * 7 + flags)
    pos, typ = _rand_box(rng, n, L, 3)
    rel = np.array([[1, 1], [1, 2], [3, 2], [2, 3]])
    nb = int(rc / ddr)
    full, part = O.rdf_loop(typ, pos[0], pos[1], pos[2], rel, L, rc, ddr, nb, nthreads=0)
    cls = (typ.astype(np.int64) - 1).astype(np.int32)       # 3 classes, no 'other'
    edges = bin_edges(ddr, nb)
    hist = ops.pair_hist(_dev(pos[None]), _dev(cls), 3, [L], O.rcut_sq(rc), edges, ddr, flags=flags)
    w = [np.full(6, 2)]
    for a, b in rel:
        r = np.zeros(6, dtype=np.int64)
        r[ops.sym_row(a - 1, b - 1, 3)] = 2 if a == b else 1
        w.append(r)
    red = ops.hist_reduce(hist, np.stack(w)).cpu().numpy()[0]
    assert np.array_equal(red[0], full)
    assert np.array_equal(red[1:], part)
    assert int(hist.sum().item()) * 2 == int(full.sum())


@pytest.mark.parametrize("n,L,rc,ddr,nb,ncls,why", [
    (2500, (40.0, 38.0, 36.0), 7.3, 0.05, None, 2, "r_cut/ddr = 146 exactly representable or not"),
    (2500, (40.0, 38.0, 36.0), 5.03, 0.1, None, 2, "r_cut/ddr not an integer, edge[nbins] < rcut2 (index nbins dropped)"),
    (2500, (40.0, 38.0, 36.0), 4.99, 0.1, 50, 2, "edge[nbins] > rcut2: the explicit rsq < rcut2 test is needed, all-fp64 kernel"),
    (1500, (30.0, 30.0, 30.0), 6.0, 0.001, None, 2, "6000 bins: edge table outside shared memory in the all-fp64 kernel"),
    (1500, (30.0, 30.0, 30.0), 6.0, 6.0, None, 2, "a single bin"),
    (2500, (40.0, 38.0, 36.0), 6.0, 1.5, None, 64, "2080 rows x 4 bins: the fp32 kernel's histogram does not fit in shared memory"),
])
def test_pair_hist_binning_paths_agree_with_oracle(ops, n, L, rc, ddr, nb, ncls, why):
    """The uniform-bin histogram has two device paths, the fp32-filtered kernel (flags 0) and the all-fp64 kernel's hit
    queue (MDP_PAIR_F64); both must give the reference's bin(rsq) = int64(sqrt(rsq)/ddr) (rdf_cn.py:68,85) for every
    pair, including the shapes where the library has to fall back to the all-fp64 kernel by itself."""
    from mdproptools_b200._lib import PAIR_F64, bin_edges
    rng = np.random.default_rng(int(rc * 1000) + n)
    pos, typ = _rand_box(rng, n, L, ncls)
    # plant pairs exactly ON bin edges and on the cutoff: x-separated partners at k*ddr and at r_cut
    for k in range(1, 40):
        pos[:, 2 * k] = pos[:, 2 * k + 1]
        pos[0, 2 * k] = pos[0, 2 * k + 1] + (k * ddr if k < 38 else rc)
    nb = int(rc / ddr) if nb is None else nb
    rel = np.array([[1, 1], [1, 2], [2, 2]] + ([[ncls, ncls], [3, ncls - 7]] if ncls > 2 else []))
    full, part = O.rdf_loop(typ, pos[0], pos[1], pos[2], rel, L, rc, ddr, nb, nthreads=0)
    cls = (typ.astype(np.int64) - 1).astype(np.int32)
    edges = bin_edges(ddr, nb)
    rows = ops.sym_rows(ncls)
    w = [np.full(rows, 2)]
    for a, b in rel:
        r = np.zeros(rows, dtype=np.int64)
        r[ops.sym_row(a - 1, b - 1, ncls)] = 2 if a == b else 1
        w.append(r)
    for flags in (0, PAIR_F64):
        for c, nc in ((cls, ncls), (None, 1)):                # multi-class and single-class kernels
            hist = ops.pair_hist(_dev(pos[None]), None if c is None else _dev(c), nc, [L], O.rcut_sq(rc), edges, ddr, flags=flags)
            if c is None:
                assert np.array_equal(hist.cpu().numpy()[0, 0] * 2, full), (why, flags)
            else:
                red = ops.hist_reduce(hist, np.stack(w)).cpu().numpy()[0]
                assert np.array_equal(red[0], full), (why, flags)
                assert np.array_equal(red[1:], part), (why, flags)


@pytest.mark.parametrize("flags", [8, 32])
def test_pair_calls_reject_unknown_flags(ops, flags):
    """Flag bits other than NO_CULL | NO_SORT | TRICLINIC | F64 are an error, not a silent choice of another kernel
    (8 selected a binning variant of the all-fp64 kernel in earlier versions)."""
    from mdproptools_b200._lib import MdpropError, bin_edges
    pos = _dev(np.random.default_rng(5).uniform(0, 10.0, (1, 3, 100)))
    with pytest.raises(MdpropError, match="unknown flag bits"):
        ops.pair_hist(pos, None, 1, [(10.0, 10.0, 10.0)], 9.0, bin_edges(0.1, 30), 0.1, flags=flags)
    with pytest.raises(MdpropError, match="unknown flag bits"):
        ops.pair_list(pos, pos, [(10.0, 10.0, 10.0)], 0.0, 9.0, 0, flags=flags)


def test_pair_hist_multiframe_and_per_frame_boxes(ops):
    from mdproptools_b200._lib import bin_edges
    rng = np.random.default_rng(11)
    F, n = 5, 1500
    Ls = [(30.0 + k, 28.0, 33.0 - k) for k in range(F)]
    pos = np.stack([rng.uniform(0, 1, (3, n)) * np.asarray(L)[:, None] for L in Ls])
    nb, ddr, rc = 160, 0.05, 8.0
    edges = bin_edges(ddr, nb)
    hist = ops.pair_hist(_dev(pos), None, 1, Ls, rc * rc, edges, ddr).cpu().numpy()
    for f in range(F):
        full, _ = O.rdf_loop(np.ones(n), pos[f, 0], pos[f, 1], pos[f, 2], np.array([[1, 1]]), Ls[f], rc, ddr, nb, nthreads=0)
        assert np.array_equal(hist[f, 0] * 2, full), f


def test_pair_hist_rectangular_vs_oracle(ops):
    from mdproptools_b200._lib import bin_edges
    rng = np.random.default_rng(3)
    L = (25.0, 27.0, 23.0)
    pa, ta = _rand_box(rng, 1234, L, 3)
    pb, tb = _rand_box(rng, 300, L, 2)
    pb[:, :50] = pa[:, :50]                        # coincident points: rsq == 0 lands in bin 0 (no self exclusion)
    rel = np.array([[1, 1], [2, 2], [3, 1], [1, 2]])
    nb, ddr, rc = 100, 0.1, 10.0
    part = O.rdf_rect(ta, pa[0], pa[1], pa[2], tb, pb[0], pb[1], pb[2], rel, L, rc, ddr, nb, nthreads=0)
    edges = bin_edges(ddr, nb)
    hist = ops.pair_hist(_dev(pa[None]), _dev((ta - 1).astype(np.int32)), 3, [L], rc * rc, edges, ddr,
                         xyz_b=_dev(pb[None]), cls_b=_dev((tb - 1).astype(np.int32)), ncls_b=2)
    w = np.zeros((len(rel), 6), dtype=np.int64)
    for k, (a, b) in enumerate(rel):
        w[k, (a - 1) * 2 + (b - 1)] = 1
    red = ops.hist_reduce(hist, w).cpu().numpy()[0]
    assert np.array_equal(red, part)
    assert part[:, 0].sum() > 0


def _tri_points(rng, n, cell, wrapped=True):
    """n points inside the triclinic cell (lx, ly, lz, xy, xz, yz) -- or, unwrapped, spilling one cell beyond it"""
    lx, ly, lz, xy, xz, yz = cell
    s = rng.uniform(0, 1, (n, 3)) if wrapped else rng.uniform(-0.4, 1.4, (n, 3))
    pos = s[:, 0:1] * np.array([lx, 0, 0]) + s[:, 1:2] * np.array([xy, ly, 0]) + s[:, 2:3] * np.array([xz, yz, lz])
    return np.ascontiguousarray(pos.T)


@pytest.mark.parametrize("n,cell,rc,ddr,flags,wrapped", [
    (1000, (21.0, 22.5, 24.0, 4.2, 2.1, -3.3), 7.0, 0.05, 4, True),
    (3000, (60.0, 40.0, 35.0, 12.0, 6.0, -6.0), 6.0, 0.05, 4, True),       # culling active, uniform image vectors
    (3000, (60.0, 40.0, 35.0, 12.0, 6.0, -6.0), 6.0, 0.05, 4 | 1, True),   # + MDP_PAIR_NO_CULL (per-pair image path)
    (3000, (60.0, 40.0, 35.0, 12.0, 6.0, -6.0), 6.0, 0.05, 4 | 3, True),   # brute force in caller order
    (777, (15.0, 15.0, 15.0, 7.5, -7.5, 7.5), 7.4, 0.1, 4, True),          # extreme tilt, r_cut close to L/2
    (1500, (30.0, 28.0, 26.0, 6.0, 3.0, -4.2), 9.0, 0.05, 4, False),       # unwrapped points: sequential shift semantics
    (257, (9.0, 9.0, 9.0, 1.0, 2.0, 3.0), 12.0, 0.25, 4, True),            # r_cut > L/2
    (31, (9.0, 9.0, 9.0, 1.0, 2.0, 3.0), 4.0, 0.25, 4, True),
    (2000, (30.0, 28.0, 26.0, 0.0, 0.0, 0.0), 9.0, 0.05, 4, True),         # zero tilt: must equal the orthogonal path
])
def test_pair_hist_triclinic_vs_oracle(ops, n, cell, rc, ddr, flags, wrapped):
    """MDP_PAIR_TRICLINIC (extension, defined by oracle.c pair_rsq_tri): bit-exact counts against the CPU restatement."""
    from mdproptools_b200._lib import bin_edges
    rng = np.random.default_rng(n * 13 + flags)
    pos = _tri_points(rng, n, cell, wrapped)
    typ = rng.integers(1, 4, n).astype(np.float64)
    rel = np.array([[1, 1], [1, 2], [3, 2]])
    nb = int(rc / ddr)
    full, part = O.rdf_loop_tri(typ, pos[0], pos[1], pos[2], rel, cell, rc, ddr, nb, nthreads=0)
    cls = (typ.astype(np.int64) - 1).astype(np.int32)
    hist = ops.pair_hist(_dev(pos[None]), _dev(cls), 3, [cell], O.rcut_sq(rc), bin_edges(ddr, nb), ddr, flags=flags)
    w = [np.full(6, 2)]
    for a, b in rel:
        r = np.zeros(6, dtype=np.int64)
        r[ops.sym_row(a - 1, b - 1, 3)] = 2 if a == b else 1
        w.append(r)
    red = ops.hist_reduce(hist, np.stack(w)).cpu().numpy()[0]
    assert np.array_equal(red[0], full)
    assert np.array_equal(red[1:], part)
    if cell[3] == cell[4] == cell[5] == 0.0:
        full_o, _ = O.rdf_loop(typ, pos[0], pos[1], pos[2], rel, cell[:3], rc, ddr, nb, nthreads=0)
        assert np.array_equal(red[0], full_o)


def test_pair_hist_triclinic_rect_and_multiframe(ops):
    from mdproptools_b200._lib import bin_edges
    rng = np.random.default_rng(21)
    F = 3
    cells = [(25.0 + k, 27.0, 23.0 - k, 5.0, -2.0 + k, 4.0) for k in range(F)]
    na, nbp = 1234, 300
    pa = np.stack([_tri_points(rng, na, c) for c in cells])
    pb = np.stack([_tri_points(rng, nbp, c) for c in cells])
    ta = rng.integers(1, 4, na).astype(np.float64)
    tb = rng.integers(1, 3, nbp).astype(np.float64)
    rel = np.array([[1, 1], [2, 2], [3, 1], [1, 2]])
    nb, ddr, rc = 100, 0.1, 10.0
    hist = ops.pair_hist(_dev(pa), _dev((ta - 1).astype(np.int32)), 3, cells, rc * rc, bin_edges(ddr, nb), ddr,
                         xyz_b=_dev(pb), cls_b=_dev((tb - 1).astype(np.int32)), ncls_b=2, flags=4)
    w = np.zeros((len(rel), 6), dtype=np.int64)
    for k, (a, b) in enumerate(rel):
        w[k, (a - 1) * 2 + (b - 1)] = 1
    red = ops.hist_reduce(hist, w).cpu().numpy()
    for f in range(F):
        part = O.rdf_rect_tri(ta, pa[f, 0], pa[f, 1], pa[f, 2], tb, pb[f, 0], pb[f, 1], pb[f, 2], rel, cells[f], rc, ddr, nb,
                              nthreads=0)
        assert np.array_equal(red[f], part), f


def test_pair_list_triclinic_shell(ops):
    rng = np.random.default_rng(22)
    cell = (22.0, 20.0, 19.0, 4.0, -3.0, 2.5)
    pa = _tri_points(rng, 150, cell)
    pb = _tri_points(rng, 900, cell)
    r_in, r_out = 2.0, 6.5
    h = O.shell_mask_tri(pa[0], pa[1], pa[2], pb[0], pb[1], pb[2], cell, r_in, r_out, False)
    lst, _ = ops.pair_list(_dev(pa[None]), _dev(pb[None]), [cell], r_in * r_in, r_out * r_out, 1, flags=4)
    got = np.zeros_like(h)
    l = lst.cpu().numpy()
    got[l[:, 1], l[:, 2]] = 1
    assert len(l) == int(h.sum())
    assert np.array_equal(got, h)


def test_pair_hist_table_mode_counts(ops):
    rng = np.random.default_rng(5)
    L = (18.0, 18.0, 18.0)
    pos, typ = _rand_box(rng, 2000, L, 2)
    rel = np.array([[1, 2], [2, 2], [1, 1]])
    rcs = [3.3, 5.125, 2.0]
    cn = O.cn_loop(typ, pos[0], pos[1], pos[2], rel, L, rcs, nthreads=0)
    rc2 = np.array([r * r for r in rcs])
    thr = np.unique(rc2)
    edges = np.concatenate(([0.0], thr))
    hist = ops.pair_hist(_dev(pos[None]), _dev((typ - 1).astype(np.int32)), 2, [L], float(thr[-1]), edges, 0.0)
    w = np.zeros((3, 3), dtype=np.int64)
    for k, (a, b) in enumerate(rel):
        w[k, ops.sym_row(a - 1, b - 1, 2)] = 2 if a == b else 1
    red = ops.hist_reduce(hist, w, cumulative=True).cpu().numpy()[0]
    upto = np.searchsorted(thr, rc2)
    got = np.array([red[k, upto[k]] for k in range(3)])
    assert np.array_equal(got, cn)


def test_bin_edges_match_reference_formula():
    from mdproptools_b200._lib import bin_edges
    rng = np.random.default_rng(0)
    for ddr, nb in [(0.05, 400), (0.07, 104), (0.1, 3), (0.013, 1000)]:
        e = bin_edges(ddr, nb)
        rsq = rng.uniform(0, (nb * ddr) ** 2 * 1.01, 200000)
        rsq = np.concatenate([rsq, e[1:], np.nextafter(e[1:], 0), np.nextafter(e[1:], np.inf)])
        ref = (np.sqrt(rsq) / ddr).astype(np.int64)
        got = np.searchsorted(e[1:], rsq, side="right")
        assert np.array_equal(np.minimum(ref, nb), got)


# ------------------------------------------------------------------------------------------------
# structural API vs golden outputs of the reference
# ------------------------------------------------------------------------------------------------
def test_calc_atomic_rdf_golden(sample_dir, gold_structural, tmp_path):
    from mdproptools_b200.structural.rdf_cn import calc_atomic_rdf
    f0 = os.path.join(sample_dir, "dump.nvt.0.dump")
    df = calc_atomic_rdf(20, 0.05, 9, MASS, REL, f0, path_or_buff=str(tmp_path / "rdf.csv"))
    assert list(df.columns) == list(gold_structural["atomic_rdf_columns"])
    assert np.array_equal(df.values, gold_structural["atomic_rdf_f0"])          # bit-identical floats
    assert os.path.exists(tmp_path / "rdf.csv")
    df2 = calc_atomic_rdf(20, 0.05, 9, MASS, REL, os.path.join(sample_dir, "dump.nvt.*.dump"), save_mode=False)
    assert np.array_equal(df2.values, gold_structural["atomic_rdf_2frames"])
    df3 = calc_atomic_rdf(12, 0.05, 9, MASS, [[32, 32], [17, 32]], f0, num_mols=NUM_MOLS, num_atoms_per_mol=NUM_ATOMS,
                          save_mode=False)
    assert list(df3.columns) == list(gold_structural["atomic_rdf_altered_columns"])
    assert np.array_equal(df3.values, gold_structural["atomic_rdf_altered_f0"])


def test_calc_atomic_rdf_consistency_error(sample_dir):
    from mdproptools_b200.structural.rdf_cn import calc_atomic_rdf
    with pytest.raises(ValueError, match="Consistency check failed"):
        calc_atomic_rdf(20, 0.05, 8, MASS, REL, os.path.join(sample_dir, "dump.nvt.0.dump"), save_mode=False)


def test_calc_atomic_cn_golden(sample_dir, gold_structural):
    from mdproptools_b200.structural.rdf_cn import calc_atomic_cn
    f0 = os.path.join(sample_dir, "dump.nvt.0.dump")
    df = calc_atomic_cn([2.325, 4.375, 2.375, 13.0], 0.05, 9, MASS, REL, f0, save_mode=False)
    assert list(df.columns) == list(gold_structural["atomic_cn_columns"])
    assert np.array_equal(df.values, gold_structural["atomic_cn_f0"])
    df2 = calc_atomic_cn([2.325, 4.375, 2.375, 13.0], 0.05, 9, MASS, REL, os.path.join(sample_dir, "dump.nvt.*.dump"),
                         save_mode=False)
    assert np.array_equal(df2.values, gold_structural["atomic_cn_2frames"])
    df3 = calc_atomic_cn([4.375, 13.0], 0.05, 9, MASS, [[32, 32], [17, 32]], f0, num_mols=NUM_MOLS,
                         num_atoms_per_mol=NUM_ATOMS, save_mode=False)
    assert np.array_equal(df3.values, gold_structural["atomic_cn_altered_f0"])


def test_molecular_rdf_cn_golden(sample_dir, gold_structural):
    from mdproptools_b200.structural.rdf_cn import calc_molecular_cn, calc_molecular_rdf
    f0 = os.path.join(sample_dir, "dump.nvt.0.dump")
    mrel = [[9, 9, 4], [1, 2, 3]]
    df = calc_molecular_rdf(20, 0.05, 9, MASS, mrel, f0, NUM_MOLS, NUM_ATOMS, save_mode=False)
    ref = gold_structural["molecular_rdf_f0"]
    assert list(df.columns) == list(gold_structural["molecular_rdf_columns"])
    assert np.array_equal(df.values[:, 0], ref[:, 0])
    # molecule centres of mass: sequential fp64 here, BLAS dot in the reference -> a COM within an ulp of a bin
    # edge may move one count (documented); everything else is bit-identical
    assert np.count_nonzero(df.values != ref) <= 4
    cn = calc_molecular_cn([2.325, 3.775, 4.375], 0.05, 9, MASS, mrel, f0, NUM_MOLS, NUM_ATOMS, save_mode=False)
    assert np.allclose(cn.values, gold_structural["molecular_cn_f0"], rtol=0, atol=1e-12)


def test_intermolecular_rdf_golden(mini_dir, gold_dynamical):
    from mdproptools_b200.structural.rdf_cn import calc_intermolecular_rdf
    num_mols = gold_dynamical["mini_num_mols"].tolist()
    df = calc_intermolecular_rdf(20, 0.05, 3, MASS, [[3, 3, 2], [1, 2, 2]], os.path.join(mini_dir, "dump.mini.0.dump"),
                                 num_mols, NUM_ATOMS, save_mode=False)
    ref = gold_dynamical["intermolecular_rdf_mini_f0"]
    assert np.count_nonzero(df.values != ref) <= 4


def test_get_clusters_golden(sample_dir, tmp_path):
    from mdproptools_b200.structural.cluster_analysis import get_clusters
    gold = json.load(open(os.path.join(GOLDEN, "ref_clusters.json")))
    wd = tmp_path / "c1"
    wd.mkdir()
    n = get_clusters(filename=os.path.join(sample_dir, "dump.nvt.*.dump"), atom_type=9, r_cut=2.3, num_mols=NUM_MOLS,
                     num_atoms_per_mol=NUM_ATOMS, full_trajectory=False, frame=1, elements=ELEMENTS,
                     alter_atom_types=False, max_force=0.75, working_dir=str(wd))
    g = gold["frame1_type9"]
    assert n == g["count"] == 33 and g["identical_to_reference_goldens"] == 33
    for name, text in g["files"].items():
        assert open(wd / name).read() == text, name             # byte-identical .xyz files
    wd2 = tmp_path / "c2"
    wd2.mkdir()
    n2 = get_clusters(filename=os.path.join(sample_dir, "dump.nvt.*.dump"), atom_type=32, r_cut=2.3, num_mols=NUM_MOLS,
                      num_atoms_per_mol=NUM_ATOMS, full_trajectory=True, elements=ELEMENTS, alter_atom_types=True,
                      max_force=0.75, working_dir=str(wd2))
    g2 = gold["full_altered32"]
    assert n2 == g2["count"]
    assert sorted(os.listdir(wd2)) == sorted(g2["files"])
    for name, text in g2["files"].items():
        assert open(wd2 / name).read() == text, name


def test_hydration_golden(water_dir, gold_hydration, tmp_path):
    import shutil
    from mdproptools_b200.structural.hydration_number import get_hydration_number
    for f in os.listdir(water_dir):
        shutil.copy(os.path.join(water_dir, f), tmp_path)
    df = get_hydration_number("dump.water.*.dump", cation_type=1, water_type=2, r_cut=5.0,
                              num_mols=gold_hydration["hyd_num_mols"].tolist(),
                              num_atoms_per_mol=gold_hydration["hyd_num_atoms"].tolist(), working_dir=str(tmp_path))
    assert np.array_equal(df["angles_distribution"].values, gold_hydration["hyd_angles"])
    assert df["hydration_factor"].values[0] == gold_hydration["hyd_factor"][0]
    assert os.path.exists(tmp_path / "angles_df.csv")


def test_number_density_golden(slab_dir, gold_density, tmp_path):
    """calc_number_density through the public API against the unmodified reference's DataFrames (bit-identical)."""
    import shutil
    from mdproptools_b200.structural.number_density import calc_number_density
    for f in os.listdir(slab_dir):
        shutil.copy(os.path.join(slab_dir, f), tmp_path)
    g = gold_density
    wd = str(tmp_path)
    df = calc_number_density("dump.slab.*.dump", 1, [2, 3, 1], 0.5, 8.0, "z", working_dir=wd)
    assert list(df.columns) == list(g["nd_pos_cols"]) and np.array_equal(df.values, g["nd_pos"])
    assert os.path.exists(tmp_path / "number_density.csv")
    df = calc_number_density("dump.slab.*.dump", 1, [2, 3], 0.5, -20.0, "z", working_dir=wd, save_mode=False)
    assert np.array_equal(df.values, g["nd_neg"])
    df = calc_number_density("dump.slab.*.dump", 1, [3, 2], 0.25, 6.0, "z", num_mols=g["nd_num_mols"].tolist(),
                             num_atoms_per_mol=g["nd_num_atoms"].tolist(), working_dir=wd, save_mode=False)
    assert np.array_equal(df.values, g["nd_alt"])
    df = calc_number_density("dump.slab.*.dump", 1, [2], 0.5, 12.0, "x", working_dir=wd, save_mode=False)
    assert np.array_equal(df.values, g["nd_x"])


def test_axis_density_kernel_vs_oracle_random(ops):
    """mdp_axis_density on seeded random frames (sizes around the block size, a frame without surface atoms, indices that
    fall outside [-nbins, nbins)) against the numpy definition."""
    rng = np.random.default_rng(11)
    for n, dist, bs in [(1, 5.0, 0.5), (255, 6.0, 0.25), (4097, -9.0, 0.5), (20000, 3.0, 0.1)]:
        F = 3
        x = rng.uniform(-4, 12, (F, n))
        key = rng.integers(1, 5, (F, n)).astype(np.float64)
        key[1][key[1] == 1.0] = 2.0                      # frame 1 has no surface atom
        nb = int(abs(dist) / bs)
        counts, mm = ops.axis_density(_dev(x), _dev(key), 1.0, [2.0, 4.0, 2.0], dist, bs, nb)
        counts, mm = counts.cpu().numpy(), mm.cpu().numpy()
        for f in range(F):
            surf = x[f][key[f] == 1.0]
            want = np.zeros((3, nb), dtype=np.int64)
            if len(surf):
                mn, mx = surf.min(), surf.max()
                assert mm[f, 0] == mn and mm[f, 1] == mx
                xs = x[f] - mn
                for i, j in enumerate([2.0, 4.0, 2.0]):
                    b = xs[(key[f] == j) & (xs < dist)] - (mx - mn) if dist > 0 else xs[(key[f] == j) & (xs > dist)]
                    k = (b / bs).astype(int)
                    k = np.where(k < 0, k + nb, k)
                    np.add.at(want[i], k[(k >= 0) & (k < nb)], 1)
            else:
                assert np.isnan(mm[f]).all()
            assert np.array_equal(counts[f], want), (n, dist, f)


def test_xcorr_fft_equals_direct_kernel(ops, monkeypatch):
    """mdp_xcorr_fft against mdp_xcorr_unbiased and the oracle's long-double direct sum: 1e-10 of max|C| (north star)."""
    import torch
    rng = np.random.default_rng(61)
    for C, T, nlags in [(1, 1, 1), (3, 9, 9), (4, 1000, 1000), (2, 4097, 1500), (5, 50000, 50000)]:
        a = np.cumsum(rng.normal(0, 1, (C, T)), axis=1) * 0.05 + rng.normal(0, 1, (C, T))
        b = a.copy()
        b[C // 2:] = rng.normal(0, 2, (C - C // 2, T))
        monkeypatch.setenv("MDP_XCORR_FFT", "0")
        ref = ops.xcorr_unbiased(_dev(a), _dev(b), nlags).cpu().numpy()
        monkeypatch.setenv("MDP_XCORR_FFT", "1")
        got = ops.xcorr_unbiased(_dev(a), _dev(b), nlags).cpu().numpy()
        for c in range(C):
            scale = np.abs(ref[c]).max() + 1e-300
            assert np.abs(got[c] - ref[c]).max() / scale < 1e-10, (C, T, c)
            if T <= 5000:
                assert np.abs(got[c] - O.xcorr_direct(a[c], b[c])[:nlags]).max() / scale < 1e-10


def test_shell_grid_search_equals_pair_list(ops, monkeypatch):
    """mdp_shell_search against mdp_pair_list (itself pinned to the oracle): same set of (frame, ia, ib) entries for
    wrapped and unwrapped coordinates, both shell modes, per-frame boxes; and the automatic fallback when the radius
    exceeds a third of the box."""
    rng = np.random.default_rng(41)
    F, na, nb = 6, 150, 4000
    Ls = np.stack([rng.uniform(20, 26, F), rng.uniform(19, 24, F), rng.uniform(22, 27, F)], axis=1)
    a = rng.uniform(0, 1, (F, 3, na)) * Ls[:, :, None]
    b = rng.uniform(0, 1, (F, 3, nb)) * Ls[:, :, None]
    b[3:] += rng.integers(-2, 3, (F - 3, 3, nb)) * Ls[3:, :, None]            # unwrapped in the later frames

    def entries(flag, r_in, r_out, mode):
        monkeypatch.setenv("MDP_SHELL_GRID", flag)
        lst, _ = ops.pair_list(_dev(a), _dev(b), Ls, r_in ** 2, r_out ** 2, mode)
        return sorted(map(tuple, lst.cpu().numpy().tolist()))

    for r_in, r_out, mode in [(0.0, 3.0, 1), (1.0, 4.5, 1), (0.0, 3.0, 0)]:
        ref, got = entries("0", r_in, r_out, mode), entries("1", r_in, r_out, mode)
        assert len(ref) > 0 and ref == got, (r_in, r_out, mode)
    assert entries("1", 0.0, 9.0, 1) == entries("0", 0.0, 9.0, 1)               # 9 A > L/3: falls back to the engine

    # dense A (31 points per cell, ~600 candidates per B point): every tile overflows the warp's candidate queue and
    # takes the cell-by-cell path with intermediate drains
    a = rng.uniform(0, 14.0, (1, 3, 2000))
    b = rng.uniform(0, 14.0, (1, 3, 16000))

    def packed(flag):
        monkeypatch.setenv("MDP_SHELL_GRID", flag)
        lst, _ = ops.pair_list(_dev(a), _dev(b), [(14.0, 14.0, 14.0)], 0.0, 9.0, 0)
        l = lst.cpu().numpy().astype(np.int64)
        return np.sort((l[:, 0] * 2000 + l[:, 1]) * 16000 + l[:, 2])

    ref, got = packed("0"), packed("1")
    assert len(ref) > 10 ** 6 and np.array_equal(ref, got)


def test_survival_runs_kernel_equals_popcount_kernel(ops, monkeypatch):
    """mdp_survival_runs against mdp_bitmask_autocorr (itself pinned to the oracle) on the same neighbour lists: dense
    random indicators (many runs, some pairs beyond the run buffer) and persistent ones; several trajectory lengths."""
    import torch
    rng = np.random.default_rng(21)
    for T, na, nb, kind in [(130, 6, 40, "dense"), (1000, 10, 60, "walk"), (2600, 4, 30, "dense"), (5000, 12, 50, "walk")]:
        if kind == "dense":
            h = rng.uniform(size=(T, na, nb)) < 0.5
        else:
            walk = np.cumsum(rng.normal(0, 0.3, (T, na, nb)), axis=0) + rng.normal(0, 1.5, (na, nb))
            h = np.abs(walk) < 1.0
        f, a, b = np.nonzero(h)
        lst = torch.from_numpy(np.stack([f, a, b], axis=1).astype(np.int32)).cuda()
        monkeypatch.setenv("MDP_SURVIVAL_RUNS", "0")
        ref, P = ops.bitmask_autocorr_from_list(lst, nb, T)
        monkeypatch.setenv("MDP_SURVIVAL_RUNS", "1")
        got, P2 = ops.bitmask_autocorr_from_list(lst, nb, T)
        assert P == P2 and torch.equal(ref, got), (T, kind)
        assert np.array_equal(got.cpu().numpy(), O.survival_counts(h.reshape(T, -1).astype(np.uint8)))


def test_device_dump_parser_matches_host_parser(sample_dir, tmp_path):
    """FrameBatches(device_parse=True) against the default host-parsed pipeline: same device batches, same host copies,
    same metadata -- on the real sample frames and on a file whose second frame the device parser must refuse (an
    exponent spelling), which the pipeline answers with the host parser."""
    import torch
    from mdproptools_b200.io.pipeline import FrameBatches
    want = ["id", "type", "x", "y", "z", "q"]
    pat = os.path.join(sample_dir, "dump.nvt.*.dump")
    ref = list(FrameBatches(pat, want, device_parse=False))
    fb = FrameBatches(pat, want, device_parse=True)
    got = list(fb)
    assert fb.device_parsed_frames == sum(len(b.metas) for b in ref) and fb.host_reparsed_frames == 0
    for a, b in zip(got, ref):
        assert [m.timestep for m in a.metas] == [m.timestep for m in b.metas]
        assert [m.box.lattice_lengths() for m in a.metas] == [m.box.lattice_lengths() for m in b.metas]
        assert torch.equal(a.wait(), b.wait()) and torch.equal(a.host, b.host)
    p = tmp_path / "two.dump"
    rows = ["%d 1 %g %g %g" % (i + 1, 0.5 * i, 1.25 * i, 2.0 * i) for i in range(40)]
    body = "\n".join(rows) + "\n"
    head = "ITEM: TIMESTEP\n%d\nITEM: NUMBER OF ATOMS\n40\nITEM: BOX BOUNDS pp pp pp\n0 9\n0 9\n0 9\nITEM: ATOMS id type x y z\n"
    p.write_text(head % 0 + body + head % 10 + body.replace("1.25 ", "1.25e-40 ", 1))     # beyond the exact fast path: host re-parse
    ref = list(FrameBatches(str(p), ["id", "x", "y", "z"], device_parse=False))
    fb = FrameBatches(str(p), ["id", "x", "y", "z"], device_parse=True)
    got = list(fb)
    assert (fb.device_parsed_frames, fb.host_reparsed_frames) == (1, 1)
    for a, b in zip(got, ref):
        assert torch.equal(a.wait(), b.wait()) and torch.equal(a.host, b.host)


# ------------------------------------------------------------------------------------------------
# dynamical API vs golden outputs of the reference
# ------------------------------------------------------------------------------------------------
def test_msd_allatom_golden(mini_dir, gold_dynamical, tmp_path):
    from mdproptools_b200.dynamical.diffusion import Diffusion
    d = Diffusion(timestep=1, units="real", outputs_dir=mini_dir, diff_dir=str(tmp_path))
    msd, msd_all, msd_int = d.get_msd_from_dump("dump.mini.*.dump", msd_type="allatom", avg_interval=True, tao_coeff=4)
    assert list(msd.columns) == list(gold_dynamical["msd_allatom_cols"])
    assert list(msd_all.columns) == list(gold_dynamical["msd_all_allatom_cols"])
    assert list(msd_int.columns) == list(gold_dynamical["msd_int_allatom_cols"])
    assert np.array_equal(msd_all.values, gold_dynamical["msd_all_allatom"])       # per-atom values: bit-identical
    assert np.allclose(msd.values, gold_dynamical["msd_allatom"], rtol=1e-12, atol=0)          # north star: <= 1e-10
    assert np.allclose(msd_int.values, gold_dynamical["msd_int_allatom"], rtol=1e-12, atol=0)
    diff = d.calc_diff(msd, initial_time={0: 1e-9}, final_time={0: 4e-9})
    assert np.allclose(diff.values, gold_dynamical["diff_allatom_window"], rtol=1e-10)
    assert os.path.exists(tmp_path / "diffusion.csv")


def test_msd_com_golden(mini_dir, gold_dynamical, tmp_path):
    from mdproptools_b200.dynamical.diffusion import Diffusion
    num_mols = gold_dynamical["mini_num_mols"].tolist()
    d = Diffusion(timestep=1, units="real", outputs_dir=mini_dir, diff_dir=str(tmp_path))
    msd, msd_all, msd_int = d.get_msd_from_dump("dump.mini.*.dump", msd_type="com", num_mols=num_mols,
                                                num_atoms_per_mol=NUM_ATOMS, mass=MASS, com_drift=True, avg_interval=True,
                                                tao_coeff=4)
    assert list(msd.columns) == list(gold_dynamical["msd_com_cols"])
    assert list(msd_all.columns) == list(gold_dynamical["msd_all_com_cols"])
    assert list(msd_int.columns) == list(gold_dynamical["msd_int_com_cols"])
    # COM sums differ from the reference's BLAS / Kahan order by ~1 ulp of a 50 A coordinate (1e-26 m);
    # squared displacements are ~1e-20 m^2, so the comparison is relative to the largest value of each column
    for got, ref in ((msd.values, gold_dynamical["msd_com"]), (msd_all.values, gold_dynamical["msd_all_com"]),
                     (msd_int.values, gold_dynamical["msd_int_com"])):
        scale = np.abs(ref).max(axis=0)
        assert np.all(np.abs(got - ref) <= 1e-10 * scale)
    diff = d.calc_diff(msd)
    assert np.allclose(diff.values, gold_dynamical["diff_com"], rtol=1e-9)
    msd2, _ = d.get_msd_from_dump("dump.mini.*.dump", msd_type="com", num_mols=num_mols, num_atoms_per_mol=NUM_ATOMS,
                                  mass=MASS, com_drift=False)
    ref = gold_dynamical["msd_com_nodrift"]
    assert np.all(np.abs(msd2.values - ref) <= 1e-10 * np.abs(ref).max(axis=0))


def test_conductivity_golden(mini_dir, gold_dynamical):
    from mdproptools_b200.dynamical.conductivity import Conductivity
    num_mols = gold_dynamical["mini_num_mols"].tolist()
    c = Conductivity("dump.mini.*.dump", num_mols, NUM_ATOMS, volume=49.182348836183905 ** 3, mass=MASS, temp=298.15,
                     timestep=1, units="real", working_dir=mini_dir)
    j = c.get_charge_flux()
    ref = gold_dynamical["cond_flux"]
    assert j.shape == ref.shape
    assert np.max(np.abs(j - ref)) <= 1e-10 * np.abs(ref).max()
    assert np.allclose(c.time, gold_dynamical["cond_time"], rtol=1e-15)
    tot = c.correlate_charge_flux(ref)
    rt = gold_dynamical["cond_tot_flux"]
    assert np.max(np.abs(tot - rt)) <= 1e-10 * np.abs(rt).max()
    integ = c.integrate_charge_flux_correlation(rt)
    ri = gold_dynamical["cond_integral"]
    assert np.max(np.abs(integ - ri)) <= 1e-10 * np.abs(ri).max()
    assert np.allclose(c.green_kubo(ri[:, -1]), gold_dynamical["cond_green_kubo_of_last"], rtol=1e-14)
    a, b = ref[0, 1], ref[1, 2]
    assert np.max(np.abs(Conductivity.correlate(a, b) - O.correlate_fft(a, b))) <= 1e-12 * np.abs(O.correlate_fft(a, b)).max()


def test_viscosity_golden(visc_dir, gold_dynamical):
    import glob as _glob
    import mdproptools_b200.dynamical.viscosity as vmod
    from mdproptools_b200.dynamical.viscosity import Viscosity
    v = Viscosity("log.visc_*", cutoff_time=500, volume=40.0 ** 3, temp=298.15, timestep=1, acf_method="wkt", units="real",
                  working_dir=visc_dir)
    real = vmod.glob.glob
    vmod.glob.glob = lambda p: sorted(real(p))       # the fixture was generated with sorted replicate order
    try:
        visc_avg, visc_data, acf_data, tvec = v.calc_avg_visc(output_all_data=True)
    finally:
        vmod.glob.glob = real
    ra, rv, rg = gold_dynamical["visc_acf"], gold_dynamical["visc_data"], gold_dynamical["visc_avg"]
    assert np.max(np.abs(np.array(acf_data) - ra)) <= 1e-10 * np.abs(ra).max()
    assert np.max(np.abs(np.array(visc_data) - rv)) <= 1e-10 * np.abs(rv).max()
    assert np.max(np.abs(np.array(visc_avg) - rg)) <= 1e-10 * np.abs(rg).max()
    assert np.array_equal(tvec, gold_dynamical["visc_time"])
    s = gold_dynamical["visc_acf_bruteforce_first200_in"]
    got = Viscosity.autocorrelate(s, "brute_force")
    ref = gold_dynamical["visc_acf_bruteforce_first200"]
    assert np.max(np.abs(got - ref)) <= 1e-12 * np.abs(ref).max()


def test_residence_time_golden(mini_dir, gold_dynamical, tmp_path):
    from mdproptools_b200.dynamical.residence_time import ResidenceTime
    num_mols = gold_dynamical["mini_num_mols"].tolist()
    rt = ResidenceTime([[0, 2.0], [1.9, 2.2], [0, 3.2]], [[32, 32, 1], [1, 27, 1]],
                       os.path.join(mini_dir, "dump.mini.*.dump"), dt=1, num_mols=num_mols, num_atoms_per_mol=NUM_ATOMS,
                       working_dir=str(tmp_path))
    rt.calc_auto_correlation()
    assert list(rt.corr_df.columns) == list(gold_dynamical["residence_cols"])
    # integer counts are exact here; the reference's FFT autocovariance carries ~1e-15 round-off
    assert np.allclose(rt.corr_df.values, gold_dynamical["residence_corr"], rtol=0, atol=1e-12)
    assert os.path.exists(tmp_path / "auto_correlation.csv")


# ------------------------------------------------------------------------------------------------
# kernels vs oracle on synthetic inputs
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [4096, 4097, 1, 2049])
def test_msd_single_origin_kernel(ops, n):
    rng = np.random.default_rng(n)
    T = 7
    traj = np.cumsum(rng.normal(0, 0.1, (T, 3, n)), axis=0) + rng.uniform(0, 50, (1, 3, n))
    per_atom, mean = O.msd_single_origin(traj, 2, 1e-10)
    t = _dev(traj)
    sums, pa = ops.msd_single_origin(t, t[2].contiguous(), 1e-10, per_atom=True)
    assert np.array_equal(pa.cpu().numpy(), per_atom)                           # per-atom values bit-identical
    assert np.allclose(sums[:, 0].cpu().numpy() / n, mean, rtol=1e-13, atol=0)
    off = np.array([0, n // 3, n // 3, n])                                        # ragged groups incl. an empty one
    gs, _ = ops.msd_single_origin(t, t[2].contiguous(), 1e-10, group_off=off)
    gs = gs.cpu().numpy()
    for g in range(3):
        ref = per_atom[:, :, off[g]:off[g + 1]].sum(axis=2)
        assert np.allclose(gs[:, g], ref, rtol=1e-13, atol=0)


def test_msd_interval_and_all_origins(ops):
    rng = np.random.default_rng(8)
    T, n = 33, 700
    traj = np.cumsum(rng.normal(0, 0.1, (T, 3, n)), axis=0)
    got = ops.msd_interval(_dev(traj[::4]), 1e-10, 1).cpu().numpy()
    assert np.allclose(got, O.msd_interval(traj, 1e-10, 4), rtol=1e-13, atol=0)
    lag = 20
    sums = ops.msd_all_origins(_dev(traj), lag).cpu().numpy()[:, 0]
    norm = (T - np.arange(lag))[:, None] * n
    ref = O.msd_all_origins(traj, lag)
    assert np.allclose(sums[1:] / norm[1:], ref[1:], rtol=1e-12, atol=0)
    assert np.all(sums[0] == 0)


@pytest.mark.parametrize("T,n,lag,groups", [
    (33, 700, 20, None),                       # one time tile, edge path only
    (300, 70, 300, None),                      # full window: several time tiles and lag blocks, 3 atom blocks (ragged)
    (517, 33, 130, [0, 1, 20, 33]),            # groups with ragged atom blocks (1 atom, 19 atoms, 13 atoms)
    (1300, 40, 1100, None),                    # more lags than one launch holds (MW_WCAP = 1024)
    (97, 1, 97, None),                         # a single atom
])
def test_msd_all_origins_windowed(ops, T, n, lag, groups):
    """Extension (no reference implementation; oracle.c orc_msd_all_origins is the definition): 1e-10 relative."""
    rng = np.random.default_rng(T + n)
    traj = 50.0 + np.cumsum(rng.normal(0, 0.1, (T, 3, n)), axis=0)
    scale = 1e-10
    sums = ops.msd_all_origins(_dev(traj), lag, scale, group_off=groups).cpu().numpy()     # [lag, G, 4]
    offs = groups if groups is not None else [0, n]
    assert sums.shape == (lag, len(offs) - 1, 4)
    for g in range(len(offs) - 1):
        a0, a1 = offs[g], offs[g + 1]
        ref = O.msd_all_origins(np.ascontiguousarray(traj[:, :, a0:a1]), lag) * scale * scale
        norm = (T - np.arange(lag))[:, None] * (a1 - a0)
        got = sums[:, g] / norm
        assert np.all(sums[0, g] == 0)
        assert np.allclose(got[1:], ref[1:], rtol=1e-10, atol=0), (g, np.abs(got[1:] / ref[1:] - 1).max())
    # accumulate semantics: a second call adds
    out = ops.msd_all_origins(_dev(traj), lag, scale, group_off=groups)
    ops.msd_all_origins(_dev(traj), lag, scale, group_off=groups, out=out)
    assert np.allclose(out.cpu().numpy(), 2 * sums, rtol=1e-14, atol=0)


def test_segment_com_kernel(ops):
    rng = np.random.default_rng(2)
    sizes = rng.integers(1, 17, 500)
    off = np.concatenate(([0], np.cumsum(sizes)))
    n = off[-1]
    attr = rng.normal(0, 10, (3, 2, n))
    w = rng.uniform(1, 30, n)
    q = rng.normal(0, 1, n)
    out, wsum, qsum = ops.segment_com(_dev(attr), _dev(w), _dev(off.astype(np.int32)), extra=_dev(q))
    ref = np.empty((3, 2, 500))
    for s in range(500):
        ws = 0.0
        for a in range(off[s], off[s + 1]):
            ws += w[a]
        for f in range(3):
            for c in range(2):
                acc = 0.0
                for a in range(off[s], off[s + 1]):
                    acc += attr[f, c, a] * w[a]
                ref[f, c, s] = acc / ws
    assert np.array_equal(out.cpu().numpy(), ref)          # sequential unfused fp64 in atom order: bit-identical
    assert np.allclose(wsum.cpu().numpy(), np.add.reduceat(w, off[:-1]), rtol=1e-14)
    assert np.allclose(qsum.cpu().numpy(), np.add.reduceat(q, off[:-1]), rtol=0, atol=1e-13)


@pytest.mark.parametrize("T", [1, 2, 127, 128, 129, 2048, 5000])
def test_xcorr_kernel_vs_long_double(ops, T, monkeypatch):
    monkeypatch.setenv("MDP_XCORR_FFT", "0")      # the direct kernel (series of >= 2048 steps take the FFT route by default)
    rng = np.random.default_rng(T)
    a = rng.normal(0, 1, (3, T))
    b = rng.normal(0, 1, (3, T))
    got = ops.xcorr_unbiased(_dev(a), _dev(b)).cpu().numpy()
    for c in range(3):
        ref = O.xcorr_direct(a[c], b[c])
        assert np.max(np.abs(got[c] - ref)) <= 1e-13 * max(1.0, np.abs(ref).max()), (T, c)
    if T > 4:
        part = ops.xcorr_unbiased(_dev(a), _dev(b), nlags=T // 2).cpu().numpy()
        assert np.array_equal(part, got[:, :T // 2])


def test_cumtrapz_kernel(ops):
    rng = np.random.default_rng(4)
    y = rng.normal(0, 1, (3, 5001))
    for lead in (True, False):
        got = ops.cumtrapz(_dev(y), 0.37, 2.5, leading_zero=lead).cpu().numpy()
        ref = np.stack([2.5 * O.cumtrapz(r, 0.37, lead) for r in y])
        assert np.allclose(got, ref, rtol=0, atol=1e-12 * np.abs(ref).max())
    # integer y, dx = 2^-3 and scale 2: every partial sum is exact, so the result is the int64 running sum bit for bit,
    # at the lengths around the 1024-thread split (1025 trapezoids: one thread takes two) and at the long end
    from tests import exact_series as ES
    for T in (2, 3, 1024, 1025, 1026, 2049, 10 ** 6 + 1, 10 ** 7):
        y = ES.ou_series(rng, 3, T, tau=100.0, sigma=1000.0)
        for lead in (True, False):
            got = ops.cumtrapz(_dev(y.astype(np.float64)), 0.125, 2.0, leading_zero=lead).cpu().numpy()
            assert np.array_equal(got, ES.cumtrapz_exact(y, 0.125, 2.0, lead)), (T, lead)


def test_pair_list_and_bitmask_autocorr(ops):
    rng = np.random.default_rng(6)
    T, na, nb_ = 70, 40, 300
    L = (14.0, 15.0, 16.0)
    base_a = rng.uniform(0, 1, (3, na)) * np.asarray(L)[:, None]
    base_b = rng.uniform(0, 1, (3, nb_)) * np.asarray(L)[:, None]
    xa = np.stack([base_a + rng.normal(0, 0.15, base_a.shape) for _ in range(T)])
    xb = np.stack([base_b + rng.normal(0, 0.15, base_b.shape) for _ in range(T)])
    r_in, r_out = 1.0, 3.0
    lst, rsq = ops.pair_list(_dev(xa), _dev(xb), [L] * T, r_in ** 2, r_out ** 2, shell_mode=1, want_rsq=True)
    h = np.stack([O.shell_mask(xa[t, 0], xa[t, 1], xa[t, 2], xb[t, 0], xb[t, 1], xb[t, 2], L, r_in, r_out, False)
                  for t in range(T)])
    got = np.zeros_like(h)
    l = lst.cpu().numpy()
    got[l[:, 0], l[:, 1], l[:, 2]] = 1
    assert len(l) == h.sum() and np.array_equal(got, h)
    # rsq values are the reference's
    k = 0
    ref_rsq = O.calc_rsq(xa[l[k, 0], :, l[k, 1]], xb[l[k, 0], 0], xb[l[k, 0], 1], xb[l[k, 0], 2], L)[l[k, 2]]
    assert rsq.cpu().numpy()[k] == ref_rsq
    cnt, npairs = ops.bitmask_autocorr_from_list(lst, nb_, T)
    ref_cnt = O.survival_counts(h.reshape(T, -1))
    assert np.array_equal(cnt.cpu().numpy(), ref_cnt)
    assert npairs == int((h.sum(axis=0) > 0).sum())


def test_ols_sums_kernel(ops):
    rng = np.random.default_rng(9)
    t = np.linspace(0, 5e-9, 1001)
    y = np.stack([3e-9 * t + rng.normal(0, 1e-20, t.size), 1e-10 * t])
    s = ops.ols_sums(_dev(t), _dev(y), 10, 900).cpu().numpy()
    for c in range(2):
        tt, yy = t[10:900], y[c, 10:900]
        assert np.allclose(s[c], [np.dot(tt, tt), np.dot(tt, yy), np.dot(yy, yy)], rtol=1e-13)


def test_large_frame_properties(ops):
    """Full-size single frame of the headline workload (100k atoms): checks that do not need the oracle to
    finish -- symmetry of the total count under culling on/off and a checksum against brute-force (no cull)."""
    from mdproptools_b200._lib import bin_edges
    rng = np.random.default_rng(20261017)
    n, L = 100_000, (167.19, 167.19, 167.19)
    pos = rng.uniform(0, 1, (3, n)) * np.asarray(L)[:, None]
    edges = bin_edges(0.05, 400)
    x = _dev(pos[None])
    h1 = ops.pair_hist(x, None, 1, [L], 400.0, edges, 0.05)
    h2 = ops.pair_hist(x, None, 1, [L], 400.0, edges, 0.05, flags=1)
    assert torch.equal(h1, h2)
    # expected number of pairs inside the cutoff for a uniform gas: N(N-1)/2 * (4/3 pi rc^3 / V)
    expect = n * (n - 1) / 2 * (4 / 3 * np.pi * 20 ** 3) / np.prod(L)
    assert abs(int(h1.sum().item()) - expect) < 5 * np.sqrt(expect)


# ------------------------------------------------------------------------------------------------
# mic="triclinic" through the public API (extension; oracle-defined)
# ------------------------------------------------------------------------------------------------
def _write_triclinic_dump(path, rng, nframes, n, cell):
    lx, ly, lz, xy, xz, yz = cell
    xlo, ylo, zlo = -1.0, 0.5, 2.0
    # LAMMPS writes the bounding box of the tilted cell (pymatgen undoes it, oracle.read_dumps restates that)
    xs = (0.0, xy, xz, xy + xz)
    with open(path, "w") as f:
        for t in range(nframes):
            pos = _tri_points(rng, n, cell) + np.array([[xlo], [ylo], [zlo]])
            ids = rng.permutation(n) + 1
            f.write(f"ITEM: TIMESTEP\n{t * 100}\nITEM: NUMBER OF ATOMS\n{n}\n")
            f.write("ITEM: BOX BOUNDS xy xz yz pp pp pp\n")
            f.write(f"{xlo + min(xs)!r} {xlo + lx + max(xs)!r} {xy!r}\n")
            f.write(f"{ylo + min(0.0, yz)!r} {ylo + ly + max(0.0, yz)!r} {xz!r}\n")
            f.write(f"{zlo!r} {zlo + lz!r} {yz!r}\n")
            f.write("ITEM: ATOMS id type x y z\n")
            for k, i in enumerate(ids):
                f.write(f"{i} {1 + (i % 3)} {float(pos[0, k])!r} {float(pos[1, k])!r} {float(pos[2, k])!r}\n")


def test_calc_atomic_rdf_triclinic_api(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mdproptools_b200.structural import rdf_cn
    rng = np.random.default_rng(31)
    cell = (24.0, 22.0, 20.0, 4.8, 2.4, -3.3)
    p = str(tmp_path / "tri.dump")
    _write_triclinic_dump(p, rng, 3, 1500, cell)
    rel = [[1, 2, 3], [1, 3, 3]]
    frames = list(O.read_dumps(p))
    for mic in ("triclinic", "reference"):
        want = O.atomic_rdf(frames, 8.0, 0.05, rel, mic=mic)
        df = rdf_cn.calc_atomic_rdf(8.0, 0.05, 3, [1.0, 2.0, 3.0], rel, p, save_mode=False, mic=mic)
        assert np.array_equal(df.values, want), mic          # equal integer counts -> bit-identical floats
    a = rdf_cn.calc_atomic_rdf(8.0, 0.05, 3, [1.0, 2.0, 3.0], rel, p, save_mode=False, mic="triclinic").values
    b = rdf_cn.calc_atomic_rdf(8.0, 0.05, 3, [1.0, 2.0, 3.0], rel, p, save_mode=False).values
    assert not np.array_equal(a, b)                           # the tilted cell is where the two conventions differ
    # a uniform fluid must give g(r) ~ 1 with the true image and the true volume
    assert abs(a[40:, 1].mean() - 1.0) < 0.02
    with pytest.raises(ValueError):
        rdf_cn.calc_atomic_rdf(8.0, 0.05, 3, [1.0, 2.0, 3.0], rel, p, save_mode=False, mic="nearest")


# ------------------------------------------------------------------------------------------------
# config C1 at full length (101 frames): known answers of the UNMODIFIED reference, SURVEY.md 8(c)
# ------------------------------------------------------------------------------------------------
C1_REL = [[9, 9, 9, 9], [1, 4, 6, 9]]


def _sha(df):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(df.values, dtype=np.float64).tobytes()).hexdigest()


def test_c1_full_atomic_rdf_kat(c1_dir, tmp_path):
    """calc_atomic_rdf over all 101 frames: the reference's DataFrame bit for bit (486 s on one core there)."""
    from mdproptools_b200.structural.rdf_cn import calc_atomic_rdf
    df = calc_atomic_rdf(20, 0.05, 9, MASS, C1_REL, os.path.join(c1_dir, "dump.nvt.*.dump"), path_or_buff=str(tmp_path / "rdf.csv"))
    assert df.shape == (400, 6)
    assert list(df.columns) == [r"r ($\AA$)", "g_full(r)", "g_9-1", "g_9-4", "g_9-6", "g_9-9"]
    assert df.iloc[40, 1:].tolist() == [1.2618212188545432, 28.56133801821835, 0.0, 89.25671173472328, 0.0]
    assert df.iloc[200, 1:].tolist() == [0.9977710416003582, 1.0339062617991446, 0.5995108632667641, 1.076978443654223,
                                         1.986950289684134]
    assert df.iloc[399, 1:].tolist() == [0.999904654025423, 1.0075979643460262, 0.9772216479509167, 0.9238303989734666,
                                         0.992322203217268]
    assert _sha(df) == "b418f238f5e58393edbe59e8419c8afe1053dada1af6959fa589ce88cfa9ccfc"


def test_c1_full_atomic_cn_kat(c1_dir, tmp_path):
    """calc_atomic_cn over all 101 frames (534 s on one core in the reference)."""
    from mdproptools_b200.structural.rdf_cn import calc_atomic_cn
    df = calc_atomic_cn([2.325, 4.375, 2.375, 13.0], 0.05, 9, MASS, C1_REL, os.path.join(c1_dir, "dump.nvt.*.dump"),
                        path_or_buff=str(tmp_path / "cn.csv"))
    got = {c: float(df[c].iloc[0]) for c in df.columns}
    assert got["cn_9-1"] == 4.322232223222324 and got["cn_9-4"] == 1.0768076807680773
    assert got["cn_9-6"] == 1.6762676267626753 and got["cn_9-9"] == 3.0483048304830462
    assert _sha(df) == "0ad5461c6508bf07e42aeb21004303b189fbf2a1ed756a2a01fc4ce1b488bb1e"


def test_c1_full_diffusion_kat(c1_dir, tmp_path):
    """MSD + diffusion over all 101 frames: the survey's MSD values of the unmodified reference and the diffusion table
    printed in the reference's example notebook (cell 17)."""
    from mdproptools_b200.dynamical.diffusion import Diffusion
    d = Diffusion(timestep=1, units="real", outputs_dir=c1_dir, diff_dir=str(tmp_path))
    msd, msd_all = d.get_msd_from_dump("dump.nvt.*.dump", msd_type="allatom")[:2]
    assert abs(msd["msd"].iloc[1] / 4.710123052923229e-19 - 1) < 1e-12
    assert abs(msd["msd"].iloc[100] / 3.6239421444312684e-17 - 1) < 1e-12
    msd, msd_all, msd_int = d.get_msd_from_dump("dump.nvt.*.dump", msd_type="com", num_mols=NUM_MOLS, num_atoms_per_mol=NUM_ATOMS,
                                                mass=MASS, com_drift=True, avg_interval=True, tao_coeff=4)
    assert abs(msd["msd1"].iloc[100] / 3.918949266310726e-17 - 1) < 1e-10
    assert abs(msd["msd3"].iloc[100] / 5.32844116327746e-18 - 1) < 1e-10
    diff = d.calc_diff(msd, diff_names=["dme", "tfsi", "mg"])
    want = {"dme": (1.330522e-09, 2.164493e-12, 0.999735), "tfsi": (1.976415e-10, 2.162102e-12, 0.988174),
            "mg": (1.585219e-10, 1.821829e-12, 0.986964)}
    for name, (dv, sd, r2) in want.items():
        row = diff.loc[name]
        assert f"{row['diffusion (m2/s)']:.6e}" == f"{dv:.6e}", (name, row.tolist())       # all 7 printed digits
        assert f"{row['std']:.6e}" == f"{sd:.6e}" and f"{row['R2']:.6f}" == f"{r2:.6f}", (name, row.tolist())
    dist = d.get_diff_dist(msd_int, dump_freq=50000, dimension=3, tao_coeff=4)
    assert "diff" in dist.columns and np.all(np.isfinite(dist["diff"].values))


# ------------------------------------------------------------------------------------------------
# N ranks == 1 rank under NCCL (needs >= 2 GPUs on the box; the driver's 1-GPU run skips it, tools/gpu_nrank_check.sh runs it)
# ------------------------------------------------------------------------------------------------
def test_nrank_equals_1rank_under_nccl(tmp_path):
    """bench.py at reduced sizes on 1 GPU and under torchrun on 2 (and 4) GPUs: the same RDF histograms (sha256 of all
    per-frame integer histograms), the same residence survival counts (sha256), the same MSD to 1e-12, the same DataFrame
    from dump files whose reads are sharded over the ranks -- frames, atoms and central atoms are only re-distributed,
    never re-computed differently."""
    import json
    import subprocess
    import sys
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs at least 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    small = ["--steps", "2", "--warmup", "1", "--frames", "24", "--msd-atoms", "400000", "--msd-frames", "200", "--gk-steps", "20000",
             "--gk-flux-frames", "1000", "--res-frames", "400", "--c5-frames", "100", "--skip-cpu", "--skip-msd-window",
             "--files-leg", "--files-copies", "2"]

    def run(n):
        cmd = ([sys.executable, "bench.py", "--gpus", "1"] if n == 1 else
               [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
                "--master-port", str(29511 + n), "bench.py", "--gpus", str(n)]) + small
        r = subprocess.run(cmd, cwd=root, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        return json.loads(r.stdout.strip().splitlines()[-1])

    one = run(1)
    for n in [k for k in (2, 4) if k <= ngpu]:
        many = run(n)
        assert many["n_gpus"] == n and many["scaling"] == "strong"
        assert many["hist_sha256"] == one["hist_sha256"]                                   # RDF counts: exact
        assert many.get("nrank_equals_1rank") is True
        assert many["residence"]["cnt_sha256"] == one["residence"]["cnt_sha256"]             # survival counts: exact
        assert many["residence"]["neighbour_entries"] == one["residence"]["neighbour_entries"]
        assert abs(many["msd"]["msd_last_frame"] / one["msd"]["msd_last_frame"] - 1) < 1e-12   # fp64 all-reduce order only
        a, b = many["green_kubo"]["charge_flux"]["abs_flux_sum"], one["green_kubo"]["charge_flux"]["abs_flux_sum"]
        assert abs(a / b - 1) < 1e-12
        # the reference's entry point on files, reads sharded over the ranks, text parsed on each rank's device
        assert many["rdf_from_files"]["df_sha256"] == one["rdf_from_files"]["df_sha256"] and many["rdf_from_files"]["ranks"] == n
        if "c1" in one:
            assert many.get("c1_sha256") is True and one.get("c1_sha256") is True


def test_api_nrank_equals_1rank_under_nccl(sample_dir, mini_dir, water_dir, slab_dir, visc_dir, tmp_path, request):
    """Every file-based public entry point (RDF/CN atomic, molecular, intermolecular; clusters with their .xyz files;
    hydration; number density; residence time; MSD all-atom and COM; charge flux and its correlations; viscosity; C1 at full
    length when the fixture is there) in one process and under torchrun on 2 GPUs, on the golden fixtures: results from
    integer counts must be identical, fp64 reductions whose order depends on the rank count equal to 1e-12
    (tests/nccl_api_worker.py).  The single-process results are what the golden tests pin to the reference."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    c1_path = os.path.join(root, "tests", "golden_large", "c1_frames.tar.gz")
    fixtures = [sample_dir, mini_dir, water_dir, slab_dir, visc_dir]
    if os.path.exists(c1_path):
        fixtures.append(request.getfixturevalue("c1_dir"))
    res = {}
    for n in (1, 2):
        out = tmp_path / f"n{n}"
        out.mkdir()
        cmd = ([sys.executable] if n == 1 else
               [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
                "--master-port", str(29561 + n)]) + [os.path.join(root, "tests", "nccl_api_worker.py"), str(out)] + fixtures
        r = subprocess.run(cmd, cwd=root, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        res[n] = np.load(out / "results.npz")
    assert sorted(res[1].files) == sorted(res[2].files) and len(res[1].files) >= 20
    for k in res[1].files:
        a, b = res[1][k], res[2][k]
        assert a.shape == b.shape, k
        if k.startswith("x_"):
            assert np.array_equal(a, b), k
        else:
            scale = np.abs(a).max() + 1e-300
            assert np.max(np.abs(a - b)) <= 1e-12 * scale, (k, float(np.max(np.abs(a - b)) / scale))


# ------------------------------------------------------------------------------------------------
# device epilogues of the cutoff searches (csrc/epilogue.cu) against numpy restatements of the reference's host code
# ------------------------------------------------------------------------------------------------
def _rand_list(rng, F, na, nb, m):
    lst = np.stack([rng.integers(0, F, m), rng.integers(0, na, m), rng.integers(0, nb, m)], axis=1).astype(np.int32)
    return np.unique(lst, axis=0)[rng.permutation(len(np.unique(lst, axis=0)))]          # distinct entries, shuffled


def test_list_group_kernel(ops):
    import torch
    rng = np.random.default_rng(5)
    for F, na, nb, m in [(1, 1, 5, 3), (4, 7, 300, 2000), (3, 50, 40, 5000), (2, 3, 10, 0)]:
        lst = _rand_list(rng, F, na, nb, m) if m else np.zeros((0, 3), dtype=np.int32)
        seg_off, key, perm = ops.list_group(torch.from_numpy(lst).cuda(), na, F)
        seg_off, key, perm = seg_off.cpu().numpy(), key.cpu().numpy(), perm.cpu().numpy()
        order = np.lexsort((lst[:, 2], lst[:, 1], lst[:, 0])) if len(lst) else np.zeros(0, dtype=np.int64)
        assert np.array_equal(perm, order) and np.array_equal(key, lst[order, 2])
        counts = np.bincount(lst[:, 0].astype(np.int64) * na + lst[:, 1], minlength=F * na) if len(lst) else np.zeros(F * na, dtype=np.int64)
        assert np.array_equal(seg_off, np.concatenate(([0], np.cumsum(counts))))


def test_hydration_count_kernel(ops):
    """cosines bit-identical to the numpy expressions of hydration_number.py:27-30 / rdf_cn.py:46-55, counters exact."""
    import torch
    rng = np.random.default_rng(8)
    F, ncat, nw = 3, 9, 120
    L = np.array([[14.0, 15.0, 13.5], [14.2, 15.1, 13.4], [13.9, 14.8, 13.6]])
    cat = rng.uniform(0, 1, (F, 3, ncat)) * L[:, :, None]
    o = rng.uniform(0, 1, (F, 3, nw)) * L[:, :, None]
    h1 = o + rng.normal(0, 0.6, o.shape)
    h2 = o + rng.normal(0, 0.6, o.shape)
    lst = _rand_list(rng, F, ncat, nw, 900)
    cos, seg_off, counts = ops.hydration_count(torch.from_numpy(lst).cuda(), _dev(cat), _dev(o), _dev(h1), _dev(h2), L, -0.72)
    cos, seg_off, counts = cos.cpu().numpy(), seg_off.cpu().numpy(), counts.cpu().numpy()
    order = np.lexsort((lst[:, 2], lst[:, 1], lst[:, 0]))
    f, ia, ib = lst[order].T
    d = np.stack([cat[f, a, ia] - o[f, a, ib] for a in range(3)], axis=1)
    for a in range(3):
        l = L[f, a]
        cond = (d[:, a] > l / 2) | (d[:, a] < -l / 2)
        d[cond, a] = d[cond, a] - np.sign(d[cond, a]) * l[cond]
    v = np.stack([(h1[f, a, ib] + h2[f, a, ib]) - 2 * o[f, a, ib] for a in range(3)], axis=1)
    want = np.sum(d * v, axis=1) / (np.linalg.norm(d, axis=1) * np.linalg.norm(v, axis=1))
    assert np.array_equal(cos, want)
    seg = f.astype(np.int64) * ncat + ia
    assert np.array_equal(counts[:, :, 0].ravel(), np.bincount(seg, minlength=F * ncat))
    assert np.array_equal(counts[:, :, 1].ravel(), np.bincount(seg[want < -0.72], minlength=F * ncat))


def test_cluster_members_kernel(ops):
    """molecule completion + signed-component force filter (cluster_analysis.py:163-182) against numpy."""
    import torch
    rng = np.random.default_rng(9)
    F, ncen, sizes = 3, 11, rng.integers(1, 17, 60)
    seg_off = np.concatenate(([0], np.cumsum(sizes))).astype(np.int32)
    n, nmol = int(seg_off[-1]), len(sizes)
    mol_of_atom = np.repeat(np.arange(nmol), sizes).astype(np.int32)
    force = rng.normal(0, 40.0, (F, 3, n))
    const, max_force = 0.043363 / 16, 0.05
    lst = _rand_list(rng, F, ncen, n, 1500)
    so, mols, cnt = ops.cluster_members(torch.from_numpy(lst).cuda(), ncen, _dev(force), torch.from_numpy(seg_off).cuda(),
                                        torch.from_numpy(mol_of_atom).cuda(), const, max_force)
    so, mols, cnt = so.cpu().numpy(), mols.cpu().numpy(), cnt.cpu().numpy()
    fsum = np.stack([[np.array([force[f, a, seg_off[m]:seg_off[m + 1]].sum() for m in range(nmol)]) for a in range(3)] for f in range(F)])
    ok = fsum.min(axis=1) * const < max_force                                   # [F, nmol]
    assert 0 < ok.sum() < ok.size
    for f in range(F):
        for c in range(ncen):
            s = f * ncen + c
            atoms = lst[(lst[:, 0] == f) & (lst[:, 1] == c)][:, 2]
            want = np.unique(mol_of_atom[atoms])
            want = want[ok[f, want]]
            assert np.array_equal(mols[so[s]: so[s] + cnt[s]], want), (f, c)


def test_unique_pair_keys_kernel(ops):
    import torch
    rng = np.random.default_rng(12)
    for na, nb, m in [(1, 1, 1), (7, 33, 500), (40, 1000, 20000), (3, 5, 0)]:
        lst = np.stack([rng.integers(0, 50, m), rng.integers(0, na, m), rng.integers(0, nb, m)], axis=1).astype(np.int32)
        got = ops.unique_pair_keys(torch.from_numpy(lst).cuda(), na, nb).cpu().numpy()
        want = np.unique(lst[:, 1].astype(np.int64) * nb + lst[:, 2])
        assert np.array_equal(got, want)


# ------------------------------------------------------------------------------------------------
# k_pair_fast (fp32 filter + fp64 exact path) against k_pair (all fp64) and the oracle over awkward geometries
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["dense", "tiny_cell", "unwrapped", "far_from_origin", "nosort", "many_bins", "coarse_bins", "rect",
                                  "clustered", "multiframe", "huge_groups"])
def test_pair_fast_equals_f64_kernel_and_oracle(ops, case):
    """The fp32-filtered kernel must give the integers of the all-fp64 kernel (and of the oracle) whatever the geometry:
    box-sized groups (MDP_PAIR_NO_SORT: the error bound collapses the fraction bits and almost every pair takes the exact
    path), cells smaller than twice the cutoff (MIXED image everywhere), coordinates many box lengths outside the cell,
    coordinates 10^5 A from the origin, thousands of bins, a handful of bins, rectangular sets, tightly clustered points
    (many pairs on identical distances), per-frame boxes."""
    import torch
    from mdproptools_b200._lib import PAIR_F64, PAIR_NO_SORT, bin_edges
    rng = np.random.default_rng(abs(hash(case)) % (2 ** 31))
    n, L, rc, ddr, flags, ncls = 3000, np.array([44.0, 41.0, 39.0]), 9.0, 0.05, 0, 2
    F = 1
    if case == "tiny_cell":
        n, L, rc = 900, np.array([13.0, 12.5, 14.0]), 6.2
    if case == "many_bins":
        ddr = 0.0025                                 # 3600 bins
    if case == "coarse_bins":
        ddr = 1.5
    if case == "multiframe":
        F = 3
    Ls = np.stack([L * (1.0 + 0.01 * f) for f in range(F)])
    pos = rng.uniform(0, 1, (F, 3, n)) * Ls[:, :, None]
    if case == "unwrapped":
        pos += rng.integers(-3, 4, (F, 3, n)) * Ls[:, :, None]
    if case == "far_from_origin":
        pos += 1.0e5
    if case == "clustered":
        centres = rng.uniform(0, 1, (F, 3, 30)) * Ls[:, :, None]
        pos = centres[:, :, rng.integers(0, 30, n)] + np.round(rng.normal(0, 0.8, (F, 3, n)), 1)   # lattice-like offsets: many ties
    if case == "nosort":
        flags = PAIR_NO_SORT
    if case == "huge_groups":
        # caller order + points thousands of box lengths apart: group boxes 10^5 A wide, the error bound exceeds a bin and the
        # kernel must route (nearly) everything it evaluates through the exact path
        flags = PAIR_NO_SORT
        pos += rng.integers(-3000, 3001, (F, 3, n)) * Ls[:, :, None]
        pos[:, :, : n // 2] = rng.uniform(0, 1, (F, 3, n // 2)) * Ls[:, :, None]          # half of them in the home cell: real hits
    typ = rng.integers(1, ncls + 1, n).astype(np.float64)
    cls = torch.from_numpy((typ - 1).astype(np.int32)).cuda()
    nb = int(rc / ddr)
    edges = bin_edges(ddr, nb)
    kw = {}
    if case == "rect":
        m = 700
        posb = rng.uniform(0, 1, (F, 3, m)) * Ls[:, :, None]
        typb = rng.integers(1, ncls + 1, m).astype(np.float64)
        kw = dict(xyz_b=_dev(posb), cls_b=torch.from_numpy((typb - 1).astype(np.int32)).cuda(), ncls_b=ncls)
    fast = ops.pair_hist(_dev(pos), cls, ncls, Ls, O.rcut_sq(rc), edges, ddr, flags=flags, **kw)
    stats = Context_stats()
    slow = ops.pair_hist(_dev(pos), cls, ncls, Ls, O.rcut_sq(rc), edges, ddr, flags=flags | PAIR_F64, **kw)
    assert torch.equal(fast, slow), case
    assert stats["pair_evals"] > 0
    if case == "huge_groups":
        assert stats["exact_path_pairs"] > 100 * 945             # (the well-sorted cases settle ~1e3 pairs in fp64)
    # and the oracle, frame 0 (symmetric cases: full histogram = sum over class pairs x 2)
    if case != "rect":
        full, _ = O.rdf_loop(typ, pos[0, 0], pos[0, 1], pos[0, 2], np.array([[1, 1]]), tuple(Ls[0]), rc, ddr, nb, nthreads=0)
        assert np.array_equal(fast[0].sum(dim=0).cpu().numpy() * 2, full)


def test_pair_engine_fuzz_fast_equals_f64():
    """The first 400 cases of tests/fuzz/fuzz_pair.py with seed 1 (random sizes, boxes incl. triclinic, cutoffs, bin widths,
    classes, distributions incl. lattices with thousands of pairs exactly on bin edges, symmetric and rectangular sets):
    k_pair_fast == k_pair bit for bit, every 10th case also == the oracle.  Case 118 of this sequence is the one that
    found a one-word overrun in the all-fp64 kernel's (since retired) direct binning; a 240 s
    run of the tool (139 220 cases, 2.3e12 pairs) is recorded in profiles/r02b_fuzz_pair.txt."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("fuzz_pair", os.path.join(root, "tests", "fuzz", "fuzz_pair.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    cases, bad = mod.main(budget=120.0, seed=1, max_cases=400)
    assert cases == 400 and bad == 0


def test_other_kernels_fuzz():
    """The first 60 cases per component of tests/fuzz/fuzz_misc.py with seed 5: shell-grid search == the general engine's list
    (wrapped, unwrapped, dense corners, central atoms among the partners), run-based survival counts == popcount kernel ==
    oracle, FFT correlation == direct sum to 1e-10, text pipeline + device parser == host parser bit for bit (random column
    orders, number spellings, CRLF, blank lines, several frames per file), per-atom MSD == oracle bit for bit.  A 30 s per
    component run (35 000 cases, no mismatch) is recorded in profiles/r02b_fuzz_misc.txt."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("fuzz_misc", os.path.join(root, "tests", "fuzz", "fuzz_misc.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    report = mod.main(budget=60.0, seed=5, max_cases=60)
    assert sorted(report) == ["fft", "msd", "parser", "shell", "survival"]
    assert all(n == 60 and bad == 0 for n, bad in report.values()), report


def test_pair_engine_fuzz_against_the_oracle():
    """The first 150 cases per component of tests/fuzz/fuzz_oracle.py with seed 9, each against the oracle's O(N^2) loops:
    symmetric and rectangular histograms (1..3 classes, both pair kernels, orthogonal and triclinic image, wrapped /
    unwrapped / clustered / lattice points), coordination numbers through the table-bin mode, neighbour lists in shell
    mode (orthogonal and triclinic, same-set exclusion).  A 30 s per component run (159 000 cases, no mismatch) is
    recorded in profiles/r02b_fuzz_oracle.txt."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("fuzz_oracle", os.path.join(root, "tests", "fuzz", "fuzz_oracle.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    report = mod.main(budget=60.0, seed=9, max_cases=150)
    assert sorted(report) == ["cn_table", "hist_rect", "hist_sym", "lists"]
    assert all(n == 150 and bad == 0 for n, bad in report.values()), report


def test_reductions_and_epilogues_fuzz():
    """The first 40 cases per component of tests/fuzz/fuzz_reduce.py with seed 3: list grouping, distinct pair keys, hydration
    cosines and counters (bit for bit), cluster membership, segment centres of mass (bit for bit), windowed and interval
    MSD, cumulative trapezoid -- against numpy / the oracle over random sizes around the tile and warp boundaries.  A 15 s
    per component run (43 800 cases, no mismatch) is recorded in profiles/r02b_fuzz_reduce.txt."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("fuzz_reduce", os.path.join(root, "tests", "fuzz", "fuzz_reduce.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    report = mod.main(budget=60.0, seed=3, max_cases=40)
    assert len(report) == 8 and all(n == 40 and bad == 0 for n, bad in report.values()), report


def Context_stats():
    from mdproptools_b200._lib import Context
    import torch
    return Context.get(torch.cuda.current_device()).pair_stats()


def test_atomic_rdf_from_arrays_equals_file_api(sample_dir, tmp_path):
    """calc_atomic_rdf_from_arrays (the in-memory front end bench.py's e2e number goes through) against calc_atomic_rdf on the
    same frames: identical DataFrames, through the vectorised normalisation (one composition, one volume) and through the
    per-frame loop (a trajectory whose box changes)."""
    from mdproptools_b200.io import dump as D
    from mdproptools_b200.structural.rdf_cn import calc_atomic_rdf, calc_atomic_rdf_from_arrays
    pat = os.path.join(sample_dir, "dump.nvt.*.dump")
    want = calc_atomic_rdf(20, 0.05, 9, MASS, C1_REL, pat, save_mode=False)
    frames = list(D.read_dumps(pat, ["id", "type", "x", "y", "z"]))
    pos = np.stack([np.stack([f.data["x"], f.data["y"], f.data["z"]]) for f in frames])
    typ = frames[0].data["type"]
    L = frames[0].box.lattice_lengths()
    got, counts = calc_atomic_rdf_from_arrays(pos, typ, L, 20, 0.05, C1_REL, return_counts=True)
    assert np.array_equal(got.values, want.values) and list(got.columns) == list(want.columns)
    assert counts.shape == (len(frames), 5, 400)
    # box changing from frame to frame: the per-frame normalisation loop; compare with the two single-frame results averaged
    Ls = np.stack([np.asarray(L), np.asarray(L) * 1.001])
    got2 = calc_atomic_rdf_from_arrays(pos, typ, Ls, 20, 0.05, C1_REL)
    one = [calc_atomic_rdf_from_arrays(pos[k:k + 1], typ, Ls[k], 20, 0.05, C1_REL).values for k in range(2)]
    assert np.array_equal(got2.values[:, 1:], (one[0][:, 1:] + one[1][:, 1:]) / 2)
