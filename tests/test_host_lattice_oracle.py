"""The closed-form lattice histograms of tests/lattice_oracle.py against the oracle's brute force (oracle/oracle.c), bit for
bit, on frames small enough to enumerate: blocks inside the box, across its boundary, crystals filling the periodic box
(even m: exact half-box ties), 1-3 classes, bin widths equal to the spacing (pairs on bin edges), cutoffs above L/2 and
cutoffs whose last index is dropped.  The GPU tests of tests/test_gpu_pair_scale.py rely on this equality at 10^12 pairs."""
import numpy as np
import pytest

from oracle import oracle as O
from tests import lattice_oracle as LO

# (name, frame, r_cut): every frame here has at most ~2200 points
FRAMES = {
    "inside": (LO.Frame([((9, 8, 7), (1.0, 2.5, 0.75))], 0.25, (12.0, 11.0, 10.0), K=2), 1.9),
    "straddling": (LO.Frame([((9, 9, 9), (5.5, 4.75, -1.25))], 0.5, (7.0, 6.5, 8.0), K=3, wrap=True), 3.3),
    "crystal_even": (LO.Frame([((8, 10, 12), (0.0, 0.0, 0.0))], 0.75, (6.0, 7.5, 9.0), K=2), 5.1),     # r_cut > L/2
    "crystal_odd": (LO.Frame([((13, 11, 9), (0.125, 0.0, 0.5))], 0.5, (6.5, 5.5, 4.5), K=3, wrap=True), 2.95),
    "two_blocks": (LO.Frame([((7, 6, 5), (0.0, 0.0, 0.0)), ((6, 6, 6), (0.25, 0.25, 0.25)), ((5, 4, 6), (2.125, 2.0, 1.0))],
                            0.5, (5.0, 5.5, 6.0), K=2, wrap=True), 2.6),
}
REL = {1: [[1, 1]], 2: [[1, 1], [1, 2], [2, 1], [2, 2]], 3: [[1, 1], [1, 3], [2, 3], [3, 3], [3, 2]]}


def _brute(fr, r_cut, ddr, tri=False):
    xyz, cls = fr.positions()
    nb = int(r_cut / ddr)
    rel = np.array(REL[fr.K])
    f = O.rdf_loop_tri if tri else O.rdf_loop
    return f(cls + 1.0, xyz[0], xyz[1], xyz[2], rel, fr.cell, r_cut, ddr, nb, nthreads=0), nb, rel


@pytest.mark.parametrize("name", sorted(FRAMES))
@pytest.mark.parametrize("ddr", ["h", 0.1, 0.07])
def test_rdf_loop_equals_closed_form(name, ddr):
    fr, r_cut = FRAMES[name]
    ddr = fr.h if ddr == "h" else ddr
    (full, part), nb, rel = _brute(fr, r_cut, ddr)
    sym = LO.hist_sym(fr, LO.uniform_bins(ddr, nb, O.rcut_sq(r_cut)))
    f2, p2 = LO.rdf_loop_counts(sym, rel, fr.K)
    assert np.array_equal(f2, full)
    assert np.array_equal(p2, part)
    if ddr == fr.h:
        assert np.count_nonzero(full) >= 3


def test_dropped_index_and_cutoff_edge():
    """r_cut / ddr = 29.5: pairs at 2.9 <= r < 2.95 reach index 29 = nbins and are dropped; pairs at exactly r_cut fail the
    strict rsq < rcut^2; both rules must be the oracle's."""
    fr, _ = FRAMES["crystal_odd"]
    ddr = 0.1
    for r_cut in (2.95, 2.5, 2.0):                        # 2.5 = 5 h and 2.0 = 4 h: lattice distances exactly on the cutoff
        (full, part), nb, rel = _brute(fr, r_cut, ddr)
        sym = LO.hist_sym(fr, LO.uniform_bins(ddr, nb, O.rcut_sq(r_cut)))
        assert np.array_equal(LO.rdf_loop_counts(sym, rel, fr.K)[0], full), r_cut
        above = LO.hist_sym(fr, LO.uniform_bins(ddr, nb + 1, O.rcut_sq(r_cut))).sum() - sym.sum()
        if r_cut == 2.95:
            assert above > 0                               # the dropped index holds pairs: the case is not vacuous


@pytest.mark.parametrize("name", ["inside", "straddling", "crystal_even", "two_blocks"])
def test_cn_loop_equals_closed_form(name):
    fr, _ = FRAMES[name]
    xyz, cls = fr.positions()
    rel = np.array(REL[fr.K])
    r_cuts = [1.0, 1.5, 2.0, 1.25, 2.75][: len(rel)]      # 1.0, 1.5, 2.0: lattice distances exactly on the threshold
    cn = O.cn_loop(cls + 1.0, xyz[0], xyz[1], xyz[2], rel, fr.cell, r_cuts, nthreads=0)
    edges, rc2 = LO.cn_thresholds(r_cuts)
    cum = np.cumsum(LO.hist_sym(fr, LO.table_bins(edges, rc2)), axis=1)
    assert np.array_equal(LO.cn_loop_counts(cum, rel, r_cuts, fr.K), cn)


@pytest.mark.parametrize("ddr", [0.5, 0.1, 0.07])
def test_rdf_rect_equals_closed_form(ddr):
    """Two interpenetrating lattices (B offset by h/2 per axis), B straddling the boundary, different class counts."""
    cell = (6.0, 6.5, 7.0)
    fa = LO.Frame([((10, 9, 11), (0.5, 1.0, 0.0))], 0.5, cell, K=2, wrap=True)
    fb = LO.Frame([((9, 10, 8), (3.75, 0.25, 1.75))], 0.5, cell, K=3, wrap=True)
    a, ca = fa.positions()
    b, cb = fb.positions()
    rel = np.array([[1, 1], [1, 3], [2, 2], [2, 3]])
    r_cut = 3.4
    nb = int(r_cut / ddr)
    part = O.rdf_rect(ca + 1.0, a[0], a[1], a[2], cb + 1.0, b[0], b[1], b[2], rel, cell, r_cut, ddr, nb, nthreads=0)
    rect = LO.hist_rect(fa, fb, LO.uniform_bins(ddr, nb, O.rcut_sq(r_cut)))
    assert np.array_equal(LO.rect_counts(rect, rel, fb.K), part)


TRI = (6.5625, 5.5625, 4.5625, 1.25, -0.75, 0.5)   # L/2 = k * 2^-5 with k odd: no displacement (a multiple of 2^-3) ties


@pytest.mark.parametrize("ddr", [0.5, 0.1, 0.07])
def test_rdf_loop_tri_equals_closed_form(ddr):
    fr = LO.Frame([((13, 11, 9), (0.0, 0.25, 0.0)), ((5, 6, 7), (1.25, 0.75, 0.5))], 0.5, TRI, K=3)
    (full, part), nb, rel = _brute(fr, 3.1, ddr, tri=True)
    sym = LO.hist_sym(fr, LO.uniform_bins(ddr, nb, O.rcut_sq(3.1)))
    f2, p2 = LO.rdf_loop_counts(sym, rel, fr.K)
    assert np.array_equal(f2, full) and np.array_equal(p2, part)


def test_rdf_rect_tri_equals_closed_form():
    fa = LO.Frame([((9, 11, 7), (0.0, 0.0, 0.0))], 0.5, TRI, K=2)
    fb = LO.Frame([((8, 7, 9), (0.25, 0.25, 0.25))], 0.5, TRI, K=1)
    a, ca = fa.positions()
    b, cb = fb.positions()
    rel = np.array([[1, 1], [2, 1]])
    ddr, r_cut = 0.1, 2.9
    nb = int(r_cut / ddr)
    part = O.rdf_rect_tri(ca + 1.0, a[0], a[1], a[2], cb + 1.0, b[0], b[1], b[2], rel, TRI, r_cut, ddr, nb, nthreads=0)
    rect = LO.hist_rect(fa, fb, LO.uniform_bins(ddr, nb, O.rcut_sq(r_cut)))
    assert np.array_equal(LO.rect_counts(rect, rel, fb.K), part)


def test_tri_half_cell_ties_follow_the_strict_compares():
    """An even triclinic crystal has exact half-cell ties: there the image, and so rsq, depends on the strict compares of
    pair_rsq_tri (a tie in z does not move dy and dx by the tilts).  The frame is unwrapped, so the closed form still holds;
    without ``ties_ok`` the module refuses it."""
    cell = (4.0, 5.0, 6.0, 1.5, 0.5, -1.0)
    with pytest.raises(AssertionError, match="half-cell tie"):
        LO.hist_sym(LO.Frame([((8, 10, 12), (0.0, 0.0, 0.0))], 0.5, cell), LO.uniform_bins(0.25, 10, 6.25))
    fr = LO.Frame([((8, 10, 12), (0.0, 0.0, 0.0))], 0.5, cell, K=2, ties_ok=True)
    for ddr in (0.5, 0.07):
        (full, part), nb, rel = _brute(fr, 3.2, ddr, tri=True)
        sym = LO.hist_sym(fr, LO.uniform_bins(ddr, nb, O.rcut_sq(3.2)))
        f2, p2 = LO.rdf_loop_counts(sym, rel, fr.K)
        assert np.array_equal(f2, full) and np.array_equal(p2, part)


@pytest.mark.parametrize("name", sorted(FRAMES))
def test_identities(name):
    """r_cut beyond every minimum-image distance: the total is n(n-1)/2; the rows of all ordered class pairs add up to the
    full row."""
    fr, _ = FRAMES[name]
    n = fr.n
    r_cut = float(np.sqrt(3.0) * max(fr.cell[:3]))
    nb = 7
    sym = LO.hist_sym(fr, LO.uniform_bins(r_cut / nb * 1.0001, nb, O.rcut_sq(r_cut)))
    assert sym.sum() == n * (n - 1) // 2
    full, part = LO.rdf_loop_counts(sym, [[a, b] for a in range(1, fr.K + 1) for b in range(1, fr.K + 1)], fr.K)
    assert np.array_equal(part.sum(axis=0), full)
    # and the class composition: unordered pairs of classes (a, b) = N_a N_b, (a, a) = N_a (N_a - 1) / 2
    c = fr.class_counts()
    for a in range(fr.K):
        for b in range(a, fr.K):
            want = c[a] * (c[a] - 1) // 2 if a == b else c[a] * c[b]
            assert sym[LO.sym_row(a, b, fr.K)].sum() == want


def test_exactness_condition_is_enforced():
    with pytest.raises(AssertionError, match="bits"):
        LO.Frame([((4, 4, 4), (0.0, 0.0, 0.0))], 2.0 ** -20, (8.0, 8.0, 8.0))
    with pytest.raises(AssertionError, match="bits"):
        LO.Frame([((4, 4, 4), (0.0, 0.0, 0.0))], 0.1, (8.0, 8.0, 8.0))
    with pytest.raises(AssertionError, match="extent"):
        LO.Frame([((9, 4, 4), (0.0, 0.0, 0.0))], 1.0, (8.0, 8.0, 8.0), wrap=True)
