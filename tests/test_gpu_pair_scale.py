"""The pair engine against the exact lattice histograms of tests/lattice_oracle.py at 10^11-10^12 pairs per frame, where
every CTA of both kernels re-bases its uint32 shared histogram into the global uint64 one mid-frame (the overflow guard,
DESIGN 4.1).  Each case runs through the default kernel (k_pair_fast for uniform bins) and through k_pair (PAIR_F64), and
every per-frame histogram must equal the closed form exactly.

Sizes follow the device's SM count.  The grids are sm_count x FAST_CTAS_PER_SM (at most; the occupancy may lower it) and
sm_count x CTAS_PER_SM, and a CTA re-bases after every GUARD pairs it evaluates.  Each case asserts the pigeonhole bound
that makes it reach the guard, so a change that makes a case too small fails here instead of passing without a re-base.
"""
import functools

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import oracle as O  # noqa: E402
from tests import lattice_oracle as LO  # noqa: E402

FAST_CTAS_PER_SM = 3     # csrc/pair_fast.cuh
CTAS_PER_SM = 2          # csrc/pair.cu
GUARD = 2 ** 30          # pairs a CTA evaluates between two re-bases of its shared histogram
KERNELS = ["fast", "f64"]


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mdproptools_b200 import ops
    from mdproptools_b200._lib import PAIR_F64, Context
    sm = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    ctx = Context.get(torch.cuda.current_device())
    return dict(ops=ops, sm=sm, flags={"fast": 0, "f64": PAIR_F64}, stats=ctx.pair_stats,
                grid={"fast": sm * FAST_CTAS_PER_SM, "f64": sm * CTAS_PER_SM})


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _hist(eng, kern, fr, rcut2, edges, ddr, frames=None, flags=0, fb=None):
    """ops.pair_hist over one frame (or the stacked positions of several) -> int64 numpy [F, rows, nbins]."""
    if frames is None:
        xyz, cls = fr.positions()
        frames = (xyz[None], np.asarray([fr.cell]))
    else:
        cls = fr.positions()[1]
    kw = {}
    if fb is not None:
        xb, cb = fb.positions()
        kw = dict(xyz_b=_dev(xb[None]), cls_b=_dev(cb), ncls_b=fb.K)
    h = eng["ops"].pair_hist(_dev(frames[0]), _dev(cls), fr.K, frames[1], rcut2, edges, ddr, flags=eng["flags"][kern] | flags, **kw)
    torch.cuda.synchronize()
    return h.cpu().numpy()


def _min_m(pairs_needed, pairs_of_m, m0):
    m = m0
    while pairs_of_m(m) < pairs_needed:
        m += 1
    return m


# ---- re-base, spread: one ~1.4 M-point frame, spacing = ddr, across the periodic boundary, every pair inside r_cut ----
@functools.lru_cache(maxsize=None)
def _spread(sm):
    h = 0.125
    m = _min_m(2 * GUARD * sm * FAST_CTAS_PER_SM, lambda m: m ** 3 * (m ** 3 - 1) // 2, 64)
    L = 2.0 ** np.ceil(np.log2(2 * m * h))                     # no pair of the block is more than L/2 apart per axis
    fr = LO.Frame([((m, m, m), (L - 7.0, L - 3.0, 5.0))], h, (L, L, L), K=3, wrap=True)
    r_cut = int(np.ceil(np.sqrt(3.0) * (m - 1) * h)) + 1      # covers every pair
    return fr, r_cut


def test_spread_frame_rebases_and_matches_closed_form(eng):
    fr, r_cut = _spread(eng["sm"])
    ddr = fr.h
    nb = int(r_cut / ddr)
    from mdproptools_b200._lib import bin_edges
    want = LO.hist_sym(fr, LO.uniform_bins(ddr, nb, O.rcut_sq(r_cut)))
    n = fr.n
    assert want.sum() == n * (n - 1) // 2                      # r_cut covers the frame
    on_edge = LO.hist_sym(fr, _on_edge_bins(ddr, O.rcut_sq(r_cut))).sum()
    assert on_edge > 10 ** 6
    for kern in KERNELS:
        # pigeonhole: some CTA evaluated >= 2 GUARD pairs of this frame, so it re-based at least twice mid-frame
        assert want.sum() >= 2 * GUARD * eng["grid"][kern], (kern, eng["sm"])
        got = _hist(eng, kern, fr, O.rcut_sq(r_cut), bin_edges(ddr, nb), ddr)
        st = eng["stats"]()
        assert np.array_equal(got[0], want), kern
        if kern == "fast":
            # every pair exactly on a bin edge is within the error bound of it: all of them took the exact path
            assert st["exact_path_pairs"] >= on_edge, st


def _on_edge_bins(ddr, rcut2):
    """one bin: the pairs whose sqrt(rsq) / ddr is an integer (exactly on a bin edge)"""
    def f(rsq):
        q = np.sqrt(rsq) / ddr
        return np.where((rsq < rcut2) & (q == np.floor(q)), 0, -1)
    f.nbins = 1
    return f


# ---- re-base, concentrated: 2^21 points 2^-6 A apart, every pair in bin 0 of one row: one shared word per CTA ----------
@functools.lru_cache(maxsize=None)
def _concentrated(K):
    return LO.Frame([((128, 128, 128), (4.0, 4.0, 4.0))], 2.0 ** -6, (16.0, 16.0, 16.0), K=K)


@pytest.mark.parametrize("kern", KERNELS)
def test_concentrated_word_passes_2_31(eng, kern):
    """k_pair_fast adds a flushed word as a signed 32-bit value, k_pair as unsigned: without re-bases the one word of bin 0
    would wrap (k_pair) or turn negative (k_pair_fast) in every CTA."""
    from mdproptools_b200._lib import bin_edges
    fr = _concentrated(1)
    n = fr.n
    assert n == 2 ** 21
    want = LO.hist_sym(fr, LO.uniform_bins(4.0, 2, O.rcut_sq(8)))
    assert want[0, 0] == n * (n - 1) // 2 and want.sum() == want[0, 0]
    word_limit = 2 ** 31 if kern == "fast" else 2 ** 32
    assert want[0, 0] >= word_limit * eng["grid"][kern], (kern, eng["sm"])     # some CTA's word passes the limit
    got = _hist(eng, kern, fr, O.rcut_sq(8), bin_edges(4.0, 2), 4.0)
    assert np.array_equal(got[0], want), (got[0], want)


# ---- frames owned by CTAs: more frames than CTAs, > GUARD in-cut pairs per frame, frames of three spacings -------------
def _owned_frames(sm):
    m = (42, 42, 42)                                           # even m: exact half-box ties
    hs = [0.25, 0.25 + 2.0 ** -10, 0.25 + 2.0 ** -9]
    frs = [LO.Frame([(m, (0.0, 0.0, 0.0))], h, tuple(k * h for k in m), K=2) for h in hs]
    return frs, 3 * sm + 1


@pytest.mark.parametrize("kern", KERNELS)
def test_frames_owned_by_ctas(eng, kern):
    from mdproptools_b200._lib import bin_edges
    frs, F = _owned_frames(eng["sm"])
    assert F > eng["grid"][kern]                                # every CTA starts at a frame of its own
    r_cut, ddr = 5.21875, 0.125                                 # just under the smallest L/2 = 5.25
    assert r_cut < min(min(fr.cell) for fr in frs) / 2
    nb = int(r_cut / ddr)
    want = [LO.hist_sym(fr, LO.uniform_bins(ddr, nb, O.rcut_sq(r_cut))) for fr in frs]
    for k in range(len(frs)):
        assert want[k].sum() > GUARD                            # a CTA that walks a frame alone re-bases in it
        assert not np.array_equal(want[k], want[k - 1])         # a flush into the wrong frame's histogram shows
    xyz = np.stack([frs[f % 3].positions()[0] for f in range(F)])
    boxes = np.stack([frs[f % 3].cell for f in range(F)])
    got = _hist(eng, kern, frs[0], O.rcut_sq(r_cut), bin_edges(ddr, nb), ddr, frames=(xyz, boxes))
    for f in range(F):
        assert np.array_equal(got[f], want[f % 3]), (kern, f)


# ---- the benchmark's shape: ~100k-point crystals, r_cut 20, 400 bins of 0.05, orthogonal and triclinic -----------------
@pytest.mark.parametrize("kern", KERNELS)
@pytest.mark.parametrize("tri", [False, True])
def test_bench_shape(eng, kern, tri):
    from mdproptools_b200._lib import PAIR_TRICLINIC, bin_edges
    if tri:
        # odd m, L = m h + 2^-5 and tilts in multiples of 2^-3: L/2 is an odd multiple of 2^-6, no displacement ties
        frs = [LO.Frame([((47, 47, 47), (0.0, 0.0, 0.0))], h, (47 * h + 2.0 ** -5,) * 3 + tilt, K=3)
               for h, tilt in ((3.5, (8.25, -4.5, 6.125)), (3.625, (-2.0, 3.375, 0.0)))]
    else:
        frs = [LO.Frame([((46, 46, 46), (0.0, 0.0, 0.0))], h, (46 * h,) * 3, K=3) for h in (3.625, 3.5, 3.75)]
    ddr, r_cut, nb = 0.05, 20, 400
    xyz = np.stack([fr.positions()[0] for fr in frs])
    boxes = np.stack([fr.cell for fr in frs])
    got = _hist(eng, kern, frs[0], O.rcut_sq(r_cut), bin_edges(ddr, nb), ddr, frames=(xyz, boxes),
                flags=PAIR_TRICLINIC if tri else 0)
    for f, fr in enumerate(frs):
        want = LO.hist_sym(fr, LO.uniform_bins(ddr, nb, O.rcut_sq(r_cut)))
        assert want.sum() > 10 ** 7
        assert np.array_equal(got[f], want), (kern, tri, f)


# ---- table bins (k_pair only): coordination thresholds over the spread frame, cumulative reduce past 2^32 ---------------
def test_table_bins_cumulative(eng):
    fr, r_cut = _spread(eng["sm"])
    ops = eng["ops"]
    r_cuts = [2.0, 5.5, 12.25, r_cut]
    edges, rc2 = LO.cn_thresholds(r_cuts)
    want = LO.hist_sym(fr, LO.table_bins(edges, rc2))
    assert want.sum() >= 2 * GUARD * eng["grid"]["f64"], eng["sm"]
    xyz, cls = fr.positions()
    hist = ops.pair_hist(_dev(xyz[None]), _dev(cls), fr.K, [fr.cell], rc2, edges, 0.0)
    assert np.array_equal(hist.cpu().numpy()[0], want)
    rows = LO.sym_rows(fr.K)
    w = np.concatenate([np.eye(rows, dtype=np.int64), np.full((1, rows), 2)])        # every row, and the full count x 2
    cum = ops.hist_reduce(hist, w, cumulative=True).cpu().numpy()[0]
    assert np.array_equal(cum[:rows], np.cumsum(want, axis=1))
    assert cum[rows, -1] == fr.n * (fr.n - 1) > 2 ** 32


# ---- rectangular: two interpenetrating lattices, B offset by h/2 per axis -------------------------------------------
@pytest.mark.parametrize("kern", KERNELS)
def test_rect_interpenetrating(eng, kern):
    from mdproptools_b200._lib import bin_edges
    h = 0.125
    m = _min_m(2 * GUARD * eng["sm"] * FAST_CTAS_PER_SM, lambda m: m ** 6, 64)
    L = 2.0 ** np.ceil(np.log2(2 * m * h + h))
    fa = LO.Frame([((m, m, m), (L - 5.0, 1.0, 2.0))], h, (L, L, L), K=2, wrap=True)
    fb = LO.Frame([((m, m, m), (L - 5.0 + h / 2, 1.0 + h / 2, 2.0 + h / 2))], h, (L, L, L), K=3, wrap=True)
    r_cut = int(np.ceil(np.sqrt(3.0) * (m - 0.5) * h)) + 1
    ddr = h
    nb = int(r_cut / ddr)
    want = LO.hist_rect(fa, fb, LO.uniform_bins(ddr, nb, O.rcut_sq(r_cut)))
    assert want.sum() == fa.n * fb.n
    assert want.sum() >= 2 * GUARD * eng["grid"][kern], (kern, eng["sm"])
    got = _hist(eng, kern, fa, O.rcut_sq(r_cut), bin_edges(ddr, nb), ddr, fb=fb)
    assert np.array_equal(got[0], want), kern


# ---- size limit: the last accepted point count and one past it ----------------------------------------------------------
@pytest.mark.parametrize("kern", KERNELS)
def test_size_limit(eng, kern):
    from mdproptools_b200._lib import MdpropError, bin_edges
    m = (127, 129, 256)                                          # 127 x 129 x 256 = 2^22 - 256: npad = 2^22 - 256
    h, ddr, r_cut = 0.5, 0.125, 0.75                             # nearest and second-nearest neighbours only
    fr = LO.Frame([(m, (0.0, 0.0, 0.0))], h, tuple(k * h for k in m))
    assert fr.n == 2 ** 22 - 256
    nb = int(r_cut / ddr)
    want = LO.hist_sym(fr, LO.uniform_bins(ddr, nb, O.rcut_sq(r_cut)))
    assert want.sum() == fr.n * 9                                # 6 + 12 neighbours per point, each pair once
    got = _hist(eng, kern, fr, O.rcut_sq(r_cut), bin_edges(ddr, nb), ddr)
    assert np.array_equal(got[0], want), kern
    over = LO.Frame([(m, (0.0, 0.0, 0.0)), ((1, 1, 1), (0.25, 0.25, 0.25))], h, fr.cell)
    assert over.n == 2 ** 22 - 255
    with pytest.raises(MdpropError, match=r"limited to 2\^22 points"):
        _hist(eng, kern, over, O.rcut_sq(r_cut), bin_edges(ddr, nb), ddr)


# ---- end to end: counts past 2^32 through the public API ----------------------------------------------------------------
def test_atomic_rdf_from_arrays_counts_past_2_32(eng):
    from mdproptools_b200.structural.rdf_cn import calc_atomic_rdf_from_arrays
    fr = _concentrated(2)
    xyz, cls = fr.positions()
    rel = [[1, 1, 2], [1, 2, 2]]
    _, counts = calc_atomic_rdf_from_arrays(xyz[None], cls + 1.0, fr.cell, 8, 4.0, rel, return_counts=True)
    sym = LO.hist_sym(fr, LO.uniform_bins(4.0, 2, O.rcut_sq(8)))
    full, part = LO.rdf_loop_counts(sym, np.asarray(rel).T, fr.K)
    assert counts.shape == (1, 4, 2)
    assert np.array_equal(counts[0, 0], full) and np.array_equal(counts[0, 1:], part)
    assert counts[0, 0, 0] == fr.n * (fr.n - 1) > 2 ** 32 and counts[0, 1:, 0].min() > 2 ** 32
