"""Host checks of the static structure factor: the per-term body of the device kernel (csrc/sk_phase.h, run by
tests/native/sk_phase_host.cpp) against long double, the k-set of structure_factor.py against the oracle's brute force,
its seeded sampling, and the oracle (tests/sk_oracle.py) against analytic cases."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from mdproptools_b200.structural import structure_factor as SF
from tests import sk_oracle as SO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MUFU = np.sqrt(2) * 2.0 ** -21.41          # the device's __sincosf on [-pi, pi] (CUDA Programming Guide), not run here


@pytest.fixture(scope="module")
def ph(tmp_path_factory):
    so = tmp_path_factory.mktemp("sk_phase") / "sk_phase_host.so"
    src = os.path.join(ROOT, "tests", "native", "sk_phase_host.cpp")
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-o", str(so), src], check=True)
    lib = ctypes.CDLL(str(so))
    c = np.zeros(4)
    lib.sk_consts(c.ctypes.data_as(ctypes.c_void_p))
    lib.consts = dict(nlim=int(c[0]), eps=float(c[1]), max_classes=int(c[2]), chunk=int(c[3]))
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _fix(ph, s):
    s = np.ascontiguousarray(s, dtype=np.float64).reshape(-1)
    u = np.empty(s.size, dtype=np.uint32)
    ph.sk_fix(_p(s), ctypes.c_longlong(s.size), _p(u))
    return u


def _edge_s(rng, n):
    """fractional coordinates: uniform, near 0 and 1 on both sides, exact integers, unwrapped (a few cells out)"""
    tiny = np.array([0.0, 1.0, -1.0, 2.0, 1e-300, -1e-300, 1e-17, -1e-17, 1 - 2.0 ** -53, 1 + 2.0 ** -52, 2.0 ** -33,
                     -2.0 ** -33, 1 - 2.0 ** -33, 0.5, -0.5, 3.75, -7.25])
    return np.concatenate([tiny, rng.uniform(0, 1, n), rng.uniform(-1e-9, 1e-9, n), 1 + rng.uniform(-1e-9, 1e-9, n),
                           rng.uniform(-5, 5, n)])


def test_constants_match_the_python_side(ph):
    from mdproptools_b200 import _lib
    assert ph.consts == dict(nlim=_lib.SK_NLIM, eps=_lib.SK_EPS, max_classes=_lib.SK_MAX_CLASSES, chunk=32)
    assert ph.consts["nlim"] >= 512


def test_fixed_point_is_floor_of_frac_times_2_32(ph):
    """u = floor(frac(s) 2^32) mod 2^32, within one unit where s - floor(s) rounds (circularly: 2^32 - 1 and 0 are neighbours)."""
    from fractions import Fraction
    s = _edge_s(np.random.default_rng(1), 2000)
    u = _fix(ph, s)
    for si, ui in zip(s.tolist(), u.tolist()):
        f = Fraction(si) - (Fraction(si).numerator // Fraction(si).denominator)
        want = int(f * (1 << 32)) % (1 << 32)
        d = (int(ui) - want) % (1 << 32)
        assert d in (0, 1, (1 << 32) - 1), (si, ui, want)
        if 0.0 <= si < 1.0 and si * 2.0 ** 32 == np.floor(si * 2.0 ** 32):
            assert ui == want, si               # exactly representable: exact


def _phase(ph, miller, u3):
    m = np.ascontiguousarray(miller, dtype=np.int32)
    u3 = np.ascontiguousarray(u3, dtype=np.uint32)
    p = np.empty((len(m), len(u3)), dtype=np.uint32)
    ph.sk_phase(_p(m), ctypes.c_longlong(len(m)), _p(u3), ctypes.c_longlong(len(u3)), _p(p))
    return p


def _miller(rng, nlim, n):
    ext = np.array([[nlim, nlim, nlim], [-nlim, -nlim, -nlim], [nlim, -nlim, nlim], [1, 0, 0], [0, 0, 1], [0, 1, -nlim],
                    [nlim, 0, 0]])
    return np.concatenate([ext, rng.integers(-nlim, nlim + 1, (n, 3))])


def test_phase_is_exact_integer_dot_product_mod_2_32(ph):
    rng = np.random.default_rng(2)
    nlim = ph.consts["nlim"]
    m = _miller(rng, nlim, 200)
    u3 = np.concatenate([rng.integers(0, 1 << 32, (300, 3), dtype=np.uint64),
                         np.array([[0, 0, 0], [(1 << 32) - 1] * 3, [1 << 31] * 3], dtype=np.uint64)]).astype(np.uint32)
    p = _phase(ph, m, u3)
    want = ((m.astype(object) @ u3.astype(object).T) + 256) % (1 << 32)
    assert np.array_equal(p.astype(object), want)


def _exact_terms(miller, s):
    """exp(2 pi i n.s) in long double: [nk, N] (re, im)"""
    ph_ = np.asarray(miller, dtype=np.longdouble) @ np.asarray(s, dtype=np.longdouble).T
    ph_ = ph_ - np.floor(ph_)
    a = ph_ * 2 * SO._PI_LD
    return np.cos(a), np.sin(a)


def test_per_term_error_within_the_contract(ph):
    """Random s (edges included) and Miller components up to +-n_lim: every term within the derived per-term bound of the
    fixed point, the 23-bit rounding and the fp32 angle, plus the fp32 rounding of the host's sin and cos; the contract adds
    the device's __sincosf and the fp32 chunk sums to that."""
    rng = np.random.default_rng(3)
    nlim = ph.consts["nlim"]
    s = np.stack([rng.permutation(_edge_s(rng, 60))[:200] for _ in range(3)], axis=1)
    m = _miller(rng, nlim, 300)
    u3 = _fix(ph, s).reshape(-1, 3)
    p = _phase(ph, m, u3).reshape(-1)
    cs = np.empty(2 * p.size, dtype=np.float32)
    ph.sk_terms(_p(p), ctypes.c_longlong(p.size), _p(cs))
    re_x, im_x = _exact_terms(m, s)
    err = np.hypot((cs[0::2] - re_x.reshape(-1)).astype(np.float64), (cs[1::2] - im_x.reshape(-1)).astype(np.float64))
    bound = 2 * np.pi * (3 * nlim * 2.0 ** -32 + 2.0 ** -24) + np.pi * 2.0 ** -23 + np.sqrt(2) * 2.0 ** -24
    assert err.max() <= bound, (err.max(), bound)
    assert bound + MUFU + np.sqrt(2) * 2.0 ** -24 * (32 * 33 / 2 - 1) / 32 <= ph.consts["eps"]


@pytest.mark.parametrize("n", [1, 31, 32, 33, 517, 2000])
def test_chunked_rho_within_the_contract(ph, n):
    """rho(k) summed as the kernel sums it (fp32 over 32 atoms, fp64 beyond) against long double: within (eps - the
    __sincosf share) N, for sizes around the chunk and Miller components up to +-n_lim."""
    rng = np.random.default_rng(4 + n)
    nlim = ph.consts["nlim"]
    s = rng.uniform(-0.2, 1.2, (n, 3))
    s[: min(n, 4)] = [[0.0, 1 - 1e-17, -1e-17], [1 - 2.0 ** -53, 0.5, 2.0 ** -40], [0.25, 0.75, 0.999999999], [0, 0, 0]][: min(n, 4)]
    m = np.ascontiguousarray(_miller(rng, nlim, 60), dtype=np.int32)
    out = np.empty(2 * len(m))
    sc = np.ascontiguousarray(s)
    ph.sk_rho(_p(m), ctypes.c_longlong(len(m)), _p(sc), ctypes.c_longlong(n), _p(out))
    re_x, im_x = _exact_terms(m, s)
    err = np.hypot((out[0::2] - re_x.sum(axis=1)).astype(np.float64), (out[1::2] - im_x.sum(axis=1)).astype(np.float64))
    assert err.max() <= (ph.consts["eps"] - MUFU) * n, (err.max() / n)


def test_fractional_coordinates_of_a_triclinic_cell(ph):
    cell = np.array([31.0, 27.5, 22.25, 6.2, -3.1, 4.4])
    rng = np.random.default_rng(5)
    s = rng.uniform(-1, 2, (500, 3))
    r = np.ascontiguousarray(s @ SO.cell_matrix(cell).T)
    got = np.empty_like(r)
    ph.sk_frac(_p(cell), _p(r), ctypes.c_longlong(len(r)), _p(got))
    assert np.abs(got - s).max() < 1e-14


# ------------------------------------------------------------------------------------------------
# k-set
# ------------------------------------------------------------------------------------------------
CELLS = {
    "cubic": (20.0, 20.0, 20.0, 0.0, 0.0, 0.0),
    "ortho": (23.0, 17.5, 31.25, 0.0, 0.0, 0.0),
    "triclinic": (25.0, 21.0, 18.0, 5.0, -2.5, 3.15),
    "c2": (167.19 / 4, 167.19 / 4, 167.19 / 4, 0.2 * 167.19 / 4, 0.1 * 167.19 / 4, -0.15 * 167.19 / 4),
}


@pytest.mark.parametrize("name", list(CELLS))
@pytest.mark.parametrize("k_max,bin_size,k_min", [(3.0, 0.05, None), (2.0, 0.1, 0.7), (1.23, 0.02, None)])
def test_kset_equals_brute_force(name, k_max, bin_size, k_min):
    cell = CELLS[name]
    miller, boff = SF.kset(cell, k_max, bin_size, k_min)
    want, wboff, nbins = SO.kset_brute(cell, k_max, bin_size, k_min)
    assert np.array_equal(miller, want) and np.array_equal(boff, wboff)
    assert miller.dtype == np.int32 and len(boff) == nbins + 1
    # half-space: no zero vector and no +-n pair twice
    keys = {tuple(v) for v in miller.tolist()}
    assert len(keys) == len(miller) and (0, 0, 0) not in keys
    assert not any(tuple(-x for x in v) in keys for v in keys)
    # range and bins
    K = SO.recip(cell)
    kn = np.linalg.norm(miller @ K.T, axis=1)
    kmn = SO.smallest_k(cell) if k_min is None else k_min
    assert np.all(kn >= kmn * (1 - 1e-12)) and np.all(kn < nbins * bin_size * (1 + 1e-12))
    b = np.repeat(np.arange(nbins), np.diff(boff))
    assert np.all(np.abs(np.floor(kn / bin_size) - b) <= (np.abs(kn / bin_size - np.round(kn / bin_size)) < 1e-9))
    # reciprocity: k.a = 2 pi h, k.b = 2 pi k, k.c = 2 pi l
    kv = miller @ K.T
    assert np.allclose(kv @ SO.cell_matrix(cell), 2 * np.pi * miller, atol=1e-9)
    # a complete half-space: with the -n partners it is every n != 0 of the shell
    if k_min is None:
        assert SF.smallest_k(cell) == SO.smallest_k(cell)


def test_smallest_k_is_the_shortest_reciprocal_vector():
    for cell in CELLS.values():
        assert SF.smallest_k(cell) == pytest.approx(np.linalg.norm(SO.recip(cell), axis=0).min(), rel=1e-15) or \
            SF.smallest_k(cell) < np.linalg.norm(SO.recip(cell), axis=0).min()
    assert SF.smallest_k(CELLS["cubic"]) == pytest.approx(2 * np.pi / 20.0, rel=1e-15)


@pytest.mark.parametrize("name", ["ortho", "triclinic"])
def test_sampling_is_seeded_bounded_and_independent_of_k_max(name):
    cell = CELLS[name]
    a, ab = SF.kset(cell, 3.0, 0.05, max_k_per_bin=40, seed=7)
    b, bb = SF.kset(cell, 3.0, 0.05, max_k_per_bin=40, seed=7)
    assert np.array_equal(a, b) and np.array_equal(ab, bb)
    full, fb = SF.kset(cell, 3.0, 0.05)
    assert np.all(np.diff(ab) == np.minimum(np.diff(fb), 40))
    assert np.diff(fb).max() > 40                              # some bins were sampled
    want, wb, _ = SO.kset_brute(cell, 3.0, 0.05, max_k_per_bin=40, seed=7)
    assert np.array_equal(a, want) and np.array_equal(ab, wb)
    c, cb = SF.kset(cell, 2.2, 0.05, max_k_per_bin=40, seed=7)     # fewer bins: the common ones are the same vectors
    assert np.array_equal(c, a[: cb[-1]]) and np.array_equal(cb, ab[: len(cb)])
    d, db = SF.kset(cell, 3.0, 0.05, max_k_per_bin=40, seed=8)
    assert np.array_equal(db, ab) and not np.array_equal(d, a)
    fs = {tuple(v) for v in full.tolist()}
    assert all(tuple(v) in fs for v in a.tolist())             # a subset of the full set


def test_miller_bound_and_class_limit_raise_value_error():
    with pytest.raises(ValueError, match="Miller"):
        SF.kset((20.0, 20.0, 7000.0, 0, 0, 0), 1.0, 0.5)
    with pytest.raises(ValueError, match="classes"):
        SF.calc_structure_factor(1.0, 0.1, [list(range(1, 40)), list(range(40, 79))], "nonexistent.dump")
    with pytest.raises(ValueError):
        SF.kset(CELLS["cubic"], 0.01, 0.1)


# ------------------------------------------------------------------------------------------------
# the oracle against analytic cases
# ------------------------------------------------------------------------------------------------
def test_two_atoms_give_one_plus_cos():
    cell = CELLS["triclinic"]
    d = np.array([3.3, -1.2, 2.0])
    pos = np.stack([np.array([1.0, 2.0, 3.0]), np.array([1.0, 2.0, 3.0]) + d])
    miller, boff, _ = SO.kset_brute(cell, 2.0, 0.1)
    re, im = SO.rho(cell, pos, miller)
    kv = miller @ SO.recip(cell).T
    assert np.allclose((re * re + im * im) / 2, 1 + np.cos(kv @ d), atol=1e-12)
    P = SO.pair_sums(re[None], im[None], boff)
    tot, part = SO.normalise(P, np.diff(boff), [2], [(0, 0)])
    ok = np.diff(boff) > 0
    want = np.array([np.mean(1 + np.cos(kv[boff[b]:boff[b + 1]] @ d)) for b in np.flatnonzero(ok)])
    assert np.allclose(tot[ok], want, atol=1e-12) and np.allclose(part[0][ok], want, atol=1e-12)
    assert np.all(np.isnan(tot[~ok]))


def test_simple_cubic_crystal_bragg_peaks():
    m, a0 = 4, 3.0
    L = m * a0
    cell = (L, L, L, 0.0, 0.0, 0.0)
    g = np.stack(np.meshgrid(*[np.arange(m)] * 3, indexing="ij"), axis=-1).reshape(-1, 3) * a0 + 0.37
    miller, boff, _ = SO.kset_brute(cell, 4.5, 0.05)
    re, im = SO.rho(cell, g, miller)
    bragg = np.all(miller % m == 0, axis=1)
    assert bragg.any() and (~bragg).any()
    amp = np.hypot(re, im)
    assert np.allclose(amp[bragg], m ** 3, atol=1e-9) and np.abs(amp[~bragg]).max() < 1e-9
    re_l, im_l = SO.rho(cell, g, miller, np.longdouble)
    assert np.abs(np.hypot(re_l, im_l)[~bragg]).max() < 1e-12


def test_sum_rule_of_the_pair_rows():
    """sum_{a<=b} w_ab P_ab = sum_k |rho_total|^2 per bin, on three classes with an empty one."""
    rng = np.random.default_rng(9)
    cell = CELLS["triclinic"]
    pos = rng.uniform(0, 1, (60, 3)) @ SO.cell_matrix(cell).T
    cls = rng.choice([0, 2, 3], 60)
    miller, boff, _ = SO.kset_brute(cell, 1.5, 0.1)
    re, im = SO.class_rho(cell, pos, cls, 4, miller)
    P = SO.pair_sums(re, im, boff)
    w = np.array([1.0 if a == b else 2.0 for a in range(4) for b in range(a, 4)])
    rt, it = SO.rho(cell, pos, miller)
    t = rt * rt + it * it
    want = np.array([t[boff[b]:boff[b + 1]].sum() for b in range(len(boff) - 1)])
    assert np.allclose((w[:, None] * P).sum(axis=0), want, rtol=1e-12, atol=1e-9)
    assert not np.any(P[SO.sym_row(1, 1, 4)]) and not np.any(P[SO.sym_row(0, 1, 4)])
