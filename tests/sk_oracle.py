"""numpy restatement of the static structure factor (mdproptools_b200/structural/structure_factor.py, csrc/sk.cu).  The
reference has no implementation, so this is the definition the library is checked against:

  cell H = [a b c], a = (lx,0,0), b = (xy,ly,0), c = (xz,yz,lz); k = 2 pi H^-T n for integer n != 0, one of each +-n pair
  (h > 0, or h = 0 and k > 0, or h = k = 0 and l > 0), kept when k_min <= |k| < nbins * bin_size, bin floor(|k| / bin_size);
  a bin with more than max_k_per_bin vectors keeps rng.choice(count, max_k_per_bin, replace=False) of them (in
  lexicographic (h, k, l) order, rng = numpy.random.default_rng((seed, bin)));
  rho_c(k) = sum_{j in c} exp(2 pi i n.s_j), s = H^-1 r;  P_ab(bin) = sum_{k in bin} Re(rho_a rho_b*);
  S_ab = P_ab / (n_k sqrt(N_a N_b));  S = sum_{a<=b} w_ab P_ab / (n_k N), w = 1 on the diagonal, 2 off it;
  per frame, then averaged over the frames in which the bin has vectors (NaN when it never has).
"""
from __future__ import annotations

import numpy as np


def cell_matrix(cell):
    lx, ly, lz, xy, xz, yz = (float(v) for v in cell)
    return np.array([[lx, xy, xz], [0.0, ly, yz], [0.0, 0.0, lz]])          # columns a, b, c


def recip(cell):
    """K with k = K @ n (2 pi H^-T)."""
    return 2.0 * np.pi * np.linalg.inv(cell_matrix(cell)).T


def kset_brute(cell, k_max, bin_size, k_min=None, max_k_per_bin=None, seed=0):
    """(miller int [nk,3] sorted by bin, lexicographic inside a bin; bin_off [nbins+1]; nbins) by a brute force over the
    bounding box of the sphere."""
    nbins = int(k_max / bin_size)
    kc = nbins * bin_size
    H = cell_matrix(cell)
    K = recip(cell)
    lim = [int(np.floor(np.linalg.norm(H[:, i]) * kc / (2 * np.pi))) for i in range(3)]
    g = np.stack(np.meshgrid(*[np.arange(-m, m + 1) for m in lim], indexing="ij"), axis=-1).reshape(-1, 3)
    h, k, l = g[:, 0], g[:, 1], g[:, 2]
    half = (h > 0) | ((h == 0) & (k > 0)) | ((h == 0) & (k == 0) & (l > 0))
    g = g[half]
    kn = knorm(g, K)
    if k_min is None:
        k_min = smallest_k(cell)
    keep = (kn >= k_min) & (kn < kc)
    g, kn = g[keep], kn[keep]
    b = np.floor(kn / bin_size).astype(np.int64)
    order = np.argsort(b, kind="stable")
    g, b = g[order], b[order]
    out, counts = [], np.zeros(nbins, dtype=np.int64)
    for bb in range(nbins):
        sel = g[b == bb]
        if max_k_per_bin is not None and len(sel) > max_k_per_bin:
            idx = np.sort(np.random.default_rng((seed, bb)).choice(len(sel), size=max_k_per_bin, replace=False))
            sel = sel[idx]
        out.append(sel)
        counts[bb] = len(sel)
    miller = np.concatenate(out) if out else np.zeros((0, 3), dtype=np.int64)
    return miller.astype(np.int64), np.concatenate(([0], np.cumsum(counts))), nbins


def smallest_k(cell):
    """smallest nonzero |k| of the cell (brute force over n in [-3, 3]^3)."""
    K = recip(cell)
    r = np.arange(-3, 4)
    g = np.stack(np.meshgrid(r, r, r, indexing="ij"), axis=-1).reshape(-1, 3)
    g = g[np.any(g != 0, axis=1)]
    return float(knorm(g, K).min())


def knorm(g, K):
    """|K n| per row, component by component in a fixed order."""
    g = g.astype(np.float64)
    kv = g[:, 0:1] * K[:, 0] + g[:, 1:2] * K[:, 1] + g[:, 2:3] * K[:, 2]
    return np.sqrt((kv[:, 0] * kv[:, 0] + kv[:, 1] * kv[:, 1]) + kv[:, 2] * kv[:, 2])


def rho(cell, pos, miller, dtype=np.float64):
    """rho(k) for positions pos [N,3] (Cartesian) in fp64 or long double: [nk] complex (as (re, im) pairs of dtype)."""
    H = np.asarray(cell_matrix(cell), dtype=dtype)
    s = np.linalg.solve(H.astype(np.float64), np.asarray(pos, dtype=np.float64).T).T if dtype == np.float64 else \
        _solve_ld(H, np.asarray(pos, dtype=dtype))
    ph = (np.asarray(miller, dtype=dtype) @ s.T.astype(dtype))                  # [nk, N] cycles
    ph = ph - np.floor(ph)
    ang = ph * (2 * np.asarray(np.pi, dtype=dtype) if dtype == np.float64 else 2 * _PI_LD)
    return np.cos(ang).sum(axis=1), np.sin(ang).sum(axis=1)


_PI_LD = np.longdouble("3.14159265358979323846264338327950288")


def _solve_ld(H, pos):
    """back substitution through the upper-triangular H in long double."""
    lx, xy, xz, ly, yz, lz = H[0, 0], H[0, 1], H[0, 2], H[1, 1], H[1, 2], H[2, 2]
    sc = pos[:, 2] / lz
    sb = (pos[:, 1] - sc * yz) / ly
    sa = (pos[:, 0] - sb * xy - sc * xz) / lx
    return np.stack([sa, sb, sc], axis=1)


def class_rho(cell, pos, cls, ncls, miller, dtype=np.float64):
    """[ncls, nk] (re, im) per class."""
    re = np.zeros((ncls, len(miller)), dtype=dtype)
    im = np.zeros((ncls, len(miller)), dtype=dtype)
    for c in range(ncls):
        sel = np.asarray(cls) == c
        if sel.any() and len(miller):
            re[c], im[c] = rho(cell, np.asarray(pos)[sel], miller, dtype)
    return re, im


def pair_sums(re, im, bin_off):
    """P[row(a,b)][bin] = sum_{k in bin} Re(rho_a conj(rho_b)), rows a <= b in the pair engine's order."""
    ncls = re.shape[0]
    nbins = len(bin_off) - 1
    rows = []
    for a in range(ncls):
        for b in range(a, ncls):
            t = re[a] * re[b] + im[a] * im[b]
            rows.append([t[bin_off[q]:bin_off[q + 1]].sum() for q in range(nbins)])
    return np.asarray(rows, dtype=np.float64).reshape(len(rows), nbins)


def sym_row(a, b, ncls):
    a, b = min(a, b), max(a, b)
    return a * ncls - a * (a - 1) // 2 + (b - a)


def normalise(P, nk, class_counts, relations):
    """One frame: (S [nbins], S_ab [R, nbins]) with NaN where n_k = 0.  relations = [(class a, class b)]."""
    ncls = len(class_counts)
    N = float(np.sum(class_counts))
    w = np.array([1.0 if a == b else 2.0 for a in range(ncls) for b in range(a, ncls)])
    nk = np.asarray(nk, dtype=np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        tot = (w[:, None] * P).sum(axis=0) / (nk * N)
        part = np.stack([P[sym_row(a, b, ncls)] / (nk * np.sqrt(float(class_counts[a]) * float(class_counts[b])))
                         for a, b in relations]) if relations else np.zeros((0, len(nk)))
    tot[nk == 0] = np.nan
    part[:, nk == 0] = np.nan
    return tot, part


def average(per_frame):
    """mean over frames ignoring NaN entries; NaN where every frame is NaN."""
    a = np.asarray(per_frame, dtype=np.float64)
    cnt = np.sum(~np.isnan(a), axis=0)
    s = np.nansum(a, axis=0)
    with np.errstate(invalid="ignore", divide="ignore"):
        out = s / cnt
    out[cnt == 0] = np.nan
    return out


def structure_factor(frames, k_max, bin_size, relations_types, k_min=None, max_k_per_bin=None, seed=0):
    """frames = [(cell, pos [N,3], types [N])] -> (k centres, S, S_ab [R, nbins], mean n_k)."""
    named = sorted(set(int(t) for pair in relations_types for t in pair))
    tot_f, part_f, nk_f = [], [], []
    for cell, pos, types in frames:
        types = np.asarray(types).astype(np.int64)
        cls = np.array([named.index(t) if t in named else len(named) for t in types])
        ncls = len(named) + 1
        miller, bin_off, nbins = kset_brute(cell, k_max, bin_size, k_min, max_k_per_bin, seed)
        re, im = class_rho(cell, pos, cls, ncls, miller)
        P = pair_sums(re, im, bin_off)
        counts = np.bincount(cls, minlength=ncls)
        rel = [(named.index(int(a)), named.index(int(b))) for a, b in relations_types]
        nk = np.diff(bin_off)
        t, p = normalise(P, nk, counts, rel)
        tot_f.append(t)
        part_f.append(p)
        nk_f.append(nk)
    nbins = int(k_max / bin_size)
    return (np.arange(nbins) + 0.5) * bin_size, average(tot_f), average(part_f), np.mean(nk_f, axis=0)
