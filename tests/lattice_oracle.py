"""Exact pair histograms of simple-cubic lattice frames, from per-axis difference counts (never from pairs).

A frame is one or more blocks.  Block b holds the points  origin_b + h * (ix, iy, iz)  for 0 <= i_a < m_a (in C order
over (ix, iy, iz)); a point's class is  ix mod K.  Coordinates may be wrapped into the orthogonal cell [0, L).

Every pair's displacement then depends only on the two blocks and the integer difference vector D = i - j, and the
number of index pairs with difference k along one axis is a trapezoid in k (split by class along x).  So the histogram
of all pairs of a 10^6-point frame (10^12 pairs) is a sum over the (2m - 1)^3 difference vectors of each block pair.

The semantics are the oracle's (oracle/oracle.c), restated for the difference vector:
  - orthogonal: per axis the single-shift minimum image with strict compares at +-L/2, rsq = (dx*dx + dy*dy) + dz*dz;
  - triclinic (cell = lx, ly, lz, xy, xz, yz): the sequential z, y, x shift of pair_rsq_tri;
  - a pair counts when rsq < rcut_sq(r_cut); uniform bins: bin = int64(sqrt(rsq) / ddr), an index >= nbins is dropped;
    table bins (coordination thresholds on rsq): bin k when edges[k] <= rsq < edges[k + 1], k < nbins.

Exactness condition (asserted by ``Frame``): every coordinate, spacing, box length and tilt is an integer multiple of
2^-q with magnitude below 2^p, and p + q <= 22.  Then every difference, shift and square, and the sum of three squares,
is an integer multiple of 2^-2q below 2^53 * 2^-2q, so each is exact in fp64 and the closed form and the brute force
compute the same rsq bit for bit.  Under the same condition, and when each axis's unwrapped extent is below L, wrapping
the block into the cell changes no pair's rsq: both the stored and the unwrapped difference lie in (-L, L), and the
single shift maps either to the minimum-image magnitude (L/2 itself, at a tie, on both sides).  The triclinic image
depends on the sign of each intermediate component at a tie (a z tie decides whether dy and dx move by the tilts), so
the same lattice stored wrapped differently can give other distances.  Triclinic frames are therefore never wrapped,
and a triclinic frame may hold no exact half-cell tie anywhere in its image sequence (asserted) unless it is built with
``ties_ok=True``: unwrapped, the stored difference is the closed form's, and the host tests use such a frame to pin the
strict compares of the tie itself.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np

EXACT_BITS = 22


def sym_rows(K: int) -> int:
    return K * (K + 1) // 2


def sym_row(a: int, b: int, K: int) -> int:
    """Row of the unordered class pair {a, b} in the symmetric histogram (the layout of ops.pair_hist)."""
    a, b = (a, b) if a <= b else (b, a)
    return a * K - a * (a - 1) // 2 + (b - a)


@dataclass(frozen=True)
class Block:
    m: tuple            # points per axis (mx, my, mz)
    origin: tuple       # coordinates of index (0, 0, 0)


def _dyadic(v: float) -> tuple:
    """(q, p): v = k * 2^-q with the smallest q >= 0 (every finite double is dyadic), and |v| < 2^p."""
    q = float(v).as_integer_ratio()[1].bit_length() - 1
    p = 0 if v == 0 else math.floor(math.log2(abs(v))) + 1
    return q, p


class Frame:
    """Blocks with spacing h and K classes in a cell (lx, ly, lz) or, triclinic, (lx, ly, lz, xy, xz, yz)."""

    def __init__(self, blocks, h, cell, K=1, wrap=False, ties_ok=False):
        self.blocks = [b if isinstance(b, Block) else Block(*b) for b in blocks]
        self.h = float(h)
        self.cell = tuple(float(c) for c in cell)
        assert len(self.cell) in (3, 6)
        self.tri = len(self.cell) == 6
        self.K = int(K)
        self.wrap = bool(wrap)
        assert not (self.tri and self.wrap), "triclinic frames are stored unwrapped"
        self.ties_ok = bool(ties_ok)
        vals = [self.h, *self.cell]
        for b in self.blocks:
            for a in range(3):
                vals += [b.origin[a], b.origin[a] + self.h * (b.m[a] - 1)]
        q = max(_dyadic(v)[0] for v in vals)
        p = max(_dyadic(v)[1] for v in vals)
        assert p + q <= EXACT_BITS, f"coordinates need {p} + {q} bits, more than {EXACT_BITS}: fp64 sums would round"
        if self.wrap:
            for a in range(3):
                lo = min(b.origin[a] for b in self.blocks)
                hi = max(b.origin[a] + self.h * (b.m[a] - 1) for b in self.blocks)
                assert hi - lo < self.cell[a], "wrapping keeps every rsq only when each axis's extent is below L"

    @property
    def n(self) -> int:
        return sum(int(np.prod(b.m)) for b in self.blocks)

    def positions(self):
        """(xyz float64 [3, N], cls int32 [N]) in block order, C order over (ix, iy, iz) inside a block."""
        xyz, cls = [], []
        for b in self.blocks:
            ix, iy, iz = np.meshgrid(*[np.arange(m) for m in b.m], indexing="ij")
            pts = np.stack([b.origin[a] + self.h * i.reshape(-1) for a, i in enumerate((ix, iy, iz))])
            if self.wrap:
                pts = np.mod(pts, np.asarray(self.cell[:3])[:, None])
                assert np.all((pts >= 0) & (pts < np.asarray(self.cell[:3])[:, None]))
            xyz.append(pts)
            cls.append((ix.reshape(-1) % self.K).astype(np.int32))
        return np.ascontiguousarray(np.concatenate(xyz, axis=1)), np.concatenate(cls)

    def class_counts(self):
        c = np.zeros(self.K, dtype=np.int64)
        for b in self.blocks:
            c += np.bincount(np.arange(b.m[0]) % self.K, minlength=self.K) * (b.m[1] * b.m[2])
        return c


# ---- binning rules -----------------------------------------------------------------------------------------------------
def uniform_bins(ddr, nbins, rcut2):
    """rsq -> int64(sqrt(rsq) / ddr) for rsq < rcut2, -1 otherwise or when the index reaches nbins."""
    def f(rsq):
        b = (np.sqrt(rsq) / ddr).astype(np.int64)
        return np.where((rsq < rcut2) & (b < nbins), b, -1)
    f.nbins = int(nbins)
    return f


def table_bins(edges, rcut2):
    """rsq -> k with edges[k] <= rsq < edges[k + 1] (edges[0] not read), for rsq < rcut2 and k < nbins."""
    edges = np.asarray(edges, dtype=np.float64)
    nb = len(edges) - 1

    def f(rsq):
        b = np.searchsorted(edges[1:], rsq, side="right").astype(np.int64)
        return np.where((rsq < rcut2) & (b < nb), b, -1)
    f.nbins = nb
    return f


# ---- closed form -------------------------------------------------------------------------------------------------------
def _axis_counts(mp: int, mq: int, KP: int = 1, KQ: int = 1):
    """ks = -(mq - 1) .. mp - 1 and c[a, b, t] = #{(i, j): 0 <= i < mp, 0 <= j < mq, i - j = ks[t], i mod KP = a,
    j mod KQ = b}: the trapezoid min(mp, mq + k) - max(0, k), split by class."""
    ks = np.arange(-(mq - 1), mp)
    c = np.zeros((KP, KQ, len(ks)), dtype=np.int64)
    for t, k in enumerate(ks):
        j = np.arange(max(0, -k), min(mq, mp - k))     # i = j + k inside [0, mp)
        c[:, :, t] = np.bincount(((j + k) % KP) * KQ + j % KQ, minlength=KP * KQ).reshape(KP, KQ)
    return ks, c


def _mic1(d, l):
    return np.where(d > l / 2, d - l, np.where(d < -(l / 2), d + l, d))


def _ordered(P: Block, Q: Block, binner, KP: int, KQ: int, cell, h, ties_ok):
    """[KP, KQ, nbins] counts of ordered pairs (p in P, q in Q), p == q included, displacement x_p - x_q."""
    kx, cx = _axis_counts(P.m[0], Q.m[0], KP, KQ)
    ky, cy = _axis_counts(P.m[1], Q.m[1])
    kz, cz = _axis_counts(P.m[2], Q.m[2])
    dxv = (P.origin[0] - Q.origin[0]) + h * kx.astype(np.float64)
    dyv = (P.origin[1] - Q.origin[1]) + h * ky.astype(np.float64)
    dzv = (P.origin[2] - Q.origin[2]) + h * kz.astype(np.float64)
    w2 = (cy[0, 0][:, None] * cz[0, 0][None, :]).astype(np.float64)       # products < 2^53: float bincount stays exact
    nb = binner.nbins
    H = np.zeros((len(kx), nb), dtype=np.int64)
    if len(cell) == 3:
        ax2 = _mic1(dxv, cell[0]) ** 2
        ay2 = _mic1(dyv, cell[1]) ** 2
        az2 = _mic1(dzv, cell[2]) ** 2
    else:
        lx, ly, lz, xy, xz, yz = cell
        dz = np.broadcast_to(dzv[None, :], w2.shape)
        dy = np.broadcast_to(dyv[:, None], w2.shape)
        ties = [np.abs(dz) == lz / 2]
        sz = np.where(dz > lz / 2, -1.0, np.where(dz < -(lz / 2), 1.0, 0.0))
        dz = dz + sz * lz
        dy = dy + sz * yz
        ties.append(np.abs(dy) == ly / 2)
        sy = np.where(dy > ly / 2, -1.0, np.where(dy < -(ly / 2), 1.0, 0.0))
        dy = dy + sy * ly
        dz2, dy2 = dz * dz, dy * dy
    for t in range(len(kx)):
        if len(cell) == 3:
            rsq = (ax2[t] + ay2)[:, None] + az2[None, :]
        else:
            dx = dxv[t] + sz * xz + sy * xy
            assert ties_ok or not (np.any(ties[0]) or np.any(ties[1]) or np.any(np.abs(dx) == lx / 2)), \
                "triclinic frame with an exact half-cell tie"
            dx = np.where(dx > lx / 2, dx - lx, np.where(dx < -(lx / 2), dx + lx, dx))
            rsq = (dx * dx + dy2) + dz2
        b = binner(rsq)
        keep = b >= 0
        s = np.bincount(b[keep], weights=w2[keep], minlength=nb)
        assert np.all(s < 2.0 ** 53)
        H[t] = s.astype(np.int64)
    return np.tensordot(cx, H, axes=([2], [0]))


def hist_sym(fr: Frame, binner):
    """Unordered pairs of the frame: int64 [K(K+1)/2, nbins], row sym_row(a, b) (what ops.pair_hist returns)."""
    K = fr.K
    ordered = np.zeros((K, K, binner.nbins), dtype=np.int64)
    for P in fr.blocks:
        for Q in fr.blocks:
            ordered += _ordered(P, Q, binner, K, K, fr.cell, fr.h, fr.ties_ok)
    b0 = int(binner(np.zeros(1))[0])
    if b0 >= 0:                                            # the self pairs (D = 0 inside one block) have rsq = 0
        for a, c in enumerate(fr.class_counts()):
            ordered[a, a, b0] -= c
    assert np.array_equal(ordered, ordered.transpose(1, 0, 2)), "rsq(D) = rsq(-D) for both images"
    out = np.zeros((sym_rows(K), binner.nbins), dtype=np.int64)
    for a in range(K):
        assert np.all(ordered[a, a] % 2 == 0)
        out[sym_row(a, a, K)] = ordered[a, a] // 2
        for b in range(a + 1, K):
            out[sym_row(a, b, K)] = ordered[a, b]
    return out


def hist_rect(fa: Frame, fb: Frame, binner):
    """Pairs (a in A, b in B), displacement x_a - x_b: int64 [KA * KB, nbins], row ka * KB + kb."""
    assert fa.cell == fb.cell and fa.h == fb.h
    out = np.zeros((fa.K, fb.K, binner.nbins), dtype=np.int64)
    for P in fa.blocks:
        for Q in fb.blocks:
            out += _ordered(P, Q, binner, fa.K, fb.K, fa.cell, fa.h, fa.ties_ok and fb.ties_ok)
    return out.reshape(fa.K * fb.K, binner.nbins)


# ---- the oracle's outputs, from the histograms (types = class + 1) -----------------------------------------------------
def rdf_loop_counts(sym, rel, K):
    """(full, part) as O.rdf_loop returns them: full = 2 per pair; part[k] counts a pair once per matching role order."""
    full = 2 * sym.sum(axis=0)
    part = np.stack([(2 if a == b else 1) * sym[sym_row(a - 1, b - 1, K)] for a, b in np.asarray(rel).reshape(-1, 2)])
    return full, part


def cn_thresholds(r_cuts):
    """(edges, rcut2) of the table-bin call that answers O.cn_loop for these cutoffs: thresholds = sorted distinct rcut^2."""
    from oracle.oracle import rcut_sq
    thr = np.unique([rcut_sq(r) for r in r_cuts])
    return np.concatenate(([0.0], thr)), float(thr[-1])


def cn_loop_counts(cum, rel, r_cuts, K):
    """O.cn_loop from a cumulative table histogram (column k = pairs with rsq < k-th threshold)."""
    from oracle.oracle import rcut_sq
    thr, _ = cn_thresholds(r_cuts)
    out = []
    for (a, b), r in zip(np.asarray(rel).reshape(-1, 2), r_cuts):
        k = int(np.searchsorted(thr[1:], rcut_sq(r)))
        out.append((2 if a == b else 1) * cum[sym_row(a - 1, b - 1, K), k])
    return np.asarray(out, dtype=np.int64)


def rect_counts(rect, rel, KB):
    """O.rdf_rect: part[k] = pairs with type_a == a and type_b == b."""
    return np.stack([rect[(a - 1) * KB + (b - 1)] for a, b in np.asarray(rel).reshape(-1, 2)])
