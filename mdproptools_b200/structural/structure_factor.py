"""Static structure factor S(k): total and partial, by the direct sum over the reciprocal-lattice vectors of the periodic
cell (extension: the reference has no implementation; tests/sk_oracle.py is the definition).

The sine transform of g(r) is truncated at half the box and rings at low k, where the charge-ordering pre-peak of ionic
liquids and electrolytes sits (0.3-1 / A); the direct sum has no such limit.  Definition:

  cell H = [a b c], a = (lx,0,0), b = (xy,ly,0), c = (xz,yz,lz), from the dump's bound extents and tilt (0 when absent);
  k = 2 pi H^-T n for integer Miller triplets n != 0, one of each +-n pair (h > 0, or h = 0 and k > 0, or h = k = 0 and
  l > 0), kept when k_min <= |k| < nbins * bin_size (nbins = int(k_max / bin_size)), in bin floor(|k| / bin_size);
  rho_c(k) = sum_{j in c} exp(i k.r_j) over the atoms of class c (classes from the relation types, as in calc_atomic_rdf);
  P_ab(bin) = sum_{k in bin} Re(rho_a(k) rho_b(k)*);
  S_ab(bin) = P_ab / (n_k sqrt(N_a N_b))  (Ashcroft-Langreth: S_aa -> 1 at large k);
  S(bin) = sum_{a <= b} w_ab P_ab / (n_k N), w = 1 on the diagonal and 2 off it (= <|rho(k)|^2> / N).
Each frame is normalised, then frames are averaged; a bin without k-vectors in a frame does not enter that bin's average,
and a bin without k-vectors in every frame is NaN.

With ``max_k_per_bin`` a bin holding more vectors keeps rng.choice(count, max_k_per_bin, replace=False) of them, counted in
lexicographic (h, k, l) order, with rng = numpy.random.default_rng((seed, bin)): a bin's sample depends on the cell, the bin
and the seed only (not on k_max), and every rank draws the same set without a broadcast.

The device computes rho in fp32 per term from 32-bit fixed-point fractional coordinates, with the phase n.s an exact integer
(csrc/sk_phase.h): |rho_c - rho_c exact| <= 1e-5 N_c for Miller components up to +-1024, which covers k = 10 / A in a 200 A
box.  Frames are sharded over ranks as in calc_atomic_rdf; per-frame fp64 sums are merged by one all-reduce of a
zero-padded [T, ...] tensor (adding zeros is exact), so every rank count gives the same bits.
"""
from __future__ import annotations

import numpy as np
import pandas as pd
import torch

from .. import ops
from .._lib import SK_MAX_CLASSES, SK_NLIM
from ..common.frames import _ClassMap, _frame_batches, file_sharded, merge_results, typed_batches


# ------------------------------------------------------------------------------------------------
# k-set: a pure function of the cell and the arguments
# ------------------------------------------------------------------------------------------------
def _recip(cell):
    lx, ly, lz, xy, xz, yz = (float(v) for v in cell)
    H = np.array([[lx, xy, xz], [0.0, ly, yz], [0.0, 0.0, lz]])
    return H, 2.0 * np.pi * np.linalg.inv(H).T


def _knorm(g, K):
    """|K n| per row of g, written out per component (a BLAS product may round differently from one shape to the next, and
    bins must not depend on how the triplets were grouped)."""
    g = g.astype(np.float64)
    kv = g[:, 0:1] * K[:, 0] + g[:, 1:2] * K[:, 1] + g[:, 2:3] * K[:, 2]
    return np.sqrt((kv[:, 0] * kv[:, 0] + kv[:, 1] * kv[:, 1]) + kv[:, 2] * kv[:, 2])


def _slabs(cell, kc, half):
    """Miller triplets with |k| < kc and their |k|, one h-slab at a time (lexicographic order); |h| <= |a| kc / 2 pi since
    k.a = 2 pi h, and likewise for k and l."""
    H, K = _recip(cell)
    lim = [int(np.floor(np.linalg.norm(H[:, i]) * kc / (2 * np.pi))) for i in range(3)]
    kk, ll = np.meshgrid(np.arange(-lim[1], lim[1] + 1), np.arange(-lim[2], lim[2] + 1), indexing="ij")
    kk, ll = kk.reshape(-1), ll.reshape(-1)
    for h in range(0 if half else -lim[0], lim[0] + 1):
        g = np.stack([np.full_like(kk, h), kk, ll], axis=1)
        if half and h == 0:
            g = g[(kk > 0) | ((kk == 0) & (ll > 0))]
        kn = _knorm(g, K)
        sel = kn < kc
        yield g[sel], kn[sel]


def smallest_k(cell):
    """The smallest nonzero |k| of the cell: it is at most the shortest reciprocal basis vector."""
    _, K = _recip(cell)
    kc = float(np.linalg.norm(K, axis=0).min()) * (1 + 1e-9)
    best = np.inf
    for g, kn in _slabs(cell, kc, half=False):
        nz = np.any(g != 0, axis=1)
        if nz.any():
            best = min(best, float(kn[nz].min()))
    return best


def kset(cell, k_max, bin_size, k_min=None, max_k_per_bin=None, seed=0):
    """(miller int32 [nk, 3] sorted by bin, lexicographic inside a bin; bin_off int64 [nbins + 1]).  Enumerated in h-slabs:
    without ``max_k_per_bin`` memory is the kept set; with it, a first pass counts each bin, the samples are drawn, and a
    second pass keeps the drawn ordinals (memory: the samples and one slab)."""
    nbins = int(k_max / bin_size)
    if nbins < 1:
        raise ValueError(f"k_max = {k_max} is below one bin of {bin_size}")
    kc = nbins * bin_size
    k_min = smallest_k(cell) if k_min is None else float(k_min)

    def binned():
        for g, kn in _slabs(cell, kc, half=True):
            sel = kn >= k_min
            yield g[sel], np.floor(kn[sel] / bin_size).astype(np.int64)

    chosen = None
    if max_k_per_bin is not None:
        counts = np.zeros(nbins, dtype=np.int64)
        for _, b in binned():
            counts += np.bincount(b, minlength=nbins)
        keys = []
        for b in np.flatnonzero(counts > int(max_k_per_bin)):
            idx = np.random.default_rng((seed, int(b))).choice(int(counts[b]), size=int(max_k_per_bin), replace=False)
            keys.append(int(b) * (1 << 40) + np.sort(idx))
        chosen = (np.sort(np.concatenate(keys)) if keys else np.zeros(0, dtype=np.int64), counts > int(max_k_per_bin))
    seen = np.zeros(nbins, dtype=np.int64)
    parts, bins = [], []
    for g, b in binned():
        if chosen is not None:
            order = np.argsort(b, kind="stable")
            first = np.searchsorted(b[order], b[order], side="left")
            ordinal = np.empty_like(b)
            ordinal[order] = np.arange(len(b)) - first
            ordinal += seen[b]
            seen += np.bincount(b, minlength=nbins)
            key = b * (1 << 40) + ordinal
            pos = np.searchsorted(chosen[0], key)
            hit = (pos < len(chosen[0])) & (chosen[0][np.minimum(pos, len(chosen[0]) - 1)] == key) if len(chosen[0]) else \
                np.zeros(len(b), dtype=bool)
            keep = ~chosen[1][b] | hit
            g, b = g[keep], b[keep]
        parts.append(g)
        bins.append(b)
    g = np.concatenate(parts) if parts else np.zeros((0, 3), dtype=np.int64)
    b = np.concatenate(bins) if bins else np.zeros(0, dtype=np.int64)
    order = np.argsort(b, kind="stable")
    g, b = g[order], b[order]
    if len(g) and int(np.abs(g).max()) > SK_NLIM:
        raise ValueError(f"k_max = {k_max} needs Miller indices up to {int(np.abs(g).max())} in this cell; the device's accuracy "
                         f"contract covers |n| <= {SK_NLIM}")
    bin_off = np.concatenate(([0], np.cumsum(np.bincount(b, minlength=nbins)))).astype(np.int64)
    return np.ascontiguousarray(g, dtype=np.int32), bin_off


class _KSetCache:
    """kset() of the last cells seen (an NVT trajectory: one entry)."""

    def __init__(self, *args):
        self.args, self.val = args, {}

    def get(self, cell):
        v = self.val.get(cell)
        if v is None:
            if len(self.val) >= 16:
                self.val.clear()
            v = self.val[cell] = kset(cell, *self.args)
        return v


def _cell(box):
    lengths = box.bound_lengths()
    tilt = box.tilt if box.tilt is not None else (0.0, 0.0, 0.0)
    return tuple(float(v) for v in tuple(lengths) + tuple(tilt))


def _save_sk(k, relation_matrix, path_or_buff, save_mode, s_tot, s_part, nk_mean):
    labels = ["k ($\\AA^{-1}$)", "S(k)"] + [f"S_{str(p[0])}-{str(p[1])}" for p in relation_matrix] + ["n_k"]
    df = pd.DataFrame(np.vstack((k, s_tot, s_part, nk_mean)).transpose(), columns=labels)
    if save_mode:
        df.to_csv(path_or_buff, index=False)
    return df


# ------------------------------------------------------------------------------------------------
# public API
# ------------------------------------------------------------------------------------------------
@file_sharded
def calc_structure_factor(k_max, bin_size, partial_relations, filename, k_min=None, max_k_per_bin=None, seed=0, num_mols=None,
                          num_atoms_per_mol=None, path_or_buff="sk.csv", save_mode=True, *, shard_files=True):
    """Total and partial static structure factor of the frames of ``filename`` (LAMMPS dump(s) with id type x y z).

    k_max, bin_size   bins [b bin_size, (b+1) bin_size) for b < int(k_max / bin_size), in 1/A
    partial_relations [[a...], [b...]] type pairs, as for calc_atomic_rdf (altered types with num_mols/num_atoms_per_mol)
    k_min             smallest |k| kept (default: the smallest nonzero |k| of the cell, i.e. all vectors)
    max_k_per_bin     keep at most this many k-vectors per bin (a seeded uniform sample, see the module docstring)
    Returns a DataFrame with columns k (bin centres), S(k), S_a-b per relation, n_k (mean k-vectors per frame and bin);
    written to ``path_or_buff`` as CSV when ``save_mode``.
    """
    nbins = int(k_max / bin_size)
    if nbins < 1:
        raise ValueError(f"k_max = {k_max} is below one bin of {bin_size}")
    relation_matrix = np.asarray(partial_relations).transpose()
    named = list(partial_relations[0]) + list(partial_relations[1])
    cmap = _ClassMap(named)                 # 'other' always present: the same class rows on every rank
    if cmap.ncls > SK_MAX_CLASSES:
        raise ValueError(f"{cmap.ncls} classes ({cmap.ncls - 1} relation types + other) exceed the kernel's {SK_MAX_CLASSES}")
    rows = ops.sym_rows(cmap.ncls)
    kcache = _KSetCache(k_max, bin_size, k_min, max_k_per_bin, seed)

    def frame_cell(meta, at):
        for t in named:
            if at.get(int(t), 0) == 0:
                raise ValueError(f"no atom of type {t} in frame {meta.index} (timestep {meta.timestep})")
        return _cell(meta.box)

    batches = _frame_batches(filename, ["id", "type", "x", "y", "z"], shard_files)
    sums, props = {}, {}
    for b in typed_batches(batches, num_mols, num_atoms_per_mol, frame_cell, cmap=cmap):
        cells, F = b.props, len(b.metas)
        xyz = b.dev[:, 2:5, :]
        k0 = 0
        while k0 < F:                       # one call per run of frames sharing a cell (all of an NVT batch)
            k1 = k0 + 1
            while k1 < F and cells[k1] == cells[k0]:
                k1 += 1
            miller, bin_off = kcache.get(cells[k0])
            cls_d = b.classes(k0, k1)
            out = ops.structure_factor(xyz[k0:k1].contiguous(), cls_d, cmap.ncls, cells[k0], miller, bin_off, nbins)
            nk = np.diff(bin_off)
            for j in range(k0, k1):
                meta = b.metas[j]
                sums[meta.index] = out[j - k0]
                props[meta.index] = (b.atom_types[j], meta.natoms, nk)
            k0 = k1
    allp, props, T = merge_results(batches, sums, props, filename, (rows, nbins), torch.float64)

    w = np.array([1.0 if a == b else 2.0 for a in range(cmap.ncls) for b in range(a, cmap.ncls)])
    prow = [ops.sym_row(cmap.cls(a), cmap.cls(b), cmap.ncls) for a, b in relation_matrix]
    s_tot = np.zeros(nbins)
    s_part = np.zeros((len(prow), nbins))
    used = np.zeros(nbins, dtype=np.int64)
    nk_sum = np.zeros(nbins)
    for idx in range(T):
        at, natoms, nk = props[idx]
        ok = nk > 0
        P = allp[idx][:, ok]
        d = nk[ok].astype(np.float64)
        s_tot[ok] += (w[:, None] * P).sum(axis=0) / (d * natoms)
        for r, (a, b) in enumerate(relation_matrix):
            s_part[r, ok] += P[prow[r]] / (d * np.sqrt(float(at[int(a)]) * float(at[int(b)])))
        used += ok
        nk_sum += nk
    with np.errstate(invalid="ignore", divide="ignore"):
        s_tot = np.where(used > 0, s_tot / used, np.nan)
        s_part = np.where(used > 0, s_part / used, np.nan)
    k = (np.arange(nbins) + 0.5) * bin_size
    return _save_sk(k, relation_matrix, path_or_buff, save_mode, s_tot, s_part, nk_sum / T)
