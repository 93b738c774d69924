"""Coherent intermediate scattering function F(k, t): total and partial, from the collective densities rho_c(k, t) over the
reciprocal-lattice vectors of the periodic cell (extension: the reference has no implementation; tests/isf_oracle.py is
the definition).

F(k, t) is the dynamical companion of S(k) (structural/structure_factor.py): its decay at the charge-ordering pre-peak and at
the main peak is the collective relaxation of an electrolyte or ionic liquid, and it is what neutron spin-echo data is
compared against.  Definition, for T >= 2 evenly spaced frames that share one cell, one atom count and one type column:

  the k-set and bins of ``structure_factor.kset`` (same arguments -> the bins of calc_structure_factor);
  z_c(k, t) = rho_c(k, t) = sum_{j in c} exp(i k.r_j(t)) per class (classes from the relation types, as in S(k)), and the
  total z_t = sum over every class, the unnamed types included;
  C_ab(k, tau) = 1/(T - tau) sum_{t < T-tau} 1/2 Re( z_a(k,t+tau) z_b(k,t)* + z_b(k,t+tau) z_a(k,t)* ),  tau < max_lag;
  F_ab(bin, tau) = sum_{k in bin} C_ab(k, tau) / (n_k sqrt(N_a N_b)),  F(bin, tau) = sum_{k in bin} C_tt(k, tau) / (n_k N);
  lag time t = tau * (timestep difference) * timestep * TIME_CONVERSION[units] in seconds.
At tau = 0 these are calc_structure_factor's S_ab and S over the same frames.  A bin without k-vectors is NaN.

Device work: rho per class, k-vector and frame by the S(k) kernel (mdp_sk_rho, csrc/sk.cu), written batch by batch into a
[classes + 1, k, T] series; the binned, symmetrised correlation of every pair through the FFT (mdp_isf_fft, csrc/isffft.cu).
rho is not centred: its time mean is physical (Bragg peaks).

Multi-GPU: every rank reads every frame; the bins are split into contiguous ranges balanced by k count (``shard_bins``), each
rank computes rho and the correlation of its bins' k-vectors only, and one fp64 all-reduce of the zero-padded
[pairs, bins, lags] sums merges them (adding zeros is exact, so every rank count gives the same bits).
"""
from __future__ import annotations

import numpy as np
import pandas as pd
import torch

from .. import dist, ops
from .._lib import SK_MAX_CLASSES
from ..common import constants
from ..common.frames import _ClassMap, _value_counts, calc_atom_type_ids
from ..io.dump import dump_files
from ..io.pipeline import FrameBatches
from ..structural.structure_factor import _cell, kset
from .series import even_times


def shard_bins(bin_off, r, w):
    """Contiguous bins [lo, hi) of rank r of w, balanced by k-vector count: rank q ends after the last bin that ends at or
    before floor((q + 1) nk / w) k-vectors (the last rank ends at the last bin).  A pure function of its arguments."""
    bin_off = np.asarray(bin_off, dtype=np.int64)
    nbins, nk = len(bin_off) - 1, int(bin_off[-1])

    def cut(q):
        if q <= 0:
            return 0
        if q >= w:
            return nbins
        return int(np.searchsorted(bin_off[1:], (q * nk) // w, side="right"))

    return cut(r), cut(r + 1)


def _series_buffer(nchan, nk, frames, device, old=None):
    """[nchan, nk, frames] complex128 on the device (the first columns of ``old`` copied over); ValueError when it does not
    fit the device's free memory."""
    need = nchan * nk * frames * 16
    free = torch.cuda.mem_get_info(device)[0]
    if need > free:
        raise ValueError(f"the rho series of {nchan} channels x {nk} k-vectors x {frames} frames ({need / 2 ** 30:.2f} GiB) "
                         f"exceeds the device's free memory ({free / 2 ** 30:.2f} GiB): lower max_k_per_bin or raise k_min")
    buf = torch.empty((nchan, nk, frames), dtype=torch.complex128, device=device)
    if old is not None:
        buf[:, :, :old.shape[2]] = old
    return buf


def lag_times(steps, nlags, timestep, units, source):
    """t (s) of lags 0 .. nlags-1 from the timesteps of all frames (in trajectory order), which must be evenly spaced."""
    even_times(steps, units, timestep, source, who="the intermediate scattering function needs")
    return np.arange(nlags) * (float(steps[1] - steps[0]) * timestep * constants.TIME_CONVERSION[units])


def isf_table(sums, bin_off, natoms, counts, relation_matrix, bin_size, t):
    """The returned table from the binned correlation sums [1 + relations, nbins, nlags] (row 0 the total pair): columns
    k, t (s), F(k,t), F_a-b per relation, n_k; one row per (bin, lag), bin-major; NaN in the rows of a bin without
    k-vectors.  counts: atoms per type."""
    nbins, L = sums.shape[1], sums.shape[2]
    nk = np.diff(np.asarray(bin_off)).astype(np.float64)
    ok = nk > 0
    f_tot = np.full((nbins, L), np.nan)
    f_part = np.full((len(relation_matrix), nbins, L), np.nan)
    f_tot[ok] = sums[0, ok] / (nk[ok, None] * natoms)
    for q, (a, b) in enumerate(relation_matrix):
        f_part[q, ok] = sums[1 + q, ok] / (nk[ok, None] * np.sqrt(float(counts[int(a)]) * float(counts[int(b)])))
    k = (np.arange(nbins) + 0.5) * bin_size
    labels = ["k ($\\AA^{-1}$)", "t (s)", "F(k,t)"] + [f"F_{str(p[0])}-{str(p[1])}" for p in relation_matrix] + ["n_k"]
    cols = [np.repeat(k, L), np.tile(t, nbins), f_tot.reshape(-1)] + [p.reshape(-1) for p in f_part] + [np.repeat(nk, L)]
    return pd.DataFrame(np.stack(cols, axis=1), columns=labels)


def calc_intermediate_scattering(k_max, bin_size, partial_relations, filename, max_lag=None, timestep=1, units="real",
                                 k_min=None, max_k_per_bin=None, seed=0, num_mols=None, num_atoms_per_mol=None,
                                 path_or_buff="isf.csv", save_mode=True):
    """Total and partial coherent intermediate scattering function of the frames of ``filename`` (LAMMPS dump(s) with
    id type x y z; evenly spaced timesteps, one cell, fixed atom count and types).

    k_max, bin_size, partial_relations, k_min, max_k_per_bin, seed, num_mols, num_atoms_per_mol   as for calc_structure_factor
    max_lag           lags tau < max_lag, in [1, T] (default T // 2)
    timestep, units   the MD timestep and the LAMMPS unit style of the lag-time axis
    Returns a DataFrame with columns k (bin centres), t (s), F(k,t), F_a-b per relation, n_k, one row per (bin, lag) in
    bin-major order; written to ``path_or_buff`` as CSV when ``save_mode``.
    """
    nbins = int(k_max / bin_size)
    if nbins < 1:
        raise ValueError(f"k_max = {k_max} is below one bin of {bin_size}")
    relation_matrix = np.asarray(partial_relations).transpose()
    altered = bool(num_mols and num_atoms_per_mol)
    named = list(partial_relations[0]) + list(partial_relations[1])
    cmap = _ClassMap(named)                 # 'other' always present: the total channel sums every atom
    ncls = cmap.ncls
    if ncls > SK_MAX_CLASSES:
        raise ValueError(f"{ncls} classes ({ncls - 1} relation types + other) exceed the kernel's {SK_MAX_CLASSES}")
    w, r = dist.world_size(), dist.rank()
    ref = None                              # (cell, natoms, type column, class counts, k-set, this rank's bins)
    rho = None
    steps = {}
    tcol = 0 if altered else 1              # altered types are a function of the ids
    for batch in FrameBatches(filename, ["id", "type", "x", "y", "z"]):     # every rank reads every frame
        dev = batch.wait()
        host = batch.host.numpy()
        for k, meta in enumerate(batch.metas):
            cell = _cell(meta.box)
            if ref is None:
                typ = calc_atom_type_ids(host[k, 0], num_mols, num_atoms_per_mol) if altered else np.array(host[k, 1], copy=True)
                at = _value_counts(typ)
                for t in named:
                    if at.get(int(t), 0) == 0:
                        raise ValueError(f"no atom of type {t} in frame {meta.index} (timestep {meta.timestep})")
                miller, bin_off = kset(cell, k_max, bin_size, k_min, max_k_per_bin, seed)
                lo, hi = shard_bins(bin_off, r, w)
                ref = (cell, meta.natoms, host[k, tcol].copy(), at, miller[bin_off[lo]:bin_off[hi]],
                       bin_off[lo:hi + 1] - bin_off[lo], lo, hi, bin_off)
                cls_d = torch.from_numpy(cmap.classes_of(typ)).to(dev.device)
                rho = _series_buffer(ncls + 1, len(ref[4]), max(2, len(dump_files(filename))), dev.device)
            elif cell != ref[0]:
                raise ValueError(f"the intermediate scattering function needs one cell for all frames: frame {meta.index} "
                                 f"(timestep {meta.timestep}) has {cell}, the first frame {ref[0]}")
            elif meta.natoms != ref[1]:
                raise ValueError(f"the intermediate scattering function needs a fixed atom count: frame {meta.index} "
                                 f"(timestep {meta.timestep}) has {meta.natoms} atoms, the first frame {ref[1]}")
            elif not np.array_equal(host[k, tcol], ref[2]):
                raise ValueError(f"the intermediate scattering function needs fixed atom types: the {'id' if altered else 'type'} "
                                 f"column of frame {meta.index} (timestep {meta.timestep}) differs from the first frame's")
            steps[meta.index] = meta.timestep
        idx = [m.index for m in batch.metas]
        if idx[-1] >= rho.shape[2]:
            rho = _series_buffer(ncls + 1, rho.shape[1], max(2 * rho.shape[2], idx[-1] + 1), rho.device, rho)
        f0 = 0
        while f0 < len(idx):                # runs of consecutive frames (all of a batch: every frame is read)
            f1 = f0 + 1
            while f1 < len(idx) and idx[f1] == idx[f1 - 1] + 1:
                f1 += 1
            ops.sk_rho(dev[f0:f1, 2:5, :].contiguous(), cls_d, ncls, ref[0], ref[4], out=rho, frame0=idx[f0])
            f0 = f1
    if ref is None:
        raise ValueError(f"no dump frames found for {filename!r}")
    T = len(steps)
    if T < 2:
        raise ValueError(f"the intermediate scattering function needs at least 2 frames, {filename!r} holds {T}")
    L = T // 2 if max_lag is None else int(max_lag)
    if not 1 <= L <= T:
        raise ValueError(f"max_lag = {max_lag} is outside [1, {T}] ({T} frames)")
    t = lag_times([steps[i] for i in range(T)], L, timestep, units, repr(filename))

    _, natoms, _, at, _, boff_loc, lo, hi, bin_off = ref
    if rho.shape[2] != T:
        rho = rho[:, :, :T].contiguous()
    tot = rho[0].clone()
    for c in range(1, ncls):                # fixed order
        tot += rho[c]
    rho[ncls] = tot
    pairs = [(ncls, ncls)] + [(cmap.cls(a), cmap.cls(b)) for a, b in relation_matrix]
    sums = torch.zeros((len(pairs), nbins, L), dtype=torch.float64, device=rho.device)
    if hi > lo:
        sums[:, lo:hi] = ops.isf_fft(rho, pairs, boff_loc, L)
    del rho, tot
    dist.all_reduce_sum_(sums)
    sums = sums.cpu().numpy()

    df = isf_table(sums, bin_off, natoms, at, relation_matrix, bin_size, t)
    if save_mode:
        df.to_csv(path_or_buff, index=False)
    return df
