"""Host plumbing shared by the time-series analyses of dump files (MSD, VACF, charge flux, Einstein and Nernst-Einstein
conductivity, F(k, t)): the columns of a read, the unwrapped positions, the molecule layout, the per-group rank split, the
lag count and the evenly spaced time axis.

Analyses that parse every frame on every rank split each group's atoms (or molecules) in contiguous blocks over the ranks
(``rank_blocks``) and sum the correlations of their blocks with one fp64 all-reduce (``all_reduce_groups``); those that
split frames round-robin merge them with ``common/frames._merge_frames``.
"""
from __future__ import annotations

import functools

import numpy as np
import torch

from .. import dist
from ..common import constants
from ..common.com_mols import atom_masses, mol_membership
from ..io import dump as _dump


class MissingCoordinatesError(AssertionError, ValueError):
    """A dump without unwrapped coordinates and without the image flags to build them (an ``AssertionError``, as in the
    reference, and a ``ValueError``)."""


def position_columns(cols):
    """Dump columns of the unwrapped positions (_prepare_unwrapped_coords :62-81): ``xu yu zu`` when ``zu`` is present, else
    ``x y z ix iy iz`` (unwrapped as x + ix * (xhi - xlo) by ``unwrapped_positions``)."""
    if "zu" in cols:
        return ["xu", "yu", "zu"]
    if "z" not in cols:
        raise MissingCoordinatesError("Missing wrapped and unwrapped coordinates (x y z xu yu zu)")
    if "iz" not in cols:
        raise MissingCoordinatesError("Missing unwrapped coordinates (xu yu zu) and box location ("
                                      "ix iy iz) for converting wrapped coordinates (x y z) into "
                                      "unwrapped coordinates. ")
    return ["x", "y", "z", "ix", "iy", "iz"]


def unwrapped_positions(dev, metas, k0, have_u):
    """[F,3,N] unwrapped positions of a parsed batch ``dev`` [F,C,N] whose columns k0.. are those of ``position_columns``
    (``have_u``: the three ``xu yu zu``; else the six ``x y z ix iy iz``)."""
    if have_u:
        return dev[:, k0:k0 + 3, :]
    L = torch.tensor([m.box.bound_lengths() for m in metas], dtype=torch.float64, device=dev.device)
    return dev[:, k0:k0 + 3, :] + dev[:, k0 + 3:k0 + 6, :] * L[:, :, None]      # x.add(ix.multiply(L)) (:78-80)


class DumpColumns:
    """The columns of one time-series read of the dump files ``pattern``, chosen before any frame is parsed: ``available``
    holds those of the first frame (ValueError when no frame matches), ``select`` returns those to parse."""

    def __init__(self, pattern):
        self.available = _dump.available_columns(pattern)
        if not self.available:
            raise ValueError(f"no dump frames found for {pattern!r}")

    def select(self, columns, positions=False, masses=False):
        """``columns``, then those of ``position_columns`` when ``positions`` (for ``unwrapped_positions`` with
        k0 = len(columns)), then ``mass`` when ``masses`` (no mass table was given: AssertionError when the dump has none)."""
        want = list(columns) + (position_columns(self.available) if positions else [])
        if masses:
            assert "mass" in self.available, "Missing atom masses in dump file."
            want.append("mass")
        return want


class MoleculeLayout:
    """The molecules in atom-id order, ``num_mols[g]`` of type g + 1 with ``num_atoms_per_mol[g]`` atoms each: ``mol_type``,
    ``mol_id`` and ``seg_off`` [M+1] of ``com_mols.mol_membership``, the molecule offsets ``type_off`` [ntypes+1] of the
    types, and the atom masses from the table ``mass`` (by atom type) or, without one, from the dump's ``mass`` column."""

    def __init__(self, num_mols, num_atoms_per_mol, mass=None):
        self.mol_type, self.mol_id, self.seg_off = mol_membership(num_mols, num_atoms_per_mol)
        self.type_off = np.concatenate(([0], np.cumsum(num_mols))).astype(np.int64)
        self.mass = mass

    def check(self, n):
        """ValueError unless the molecules hold exactly the n atoms of a frame."""
        if self.seg_off[-1] != n:
            raise ValueError(f"Length of values ({self.seg_off[-1]}) does not match length of index ({n})")

    def masses(self, types, mass_row=None, device=None):
        """Per-atom masses, float64: ``mass[type - 1]`` with a table, else a copy of the dump's ``mass_row`` (which may be a
        view of a staging buffer); on ``device`` if given."""
        m = np.array(atom_masses(types, self.mass) if self.mass else mass_row, dtype=np.float64)
        return m if device is None else torch.from_numpy(m).to(device)

    def type_members(self):
        """The molecule indices of each type, in type order (the groups of ``rank_blocks``)."""
        return [np.arange(a, b) for a, b in zip(self.type_off[:-1], self.type_off[1:])]

    @functools.cached_property
    def seg_d(self):
        """``seg_off`` as the int32 vector of the segmented reductions on the current device (uploaded once)."""
        return torch.from_numpy(self.seg_off.astype(np.int32)).cuda()


def rank_blocks(members, device, r=None, w=None):
    """This rank's contiguous ``dist.shard_range`` block of every group of ``members`` (per-group index arrays),
    concatenated in group order -> (int64 indices on ``device``, the number of them in each group)."""
    local = [np.asarray(idx)[slice(*dist.shard_range(len(idx), r, w))] for idx in members]
    return torch.from_numpy(np.concatenate(local).astype(np.int64)).to(device), [len(idx) for idx in local]


def all_reduce_groups(correlate, chans, ngroups, nlags):
    """``correlate(chans)`` -- the [ngroups, nlags] fp64 sums of this rank's channels -- summed over the ranks with one
    all-reduce.  A rank without channels (its blocks of every group are empty) still joins it with zeros."""
    sums = correlate(chans) if chans.shape[0] else torch.zeros((ngroups, nlags), dtype=torch.float64, device=chans.device)
    return dist.all_reduce_sum_(sums)


def lag_count(max_lag, T):
    """The number of lags of a correlation over T frames: ``max_lag`` clipped to T, by default T // 2; ValueError below 1."""
    L = T // 2 if max_lag is None else min(int(max_lag), T)
    if L < 1:
        raise ValueError(f"max_lag must be at least 1 ({T} frames)")
    return L


def even_times(steps, units, timestep, source, who="the Einstein and Nernst-Einstein conductivity need"):
    """Times in seconds of the frames' timesteps (in trajectory order), which must be evenly spaced: ValueError naming
    ``who`` otherwise, and naming ``source`` when there is no frame."""
    steps = np.asarray(steps, dtype=np.float64)
    if len(steps) == 0:
        raise ValueError(f"no dump frames found for {source}")
    d = np.diff(steps)
    if len(d) and not (d[0] > 0 and (d == d[0]).all()):
        raise ValueError(f"{who} evenly spaced frames (timesteps "
                         f"{steps[:3].tolist()}...: spacings {sorted(set(d.tolist()))[:4]})")
    return steps * constants.TIME_CONVERSION[units] * timestep


def fit_window(t, initial_time=None, final_time=None):
    """Mask of the lag times ``t`` (l * dt, l < L) inside [initial_time, final_time]; by default the lags max(1, L // 10)
    to L - 1, which leaves out the first tenth of the curve.  ValueError when the window holds fewer than 2 lag times."""
    L = len(t)
    lo = t[min(max(1, L // 10), L - 1)] if initial_time is None else initial_time
    hi = t[L - 1] if final_time is None else final_time
    mask = (t >= lo) & (t <= hi)
    if L < 2 or mask.sum() < 2:
        raise ValueError(f"the fit window [{lo}, {hi}] holds {int(mask.sum()) if L >= 2 else 0} lag times; "
                         "at least 2 are needed")
    return mask
