"""Radial distribution functions and coordination numbers from LAMMPS dump files -- drop-in for
``mdproptools.structural.rdf_cn`` (reference file mdproptools/structural/rdf_cn.py; citations below are
lines of that file).

Public functions keep the reference's names, positional order, defaults, return types and side-effect
files: calc_atomic_rdf (:385), calc_atomic_cn (:533), calc_molecular_rdf (:654), calc_molecular_cn (:759),
calc_intermolecular_rdf (:857).

Division of labour
  device  all pair arithmetic (_calc_rsq/_remove_outliers/_rdf_loop/_cn_loop/_rdf_mol_loop/_cn_mol_loop,
          :35-162) -> per-frame *integer* histograms via libmdprop_b200 (csrc/pair.cu); molecule centres of
          mass (_define_mol_cols, :218-241) via the segmented reduction kernel;
  host    everything that only defines how integers become the final floats (_calc_props :244-294,
          _normalize_rdf :297-329, _normalize_cn :332-338, _save_* :341-382), restated in numpy in the
          reference's operation order so that equal counts give bit-identical DataFrames.
Frames are sharded round-robin over the ranks of an initialised torch.distributed group; the per-frame
integer histograms are merged with one int64 all-reduce.

Extension (keyword ``mic``, default "reference"): the reference has no triclinic minimum image -- it wraps tilted
cells as if they were orthogonal with the lattice-vector lengths and takes volume = prod(lengths) (:260-261).
``mic="reference"`` reproduces exactly that; ``mic="triclinic"`` uses the general triclinic image of
MDP_PAIR_TRICLINIC (include/mdprop_b200.h) with the cell (lx, ly, lz, xy, xz, yz) from the dump header and the true
cell volume lx*ly*lz.  For orthogonal boxes the two are identical bit for bit.

Documented divergences from the reference:
  * a bin index >= num_bins (possible when r_cut/bin_size is not an integer) is dropped instead of
    written out of bounds (the reference corrupts memory, SURVEY 5);
  * molecule centres of mass use sequential fp64 accumulation in atom-id order (the reference's BLAS dot
    has a library-dependent order; differences are <= 1 ulp of the coordinate).
"""
from __future__ import annotations

import numpy as np
import pandas as pd
import torch

from .. import dist, ops
from .._lib import PAIR_TRICLINIC, bin_edges
from ..common.frames import _ClassMap, _frame_batches, _value_counts, file_sharded, merge_results, typed_batches
from ..common.frames import calc_atom_type_ids  # noqa: F401  (public under this module's path, as in the reference)
from ..io.pipeline import ArrayBatches

CON_CONSTANT = 1.660538921  # :30

VERBOSE = False   # the reference prints per-frame progress; off by default here


def _log(*a):
    if VERBOSE:
        print(*a)


# ------------------------------------------------------------------------------------------------
# host-side restatements
# ------------------------------------------------------------------------------------------------
def _num_bins(r_cut, bin_size):
    """_initialize (:165-180)."""
    if isinstance(r_cut, list):
        nb = [int(i / bin_size) for i in r_cut]
        radii = [(np.arange(i) + 0.5) * bin_size for i in nb]
    else:
        nb = int(r_cut / bin_size)
        radii = (np.arange(nb) + 0.5) * bin_size
    return nb, radii


def _rcut_sq(r_cut) -> float:
    """``r_cut ** 2`` as the numba kernels evaluate it (:66): exact for ints, x*x for floats."""
    if isinstance(r_cut, (int, np.integer)):
        return float(int(r_cut) ** 2)
    r = float(r_cut)
    return r * r


def _calc_props(box_lengths, n_objects, atom_types, object_types, num_types, mass, partial_relations, atom_types_col,
                num_atoms_per_mol=None):
    """_calc_props (:244-294): densities and the consistency checks (same exceptions)."""
    num_relations = len(partial_relations[0])
    volume = np.prod(box_lengths)
    set_id = set(atom_types.keys())
    if atom_types_col == "type":
        if num_types != len(set_id):
            raise ValueError(
                f"""Consistency check failed: Number of specified
                            atomic types is different from the calculated value
                            specified= {num_types}, calculated= {len(set_id)}"""
            )
    elif atom_types_col == "id":
        if np.sum(num_atoms_per_mol) != len(set_id):
            raise ValueError(
                f"""Consistency check failed: Number of specified
                            atomic types is different from the calculated value
                            specified= {num_atoms_per_mol},
                            calculated= {len(set_id)}"""
            )
    total_mass = np.sum([float(mass[i]) * float(atom_types[i + 1]) for i in range(num_types)])
    total_density = float((total_mass / volume) * CON_CONSTANT)
    _log("{0:s}{1:10.8f}".format("Average density=", float(total_density)))
    rho = n_objects / volume
    rho_pairs = np.zeros(num_relations)
    for index, object_type in enumerate(partial_relations[1]):
        rho_pairs[index] = object_types[object_type] / volume
        if rho_pairs[index] < 1.0e-22:
            raise ValueError("Error: Density is zero for mol type: " + str(object_type))
    return rho, rho_pairs


def _rdf_denominators(bin_size, rho_pairs, atom_types, partial_relations, num_relations, num_bins, num_atoms=None, rho=None):
    """The divisors of _normalize_rdf (:297-329), built with the reference's expressions in the reference's order, so that
    ``counts / divisor`` is bit-identical to the reference whether it is evaluated per frame or for a batch of frames."""
    shell_volume = (
        4 / 3 * np.pi * bin_size ** 3 * (np.arange(1, num_bins + 1) ** 3 - np.arange(num_bins) ** 3)
    )
    den_full = None if num_atoms is None else num_atoms * rho * shell_volume
    ref_atoms = np.asarray(partial_relations[0]).reshape((num_relations, 1))
    ref_atoms_matrix = np.tile(ref_atoms, num_bins)
    num_atoms_matrix = np.vectorize(atom_types.get)(ref_atoms_matrix)
    rho_pairs_matrix = np.tile(rho_pairs.reshape((num_relations, 1)), num_bins)
    shell_volume_matrix = np.tile(shell_volume, (num_relations, 1))
    return den_full, num_atoms_matrix * rho_pairs_matrix * shell_volume_matrix


def _normalize_rdf(bin_size, rho_pairs, atom_types, partial_relations, num_relations, num_bins, rdf_part, rdf_full=None,
                   num_atoms=None, rho=None):
    """_normalize_rdf (:297-329)."""
    den_full, den_part = _rdf_denominators(bin_size, rho_pairs, atom_types, partial_relations, num_relations, num_bins,
                                           num_atoms if rdf_full is not None else None, rho)
    if rdf_full is not None:
        rdf_full = rdf_full / den_full
    rdf_part = rdf_part / den_part
    return rdf_full, rdf_part


def _normalize_cn(atom_types, partial_relations, cn):
    """_normalize_cn (:332-338)."""
    num_ref_atoms = [atom_types[i] for i in partial_relations[0]]
    return cn / num_ref_atoms


def _save_rdf(radii, relation_matrix, path_or_buf, save_mode, rdf_part_sum, rdf_full_sum=None):
    """_save_rdf (:341-365)."""
    if rdf_full_sum is not None:
        result_tuple = (radii, rdf_full_sum, rdf_part_sum)
        final_label = ["r ($\\AA$)", "g_full(r)"]
    else:
        result_tuple = (radii, rdf_part_sum)
        final_label = ["r ($\\AA$)"]
    final_array = np.vstack(result_tuple).transpose()
    final_labels = final_label + [f"g_{str(pair[0])}-{str(pair[1])}" for pair in relation_matrix]
    final_df = pd.DataFrame(final_array, columns=final_labels)
    if save_mode:
        final_df.to_csv(path_or_buf, index=False)
        _log("Results are written to pd.DataFrame and csv file")
    else:
        _log(final_df)
    return final_df


def _save_cn(relation_matrix, path_or_buff, cn_sum, save_mode):
    """_save_cn (:368-382)."""
    final_array = np.vstack(cn_sum).transpose()
    final_labels = [f"cn_{str(pair[0])}-{str(pair[1])}" for pair in relation_matrix]
    final_df = pd.DataFrame(final_array, columns=final_labels)
    if save_mode:
        final_df.to_csv(path_or_buff, index=False)
        _log("CN results are written to pd.DataFrame and csv file")
    else:
        _log(final_df)
    return final_df


def _sym_weights(cmap: _ClassMap, relation_matrix, with_full: bool):
    """hist_reduce weights for the symmetric kernel: g_full counts every pair twice (:85-86); relation (a,b)
    counts a pair once per matching role order (:89-96) -> 2 on the like row, 1 on the unlike row."""
    rows = ops.sym_rows(cmap.ncls)
    w = []
    if with_full:
        w.append(np.full(rows, 2, dtype=np.int32))
    for a, b in relation_matrix:
        r = np.zeros(rows, dtype=np.int32)
        r[ops.sym_row(cmap.cls(a), cmap.cls(b), cmap.ncls)] = 2 if int(a) == int(b) else 1
        w.append(r)
    return np.stack(w)


def _rect_weights(cmap_a: _ClassMap, cmap_b: _ClassMap, relation_matrix):
    rows = cmap_a.ncls * cmap_b.ncls
    w = []
    for a, b in relation_matrix:
        r = np.zeros(rows, dtype=np.int32)
        r[cmap_a.cls(a) * cmap_b.ncls + cmap_b.cls(b)] = 1
        w.append(r)
    return np.stack(w)


def _cn_edges(r_cut_list):
    """Sorted distinct squared cutoffs as a histogram edge table; bin k = #{thresholds <= rsq}."""
    rc2 = np.array([_rcut_sq(r) for r in r_cut_list], dtype=np.float64)
    thr = np.unique(rc2)                       # ascending
    edges = np.concatenate(([0.0], thr))       # edges[k>=1] = thr[k-1]
    # a pair with rsq < rc2[kl] lies in bins 0 .. (index of rc2[kl] in thr); cumulative bin index per relation
    upto = np.searchsorted(thr, rc2)           # bins 0..upto inclusive
    return edges, float(thr[-1]), upto


# ------------------------------------------------------------------------------------------------
# minimum-image convention
# ------------------------------------------------------------------------------------------------
def _mic_flags(mic) -> int:
    if mic == "reference":
        return 0
    if mic == "triclinic":
        return PAIR_TRICLINIC
    raise ValueError(f"mic must be 'reference' or 'triclinic', got {mic!r}")


def _frame_box(box, flags):
    """(lengths whose product is the normalisation volume, the row handed to the pair kernel)."""
    if flags & PAIR_TRICLINIC:
        lengths = box.bound_lengths()
        tilt = box.tilt if box.tilt is not None else (0.0, 0.0, 0.0)
        return lengths, tuple(lengths) + tuple(tilt)
    lengths = box.lattice_lengths()          # :260
    return lengths, lengths


class _PropsCache:
    """_frame_box + _calc_props of a frame, remembered for the next frames with the same box, atom count and type table
    (every frame of an NVT trajectory): ~0.1 ms of small numpy calls per frame otherwise -- as much as the pair kernel
    itself needs for a 10^5-atom frame.  The checks of _calc_props run (and raise) on the first frame of each kind."""

    def __init__(self, flags, num_types, mass, partial_relations, col, num_atoms_per_mol):
        self.args = (num_types, mass, partial_relations, col, num_atoms_per_mol)
        self.flags, self.key, self.val = flags, None, None

    def get(self, meta, at):
        b = meta.box
        key = (meta.natoms, id(at), tuple(map(tuple, b.bounds)), None if b.tilt is None else tuple(b.tilt))
        if key != self.key:
            lengths, boxrow = _frame_box(b, self.flags)
            num_types, mass, rel, col, napm = self.args
            rho, rho_pairs = _calc_props(lengths, meta.natoms, at, at, num_types, mass, rel, col, napm)
            self.key, self.val = key, (at, boxrow, rho, rho_pairs)           # (holding `at` keeps its id unique)
        return self.val[1:]


def _mol_segments(num_mols, num_atoms_per_mol):
    """Molecule membership implied by id order (:222-230): (mol_type[M], seg_off[M+1])."""
    mt = np.repeat(np.arange(1, len(num_mols) + 1), num_mols)
    sizes = np.repeat(np.asarray(num_atoms_per_mol), num_mols)
    off = np.concatenate(([0], np.cumsum(sizes)))
    return mt, off


# ------------------------------------------------------------------------------------------------
# frame loops of the file-based entry points
# ------------------------------------------------------------------------------------------------
def _atomic_counts(filename, num_types, mass, partial_relations, num_mols, num_atoms_per_mol, flags, shard_files, rcut2, edges,
                   ddr, cumulative):
    """The frame loop of calc_atomic_rdf (``cumulative=False``: rows g_full and the relations; props (at, rho, rho_pairs,
    natoms) per frame) and calc_atomic_cn (``cumulative=True``: the relations, cumulative over the cutoff table; props at
    per frame) -> (counts [T, rows, bins], props of every frame, T)."""
    relation_matrix = np.asarray(partial_relations).transpose()
    altered = bool(num_mols and num_atoms_per_mol)
    pcache = _PropsCache(flags, num_types, mass, partial_relations, "id" if altered else "type", num_atoms_per_mol)

    def frame_props(meta, at):
        if not cumulative:
            _log("The timestep of the current file is: " + str(meta.timestep))
        return pcache.get(meta, at)

    batches = _frame_batches(filename, ["id", "type", "x", "y", "z"], shard_files)
    named = list(partial_relations[0]) + list(partial_relations[1])
    counts, props = {}, {}
    weights = None          # fixed by the types present in this rank's first frame
    for b in typed_batches(batches, num_mols, num_atoms_per_mol, frame_props, named=named):
        if weights is None:
            weights = _sym_weights(b.cmap, relation_matrix, with_full=not cumulative)
        boxes = np.array([p[0] for p in b.props], dtype=np.float64)
        xyz = b.dev[:, 2:5, :].contiguous()
        hist = ops.pair_hist(xyz, b.classes(0, len(b.metas)), b.cmap.ncls, boxes, rcut2, edges, ddr, flags=flags)
        red = ops.hist_reduce(hist, weights, cumulative=cumulative)
        for k, meta in enumerate(b.metas):
            counts[meta.index] = red[k]
            props[meta.index] = b.atom_types[k] if cumulative else (b.atom_types[k], *b.props[k][1:], meta.natoms)
    rows = len(partial_relations[0]) + (0 if cumulative else 1)
    return merge_results(batches, counts, props, filename, (rows, len(edges) - 1))


def _molecular_counts(filename, num_types, mass, partial_relations, num_mols, num_atoms_per_mol, inter, flags, shard_files,
                      rcut2, edges, ddr, cumulative):
    """The frame loop of the atom/molecule-COM entry points (:654-902): relation counts between the atoms (with ``inter``
    the molecule centres) of the types partial_relations[0] and the centres of the molecule types partial_relations[1],
    cumulative over the cutoff table with ``cumulative`` -> (counts [T, R, bins], props (at, rho_pairs) of every frame, T)."""
    relation_matrix = np.asarray(partial_relations).transpose()
    mol_type, seg_off = _mol_segments(num_mols, num_atoms_per_mol)
    cmap_a = _ClassMap(partial_relations[0])
    cmap_b = _ClassMap(partial_relations[1])
    weights = _rect_weights(cmap_a, cmap_b, relation_matrix)
    mol_types_count = _value_counts(mol_type)
    batches = _frame_batches(filename, ["id", "type", "x", "y", "z"], shard_files)
    counts, props = {}, {}
    for batch in batches:
        dev = batch.wait()
        device = dev.device
        F = len(batch.metas)
        host = batch.host.numpy()
        n = host.shape[2]
        if seg_off[-1] != n:
            raise ValueError(f"Length of values ({seg_off[-1]}) does not match length of index ({n})")
        boxes = np.empty((F, 6 if flags else 3))
        cls_a = np.empty((F, n), dtype=np.int32)
        for k, meta in enumerate(batch.metas):
            lengths, boxes[k] = _frame_box(meta.box, flags)
            at = mol_types_count if inter else _value_counts(host[k, 1])
            if not inter:
                cls_a[k] = cmap_a.classes_of(host[k, 1])
            rho, rho_pairs = _calc_props(lengths, len(mol_type), at, mol_types_count, num_types, mass, partial_relations, "type",
                                         num_atoms_per_mol)
            props[meta.index] = (at, rho_pairs)
        xyz = dev[:, 2:5, :].contiguous()
        # masses per atom from the type column of the first frame of the batch (:231); types are static per id
        m_atom = torch.from_numpy(np.array([mass[int(t - 1)] for t in host[0, 1]], dtype=np.float64)).to(device)
        com, _, _ = ops.segment_com(xyz, m_atom, torch.from_numpy(seg_off.astype(np.int32)).to(device))   # [F,3,M]
        cls_m = torch.from_numpy(cmap_b.classes_of(mol_type)).to(device)
        if inter:
            xyz_a, cls_a_d = com, torch.from_numpy(cmap_a.classes_of(mol_type)).to(device)
        else:
            xyz_a, cls_a_d = xyz, torch.from_numpy(cls_a).to(device)
        hist = ops.pair_hist(xyz_a, cls_a_d, cmap_a.ncls, boxes, rcut2, edges, ddr, xyz_b=com, cls_b=cls_m, ncls_b=cmap_b.ncls,
                             flags=flags)
        red = ops.hist_reduce(hist, weights, cumulative=cumulative)
        for k, meta in enumerate(batch.metas):
            counts[meta.index] = red[k]
    return merge_results(batches, counts, props, filename, (len(partial_relations[0]), len(edges) - 1))


# ------------------------------------------------------------------------------------------------
# public API
# ------------------------------------------------------------------------------------------------
@file_sharded
def calc_atomic_rdf(r_cut, bin_size, num_types, mass, partial_relations, filename, num_mols=None, num_atoms_per_mol=None,
                    path_or_buff="rdf.csv", save_mode=True, mic="reference", *, shard_files=True):
    """Full and partial atom-atom RDF; see the reference docstring (:397-452) for the arguments."""
    flags = _mic_flags(mic)
    num_bins, radii = _num_bins(r_cut, bin_size)
    num_relations = len(partial_relations[0])
    relation_matrix = np.asarray(partial_relations).transpose()
    edges = bin_edges(bin_size, num_bins)
    rcut2 = _rcut_sq(r_cut)
    allc, props, T = _atomic_counts(filename, num_types, mass, partial_relations, num_mols, num_atoms_per_mol, flags,
                                    shard_files, rcut2, edges, bin_size, cumulative=False)
    rdf_full_sum = np.zeros(num_bins)
    rdf_part_sum = np.zeros((num_relations, num_bins))
    den_cache = {}   # frames of one composition and volume share the divisors of _normalize_rdf (the NVT case: one entry)
    for idx in range(T):
        at, rho, rho_pairs, natoms = props[idx]
        key = (natoms, rho, np.asarray(rho_pairs).tobytes(), tuple(sorted(at.items())))
        den = den_cache.get(key)
        if den is None:
            den = den_cache[key] = _rdf_denominators(bin_size, rho_pairs, at, partial_relations, num_relations, num_bins,
                                                     natoms, rho)
        rdf_full_sum += allc[idx, 0].astype(np.float64) / den[0]
        rdf_part_sum += allc[idx, 1:].astype(np.float64) / den[1]
    rdf_full_sum = rdf_full_sum / T
    rdf_part_sum = rdf_part_sum / T
    return _save_rdf(radii, relation_matrix, path_or_buff, save_mode, rdf_part_sum, rdf_full_sum=rdf_full_sum)


@file_sharded
def calc_atomic_cn(r_cut, bin_size, num_types, mass, partial_relations, filename, num_mols=None, num_atoms_per_mol=None,
                   path_or_buff="cn.csv", save_mode=True, mic="reference", *, shard_files=True):
    """Atom-atom coordination numbers, one cutoff per relation (:533-651)."""
    flags = _mic_flags(mic)
    _num_bins(r_cut, bin_size)
    num_relations = len(partial_relations[0])
    relation_matrix = np.asarray(partial_relations).transpose()
    edges, rcut2_max, upto = _cn_edges(r_cut)
    allc, props, T = _atomic_counts(filename, num_types, mass, partial_relations, num_mols, num_atoms_per_mol, flags,
                                    shard_files, rcut2_max, edges, 0.0, cumulative=True)
    cn_sum = np.zeros(num_relations)
    for idx in range(T):
        cn = np.array([allc[idx, kl, upto[kl]] for kl in range(num_relations)], dtype=np.float64)
        cn_sum += _normalize_cn(props[idx], partial_relations, cn)
    cn_sum = cn_sum / T
    return _save_cn(relation_matrix, path_or_buff, cn_sum, save_mode)


@file_sharded
def calc_molecular_rdf(r_cut, bin_size, num_types, mass, partial_relations, filename, num_mols, num_atoms_per_mol,
                       path_or_buff="rdf_mol.csv", save_mode=True, _inter=False, mic="reference", *, shard_files=True):
    """Partial RDF between atoms and molecule centres of mass (:654-756)."""
    flags = _mic_flags(mic)
    num_bins, radii = _num_bins(r_cut, bin_size)
    edges = bin_edges(bin_size, num_bins)
    rcut2 = _rcut_sq(r_cut)
    allc, props, T = _molecular_counts(filename, num_types, mass, partial_relations, num_mols, num_atoms_per_mol, _inter,
                                       flags, shard_files, rcut2, edges, bin_size, cumulative=False)
    R = len(partial_relations[0])
    rdf_part_sum = np.zeros((R, num_bins))
    for idx in range(T):
        at, rho_pairs = props[idx]
        _, rdf_part = _normalize_rdf(bin_size, rho_pairs, at, partial_relations, R, num_bins, allc[idx].astype(np.float64))
        rdf_part_sum += rdf_part
    rdf_part_sum = rdf_part_sum / T
    return _save_rdf(radii, np.asarray(partial_relations).transpose(), path_or_buff, save_mode, rdf_part_sum)


@file_sharded
def calc_molecular_cn(r_cut, bin_size, num_types, mass, partial_relations, filename, num_mols, num_atoms_per_mol,
                      path_or_buff="cn_mol.csv", save_mode=True, mic="reference", *, shard_files=True):
    """Coordination numbers between atoms and molecule centres of mass (:759-854)."""
    flags = _mic_flags(mic)
    _num_bins(r_cut, bin_size)
    edges, rcut2_max, upto = _cn_edges(r_cut)
    allc, props, T = _molecular_counts(filename, num_types, mass, partial_relations, num_mols, num_atoms_per_mol, False, flags,
                                       shard_files, rcut2_max, edges, 0.0, cumulative=True)
    R = len(partial_relations[0])
    cn_sum = np.zeros(R)
    for idx in range(T):
        at, _ = props[idx]
        cn = np.array([allc[idx, kl, upto[kl]] for kl in range(R)], dtype=np.float64)
        cn_sum += _normalize_cn(at, partial_relations, cn)
    cn_sum = cn_sum / T
    return _save_cn(np.asarray(partial_relations).transpose(), path_or_buff, cn_sum, save_mode)


def calc_atomic_rdf_from_arrays(positions, types, box_lengths, r_cut, bin_size, partial_relations, batch_frames=64,
                                return_counts=False, mic="reference", frame_range=None):
    """Array front end of :func:`calc_atomic_rdf` for trajectories that are already in memory.

    positions   float64 [T, 3, N] host array (numpy, or a pinned torch tensor for async copies), rows in id order
    types       [N] or [T, N] atom types (ints or floats, as the dump's ``type`` column)
    box_lengths [3] or [T, 3] box lengths as ``dump.box.to_lattice().lengths`` gives them; with ``mic="triclinic"``
                [6] or [T, 6] = (lx, ly, lz, xy, xz, yz) and the normalisation volume is lx*ly*lz
    Everything else as in calc_atomic_rdf; same per-frame normalisation (rdf_cn.py:297-329, 502-521), same DataFrame.
    Frames stream through pinned staging buffers: the copy of batch k+1 overlaps the kernels of batch k.
    With ``return_counts`` the raw integer histograms [T, 1+R, nbins] (g_full row first) are returned as well.

    Under an initialised process group the T frames are split in contiguous blocks over the ranks (``dist.shard_range``);
    ``positions`` then holds either all T frames on every rank, or only this rank's block with ``frame_range=(lo, hi, T)``
    saying which block of a T-frame trajectory it is.  The per-frame integer histograms are all-gathered (exact) and every
    rank returns the same DataFrame.
    """
    pos = positions if isinstance(positions, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(positions, dtype=np.float64))
    T, _, N = pos.shape
    if frame_range is not None:
        lo, hi, T = (int(v) for v in frame_range)
        if (lo, hi) != dist.shard_range(T) or pos.shape[0] != hi - lo:
            raise ValueError(f"frame_range {frame_range} is not this rank's block {dist.shard_range(T)} of {T} frames")
    else:
        lo, hi = dist.shard_range(T)
        pos = pos[lo:hi]
    num_bins, radii = _num_bins(r_cut, bin_size)
    num_relations = len(partial_relations[0])
    relation_matrix = np.asarray(partial_relations).transpose()
    dev = torch.device("cuda", torch.cuda.current_device())
    batches = iter(ArrayBatches(pos, batch_frames, dev)) if hi > lo else iter(())   # (a rank beyond the last frame has no block)
    first = next(batches, None)                                   # the copy of the first batch starts now, under the host prep
    types = np.asarray(types)
    at_all = _value_counts(types)                                 # one pass over the types serves the class map too
    cmap = _ClassMap(list(partial_relations[0]) + list(partial_relations[1]), present_types=list(at_all))
    weights = _sym_weights(cmap, relation_matrix, with_full=True)
    edges = bin_edges(bin_size, num_bins)
    rcut2 = _rcut_sq(r_cut)
    flags = _mic_flags(mic)
    boxes = np.broadcast_to(np.asarray(box_lengths, dtype=np.float64), (T, 6 if flags else 3))
    static_types = types.ndim == 1
    if static_types:
        cls_static = torch.from_numpy(cmap.classes_of(types)).to(dev)
        at_static = at_all
    out = torch.empty((hi - lo, 1 + num_relations, num_bins), dtype=torch.int64, device=dev)

    def _all_batches():
        if first is not None:
            yield first
            yield from batches

    for f0, f1, x in _all_batches():                             # copy of batch k+1 overlaps the kernels of batch k
        cls = cls_static if static_types else torch.from_numpy(np.stack([cmap.classes_of(t) for t in types[lo + f0:lo + f1]])).to(dev)
        hist = ops.pair_hist(x, cls, cmap.ncls, boxes[lo + f0:lo + f1], rcut2, edges, bin_size, flags=flags)
        out[f0:f1] = ops.hist_reduce(hist, weights)
    counts = dist.all_gather_blocks(out, T).cpu().numpy()
    rdf_full_sum = np.zeros(num_bins)
    rdf_part_sum = np.zeros((num_relations, num_bins))
    den_cache = {}   # frames with the same composition and volume share their divisors (the usual NVT case: one entry)
    volumes = np.prod(boxes[:, :3], axis=1)
    if static_types and T > 1 and np.all(volumes == volumes[0]):
        # one composition, one volume: the per-frame loop below divides every frame by the same arrays and adds the frames in
        # order -- which is what an axis-0 reduction of the divided [T, ...] array does (numpy accumulates rows sequentially
        # along a non-contiguous axis: same additions in the same order, bit-identical; 1000 frames: 10 ms -> 1 ms)
        rho = N / volumes[0]
        rho_pairs = np.array([at_static[b] / volumes[0] for b in partial_relations[1]])
        den = _rdf_denominators(bin_size, rho_pairs, at_static, partial_relations, num_relations, num_bins, N, rho)
        rdf_full_sum = np.add.reduce(counts[:, 0].astype(np.float64) / den[0], axis=0)
        rdf_part_sum = np.add.reduce(counts[:, 1:].astype(np.float64) / den[1], axis=0)
        df = _save_rdf(radii, relation_matrix, None, False, rdf_part_sum / T, rdf_full_sum=rdf_full_sum / T)
        return (df, counts) if return_counts else df
    for t in range(T):
        at = at_static if static_types else _value_counts(types[t])
        volume = np.prod(boxes[t, :3])
        key = (volume,) if static_types else (volume, tuple(sorted(at.items())))
        den = den_cache.get(key)
        if den is None:
            rho = N / volume
            rho_pairs = np.array([at[b] / volume for b in partial_relations[1]])
            den = den_cache[key] = _rdf_denominators(bin_size, rho_pairs, at, partial_relations, num_relations, num_bins, N, rho)
        rdf_full_sum += counts[t, 0].astype(np.float64) / den[0]
        rdf_part_sum += counts[t, 1:].astype(np.float64) / den[1]
    df = _save_rdf(radii, relation_matrix, None, False, rdf_part_sum / T, rdf_full_sum=rdf_full_sum / T)
    return (df, counts) if return_counts else df


def calc_intermolecular_rdf(r_cut, bin_size, num_types, mass, partial_relations, filename, num_mols, num_atoms_per_mol,
                            path_or_buff="rdf_mol.csv", save_mode=True, mic="reference"):
    """Molecule-COM / molecule-COM partial RDF, self pairs included as in the reference (:857-902)."""
    return calc_molecular_rdf(r_cut, bin_size, num_types, mass, partial_relations, filename, num_mols, num_atoms_per_mol,
                              path_or_buff=path_or_buff, save_mode=save_mode, _inter=True, mic=mic)
