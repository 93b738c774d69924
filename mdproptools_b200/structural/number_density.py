"""Number-density profile normal to an interface -- drop-in for ``mdproptools.structural.number_density``
(reference mdproptools/structural/number_density.py:30-154; citations are lines of that file).

Per frame the reference shifts the chosen coordinate by the minimum over the surface atoms (:77-86), selects, for every
requested atom type, the atoms on the requested side of ``dist_from_interface`` and histograms their distance -- measured
from the top of the surface slab for a positive distance (:88-99), from its bottom for a negative one (:100-110) -- with
``(b / bin_size).astype(int)``; the counts are divided by the bin volume (cross-section x bin_size, :115-132), averaged
over the frames and written like an RDF table (:138-145).  Here the masked min/max and the histograms are one call of
``mdp_axis_density`` per batch of frames (same fp64 operation order, integer counts); the normalisation is host numpy in
the reference's order.  Frames are split over ranks and merged with one int64 all-reduce.

Divergences (the reference cannot run on numpy >= 1.24: ``np.int`` :50, ``np.product`` :118):
* a negative bin index counts in bin ``num_bins + k``, exactly as numpy's negative indexing does at :99;
* an index outside ``[-num_bins, num_bins)`` raises IndexError in the reference; here such atoms are not counted.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from .. import dist, ops
from ..common.frames import _merge_frames, calc_atom_type_ids
from ..io.pipeline import FrameBatches
from .rdf_cn import _log, _num_bins, _save_rdf

_AXES = {"x": 2, "y": 3, "z": 4}


def calc_number_density(dump_pattern, surface_atom, atom_types, bin_size, dist_from_interface, axis_norm_interface,
                        num_mols=None, num_atoms_per_mol=None, working_dir=None, results_file="number_density.csv",
                        save_mode=True):
    if not working_dir:
        working_dir = os.getcwd()
    if axis_norm_interface not in _AXES:
        raise KeyError(axis_norm_interface)
    atom_types = list(atom_types)
    partial_relations = np.array((np.full(shape=len(atom_types), fill_value=surface_atom, dtype=int), atom_types))   # :47-52
    num_bins, radii = _num_bins(abs(dist_from_interface), bin_size)                                                    # :53-58
    num_relations = len(atom_types)
    altered = bool(num_mols and num_atoms_per_mol)
    w, me = dist.world_size(), dist.rank()
    batches = FrameBatches(os.path.join(working_dir, dump_pattern), ["id", "type", "x", "y", "z"],
                           frame_select=(lambda i: i % w == me) if w > 1 else None)
    per_frame, areas = {}, {}
    dev = torch.device("cuda", torch.cuda.current_device())
    for batch in batches:
        d = batch.wait()
        host = batch.host.numpy()
        if altered:       # altered types come from the id column of the id-sorted frame (:64-70)
            key = torch.from_numpy(np.stack([calc_atom_type_ids(host[k, 0], num_mols, num_atoms_per_mol).astype(np.float64)
                                             for k in range(len(batch.metas))])).to(d.device)
        else:
            key = d[:, 1, :].contiguous()
        coord = d[:, _AXES[axis_norm_interface], :].contiguous()
        counts, _ = ops.axis_density(coord, key, surface_atom, atom_types, dist_from_interface, bin_size, num_bins)
        for k, meta in enumerate(batch.metas):
            per_frame[meta.index] = counts[k]
            lengths = dict(zip("xyz", meta.box.lattice_lengths()))                                                    # :113-118
            areas[meta.index] = float(np.prod([lengths[a] for a in lengths if a != axis_norm_interface]))
            _log("Finished computing density profile for timestep", meta.timestep)
    T = batches.total_frames or 0
    if T == 0:
        raise ValueError(f"no dump frames found for {dump_pattern!r}")
    counts = _merge_frames(per_frame, T, (num_relations, num_bins), dev).cpu().numpy()
    area = torch.zeros((T,), dtype=torch.float64, device=dev)
    for idx, a in areas.items():
        area[idx] = a
    dist.all_reduce_sum_(area)
    area = area.cpu().numpy()
    rho_part_sum = np.zeros((num_relations, num_bins))
    for t in range(T):                                                                                                # :119-133
        rho_part_sum += counts[t].astype(np.float64) / (area[t] * bin_size)
    rho_part_sum = rho_part_sum / T                                                                                    # :138
    path = os.path.join(working_dir, results_file)
    if dist.rank() != 0:
        save_mode = False
    return _save_rdf(radii, np.asarray(partial_relations).transpose(), path, save_mode, rho_part_sum)
