"""Cluster extraction around a central atom type -- drop-in for
``mdproptools.structural.cluster_analysis.get_clusters`` (reference mdproptools/structural/cluster_analysis.py;
citations are lines of that file).

The O(n_central x N) cutoff search of every frame (:143-161, ``_calc_rsq`` + ``rsq < r_cut**2``) runs on the
device as one rectangular neighbour-list call per batch of frames (``mdp_pair_list``, csrc/pair.cu), and so do
the molecule completion and the signed force filter (:163-182): ``mdp_cluster_members`` (csrc/epilogue.cu) returns,
per frame and central atom, the sorted molecules that own a neighbour atom and whose min(sum fx, sum fy, sum fz)
times FORCE_CONSTANT is below ``max_force``.  What is left -- the output ordering (:185-207), the re-imaging relative
to the central atom (:31-44) and the .xyz writer (:213-233) -- is per-cluster file output on the host.

Not supported (raises): element names read from an ``element`` column of the dump (pass ``elements``).

``get_unique_configurations`` (:238-457, SURVEY 8(f) item 3) is host-side bookkeeping on the few-hundred-atom cluster
files; it is restated here without pymatgen (``molecules`` may be pymatgen Molecules, anything with ``.species``, plain
lists of element symbols, or paths of .pdb/.xyz files).
"""
from __future__ import annotations

import ctypes
import glob
import os
import shutil
import warnings
from collections import Counter

import numpy as np
import pandas as pd
import torch

from .. import _lib, dist, ops
from ..common.frames import calc_atom_type_ids
from ..io import dump as _dump
from ..io.pipeline import FrameBatches
from .rdf_cn import _mol_segments

FORCE_CONSTANT = 0.043363 / 16.0  # :28


def _count_frames(filename: str) -> int:
    L = _lib.lib()
    n = 0
    for f in _dump.dump_files(filename):
        buf = _dump._read_bytes(f)
        n += int(L.mdp_dump_scan(buf, len(buf), None, 0))
    return n


def _remove_boundary_effects(head_xyz, xyz, lx, ly, lz):
    """_remove_boundary_effects (:31-44): shift an atom by one box length when its displacement from the
    central atom exceeds half a box (strict compares, single shift)."""
    out = xyz.copy()
    d = xyz - head_xyz
    for k, l in enumerate((lx, ly, lz)):
        cond = (d[:, k] > l / 2) | (d[:, k] < -l / 2)
        out[cond, k] = out[cond, k] - np.sign(d[cond, k]) * l
    return out


def _write_xyz(path, elements, xyz):
    """pandas.to_csv(sep='\\t', float_format='%15.10f', header=False, index=False) of (element, x, y, z) (:229-232)."""
    with open(path, "w") as f:
        f.write("{}\n\n".format(len(elements)))
        for e, (x, y, z) in zip(elements, xyz):
            f.write("%s\t%15.10f\t%15.10f\t%15.10f\n" % (e, x, y, z))


def get_clusters(filename, atom_type, r_cut, num_mols, num_atoms_per_mol, full_trajectory=False, frame=None, elements=None,
                 alter_atom_types=False, max_force=0.75, working_dir=None):
    """Extract the molecules within ``r_cut`` of every atom of ``atom_type`` and write them as
    ``Cluster_<frame>_<k>.xyz``; returns the number of clusters written (reference docstring :60-96)."""
    if elements:
        elements = {i + 1: j for i, j in enumerate(elements)}
    if not working_dir:
        working_dir = os.getcwd()
    cols_present = _dump.available_columns(filename)
    if "element" not in cols_present and not elements:
        raise ValueError("The elements of the atoms in the system should be provided if they "
                         "are not in the dump files.")
    if not elements:
        raise NotImplementedError("element names from a dump column are not supported; pass `elements`")

    total = _count_frames(filename)
    if full_trajectory:
        selected = list(range(total))
    else:
        selected = [range(total)[frame]]
    n_sel = len(selected)
    pos_of = {g: k for k, g in enumerate(selected)}
    w, r = dist.world_size(), dist.rank()
    mine = set(g for k, g in enumerate(selected) if k % w == r)

    mol_type_m, seg_off = _mol_segments(num_mols, num_atoms_per_mol)
    sizes = np.diff(seg_off)
    mol_of_atom = np.repeat(np.arange(len(mol_type_m)), sizes)
    first_col = cols_present[0]
    want = ["id", "type", "x", "y", "z", "fx", "fy", "fz"]
    if first_col not in want:
        want.append(first_col)
    rc2 = r_cut ** 2
    cluster_count = 0
    batches = FrameBatches(filename, want, frame_select=lambda i: i in mine)
    for batch in batches:
        dev = batch.wait()
        host = batch.host.numpy()
        F, _, n = host.shape
        if seg_off[-1] != n:
            raise ValueError(f"Length of values ({seg_off[-1]}) does not match length of index ({n})")
        ci = {c: batch.col(c) for c in want}
        # central atoms (same rows in every frame of the batch unless the type column changes)
        per_frame = []
        for k in range(F):
            typ = host[k, ci["type"]]
            if alter_atom_types:
                # the reference feeds df.values to _calc_atom_type, i.e. the FIRST dump column (:137-139)
                typ = calc_atom_type_ids(host[k, ci[first_col]], num_mols, num_atoms_per_mol)
            per_frame.append(np.nonzero(typ == atom_type)[0])
        same = all(np.array_equal(per_frame[0], p) for p in per_frame[1:])
        xyz = dev[:, [ci["x"], ci["y"], ci["z"]], :].contiguous()
        groups = [(0, F)] if same else [(k, k + 1) for k in range(F)]
        # per frame and central atom: the molecules that own a neighbour atom and pass the force filter, on the device
        # (search: mdp_pair_list; molecule completion + signed-component force filter :163-182: mdp_cluster_members)
        members = [None] * F                                         # per frame: (seg_off, mols, counts) host arrays
        fdev = dev[:, [ci["fx"], ci["fy"], ci["fz"]], :].contiguous()
        seg_d = torch.from_numpy(seg_off.astype(np.int32)).to(dev.device)
        moa_d = torch.from_numpy(mol_of_atom.astype(np.int32)).to(dev.device)
        for k0, k1 in groups:
            cen = per_frame[k0]
            if len(cen) == 0:
                continue
            idx = torch.from_numpy(cen).to(dev.device)
            xa = xyz[k0:k1].index_select(2, idx).contiguous()
            boxes = np.array([batch.metas[k].box.bound_lengths() for k in range(k0, k1)])
            lst, _ = ops.pair_list(xa, xyz[k0:k1].contiguous(), boxes, 0.0, rc2, shell_mode=0)
            so, mols_d, cnt_d = ops.cluster_members(lst, len(cen), fdev[k0:k1].contiguous(), seg_d, moa_d, FORCE_CONSTANT, max_force)
            so, mols_h, cnt_h = so.cpu().numpy(), mols_d.cpu().numpy(), cnt_d.cpu().numpy()
            for fidx in range(k1 - k0):
                members[k0 + fidx] = (so[fidx * len(cen):(fidx + 1) * len(cen)], mols_h, cnt_h[fidx * len(cen):(fidx + 1) * len(cen)])
        for k, meta in enumerate(batch.metas):
            lx, ly, lz = meta.box.bound_lengths()
            x = np.stack([host[k, ci["x"]], host[k, ci["y"]], host[k, ci["z"]]], axis=1)
            elem = np.array([elements.get(int(t)) for t in host[k, ci["type"]]], dtype=object)
            cen = per_frame[k]
            index = pos_of[meta.index]
            frame_number = "{}{}".format("0" * (len(str(n_sel)) - len(str(index))), index)
            for counter, row in enumerate(cen):
                so, mols_h, cnt_h = members[k]
                mols = mols_h[so[counter]: so[counter] + cnt_h[counter]].astype(np.int64)   # sorted == (mol_type, mol_id) order
                own = mol_of_atom[row]
                kept_atoms = np.concatenate([np.arange(seg_off[m], seg_off[m + 1]) for m in mols]) if len(mols) else \
                    np.zeros(0, dtype=np.int64)
                own_rest = kept_atoms[(mol_of_atom[kept_atoms] == own) & (kept_atoms != row)]
                others = kept_atoms[mol_of_atom[kept_atoms] != own]
                order_rows = np.concatenate(([row], own_rest, others)).astype(np.int64)
                # the final inner merge on id drops the central atom when its own molecule failed the filter (:213-218)
                keep = np.isin(order_rows, kept_atoms)
                shifted = _remove_boundary_effects(x[row], x[order_rows], lx, ly, lz)
                fname = "Cluster_{}_{}{}.xyz".format(frame_number, "0" * (len(str(len(cen))) - len(str(counter))), counter)
                _write_xyz(os.path.join(working_dir, fname), elem[order_rows][keep], shifted[keep])
                cluster_count += 1
    if w > 1:
        t = torch.tensor([cluster_count], dtype=torch.int64, device="cuda")
        dist.all_reduce_sum_(t)
        cluster_count = int(t.item())
    return cluster_count


# ------------------------------------------------------------------------------------------------
# unique configurations (:238-457)
# ------------------------------------------------------------------------------------------------
def _read_xyz(path):
    """(symbols, coords) of an .xyz file: atom count, comment line, then ``sym x y z`` rows."""
    with open(path) as f:
        lines = f.read().splitlines()
    n = int(lines[0].split()[0])
    sym, xyz = [], np.empty((n, 3))
    for k, ln in enumerate(lines[2:2 + n]):
        p = ln.split()
        sym.append(p[0])
        xyz[k] = (float(p[1]), float(p[2]), float(p[3]))
    return sym, xyz


def _species_of(mol):
    """Element symbols of one entry of ``molecules``: pymatgen Molecule (``.species``), list of symbols, or a file."""
    if isinstance(mol, (str, os.PathLike)):
        path = str(mol)
        if path.lower().endswith(".pdb"):
            with open(path) as f:
                return [ln[76:78].strip().capitalize() for ln in f if ln.startswith(("HETATM", "ATOM"))]
        return _read_xyz(path)[0]
    if hasattr(mol, "species"):
        return [str(x) for x in mol.species]
    return [str(x) for x in mol]


def get_unique_configurations(cluster_pattern, r_cut, molecules, mol_num, type_coord_atoms=None, working_dir=None,
                              find_top=True, perc=None, cum_perc=90, mol_names=None, zip=True):
    """Group the ``Cluster_*.xyz`` files written by :func:`get_clusters` into configurations -- same arguments, result
    DataFrames, csv files (clusters.csv, configurations.csv, top_conf.csv), ``conf_N.xyz`` copies and optional
    ``Clusters.zip`` as the reference (:238-457).

    Per cluster file: the atoms within ``r_cut`` of the first atom (the atom of interest; ``<=``, Molecule.get_neighbors
    :346), optionally restricted to ``type_coord_atoms`` (:349-352); the atoms after the central molecule are cut into
    molecules by matching the element sequences of ``molecules`` in order (:360-373); for every molecule type the number
    of molecules and, per molecule, the coordinating atoms written as ``<count><first letter of the element>`` sorted by
    letter, the per-molecule strings sorted and joined by ``:`` (:387-397).  Configurations = distinct rows of
    (numbers, strings), counted and ranked (:420-428); the top ones by cumulative share ``cum_perc`` (or share >=
    ``perc``) get the first cluster file (by name) showing them copied to ``conf_<rank>.xyz`` (:429-447).
    """
    working_dir = working_dir or os.getcwd()
    cluster_files = glob.glob(f"{working_dir}/{cluster_pattern}")
    main_atoms = [_species_of(m) for m in molecules]
    n_types = len(main_atoms)
    n_central = len(main_atoms[mol_num])
    rows = {"cluster": [], "num_mols": [], "coordinating_atoms": []}
    for path in cluster_files:
        sym, xyz = _read_xyz(path)
        rows["cluster"].append(os.path.basename(path))
        d0 = np.sqrt(np.sum((xyz - xyz[0]) ** 2, axis=1))
        near = [j for j in range(1, len(sym)) if d0[j] <= r_cut]
        if near and type_coord_atoms:
            near = [j for j in near if sym[j] in type_coord_atoms]
        rest = sym[n_central:]
        sites = [[] for _ in range(n_types)]        # per molecule type: one list of coordinating symbols per molecule
        idx = 0
        while idx < len(rest):
            for t, atoms in enumerate(main_atoms):
                if rest[idx: idx + len(atoms)] == atoms:
                    lo = idx + n_central
                    sites[t].append([sym[j] for j in near if lo <= j < lo + len(atoms)])
                    idx += len(atoms)
                    break
            # (like the reference, a tail that matches no molecule would loop forever; get_clusters never writes one)
        rows["num_mols"].append([len(s) for s in sites])
        labels = []
        for t in range(n_types):
            per_mol = []
            for coord in sites[t]:
                c = Counter(x[0] for x in coord if x)
                per_mol.append("".join(f"{c[k]}{k}" for k in sorted(c)))
            labels.append(":".join(sorted(per_mol)))
        rows["coordinating_atoms"].append(labels)
    if mol_names:
        num_cols = [f"num_{i}" for i in mol_names]
        atom_cols = [f"atoms_{i}" for i in mol_names]
    else:
        num_cols = [f"num_{i + 1}" for i in range(n_types)]
        atom_cols = [f"atoms_{i + 1}" for i in range(n_types)]
    df = pd.concat([pd.DataFrame({"cluster": rows["cluster"]}), pd.DataFrame(rows["num_mols"], columns=num_cols),
                    pd.DataFrame(rows["coordinating_atoms"], columns=atom_cols)], axis=1)
    df1 = df.groupby([c for c in df.columns if c != "cluster"]).size().rename("count").reset_index()
    df1.sort_values("count", ascending=False, inplace=True)
    df1["%"] = df1["count"] * 100 / sum(df1["count"])
    if find_top:
        if cum_perc and perc:
            warnings.warn("Two percentage types are provided for determining the top configurations; using cum_perc")
        if cum_perc:
            top = df1[df1["%"].cumsum() <= cum_perc]
        elif perc:
            top = df1[df1["%"] >= perc]
        else:
            raise ValueError("No percentage type is provided for determining the top configurations")
        df = df.sort_values("cluster").reset_index(drop=True)
        top = top.merge(df[["cluster"] + atom_cols], on=atom_cols).drop_duplicates(atom_cols)
        for rank, cluster in enumerate(top["cluster"]):
            shutil.copy(f"{working_dir}/{cluster}", f"{working_dir}/conf_{rank + 1}.xyz")
        top.to_csv(f"{working_dir}/top_conf.csv", index=False)
    df.to_csv(f"{working_dir}/clusters.csv", index=False)
    df1.to_csv(f"{working_dir}/configurations.csv", index=False)
    if zip:
        clusters_dir = f"{working_dir}/Clusters"
        os.mkdir(clusters_dir)
        for path in cluster_files:
            shutil.move(path, f"{clusters_dir}/{os.path.basename(path)}")
        shutil.make_archive(f"{working_dir}/Clusters", "zip", clusters_dir)
        shutil.rmtree(clusters_dir)
    return df, df1
