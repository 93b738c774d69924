"""Reorientation: first- and second-rank orientational correlation functions of molecule-fixed unit vectors and their
correlation times (extension: the reference has no implementation; tests/reorient_oracle.py is the definition).

C1 of a dipole direction is compared with dielectric relaxation, C2 of a bond vector with NMR relaxation and OKE / 2D-IR
anisotropy.  Definition, for T >= 2 evenly spaced frames with a fixed atom count:

  molecules in atom-id order (``MoleculeLayout``); a vector definition ``name -> (mol_type, kind, atoms)`` names 1-based
  atom positions i, j (, k) inside every molecule of type ``mol_type`` (1-based);
  d_j = mic(r_j - r_i), d_k = mic(r_k - r_i) in the frame's restricted triclinic cell;
  w = d_j (``"bond"``), (d_j + d_k)/2 (``"bisector"``), d_j x d_k (``"normal"``);  u = w / |w|;
  C_l(tau) = 1/M sum_m 1/(T - tau) sum_{t < T-tau} P_l(u_m(t).u_m(t+tau)),  l = 1, 2,  tau < max_lag (default T // 2);
  tau_l = the trapezoid running integral of C_l read at t_end, the first lag >= 1 where C_l <= 0 (else the last lag).

Device work: mdp_orient_series (csrc/orient.cu) turns every batch of parsed frames into 8 channels per molecule -- u and
the 5 orthonormal components of u u^T - I/3 -- written time-major into one [sum_v 8 M_v, T] series; one grouped FFT
autocorrelation (mdp_group_acf_fft) then gives, per definition, sum_m u.u' over the 3 M_v rank-1 channels and sum_m Q:Q'
over the 5 M_v rank-2 channels, and P2(u.u') = 1.5 Q:Q' exactly.  No per-lag Legendre evaluation.

Multi-GPU: every rank reads every frame and keeps a contiguous block of each definition's molecules (``rank_blocks``); the
group sums are merged with one fp64 all-reduce.
"""
from __future__ import annotations

import numpy as np
import pandas as pd
import torch

from .. import ops
from .._lib import ORIENT_KINDS
from ..io.dump import dump_files
from ..io.pipeline import FrameBatches
from ..structural.structure_factor import _cell
from .series import DumpColumns, MoleculeLayout, all_reduce_groups, even_times, lag_count, rank_blocks

NATOMS_OF_KIND = {"bond": 2, "bisector": 3, "normal": 3}


def vector_rows(vectors, num_mols, num_atoms_per_mol):
    """Checked vector definitions -> per definition (name, kind code, 0-based atom rows [M, 3] of every molecule of its
    type; a bond's third row repeats its first).  ValueError for an unknown kind, the wrong number of atoms, an atom
    position outside the molecule, repeated atoms or a molecule type out of range.  Host only."""
    if not vectors:
        raise ValueError("no vector definitions given")
    start = np.concatenate(([0], np.cumsum(np.asarray(num_mols, dtype=np.int64) * np.asarray(num_atoms_per_mol, dtype=np.int64))))
    out = []
    for name, spec in vectors.items():
        try:
            mol_type, kind, atoms = spec
        except (TypeError, ValueError):
            raise ValueError(f"vector {name!r}: expected (mol_type, kind, atoms), got {spec!r}") from None
        if kind not in ORIENT_KINDS:
            raise ValueError(f"vector {name!r}: unknown kind {kind!r} (one of {', '.join(ORIENT_KINDS)})")
        atoms = [int(a) for a in atoms]
        if len(atoms) != NATOMS_OF_KIND[kind]:
            raise ValueError(f"vector {name!r}: a {kind} takes {NATOMS_OF_KIND[kind]} atoms, got {len(atoms)}")
        if not 1 <= int(mol_type) <= len(num_mols) or int(num_mols[int(mol_type) - 1]) < 1:
            raise ValueError(f"vector {name!r}: molecule type {mol_type} outside 1..{len(num_mols)} or without molecules")
        g = int(mol_type) - 1
        na = int(num_atoms_per_mol[g])
        for a in atoms:
            if not 1 <= a <= na:
                raise ValueError(f"vector {name!r}: atom position {a} outside 1..{na} of molecule type {mol_type}")
        if len(set(atoms)) != len(atoms):
            raise ValueError(f"vector {name!r}: repeated atoms {atoms}")
        first = start[g] + na * np.arange(int(num_mols[g]), dtype=np.int64)
        pos = np.asarray(atoms + [atoms[0]] * (3 - len(atoms)), dtype=np.int64) - 1
        out.append((str(name), ORIENT_KINDS[kind], first[:, None] + pos[None, :]))
    return out


def _channel_buffer(rows, frames, device, old=None):
    """[rows, frames] float64 on the device (the first columns of ``old`` copied over); ValueError when it does not fit the
    device's free memory."""
    need = rows * frames * 8
    free = torch.cuda.mem_get_info(device)[0]
    if need > free:
        raise ValueError(f"the orientation channels of {rows} series x {frames} frames ({need / 2 ** 30:.2f} GiB) exceed the "
                         f"device's free memory ({free / 2 ** 30:.2f} GiB): use fewer vectors or more GPUs")
    buf = torch.empty((rows, frames), dtype=torch.float64, device=device)
    if old is not None:
        buf[:, :old.shape[1]] = old
    return buf


def calc_reorientation(filename, vectors, num_mols, num_atoms_per_mol, max_lag=None, timestep=1, units="real",
                       path_or_buff="reorientation.csv", save_mode=True):
    """First- and second-rank orientational correlation functions of the vectors ``vectors`` (dict name -> (mol_type,
    kind, atoms); kind ``"bond"`` (i, j), ``"bisector"`` (i, j, k) or ``"normal"`` (i, j, k); 1-based mol_type and atom
    positions inside the molecule) over the frames of the LAMMPS dump(s) ``filename`` (``x y z``, or ``xu yu zu`` without
    wrapped columns; evenly spaced timesteps, fixed atom count).  Molecules are ``num_mols[g]`` of type g + 1 with
    ``num_atoms_per_mol[g]`` atoms each, in atom-id order.

    max_lag           lags tau < max_lag (default T // 2; clipped to T)
    timestep, units   the MD timestep and the LAMMPS unit style of the lag-time axis
    Returns a DataFrame with columns ``Time (s)`` (from 0), then ``C1_<name>`` and ``C2_<name>`` per vector in dict order;
    written to ``path_or_buff`` as CSV when ``save_mode``.  ValueError for a bad definition (before any frame is read), a
    dump without positions, a molecule layout that does not hold the frame's atoms, a changing atom count, uneven frames,
    fewer than 2 frames, max_lag < 1, channels that do not fit the device, or a degenerate vector (zero length or not
    finite in some frame: its C_l(0) is not finite)."""
    defs = vector_rows(vectors, num_mols, num_atoms_per_mol)
    if max_lag is not None and int(max_lag) < 1:
        raise ValueError(f"max_lag must be at least 1, got {max_lag}")
    layout = MoleculeLayout(num_mols, num_atoms_per_mol)
    plan = DumpColumns(filename)
    have = set(plan.available)
    if {"x", "y", "z"} <= have:
        cols = ["x", "y", "z"]
    elif {"xu", "yu", "zu"} <= have:
        cols = ["xu", "yu", "zu"]
    else:
        raise ValueError(f"the reorientation needs the dump columns x y z or xu yu zu ({filename!r} has {sorted(have)})")
    dev = torch.device("cuda", torch.cuda.current_device())
    # this rank's block of every definition's molecules; channel rows [8][m_v] per definition, stacked
    local, row0 = [], 0
    for name, kind, rows in defs:
        sel, (m,) = rank_blocks([np.arange(len(rows))], "cpu")
        local.append((name, kind, np.ascontiguousarray(rows[sel.numpy()], dtype=np.int32), m, row0, len(rows)))
        row0 += 8 * m
    natoms, buf, steps = None, None, {}
    for batch in FrameBatches(filename, cols):                                # every rank reads every frame
        xyz = batch.wait()
        for meta in batch.metas:
            if natoms is None:
                natoms = meta.natoms
                layout.check(natoms)
                buf = _channel_buffer(row0, max(2, len(dump_files(filename))), dev)
            elif meta.natoms != natoms:
                raise ValueError(f"the reorientation needs a fixed atom count: frame {meta.index} (timestep {meta.timestep}) "
                                 f"has {meta.natoms} atoms, the first frame {natoms}")
            steps[meta.index] = meta.timestep
        idx = [m.index for m in batch.metas]
        if idx[-1] >= buf.shape[1]:
            buf = _channel_buffer(row0, max(2 * buf.shape[1], idx[-1] + 1), dev, buf)
        cells = np.array([_cell(m.box) for m in batch.metas], dtype=np.float64)
        f0 = 0
        while f0 < len(idx):                # runs of consecutive frames (all of a batch: every frame is read)
            f1 = f0 + 1
            while f1 < len(idx) and idx[f1] == idx[f1 - 1] + 1:
                f1 += 1
            for _, kind, rows, m, r0, _ in local:
                if m:
                    ops.orient_series(xyz[f0:f1], cells[f0:f1], kind, rows, buf[r0:r0 + 8 * m].view(8, m, buf.shape[1]),
                                      frame0=idx[f0])
            f0 = f1
    if natoms is None:
        raise ValueError(f"no dump frames found for {filename!r}")
    T = len(steps)
    if T < 2:
        raise ValueError(f"the reorientation needs at least 2 frames, {filename!r} holds {T}")
    times = even_times([steps[i] for i in range(T)], units, timestep, repr(filename), who="the reorientation needs")
    L = lag_count(max_lag, T)
    if buf.shape[1] != T:
        buf = buf[:, :T].contiguous()
    goff = np.concatenate(([0], np.cumsum([k * d[3] for d in local for k in (3, 5)]))).astype(np.int64)   # (3 m_v, 5 m_v)
    sums = all_reduce_groups(lambda c: ops.group_acf_fft(c, goff, L), buf, len(goff) - 1, L)
    del buf
    sums = sums.cpu().numpy()
    out = {"Time (s)": times[:L] - times[0]}
    for v, (name, _, _, _, _, M) in enumerate(local):
        c1, c2 = sums[2 * v] / M, 1.5 * sums[2 * v + 1] / M
        if not (np.isfinite(c1[0]) and np.isfinite(c2[0])):
            raise ValueError(f"vector {name!r}: C_l(0) is not finite -- the vector is degenerate (zero length) or not finite "
                             f"in some frame")
        out[f"C1_{name}"], out[f"C2_{name}"] = c1, c2
    df = pd.DataFrame(out)
    if save_mode:
        df.to_csv(path_or_buff, index=False)
    return df


def calc_reorientation_times(corr):
    """Correlation times of every ``C*`` column of ``calc_reorientation``: tau = the trapezoid running integral (one device
    call over all columns) read at t_end, the first lag >= 1 where the curve is <= 0, or the last lag when it never gets
    there.  Returns a DataFrame indexed by column name with columns ``tau (s)`` and ``t_end (s)``."""
    names = [c for c in corr.columns if c.startswith("C")]
    t = corr["Time (s)"].to_numpy(dtype=np.float64)
    if len(t) < 2:
        raise ValueError(f"the correlation times need at least 2 lag times, got {len(t)}")
    c = np.array(corr[names].to_numpy(dtype=np.float64).T, order="C")
    run = ops.cumtrapz(torch.from_numpy(c).cuda(), float(t[1] - t[0]), 1.0, leading_zero=True).cpu().numpy()
    ends = [t_end_index(row) for row in c]
    return pd.DataFrame([(run[k, e], t[e]) for k, e in enumerate(ends)], columns=["tau (s)", "t_end (s)"], index=names)


def t_end_index(c):
    """The lag at which a correlation curve's integral is read: the first lag >= 1 where c <= 0, else the last lag."""
    hit = np.nonzero(np.asarray(c)[1:] <= 0)[0]
    return int(hit[0]) + 1 if len(hit) else len(c) - 1
