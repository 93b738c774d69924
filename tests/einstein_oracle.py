"""Test-side definition of the Einstein and Nernst-Einstein conductivity (``Conductivity.einstein`` / ``nernst``; the
reference's methods are empty, so there is no reference output to pin them to and their parity is unpinned).

TEST INFRASTRUCTURE ONLY, imported by tests/test_host_einstein.py and tests/test_gpu_einstein.py:
  * ``cross_msd_direct``: the long-double direct sum of mdp_cross_msd_fft (tests/native/cross_msd_direct.c, compiled
    into a temporary directory on first use);
  * ``einstein_conductivity`` / ``nernst_einstein``: numpy restatements of the two methods, built on the oracle's dump
    reader (``oracle.read_dumps``), centre-of-mass restatement (``oracle.com_unwrapped``) and the direct sum above.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as O

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "native", "cross_msd_direct.c")
_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(tempfile.mkdtemp(prefix="cross_msd_direct_"), "cross_msd_direct.so")
        base = ["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-o", so, _SRC]
        if subprocess.run(base[:1] + ["-fopenmp"] + base[1:], capture_output=True).returncode != 0:
            subprocess.run(base, check=True, capture_output=True)      # no OpenMP: the serial build
        _LIB = ctypes.CDLL(so)
    return _LIB


def cross_msd_direct(a, b, group_off, nlags):
    """long-double direct sum of mdp_cross_msd_fft: a, b [C,T] (b None: b = a), group_off [G+1] -> [G, nlags]."""
    a = np.ascontiguousarray(np.atleast_2d(a), dtype=np.float64)
    bb = None if b is None else np.ascontiguousarray(np.atleast_2d(b), dtype=np.float64)
    go = np.ascontiguousarray(group_off, dtype=np.int64)
    G = len(go) - 1
    out = np.empty((G, int(nlags)))
    dp = ctypes.POINTER(ctypes.c_double)
    _lib().orc_cross_msd_direct(a.ctypes.data_as(dp), None if bb is None else bb.ctypes.data_as(dp),
                                ctypes.c_int64(a.shape[1]), go.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
                                ctypes.c_int64(G), ctypes.c_int64(int(nlags)), out.ctypes.data_as(dp))
    return out


def _unwrapped_com_series(pattern, num_mols, num_atoms_per_mol, mass, unwrap):
    """per frame (timestep, molecular COM [3, M], molecular charge [M]) of unwrapped positions: ``xu yu zu`` columns
    (unwrap="xu") or x + ix * (xhi - xlo) (unwrap="image", _prepare_unwrapped_coords diffusion.py:62-81)."""
    steps, coms, q = [], [], None
    for fr in O.read_dumps(pattern):
        cols = fr.sorted_by_id()
        if unwrap == "image":
            L = fr.bound_lengths
            for k, ax in enumerate("xyz"):
                cols[ax + "u"] = cols[ax] + cols["i" + ax] * L[k]
        c = O.com_unwrapped(cols, num_mols, num_atoms_per_mol, mass, charge=True)
        steps.append(fr.timestep)
        coms.append(np.stack([c["xu"], c["yu"], c["zu"]]))
        q = c["q"]
    return np.asarray(steps, dtype=np.float64), np.stack(coms), q


def _fit_slope(t, y, max_lag, initial_time, final_time):
    """polyfit (degree 1, with intercept) over the lag window: default lags max(1, max_lag // 10) .. max_lag - 1."""
    lo = t[max(1, max_lag // 10)] if initial_time is None else initial_time
    hi = t[max_lag - 1] if final_time is None else final_time
    m = (t >= lo) & (t <= hi)
    return np.polyfit(t[m], y[m], 1)[0]


def einstein_conductivity(pattern, num_mols, num_atoms_per_mol, volume_si, temp, dt_si, mass, dist_conv, charge_conv, kb,
                          max_lag=None, initial_time=None, final_time=None, unwrap="xu"):
    """Conductivity.einstein: sigma_E[ntypes+1] (S/m) and the dipole MSD [ntypes+1, max_lag]; dt_si = frame spacing (s)."""
    _, com, q = _unwrapped_com_series(pattern, num_mols, num_atoms_per_mol, mass, unwrap)
    T = com.shape[0]
    off = np.concatenate(([0], np.cumsum(num_mols))).astype(np.int64)
    qs = q * charge_conv
    M = np.stack([np.einsum("tcm,m->ct", com[:, :, off[g]:off[g + 1]] * dist_conv, qs[off[g]:off[g + 1]])
                  for g in range(len(num_mols))], axis=1)                                  # [3, G, T]
    tot = M.sum(axis=1)
    max_lag = T // 2 if max_lag is None else max_lag
    rows = np.concatenate([M.transpose(1, 0, 2), tot[None]], axis=0)                     # [G+1, 3, T]
    msd = np.stack([cross_msd_direct(rows[i], tot, [0, 3], max_lag)[0] for i in range(len(rows))])
    t = np.arange(max_lag) * dt_si
    slopes = np.array([_fit_slope(t, r, max_lag, initial_time, final_time) for r in msd])
    return slopes / (6 * kb * temp * volume_si), msd


def nernst_einstein(pattern, num_mols, num_atoms_per_mol, volume_si, temp, dt_si, mass, dist_conv, charge_conv, kb,
                    max_lag=None, initial_time=None, final_time=None, unwrap="xu"):
    """Conductivity.nernst: (sigma_NE[ntypes+1] in S/m, D[ntypes] in m^2/s)."""
    _, com, q = _unwrapped_com_series(pattern, num_mols, num_atoms_per_mol, mass, unwrap)
    T = com.shape[0]
    off = np.concatenate(([0], np.cumsum(num_mols))).astype(np.int64)
    chans = (com * dist_conv).transpose(2, 1, 0).reshape(-1, T)                          # [M * 3, T]
    max_lag = T // 2 if max_lag is None else max_lag
    msd = cross_msd_direct(chans, None, 3 * off, max_lag) / np.asarray(num_mols, dtype=np.float64)[:, None]
    t = np.arange(max_lag) * dt_si
    D = np.array([_fit_slope(t, r, max_lag, initial_time, final_time) for r in msd]) / 6
    qs = q * charge_conv
    q2 = np.array([np.sum(qs[off[g]:off[g + 1]] ** 2) for g in range(len(num_mols))])
    cond = D * q2 / (volume_si * kb * temp)
    return np.append(cond, cond.sum()), D
