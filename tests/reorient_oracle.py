"""numpy restatement of the reorientation correlations (``dynamical/reorientation.py``; csrc/orient.h, csrc/orient.cu).  The
reference has no implementation, so this is the definition the library is checked against:

  molecules in atom-id order (num_mols[g] of type g + 1 with num_atoms_per_mol[g] atoms each); a vector definition
  (mol_type, kind, atoms) names 1-based atom positions i, j (, k) inside each molecule of that type;
  d_j = mic(r_j - r_i), d_k = mic(r_k - r_i) in the frame's triclinic cell H = [a b c], a = (lx,0,0), b = (xy,ly,0),
  c = (xz,yz,lz), here in fractional form: s = H^-1 d, d - H rint(s) (the nearest image for vectors short next to half the
  cell, which is what the library's sequential reduction gives too);
  w = d_j (bond), (d_j + d_k)/2 (bisector), d_j x d_k (normal);  u = w / |w|;
  C_l(tau) = 1/M sum_m 1/(T - tau) sum_{t < T-tau} P_l(u_m(t).u_m(t+tau)),  l = 1, 2,  tau < L (default T // 2),
  evaluated directly for every origin and lag in long double -- no channel decomposition, no FFT;
  tau_l = the trapezoid running integral of C_l read at t_end, the first lag >= 1 where C_l <= 0 (the last lag when C_l
  never reaches 0).

``channels`` restates the 8 channels of csrc/orient.h for the host checks of the kernel body only.
TEST INFRASTRUCTURE ONLY, imported by tests/test_host_reorientation.py and tests/test_gpu_reorientation.py.
"""
from __future__ import annotations

import numpy as np

from oracle import oracle as O

LD = np.longdouble
KINDS = {"bond": 2, "bisector": 3, "normal": 3}


def read_positions(pattern):
    """(timesteps [T], positions [T, 3, N] in id order, cells [T, 6] = (lx, ly, lz, xy, xz, yz)): ``x y z``, or ``xu yu zu``
    when the dump has no wrapped columns."""
    steps, pos, cells = [], [], []
    for fr in O.read_dumps(pattern):
        c = fr.sorted_by_id()
        names = ("x", "y", "z") if "x" in c else ("xu", "yu", "zu")
        pos.append(np.stack([c[k] for k in names]))
        tilt = fr.tilt if fr.tilt is not None else (0.0, 0.0, 0.0)
        cells.append(np.array(list(fr.bound_lengths) + list(tilt), dtype=np.float64))
        steps.append(fr.timestep)
    return np.asarray(steps, dtype=np.float64), np.stack(pos), np.stack(cells)


def mol_rows(num_mols, num_atoms_per_mol, mol_type, atoms):
    """[M, len(atoms)] 0-based atom rows of the definition's atoms in every molecule of type ``mol_type`` (1-based)."""
    start = int(np.dot(num_mols[:mol_type - 1], num_atoms_per_mol[:mol_type - 1]))
    na = num_atoms_per_mol[mol_type - 1]
    first = start + na * np.arange(num_mols[mol_type - 1])
    return first[:, None] + (np.asarray(atoms) - 1)[None, :]


def cell_matrix(cell):
    lx, ly, lz, xy, xz, yz = [LD(float(v)) for v in cell]
    return np.array([[lx, xy, xz], [LD(0), ly, yz], [LD(0), LD(0), lz]], dtype=LD)      # columns a, b, c


def mic(d, cell):
    """d [..., 3] -> its nearest image in the cell, in long double (fractional form)."""
    H = cell_matrix(cell)
    d = np.asarray(d, dtype=LD)
    sz = d[..., 2] / H[2, 2]
    sy = (d[..., 1] - sz * H[1, 2]) / H[1, 1]
    sx = (d[..., 0] - sy * H[0, 1] - sz * H[0, 2]) / H[0, 0]
    n = np.stack([np.rint(sx), np.rint(sy), np.rint(sz)], axis=-1)
    return d - n @ H.T


def unit_vectors(pos, cells, rows, kind):
    """u [T, M, 3] (long double) of the vectors whose atoms are ``rows`` [M, 2 or 3] in positions pos [T, 3, N]."""
    out = []
    for t in range(pos.shape[0]):
        r = np.asarray(pos[t], dtype=LD).T                                 # [N, 3]
        dj = mic(r[rows[:, 1]] - r[rows[:, 0]], cells[t])
        if kind == "bond":
            w = dj
        else:
            dk = mic(r[rows[:, 2]] - r[rows[:, 0]], cells[t])
            w = (dj + dk) / 2 if kind == "bisector" else np.cross(dj, dk)
        out.append(w / np.sqrt((w * w).sum(axis=1))[:, None])
    return np.stack(out)


def channels(u):
    """[8, ...] channels of unit vectors u [..., 3]: ux, uy, uz, then the orthonormal traceless-tensor components."""
    u = np.asarray(u, dtype=LD)
    x, y, z = u[..., 0], u[..., 1], u[..., 2]
    s2, s6 = np.sqrt(LD(2)), np.sqrt(LD(6))
    return np.stack([x, y, z, (x * x - y * y) / s2, (2 * z * z - x * x - y * y) / s6, s2 * x * y, s2 * x * z, s2 * y * z])


def legendre_corr(u, nlags):
    """(C1, C2) [nlags] float64 of unit vectors u [T, M, 3]: P_l(u(t).u(t+tau)) summed directly over every origin."""
    u = np.asarray(u, dtype=LD)
    T, M = u.shape[0], u.shape[1]
    c1, c2 = np.zeros(nlags, dtype=LD), np.zeros(nlags, dtype=LD)
    for tau in range(nlags):
        x = (u[tau:] * u[:T - tau]).sum(axis=2)                            # [T - tau, M]
        c1[tau] = x.sum() / (T - tau) / M
        c2[tau] = (LD(1.5) * x * x - LD(0.5)).sum() / (T - tau) / M
    return c1.astype(np.float64), c2.astype(np.float64)


def calc_reorientation(pattern, vectors, num_mols, num_atoms_per_mol, dt_step_si, max_lag=None):
    """calc_reorientation: a dict of columns (``Time (s)`` first, then C1_<name>, C2_<name> per vector in dict order);
    dt_step_si = seconds per LAMMPS step."""
    steps, pos, cells = read_positions(pattern)
    T = len(steps)
    L = T // 2 if max_lag is None else min(int(max_lag), T)
    out = {"Time (s)": (steps[:L] - steps[0]) * dt_step_si}
    for name, (mol_type, kind, atoms) in vectors.items():
        c1, c2 = legendre_corr(unit_vectors(pos, cells, mol_rows(num_mols, num_atoms_per_mol, mol_type, atoms), kind), L)
        out[f"C1_{name}"], out[f"C2_{name}"] = c1, c2
    return out


def t_end_index(c):
    """The first lag >= 1 where c <= 0, else the last lag."""
    c = np.asarray(c)
    hit = np.nonzero(c[1:] <= 0)[0]
    return int(hit[0]) + 1 if len(hit) else len(c) - 1


def correlation_time(t, c):
    """(tau, t_end) of one curve: the trapezoid integral of c from 0 to t_end."""
    k = t_end_index(c)
    c = np.asarray(c, dtype=np.float64)
    return float(np.sum(0.5 * (c[1:k + 1] + c[:k]) * (t[1] - t[0]))), float(t[k])
