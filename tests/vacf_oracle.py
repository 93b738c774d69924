"""numpy restatement of the velocity autocorrelation, Green-Kubo self-diffusion and vibrational density of states
(``Diffusion.get_vacf``, ``calc_diff_green_kubo``, ``get_vdos``; csrc/msdfft.cu mdp_group_acf_fft).  The reference has no
implementation, so this is the definition the library is checked against:

  C_g(tau) = sum_{c in g} 1/(T - tau) sum_{t < T-tau} a_c(t+tau) a_c(t)        (acf_direct, in long double);
  per group (type or molecule type) the columns vxvx, vyvy, vzvz = C of the axis / N_g and vacf = their sum; for
  ``allatom`` also vacf = the sum over every type / N; velocities times VELOCITY_CONVERSION, not centred;
  D = mean over the fit window of the trapezoid running integral / dimension, std its standard deviation / dimension;
  S(nu_k) = 2 dt X_k / C_0 with X_k the explicit cosine sum of the (windowed) DCT-I and nu_k = k / (2 (L-1) dt).

TEST INFRASTRUCTURE ONLY, imported by tests/test_host_vacf.py and tests/test_gpu_vacf.py.
"""
from __future__ import annotations

import numpy as np

from oracle import oracle as O


def acf_direct(a, group_off, nlags, dtype=np.longdouble):
    """a [C, T], group_off [G+1] -> [G, nlags] float64: the grouped all-origins autocorrelation summed in ``dtype``."""
    a = np.asarray(np.atleast_2d(a), dtype=dtype)
    T = a.shape[1]
    go = np.asarray(group_off, dtype=np.int64)
    out = np.zeros((len(go) - 1, int(nlags)), dtype=dtype)
    for tau in range(int(nlags)):
        s = (a[:, tau:] * a[:, :T - tau]).sum(axis=1) / (T - tau)
        for g in range(len(go) - 1):
            out[g, tau] = s[go[g]:go[g + 1]].sum()
    return out.astype(np.float64)


def read_velocities(pattern, vel_conv, vacf_type="allatom", num_mols=None, num_atoms_per_mol=None, mass=None):
    """(timesteps [T], velocities [T, 3, n] in SI, labels, counts, members) of every frame: per atom (``allatom``, groups = atom
    types in ascending order) or per molecule centre of mass (``com``, groups = molecule types 1..)."""
    steps, vel, types0 = [], [], None
    for fr in O.read_dumps(pattern):
        cols = fr.sorted_by_id()
        if types0 is None:
            types0 = cols["type"].copy()
        assert np.array_equal(cols["type"], types0)
        if vacf_type == "com":
            c = O.com_unwrapped(cols, num_mols, num_atoms_per_mol, mass, attrs=("vx", "vy", "vz"))
        else:
            c = cols
        vel.append(np.stack([c["vx"], c["vy"], c["vz"]]) * vel_conv)
        steps.append(fr.timestep)
    if vacf_type == "com":
        off = np.concatenate(([0], np.cumsum(num_mols)))
        members = [np.arange(off[g], off[g + 1]) for g in range(len(num_mols))]
        labels = [str(g + 1) for g in range(len(num_mols))]
    else:
        tids = np.unique(types0)
        members = [np.nonzero(types0 == t)[0] for t in tids]
        labels = [str(int(t)) for t in tids]
    return np.asarray(steps, dtype=np.float64), np.stack(vel), labels, members


def get_vacf(pattern, dt_step_si, vel_conv, max_lag=None, vacf_type="allatom", num_mols=None, num_atoms_per_mol=None,
             mass=None):
    """Diffusion.get_vacf: a dict of columns (``Time (s)`` first); dt_step_si = seconds per LAMMPS step."""
    steps, vel, labels, members = read_velocities(pattern, vel_conv, vacf_type, num_mols, num_atoms_per_mol, mass)
    T = len(steps)
    L = T // 2 if max_lag is None else min(int(max_lag), T)
    out = {"Time (s)": (steps[:L] - steps[0]) * dt_step_si}
    total = np.zeros(L)
    for lab, idx in zip(labels, members):
        chans = vel[:, :, idx].transpose(1, 2, 0).reshape(-1, T)                   # [3 * n_g, T], axis-major
        s = acf_direct(chans, [0, len(idx), 2 * len(idx), 3 * len(idx)], L)
        for k, name in enumerate(["vxvx", "vyvy", "vzvz"]):
            out[f"{name}{lab}"] = s[k] / len(idx)
        out[f"vacf{lab}"] = s.sum(axis=0) / len(idx)
        total += s.sum(axis=0)
    if vacf_type == "allatom":
        out["vacf"] = total / sum(len(idx) for idx in members)
    return out


def green_kubo(t, c, dimension=3, initial_time=None, final_time=None):
    """(D, std, running integral) of one VACF column c over lag times t."""
    run = np.concatenate(([0.0], np.cumsum(0.5 * (c[1:] + c[:-1]) * (t[1] - t[0]))))
    L = len(t)
    lo = t[min(max(1, L // 10), L - 1)] if initial_time is None else initial_time
    hi = t[L - 1] if final_time is None else final_time
    m = (t >= lo) & (t <= hi)
    return run[m].mean() / dimension, run[m].std() / dimension, run


def vdos(c, dt, window="hann"):
    """(nu, S) by the explicit cosine sum of the DCT-I."""
    c = np.asarray(c, dtype=np.float64)
    L = len(c)
    l = np.arange(L)
    w = 0.5 * (1 + np.cos(np.pi * l / (L - 1))) if window == "hann" else np.ones(L)
    y = w * c
    X = np.array([y[0] + (-1) ** k * y[L - 1] + 2 * np.sum(y[1:L - 1] * np.cos(np.pi * k * l[1:L - 1] / (L - 1)))
                  for k in range(L)])
    return l / (2 * (L - 1) * dt), 2 * dt * X / c[0]
