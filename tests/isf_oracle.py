"""numpy restatement of the coherent intermediate scattering function (mdproptools_b200/dynamical/intermediate_scattering.py,
csrc/isffft.cu).  The reference has no implementation, so this is the definition the library is checked against:

  the k-set and bins of tests/sk_oracle.py; rho_c(k, t) = sum_{j in c} exp(i k.r_j(t)) per frame t < T (one cell);
  C_ab(k, tau) = 1/(T - tau) sum_{t < T-tau} 1/2 Re( z_a(k,t+tau) z_b(k,t)* + z_b(k,t+tau) z_a(k,t)* ),  z_c = rho_c;
  F_ab(bin, tau) = sum_{k in bin} C_ab(k, tau) / (n_k sqrt(N_a N_b));
  F(bin, tau) = sum_{k in bin} C_tt(k, tau) / (n_k N),  z_t = sum over every class (the unnamed types included);
  NaN for a bin without k-vectors.
"""
from __future__ import annotations

import numpy as np

from tests import sk_oracle as SO


def direct_corr(re, im, pairs, bin_off, nlags, dtype=np.longdouble):
    """re, im [nchan, nk, T] -> [npairs, nbins, nlags]: sum over each bin's k of C_ab(k, tau), by the direct sum in ``dtype``."""
    re = np.asarray(re, dtype=dtype)
    im = np.asarray(im, dtype=dtype)
    T = re.shape[2]
    nbins = len(bin_off) - 1
    out = np.zeros((len(pairs), nbins, nlags), dtype=dtype)
    for q, (a, b) in enumerate(pairs):
        for tau in range(nlags):
            m = T - tau
            # 1/2 Re(x y*) + 1/2 Re(y' x'*), Re(x y*) = x.re y.re + x.im y.im
            s = 0.5 * ((re[a, :, tau:] * re[b, :, :m] + im[a, :, tau:] * im[b, :, :m]).sum(axis=1)
                       + (re[b, :, tau:] * re[a, :, :m] + im[b, :, tau:] * im[a, :, :m]).sum(axis=1)) / m
            for bb in range(nbins):
                out[q, bb, tau] = s[bin_off[bb]:bin_off[bb + 1]].sum()
    return out


def series(cell, frames_pos, cls, ncls, miller, dtype=np.float64):
    """rho per class, k and frame: (re, im) [ncls, nk, T] from positions [T, N, 3]."""
    T = len(frames_pos)
    re = np.zeros((ncls, len(miller), T), dtype=dtype)
    im = np.zeros_like(re)
    for t, pos in enumerate(frames_pos):
        r, i = SO.class_rho(cell, pos, cls, ncls, miller, dtype)
        re[:, :, t], im[:, :, t] = r, i
    return re, im


def isf(cell, frames_pos, types, k_max, bin_size, relations_types, max_lag=None, k_min=None, max_k_per_bin=None, seed=0):
    """One cell, positions [T, N, 3], fixed types [N] -> (k centres, F [nbins, L], F_ab [R, nbins, L], n_k [nbins]) with the
    correlation summed in long double."""
    named = sorted(set(int(t) for pair in relations_types for t in pair))
    types = np.asarray(types).astype(np.int64)
    cls = np.array([named.index(t) if t in named else len(named) for t in types])
    ncls = len(named) + 1
    miller, bin_off, nbins = SO.kset_brute(cell, k_max, bin_size, k_min, max_k_per_bin, seed)
    re, im = series(cell, frames_pos, cls, ncls, miller)
    re = np.concatenate([re, re.sum(axis=0, keepdims=True)])
    im = np.concatenate([im, im.sum(axis=0, keepdims=True)])
    T = len(frames_pos)
    L = T // 2 if max_lag is None else int(max_lag)
    rel = [(named.index(int(a)), named.index(int(b))) for a, b in relations_types]
    P = direct_corr(re, im, [(ncls, ncls)] + rel, bin_off, L).astype(np.float64)
    counts = np.bincount(cls, minlength=ncls)
    nk = np.diff(bin_off).astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        F = P[0] / (nk[:, None] * len(types))
        Fab = np.stack([P[1 + r] / (nk[:, None] * np.sqrt(float(counts[a]) * float(counts[b]))) for r, (a, b) in enumerate(rel)]) \
            if rel else np.zeros((0, nbins, L))
    F[nk == 0] = np.nan
    Fab[:, nk == 0] = np.nan
    return (np.arange(nbins) + 0.5) * bin_size, F, Fab, nk


def rigid_translation(cell, pos0, cls, ncls, miller, shift, pairs, bin_off, nlags):
    """Closed form for r_j(t) = r_j(0) + shift * t: rho_c(k, t) = exp(i k.shift t) rho_c(k, 0), so
    C_ab(k, tau) = Re(rho_a(k,0) rho_b(k,0)*) cos(k.shift tau), whatever T; summed per bin -> [npairs, nbins, nlags]."""
    re, im = SO.class_rho(cell, pos0, cls, ncls, miller)
    re = np.concatenate([re, re.sum(axis=0, keepdims=True)])
    im = np.concatenate([im, im.sum(axis=0, keepdims=True)])
    s = np.linalg.solve(SO.cell_matrix(cell), np.asarray(shift, dtype=np.float64))
    kv = 2 * np.pi * (np.asarray(miller, dtype=np.float64) @ s)                          # k.shift per k-vector
    tau = np.arange(nlags)
    out = np.zeros((len(pairs), len(bin_off) - 1, nlags))
    for q, (a, b) in enumerate(pairs):
        c = (re[a] * re[b] + im[a] * im[b])[:, None] * np.cos(kv[:, None] * tau[None, :])
        for bb in range(len(bin_off) - 1):
            out[q, bb] = c[bin_off[bb]:bin_off[bb + 1]].sum(axis=0)
    return out
