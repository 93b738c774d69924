"""Residence-time survival correlation -- drop-in for ``mdproptools.dynamical.residence_time.ResidenceTime``
(reference mdproptools/dynamical/residence_time.py; citations are lines of that file).

Reference algorithm: per frame and relation (k, l), for every central atom of type k the indicator
h_ij(t) = r_in^2 < rsq_ij <= r_out^2 against every atom of type l (:100-104); then for every (i, j) column the
unbiased autocovariance of h (statsmodels acovf, FFT, no demeaning, :135-137), summed over all pairs, divided
by N_k N_l (:140) and normalised by its lag-0 value (:142).

Here: loop 1 is one rectangular neighbour-list call per batch of frames (mdp_pair_list, shell mode), the
indicators of the pairs that are ever neighbours become per-pair time bitmasks, and loop 2 is the exact
integer count  cnt[tau] = sum_pairs popcount(m & (m >> tau))  (mdp_bitmask_autocorr); the floats are formed
at the very end:  C(tau) = (cnt[tau] / (T - tau)) / (N_k N_l),  C /= C(0).
Multi-GPU: the search is split by FRAMES (rank r parses and searches frames r, r + w, ...: sorting the neighbour
set of every frame is the expensive part and does not shrink with the central set), the entries are routed to the
rank that owns their central atom (dist.exchange_rows, all-to-all over NVLink), the correlation is split by
CENTRAL ATOMS (a pair's time bitmask never crosses ranks) and cnt is merged with one int64 all-reduce (exact).

Divergence: with ``num_mols=None`` the reference crashes (it feeds 4-column rows to ``_calc_rsq(..., 0)``);
here the plain ``type`` column is used in that case.
"""
from __future__ import annotations

import os

import numpy as np
import pandas as pd
import torch

from .. import dist, ops
from ..common.frames import _merge_frames, calc_atom_type_ids
from ..io import dump as _dump
from ..io.pipeline import FrameBatches


class ResidenceTime:
    def __init__(self, r_cut, partial_relations, filename, dt=1, num_mols=None, num_atoms_per_mol=None, working_dir=None):
        self.r_cut = r_cut
        self.relation_matrix = np.asarray(partial_relations).transpose()
        self.atom_pairs = []
        self.filename = filename
        self.dt = dt * 10 ** -3  # input dt in fs - convert to ps (:55)
        self.corr_df = None
        self.res_time_df = None
        self.num_mols = num_mols
        self.num_atoms_per_mol = num_atoms_per_mol
        self.working_dir = working_dir or os.getcwd()

    @staticmethod
    def _stretched_exp_function(x, a, tau_res, tau_short, beta):
        return a * np.exp(-((x / tau_res) ** beta)) + (1 - a) * np.exp(-x / tau_short)

    @staticmethod
    def _integrate_sum_exp(a, tau_res, tau_short, beta):
        from scipy.special import gamma

        return (a * tau_res * gamma(1 + 1 / beta)) + (1 - a) * tau_short

    def calc_auto_correlation(self):
        want = ["id", "type", "x", "y", "z"]
        altered = bool(self.num_mols and self.num_atoms_per_mol)
        R = len(self.relation_matrix)
        lists = [[] for _ in range(R)]
        rows_k, rows_l = [None] * R, [None] * R
        w, me = dist.world_size(), dist.rank()
        dev = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
        own = {}                                # global frame index -> timestep of the frames searched here
        batches = FrameBatches(self.filename, want, frame_select=(lambda i: i % w == me) if w > 1 else None)
        for batch in batches:
            d = batch.wait()
            host = batch.host.numpy()
            for k, meta in enumerate(batch.metas):
                own[meta.index] = meta.timestep
                # altered types are derived from the id column of the id-sorted frame (:80-90)
                typ = calc_atom_type_ids(host[k, 0], self.num_mols, self.num_atoms_per_mol) if altered else host[k, 1]
                for kl in range(R):
                    a, b = self.relation_matrix[kl]
                    ra, rb = np.nonzero(typ == a)[0], np.nonzero(typ == b)[0]
                    if rows_k[kl] is None:
                        rows_k[kl], rows_l[kl] = ra, rb
                    elif not (np.array_equal(rows_k[kl], ra) and np.array_equal(rows_l[kl], rb)):
                        raise ValueError("atom types change between frames; residence time needs a fixed pair set")
            xyz = d[:, 2:5, :]
            boxes = np.array([m.box.lattice_lengths() for m in batch.metas])        # (:79)
            fidx = torch.tensor([m.index for m in batch.metas], dtype=torch.int32, device=d.device)
            for kl in range(R):
                a, b = self.relation_matrix[kl]
                ra, rb = rows_k[kl], rows_l[kl]
                if len(ra) == 0 or len(rb) == 0:
                    continue
                xa = xyz.index_select(2, torch.from_numpy(ra).to(d.device)).contiguous()
                xb = xyz.index_select(2, torch.from_numpy(rb).to(d.device)).contiguous()
                lst, _ = ops.pair_list(xa, xb, boxes, self.r_cut[kl][0] ** 2, self.r_cut[kl][1] ** 2, shell_mode=1,
                                       exclude_same_index=False)
                if len(lst):
                    lst = lst.clone()
                    if a == b:                                                   # h[idx] = False (:103-104)
                        lst = lst[lst[:, 1] != lst[:, 2]]
                    lst[:, 0] = fidx[lst[:, 0].long()]                           # batch-local -> trajectory frame index
                    lists[kl].append(lst)
        T = batches.total_frames or 0
        if T == 0:
            raise ValueError(f"no dump frames found for {self.filename!r}")
        # every rank needs every frame's time and the sizes of the two sets (a rank may have had no frame at all)
        tt = _merge_frames(own, T, (), dev)
        nkl = torch.tensor([[len(rows_k[kl]), len(rows_l[kl])] if rows_k[kl] is not None else [0, 0] for kl in range(R)],
                           dtype=torch.int64, device=dev).reshape(R, 2)
        if w > 1:
            dist.all_reduce_max_(nkl)
        times = [float(v) * self.dt for v in tt.cpu().numpy()]
        nkl = nkl.cpu().numpy()
        correlation = {"Time (ps)": times}
        for kl in range(R):
            a, b = self.relation_matrix[kl]
            atom_pair = f"{a}-{b}"
            n_k, n_l = int(nkl[kl, 0]), int(nkl[kl, 1])
            lst = torch.cat(lists[kl], dim=0) if lists[kl] else torch.zeros((0, 3), dtype=torch.int32, device=dev)
            if w > 1:
                lst = dist.exchange_rows(lst, dist.owner_of_rows(lst[:, 1], n_k, w))
            if len(lst):
                cnt, _ = ops.bitmask_autocorr_from_list(lst.contiguous(), n_l, T, n_a=n_k)
            else:
                cnt = torch.zeros((T,), dtype=torch.int64, device=dev)
            if w > 1:
                dist.all_reduce_sum_(cnt)
            cnt = cnt.cpu().numpy().astype(np.float64)
            total_number_of_columns = n_k * n_l
            corr_array = (cnt / (T - np.arange(T))) / total_number_of_columns       # acovf unbiased, (:135-140)
            corr_array = corr_array / corr_array[0]                                 # (:142)
            correlation[atom_pair] = corr_array
        self.atom_pairs = [f"{a}-{b}" for a, b in self.relation_matrix] * T
        self.corr_df = pd.DataFrame.from_dict(correlation)
        if dist.rank() == 0:
            self.corr_df.to_csv(self.working_dir + "/auto_correlation.csv")
        return self.corr_df

    def fit_auto_correlation(self, cut_percent=0.9, plot=True):
        """Stretched-exponential fit of every correlation column (:150-208); host scipy."""
        from scipy.optimize import curve_fit

        residence_time = {}
        corr_data = self.corr_df.head(int(len(self.corr_df) * cut_percent))
        for col in corr_data:
            if col == "Time (ps)":
                continue
            x = corr_data["Time (ps)"].values
            y = corr_data[col].values
            popt, _ = curve_fit(self._stretched_exp_function, x, y, bounds=([0, 0, 0, 0.1], [np.inf, np.inf, np.inf, 1]),
                                maxfev=5000)
            a, tau_res, tau_short, beta = popt
            residence_time[col] = [a, tau_res, tau_short, beta, self._integrate_sum_exp(a, tau_res, tau_short, beta)]
            if plot:
                try:
                    import matplotlib
                    matplotlib.use("Agg")
                    import matplotlib.pyplot as plt
                except ImportError as exc:
                    raise ImportError("plot=True needs matplotlib") from exc
                fig, ax = plt.subplots(figsize=(8, 6))
                ax.scatter(x, y, color="red", label="original")
                ax.plot(x, self._stretched_exp_function(x, a, tau_res, tau_short, beta), color="black", label="fit")
                ax.legend(frameon=False)
                ax.set_xlabel("Time (ps)")
                ax.set_ylabel("C(t)")
                fig.savefig(self.working_dir + f"/{col}_fit.png", bbox_inches="tight", pad_inches=0.1)
                plt.close(fig)
        self.res_time_df = pd.DataFrame(residence_time)
        self.res_time_df.index = ["a", "tau_res", "tau_short", "beta", "r (ps)"]
        self.res_time_df.to_csv(self.working_dir + "/residence_time.csv")
        return residence_time
