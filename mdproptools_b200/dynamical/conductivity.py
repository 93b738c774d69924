"""Green-Kubo ionic conductivity -- drop-in for ``mdproptools.dynamical.conductivity.Conductivity``
(reference mdproptools/dynamical/conductivity.py and _conductivity.py; citations are lines of
conductivity.py unless prefixed).

Device work: the charge-flux stage (per frame: molecular COM velocity, molecular charge, per-type
J = sum q v, _conductivity.py:7-36) as a streaming segmented reduction over ``[T][3][N]`` velocities
(csrc/reduce.cu), the ntypes^2 x 3 unbiased cross-correlations (:97-114, :197-214) as batched direct fp64
correlations and the cumulative trapezoid (:216-232) (csrc/corr.cu).  ``detect_time_range`` (:116-165) is
discrete window selection and stays on the host, fed with the device results.

Einstein (Helfand) and Nernst-Einstein conductivity (``einstein``, ``nernst``; the reference's methods are empty): the
translational dipole M = sum q_mol r_com per type is the charge-flux reduction applied to unwrapped positions, and
both the dipole MSD and the per-type centre-of-mass MSD over all time origins go through the FFT kernel
mdp_cross_msd_fft (csrc/msdfft.cu).  The straight-line fits (with intercept) run on the host.

Multi-GPU: frames are split round-robin for the flux and dipole stages (all-reduce of the zero-padded J or M), the
correlation channels (or dipole MSD groups) are split over ranks and summed with one fp64 all-reduce; ``nernst`` parses
every frame on every rank and shards the molecules of each type.
"""
from __future__ import annotations

import os

import numpy as np
import pandas as pd
import torch

from .. import dist, ops
from ..common import constants
from ..common.com_mols import atom_masses, mol_membership
from ..io import dump as _dump
from ..io.pipeline import FrameBatches
from .diffusion import fit_window, position_columns, unwrapped_positions


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


class Conductivity:
    def __init__(self, filename, num_mols, num_atoms_per_mol, volume, mass=None, temp=298.15, timestep=1, units="real",
                 working_dir=None):
        self.working_dir = working_dir or os.getcwd()
        self.filename = filename
        self.mass = mass
        self.num_mols = num_mols
        self.num_atoms_per_mol = num_atoms_per_mol
        self.units = units
        self.volume = volume * constants.DISTANCE_CONVERSION[self.units] ** 3  # volume in m^3 (:92)
        self.temp = temp
        self.timestep = timestep
        self.time = []  # time data used to calculate GK integral

    # -- correlators --------------------------------------------------------------------------------
    @staticmethod
    def correlate(a, b):
        """Unbiased correlation c[tau] = sum_t a[t+tau] b[t] / (T - tau) (:97-114), direct sum on the device."""
        a = torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).cuda().reshape(1, -1)
        b = torch.as_tensor(np.ascontiguousarray(b, dtype=np.float64)).cuda().reshape(1, -1)
        return ops.xcorr_unbiased(a, b)[0].cpu().numpy()

    @staticmethod
    def detect_time_range(flux, tol):
        """Host restatement of :116-165: block-wise std of the correlation function, normalised by the std of
        the block stds, thresholded at ``tol``, median-filtered; the longest run of quiet blocks wins."""
        flux = pd.Series(flux, name="flux")
        time_step = max(int(len(flux) / 10000), 5)
        ind = [i // time_step for i in range(len(flux))]
        flux_std = flux.groupby(ind).transform("std")
        std = flux_std.std()
        div = std if std else 1
        flux_std = flux_std / div
        flux_std = (flux_std < tol).astype("int").to_frame()
        flux_std = (
            flux_std.rolling(window=4 * time_step + 1, min_periods=3 * time_step + 1, center=True)
            .median().fillna(0)["flux"].to_list()
        )
        s_e_list = []
        found_start = False
        for k, v in enumerate(flux_std):
            if v == 1 and not found_start:
                s_e_list.append((k,))
                found_start = True
            elif v < 1 and found_start:
                s_e_list[-1] = s_e_list[-1] + (k,)
                found_start = False
        if s_e_list and len(s_e_list[-1]) == 1:
            s_e_list[-1] = s_e_list[-1] + (len(flux_std) - 1,)
        max_s_e = 0
        max_s_e_ind = None
        for s_e_ind, s_e in enumerate(s_e_list):
            if s_e[1] - s_e[0] > max_s_e:
                max_s_e = s_e[1] - s_e[0]
                max_s_e_ind = s_e_ind
        return s_e_list[max_s_e_ind]   # TypeError when no window exists, as in the reference

    # -- pipeline stages ------------------------------------------------------------------------------
    def get_charge_flux(self):
        """J[3, ntypes, T] (:167-195)."""
        pattern = f"{self.working_dir}/{self.filename}"
        cols = _dump.available_columns(pattern)
        want = ["id", "type", "q", "vx", "vy", "vz"]
        if not self.mass:
            assert "mass" in cols, "Missing atom masses in dump file."
            want.append("mass")
        mol_type, _, seg_off = mol_membership(self.num_mols, self.num_atoms_per_mol)
        ntypes = len(self.num_mols)
        type_off = np.concatenate(([0], np.cumsum(self.num_mols))).astype(np.int64)
        w, r = dist.world_size(), dist.rank()
        sel = (lambda i: i % w == r) if w > 1 else None
        batches = FrameBatches(pattern, want, frame_select=sel)
        pieces, times = [], {}
        dev = torch.device("cuda", torch.cuda.current_device())    # a rank without frames still joins the collectives
        seg_d = torch.from_numpy(seg_off.astype(np.int32)).to(dev)
        vs, qs = constants.VELOCITY_CONVERSION[self.units], constants.CHARGE_CONVERSION[self.units]
        for batch in batches:
            d = batch.wait()
            host = batch.host.numpy()
            n = host.shape[2]
            if seg_off[-1] != n:
                raise ValueError(f"Length of values ({seg_off[-1]}) does not match length of index ({n})")
            mcol = None if self.mass else batch.col("mass")

            def masses(k):
                return atom_masses(host[k, 1], self.mass) if self.mass else host[k, mcol]

            vel = d[:, 3:6, :].contiguous()
            # the kernel sums each molecule's charge and mass once per call; the reference does it per frame
            # (_conductivity.py:11-18), so one call serves the batch only when q, type and mass do not change inside it
            # (fixed-charge force fields); fluctuating charges (QEq, polarisable models) take one call per frame
            static = bool((host[:, 2] == host[0, 2]).all() and (host[:, 1] == host[0, 1]).all()
                          and (mcol is None or (host[:, mcol] == host[0, mcol]).all()))
            if static:
                j = ops.charge_flux(vel, torch.from_numpy(np.ascontiguousarray(masses(0))).to(dev), d[0, 2].contiguous(),
                                    seg_d, type_off, vs, qs)
            else:
                j = torch.cat([ops.charge_flux(vel[k:k + 1], torch.from_numpy(np.ascontiguousarray(masses(k))).to(dev),
                                               d[k, 2].contiguous(), seg_d, type_off, vs, qs)
                               for k in range(vel.shape[0])], dim=2)
            pieces.append(([m.index for m in batch.metas], j))
            for m in batch.metas:
                times[m.index] = m.timestep * constants.TIME_CONVERSION[self.units] * self.timestep
        T = batches.total_frames or 0
        if T == 0:
            raise ValueError(f"no dump frames found for {pattern!r}")
        J = torch.zeros((3, ntypes, T), dtype=torch.float64, device=dev)
        tt = torch.zeros((T,), dtype=torch.float64, device=dev)
        for idxs, j in pieces:
            ii = torch.tensor(idxs, device=dev)
            J[:, :, ii] = j
            tt[ii] = torch.tensor([times[i] for i in idxs], dtype=torch.float64, device=dev)
        dist.all_reduce_sum_(J)
        dist.all_reduce_sum_(tt)
        self.time = tt.cpu().tolist()
        self._flux_dev = J
        return J.cpu().numpy()

    def correlate_charge_flux(self, flux):
        """tot_flux[i] = sum_j sum_c corr(J_c,i , J_c,j); last row = grand total (:197-214)."""
        flux_d = torch.as_tensor(np.ascontiguousarray(flux, dtype=np.float64)).cuda()
        _, ntypes, T = flux_d.shape
        chans = [(k, i, j) for i in range(ntypes) for j in range(ntypes) for k in range(3)]
        lo, hi = dist.shard_range(len(chans))
        tot = torch.zeros((ntypes + 1, T), dtype=torch.float64, device=flux_d.device)
        if hi > lo:
            a = torch.stack([flux_d[k, i] for (k, i, j) in chans[lo:hi]]).contiguous()
            b = torch.stack([flux_d[k, j] for (k, i, j) in chans[lo:hi]]).contiguous()
            corr = ops.xcorr_unbiased(a, b)
            for row, (k, i, j) in zip(corr, chans[lo:hi]):       # fixed order: i, then j, then axis
                tot[i] += row
                tot[-1] += row
        dist.all_reduce_sum_(tot)
        return tot.cpu().numpy()

    def integrate_charge_flux_correlation(self, tot_flux):
        """Cumulative trapezoid with a leading zero, dx = time[1] - time[0] (:216-232)."""
        delta = self.time[1] - self.time[0]
        y = torch.as_tensor(np.ascontiguousarray(tot_flux, dtype=np.float64)).cuda()
        return ops.cumtrapz(y, delta, 1.0, leading_zero=True).cpu().numpy()

    def fit_curve(self, tot_flux, integral, tol):
        """(:234-257)"""
        ave = np.zeros((len(integral)))
        time_range = np.zeros((len(integral)), dtype=object)
        for i in range(len(integral)):
            time_range_ind = self.detect_time_range(tot_flux[i], tol=tol)
            ave[i] = np.average(integral[i][time_range_ind[0]: time_range_ind[1]])
            time_range[i] = (self.time[time_range_ind[0]], self.time[time_range_ind[1]])
        return ave, time_range

    def green_kubo(self, ave):
        """sigma = <integral> / 3 / k_B / T / V (:259-274)."""
        cond = np.zeros((len(ave)))
        for i in range(len(ave)):
            cond[i] = ave[i] / 3 / constants.BOLTZMANN / self.temp / self.volume
        return cond

    def calc_cond(self, tol=1e-4, plot=False, save=False):
        """Wrapper (:276-398): flux -> correlation -> integral -> plateau window -> conductivity (S/m)."""
        j = self.get_charge_flux()
        tot_flux = self.correlate_charge_flux(j)
        integral = self.integrate_charge_flux_correlation(tot_flux)
        ave, time_range = self.fit_curve(tot_flux, integral, tol)
        cond = self.green_kubo(ave)
        if plot:
            self._plot(tot_flux, integral, time_range)
        if save and dist.rank() == 0:
            charge_flux = np.append(np.array([self.time]), tot_flux, axis=0)
            integral_t = np.append(np.array([self.time]), integral, axis=0)
            start_time = [i[0] for i in time_range]
            end_time = [i[1] for i in time_range]
            cond_t = np.asarray([start_time, end_time, cond])
            mol_names = ",".join([str(i + 1) for i in range(len(tot_flux) - 1)]) + ",tot"
            col_names = "t" + "," + mol_names
            np.savetxt(f"{self.working_dir}/charge_flux.csv", charge_flux.T, delimiter=",", header=col_names, comments="")
            np.savetxt(f"{self.working_dir}/integral.csv", integral_t.T, delimiter=",", header=col_names, comments="")
            np.savetxt(f"{self.working_dir}/conductivity.csv", cond_t.T, delimiter=",", header="start_t,end_t,cond",
                       comments="")
            cond = cond_t   # the reference returns the stacked array when save=True (:376)
        return cond

    def _plot(self, tot_flux, integral, time_range):
        try:
            import matplotlib
            matplotlib.use("Agg")
            import matplotlib.pyplot as plt
        except ImportError as exc:
            raise ImportError("plot=True needs matplotlib") from exc
        t = np.array(self.time) * 10 ** 9
        fig, ax = plt.subplots(1, 2, figsize=(20, 5))
        for i in range(len(tot_flux) - 1):
            ax[0].plot(t, tot_flux[i], linewidth=2)
            ax[1].plot(t, integral[i], linewidth=2, label=i + 1)
        ax[0].plot(t, tot_flux[-1], linewidth=2, color="black")
        ax[1].plot(t, integral[-1], linewidth=2, color="black", label="total")
        for a in ax:
            a.axvline(time_range[-1][0] * 10 ** 9, color="black", linestyle="--")
            a.axvline(time_range[-1][1] * 10 ** 9, color="black", linestyle="--")
            a.set_xscale("log")
            a.set_xlabel("Time, 10^9 (s)")
        ax[1].legend(frameon=False)
        fig.savefig(f"{self.working_dir}/conductivity.png", bbox_inches="tight", pad_inches=0.1)
        plt.close(fig)

    # -- Einstein and Nernst-Einstein conductivity ------------------------------------------------------------
    def _fixed_charge_frames(self, frame_select=None):
        """Unwrapped positions of every (selected) frame, batch by batch: yields (frame indices, timesteps, pos [F,3,N]
        device) and returns nothing; afterwards ``self._fixed`` holds (q, type, mass) of the first frame seen (host arrays,
        None when this rank saw no frame).  Charges, types and masses must not change between frames (the Helfand moment of
        fluctuating charges is not the integral of the flux): ValueError otherwise, also across ranks."""
        pattern = f"{self.working_dir}/{self.filename}"
        cols = _dump.available_columns(pattern)
        if not cols:
            raise ValueError(f"no dump frames found for {pattern!r}")
        pos_cols = position_columns(cols)
        want = ["id", "type", "q"] + pos_cols
        if not self.mass:
            assert "mass" in cols, "Missing atom masses in dump file."
            want.append("mass")
        _, _, seg_off = mol_membership(self.num_mols, self.num_atoms_per_mol)
        self._fixed = None
        for batch in FrameBatches(pattern, want, frame_select=frame_select):
            d = batch.wait()
            host = batch.host.numpy()
            if seg_off[-1] != host.shape[2]:
                raise ValueError(f"Length of values ({seg_off[-1]}) does not match length of index ({host.shape[2]})")
            mcol = None if self.mass else batch.col("mass")
            if self._fixed is None:
                q0, t0 = host[0, 2].copy(), host[0, 1].copy()
                self._fixed = (q0, t0, atom_masses(t0, self.mass) if self.mass else host[0, mcol].copy())
            q0, t0, m0 = self._fixed
            if not ((host[:, 2] == q0).all() and (host[:, 1] == t0).all() and (mcol is None or (host[:, mcol] == m0).all())):
                raise ValueError("charges, types and masses must be the same in every frame for the Einstein and "
                                 "Nernst-Einstein conductivity")
            yield ([m.index for m in batch.metas], [m.timestep for m in batch.metas],
                   unwrapped_positions(d, batch.metas, 3, len(pos_cols) == 3).contiguous())
        if dist.world_size() > 1:                     # the same charges, types and masses on every rank
            n = int(seg_off[-1])
            dev = torch.device("cuda", torch.cuda.current_device())
            ref = (torch.from_numpy(np.concatenate(self._fixed)).to(dev) if self._fixed is not None
                   else torch.full((3 * n,), -np.inf, dtype=torch.float64, device=dev))
            hi = dist.all_reduce_max_(ref.clone())
            lo = dist.all_reduce_max_(torch.where(torch.isinf(ref), ref, -ref))
            if not torch.equal(hi, -lo):
                raise ValueError("charges, types and masses must be the same in every frame for the Einstein and "
                                 "Nernst-Einstein conductivity")
            if self._fixed is None:
                h = hi.cpu().numpy()
                self._fixed = (h[:n], h[n:2 * n], h[2 * n:])

    def _set_even_time(self, steps):
        """self.time from the timesteps of all frames (in trajectory order); they must be evenly spaced."""
        self.time = even_times(steps, self.units, self.timestep, f"{self.working_dir}/{self.filename!r}").tolist()

    def get_translational_dipole(self):
        """M[3, ntypes, T] in C m: per type, the sum over molecules of charge x unwrapped centre of mass (SI).  Positions
        are ``xu yu zu`` or x + ix (xhi - xlo) (as ``Diffusion``); charges, types and masses must be fixed and the frames
        evenly spaced (ValueError otherwise).  Sets ``self.time``."""
        _, _, seg_off = mol_membership(self.num_mols, self.num_atoms_per_mol)
        ntypes = len(self.num_mols)
        type_off = np.concatenate(([0], np.cumsum(self.num_mols))).astype(np.int64)
        w, r = dist.world_size(), dist.rank()
        dev = torch.device("cuda", torch.cuda.current_device())
        seg_d = torch.from_numpy(seg_off.astype(np.int32)).to(dev)
        ds, qs = constants.DISTANCE_CONVERSION[self.units], constants.CHARGE_CONVERSION[self.units]
        pieces, steps = [], {}
        frames = self._fixed_charge_frames((lambda i: i % w == r) if w > 1 else None)
        md = qd = None
        for idxs, ts, pos in frames:
            if md is None:
                md = torch.from_numpy(np.ascontiguousarray(self._fixed[2])).to(dev)
                qd = torch.from_numpy(np.ascontiguousarray(self._fixed[0])).to(dev)
            # the charge-flux reduction (csrc/reduce.cu) of positions instead of velocities
            pieces.append((idxs, ops.charge_flux(pos, md, qd, seg_d, type_off, ds, qs)))
            steps.update(zip(idxs, ts))
        T = torch.zeros((1,), dtype=torch.float64, device=dev)
        T[0] = max(steps) + 1 if steps else 0
        dist.all_reduce_max_(T)
        T = int(T.item())
        if T == 0:
            raise ValueError(f"no dump frames found for {self.working_dir}/{self.filename!r}")
        M = torch.zeros((3, ntypes, T), dtype=torch.float64, device=dev)
        st = torch.zeros((T,), dtype=torch.float64, device=dev)
        for idxs, m in pieces:
            ii = torch.tensor(idxs, device=dev)
            M[:, :, ii] = m
            st[ii] = torch.tensor([float(steps[i]) for i in idxs], dtype=torch.float64, device=dev)
        dist.all_reduce_sum_(M)
        dist.all_reduce_sum_(st)
        self._set_even_time(st.cpu().numpy())
        return M.cpu().numpy()

    def correlate_translational_dipole(self, dipole, max_lag=None):
        """[ntypes+1, max_lag] in C^2 m^2: row i = sum_j sum_axes <dM_i(lag) . dM_j(lag)> over all time origins, last row
        <|dM_tot(lag)|^2> (the row convention of ``correlate_charge_flux``).  By linearity row i is the cross MSD of the
        three channel pairs (M_i,c , M_tot,c): one mdp_cross_msd_fft call of 3 (ntypes+1) channels.  max_lag defaults to
        T // 2."""
        m = torch.as_tensor(np.ascontiguousarray(dipole, dtype=np.float64)).cuda()
        _, ntypes, T = m.shape
        max_lag = T // 2 if max_lag is None else min(int(max_lag), T)
        if max_lag < 1:
            raise ValueError(f"max_lag must be at least 1 ({T} frames)")
        tot = m[:, 0].clone()
        for i in range(1, ntypes):                      # fixed order
            tot += m[:, i]
        rows = torch.cat([m.permute(1, 0, 2), tot[None]], dim=0)       # [ntypes+1, 3, T]
        lo, hi = dist.shard_range(ntypes + 1)
        out = torch.zeros((ntypes + 1, max_lag), dtype=torch.float64, device=m.device)
        if hi > lo:
            a = rows[lo:hi].reshape(-1, T).contiguous()
            b = tot[None].expand(hi - lo, 3, T).reshape(-1, T).contiguous()
            out[lo:hi] = ops.cross_msd_fft(a, b, np.arange(0, 3 * (hi - lo) + 1, 3), max_lag)
        dist.all_reduce_sum_(out)
        return out.cpu().numpy()

    def _fit_window(self, max_lag, initial_time, final_time):
        """Lag times l * dt (l < max_lag) and the mask of the fit window (``fit_window``: by default the lags
        max(1, max_lag // 10) to max_lag - 1)."""
        dt = self.time[1] - self.time[0] if len(self.time) > 1 else 0.0
        t = np.arange(max_lag) * dt
        return t, fit_window(t, initial_time, final_time)

    @staticmethod
    def _slope(t, y):
        """Ordinary least squares with intercept: the slope of y against t."""
        tc = t - t.mean()
        return float(np.dot(tc, y - y.mean()) / np.dot(tc, tc))

    def einstein(self, max_lag=None, initial_time=None, final_time=None, save=False):
        """Einstein (Helfand) conductivity sigma_E[ntypes+1] in S/m: the slope of each row of the translational-dipole
        MSD (``correlate_translational_dipole``) against the lag time, fitted with intercept over
        initial_time <= t <= final_time, divided by 6 k_B T V.  Row i is the share of type i, the last row the total.
        ``save`` writes dipole_msd.csv and einstein_conductivity.csv into ``working_dir``."""
        dipole = self.get_translational_dipole()
        msd = self.correlate_translational_dipole(dipole, max_lag)
        max_lag = msd.shape[1]
        t, mask = self._fit_window(max_lag, initial_time, final_time)
        cond = np.array([self._slope(t[mask], row[mask]) for row in msd]) / (
            6 * constants.BOLTZMANN * self.temp * self.volume)
        if save and dist.rank() == 0:
            names = "t," + ",".join(str(i + 1) for i in range(len(msd) - 1)) + ",tot"
            np.savetxt(f"{self.working_dir}/dipole_msd.csv", np.append(t[None], msd, axis=0).T, delimiter=",", header=names,
                       comments="")
            win = np.asarray([[t[mask][0]] * len(cond), [t[mask][-1]] * len(cond), cond])
            np.savetxt(f"{self.working_dir}/einstein_conductivity.csv", win.T, delimiter=",", header="start_t,end_t,cond",
                       comments="")
        return cond

    def nernst(self, max_lag=None, initial_time=None, final_time=None, save=False):
        """Nernst-Einstein conductivity sigma_NE[ntypes+1] in S/m: row g = D_g sum_{m in g} q_m^2 / (V k_B T), the last
        row the sum.  D_g is slope / 6 of the all-origins centre-of-mass MSD of type g, fitted as in ``einstein`` (same
        window defaults, so sigma_NE / sigma_E is the Haven ratio); q_m is the molecule's charge summed in atom order.
        ``save`` writes nernst_einstein.csv (type, diffusion (m2/s), cond)."""
        _, _, seg_off = mol_membership(self.num_mols, self.num_atoms_per_mol)
        ntypes = len(self.num_mols)
        type_off = np.concatenate(([0], np.cumsum(self.num_mols))).astype(np.int64)
        dev = torch.device("cuda", torch.cuda.current_device())
        seg_d = torch.from_numpy(seg_off.astype(np.int32)).to(dev)
        # every rank parses every frame; the molecules of each type are split in contiguous blocks over the ranks
        shards = [dist.shard_range(int(n)) for n in self.num_mols]
        sel = np.concatenate([np.arange(type_off[g] + lo, type_off[g] + hi) for g, (lo, hi) in enumerate(shards)])
        sel_d = torch.from_numpy(sel.astype(np.int64)).to(dev)
        coms, steps, md = [], [], None
        for _, ts, pos in self._fixed_charge_frames():
            if md is None:
                md = torch.from_numpy(np.ascontiguousarray(self._fixed[2])).to(dev)
            com, _, _ = ops.segment_com(pos, md, seg_d)                          # [F, 3, M]
            coms.append(com.index_select(2, sel_d))
            steps += ts
        self._set_even_time(steps)
        T = len(steps)
        max_lag = T // 2 if max_lag is None else min(int(max_lag), T)
        t, mask = self._fit_window(max(max_lag, 1), initial_time, final_time)
        conv = constants.DISTANCE_CONVERSION[self.units]
        com = torch.cat(coms, dim=0) * conv                                     # [T, 3, Mloc] in m
        chans = com.permute(2, 1, 0).reshape(-1, T).contiguous()                # [Mloc * 3, T]
        goff = 3 * np.concatenate(([0], np.cumsum([hi - lo for lo, hi in shards]))).astype(np.int64)
        if chans.shape[0]:
            msd = ops.cross_msd_fft(chans, None, goff, max_lag)
        else:                                       # a rank without molecules still joins the all-reduce
            msd = torch.zeros((ntypes, max_lag), dtype=torch.float64, device=dev)
        dist.all_reduce_sum_(msd)
        msd = msd.cpu().numpy() / np.asarray(self.num_mols, dtype=np.float64)[:, None]
        diff = np.array([self._slope(t[mask], row[mask]) for row in msd]) / 6
        qmol = np.add.reduceat(self._fixed[0], seg_off[:-1]) * constants.CHARGE_CONVERSION[self.units]
        q2 = np.array([np.sum(qmol[type_off[g]:type_off[g + 1]] ** 2) for g in range(ntypes)])
        cond = diff * q2 / (self.volume * constants.BOLTZMANN * self.temp)
        cond = np.append(cond, cond.sum())
        if save and dist.rank() == 0:
            with open(f"{self.working_dir}/nernst_einstein.csv", "w") as f:
                f.write("type,diffusion (m2/s),cond\n")
                for g in range(ntypes):
                    f.write(f"{g + 1},{diff[g]!r},{cond[g]!r}\n")
                f.write(f"tot,,{cond[-1]!r}\n")
        return cond
