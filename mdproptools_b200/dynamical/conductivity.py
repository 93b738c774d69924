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
from ..common.frames import _frame_batches, _merge_frames
from ..io.pipeline import FrameBatches
from .series import (DumpColumns, MoleculeLayout, all_reduce_groups, even_times, fit_window, lag_count, rank_blocks,
                     unwrapped_positions)


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
        want = DumpColumns(pattern).select(["id", "type", "q", "vx", "vy", "vz"], masses=not self.mass)
        layout = MoleculeLayout(self.num_mols, self.num_atoms_per_mol, self.mass)
        batches = _frame_batches(pattern, want, shard_files=False)
        fluxes, times = {}, {}
        dev = torch.device("cuda", torch.cuda.current_device())    # a rank without frames still joins the collectives
        vs, qs = constants.VELOCITY_CONVERSION[self.units], constants.CHARGE_CONVERSION[self.units]
        for batch in batches:
            d = batch.wait()
            host = batch.host.numpy()
            layout.check(host.shape[2])
            mcol = None if self.mass else batch.col("mass")

            def masses(k):
                return layout.masses(host[k, 1], None if mcol is None else host[k, mcol], dev)

            vel = d[:, 3:6, :].contiguous()
            # the kernel sums each molecule's charge and mass once per call; the reference does it per frame
            # (_conductivity.py:11-18), so one call serves the batch only when q, type and mass do not change inside it
            # (fixed-charge force fields); fluctuating charges (QEq, polarisable models) take one call per frame
            static = bool((host[:, 2] == host[0, 2]).all() and (host[:, 1] == host[0, 1]).all()
                          and (mcol is None or (host[:, mcol] == host[0, mcol]).all()))
            if static:
                j = ops.charge_flux(vel, masses(0), d[0, 2].contiguous(), layout.seg_d, layout.type_off, vs, qs)
            else:
                j = torch.cat([ops.charge_flux(vel[k:k + 1], masses(k), d[k, 2].contiguous(), layout.seg_d, layout.type_off,
                                               vs, qs) for k in range(vel.shape[0])], dim=2)
            idxs = tuple(m.index for m in batch.metas)
            fluxes[idxs] = j.permute(2, 0, 1)                                            # [F, 3, ntypes]
            times[idxs] = torch.tensor([m.timestep * constants.TIME_CONVERSION[self.units] * self.timestep
                                        for m in batch.metas], dtype=torch.float64, device=dev)
        J = _merge_frames(fluxes, batches.total_frames, (3, len(self.num_mols)), dev, torch.float64)     # [T, 3, ntypes]
        self.time = _merge_frames(times, batches.total_frames, (), dev, torch.float64).cpu().tolist()
        J = J.permute(1, 2, 0).contiguous()
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
    def _fixed_charge_frames(self, layout, round_robin=False):
        """Unwrapped positions of every frame (``round_robin``: of this rank's frames) of the molecules ``layout``, batch by
        batch: yields (frame indices, timesteps, pos [F,3,N], atom masses [N], charges [N]; on the device) and returns
        nothing; afterwards ``self._fixed`` holds (q, type, mass) of the first frame seen (host arrays, None when this rank
        saw no frame) and ``self._total_frames`` the number of frames of the trajectory.  Charges, types and masses must not
        change between frames (the Helfand moment of fluctuating charges is not the integral of the flux): ValueError
        otherwise, also across ranks."""
        pattern = f"{self.working_dir}/{self.filename}"
        want = DumpColumns(pattern).select(["id", "type", "q"], positions=True, masses=not self.mass)
        self._fixed = None
        batches = _frame_batches(pattern, want, shard_files=False) if round_robin else FrameBatches(pattern, want)
        for batch in batches:
            d = batch.wait()
            host = batch.host.numpy()
            layout.check(host.shape[2])
            mcol = None if self.mass else batch.col("mass")
            if self._fixed is None:
                q0, t0 = host[0, 2].copy(), host[0, 1].copy()
                self._fixed = (q0, t0, layout.masses(t0, None if mcol is None else host[0, mcol]))
                md, qd = torch.from_numpy(self._fixed[2]).to(d.device), torch.from_numpy(q0).to(d.device)
            q0, t0, m0 = self._fixed
            if not ((host[:, 2] == q0).all() and (host[:, 1] == t0).all() and (mcol is None or (host[:, mcol] == m0).all())):
                raise ValueError("charges, types and masses must be the same in every frame for the Einstein and "
                                 "Nernst-Einstein conductivity")
            yield (tuple(m.index for m in batch.metas), [m.timestep for m in batch.metas],
                   unwrapped_positions(d, batch.metas, 3, want[3] == "xu").contiguous(), md, qd)
        self._total_frames = batches.total_frames
        if dist.world_size() > 1:                     # the same charges, types and masses on every rank
            n = int(layout.seg_off[-1])
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
        layout = MoleculeLayout(self.num_mols, self.num_atoms_per_mol, self.mass)
        dev = torch.device("cuda", torch.cuda.current_device())
        ds, qs = constants.DISTANCE_CONVERSION[self.units], constants.CHARGE_CONVERSION[self.units]
        dipoles, steps = {}, {}
        for idxs, ts, pos, md, qd in self._fixed_charge_frames(layout, round_robin=True):
            # the charge-flux reduction (csrc/reduce.cu) of positions instead of velocities
            m = ops.charge_flux(pos, md, qd, layout.seg_d, layout.type_off, ds, qs)
            dipoles[idxs] = m.permute(2, 0, 1)                                           # [F, 3, ntypes]
            steps[idxs] = torch.tensor([float(s) for s in ts], dtype=torch.float64, device=dev)
        M = _merge_frames(dipoles, self._total_frames, (3, len(self.num_mols)), dev, torch.float64)      # [T, 3, ntypes]
        self._set_even_time(_merge_frames(steps, self._total_frames, (), dev, torch.float64).cpu().numpy())
        return M.permute(1, 2, 0).contiguous().cpu().numpy()

    def correlate_translational_dipole(self, dipole, max_lag=None):
        """[ntypes+1, max_lag] in C^2 m^2: row i = sum_j sum_axes <dM_i(lag) . dM_j(lag)> over all time origins, last row
        <|dM_tot(lag)|^2> (the row convention of ``correlate_charge_flux``).  By linearity row i is the cross MSD of the
        three channel pairs (M_i,c , M_tot,c): one mdp_cross_msd_fft call of 3 (ntypes+1) channels.  max_lag defaults to
        T // 2."""
        m = torch.as_tensor(np.ascontiguousarray(dipole, dtype=np.float64)).cuda()
        _, ntypes, T = m.shape
        max_lag = lag_count(max_lag, T)
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
        layout = MoleculeLayout(self.num_mols, self.num_atoms_per_mol, self.mass)
        ntypes = len(self.num_mols)
        dev = torch.device("cuda", torch.cuda.current_device())
        # every rank parses every frame; the molecules of each type are split in contiguous blocks over the ranks
        sel_d, nloc = rank_blocks(layout.type_members(), dev)
        coms, steps = [], []
        for _, ts, pos, md, _ in self._fixed_charge_frames(layout):
            com, _, _ = ops.segment_com(pos, md, layout.seg_d)                 # [F, 3, M]
            coms.append(com.index_select(2, sel_d))
            steps += ts
        self._set_even_time(steps)
        T = len(steps)
        max_lag = lag_count(max_lag, T)
        t, mask = self._fit_window(max_lag, initial_time, final_time)
        conv = constants.DISTANCE_CONVERSION[self.units]
        com = torch.cat(coms, dim=0) * conv                                     # [T, 3, Mloc] in m
        chans = com.permute(2, 1, 0).reshape(-1, T).contiguous()                # [Mloc * 3, T]
        goff = 3 * np.concatenate(([0], np.cumsum(nloc))).astype(np.int64)
        msd = all_reduce_groups(lambda c: ops.cross_msd_fft(c, None, goff, max_lag), chans, ntypes, max_lag)
        msd = msd.cpu().numpy() / np.asarray(self.num_mols, dtype=np.float64)[:, None]
        diff = np.array([self._slope(t[mask], row[mask]) for row in msd]) / 6
        qmol = np.add.reduceat(self._fixed[0], layout.seg_off[:-1]) * constants.CHARGE_CONVERSION[self.units]
        q2 = np.array([np.sum(qmol[a:b] ** 2) for a, b in zip(layout.type_off[:-1], layout.type_off[1:])])
        cond = diff * q2 / (self.volume * constants.BOLTZMANN * self.temp)
        cond = np.append(cond, cond.sum())
        if save and dist.rank() == 0:
            with open(f"{self.working_dir}/nernst_einstein.csv", "w") as f:
                f.write("type,diffusion (m2/s),cond\n")
                for g in range(ntypes):
                    f.write(f"{g + 1},{diff[g]!r},{cond[g]!r}\n")
                f.write(f"tot,,{cond[-1]!r}\n")
        return cond
