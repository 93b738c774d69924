"""Mean-square displacement and Einstein diffusion coefficients -- drop-in for
``mdproptools.dynamical.diffusion.Diffusion`` (reference mdproptools/dynamical/diffusion.py; citations are
lines of that file).

Device work (csrc/reduce.cu): molecule centres of mass of unwrapped coordinates (calc_com), the squared
displacements from the Time==0 frame and their per-group sums (:212-218) as a streaming fp64 reduction over
``[T][3][N]`` SoA frames, the strided-interval MSD (:225-237), the OLS sums of calc_diff (:323-329), and --
beyond the reference -- the windowed MSD over all time origins (``get_msd_all_origins``).
Green-Kubo route (``get_vacf``, ``calc_diff_green_kubo``, ``get_vdos``; no reference counterpart): the velocity
autocorrelation over all time origins per (type, axis) group through the grouped FFT autocorrelation mdp_group_acf_fft
(csrc/msdfft.cu) and its running integral (mdp_cumtrapz); the vibrational density of states is a DCT-I of each VACF.
Host work: unit tables, DataFrame shaping/column names (:211-222), artefact files.

Multi-GPU: atoms (or molecules) are split in contiguous blocks over the ranks; per-frame partial sums are
merged with one fp64 all-reduce (SURVEY 8e).  Every rank parses the dump files (parsing is replicated).
"""
from __future__ import annotations

import os

import numpy as np
import pandas as pd
import torch

from .. import dist, ops
from ..common import constants
from ..io.log import concat_log
from ..io.pipeline import ArrayBatches, FrameBatches
from .series import (DumpColumns, MoleculeLayout, all_reduce_groups, even_times, fit_window, lag_count, rank_blocks,
                     unwrapped_positions)
from .series import MissingCoordinatesError, position_columns  # noqa: F401  (public under this path)


VDOS_WINDOWS = ("hann", "none")


def vdos_transform(c, dt, window="hann"):
    """(nu [L], S [L]) of one autocorrelation c [L] (a float64 torch tensor on any device) with lag step dt, L >= 2:
    the DCT-I  X_k = w_0 c_0 + (-1)^k w_{L-1} c_{L-1} + 2 sum_{l=1}^{L-2} w_l c_l cos(pi k l / (L-1)),
    S(nu_k) = 2 dt X_k / c_0 at nu_k = k / (2 (L-1) dt), with w_l = 0.5 (1 + cos(pi l / (L-1))) ("hann") or 1 ("none").
    The DCT-I is the real part of the FFT of the even extension (c_0 .. c_{L-1} .. c_1).  The trapezoid area of S over nu
    is w_0 = 1, and S(0) c_0 / 4 is the trapezoid integral of w c."""
    if window not in VDOS_WINDOWS:
        raise ValueError(f"window must be one of {VDOS_WINDOWS}, got {window!r}")
    L = c.shape[0]
    lag = torch.arange(L, dtype=torch.float64, device=c.device)
    w = 0.5 * (1.0 + torch.cos(np.pi * lag / (L - 1))) if window == "hann" else torch.ones_like(lag)
    y = w * c
    ext = torch.cat([y, y[1:L - 1].flip(0)])                             # length 2 (L - 1)
    X = torch.fft.rfft(ext).real                                         # L values
    return lag / (2 * (L - 1) * dt), 2.0 * dt * X / c[0]


class Diffusion:
    """Same constructor and methods as the reference class (:32-60)."""

    def __init__(self, timestep=1, units="real", outputs_dir=None, diff_dir=None):
        self.units = units
        if self.units not in constants.SUPPORTED_UNITS:
            raise KeyError("Unit type not supported. Supported units are: " + str(constants.SUPPORTED_UNITS))
        self.outputs_dir = outputs_dir or os.getcwd()
        self.diff_dir = diff_dir or os.getcwd()
        self.timestep = timestep

    # ------------------------------------------------------------------------------------------
    def _load_unwrapped(self, filename, extra_cols=(), masses=False):
        """Read every frame; returns (times[T], metas, coords device [T,3,N], host columns of frame 0).  ``masses``: the
        dump's ``mass`` column is read too (``DumpColumns.select``).

        _prepare_unwrapped_coords (:62-81): when ``zu`` is absent, xu = x + ix * (xhi - xlo) etc."""
        pattern = f"{self.outputs_dir}/{filename}"
        plan = DumpColumns(pattern)
        assert "id" in plan.available, "Missing atom id's in dump file."
        want = plan.select(["id", *extra_cols], positions=True, masses=masses)
        k0 = 1 + len(extra_cols)
        chunks, metas, first_host = [], [], None
        for batch in FrameBatches(pattern, want):
            dev = batch.wait()
            if first_host is None:
                first_host = {c: batch.host[0, k].numpy().copy() for k, c in enumerate(want)}
            chunks.append(unwrapped_positions(dev, batch.metas, k0, want[k0] == "xu").contiguous())
            metas += batch.metas
        coords = torch.cat(chunks, dim=0) if len(chunks) > 1 else chunks[0]
        times = np.array([m.timestep * self.timestep * constants.TIME_CONVERSION[self.units] for m in metas])
        order = np.argsort(times, kind="stable")                          # set_index(...).sort_index() (:207)
        if not np.array_equal(order, np.arange(len(times))):
            coords = coords[torch.from_numpy(order).to(coords.device)].contiguous()
            times = times[order]
            metas = [metas[k] for k in order]
        return times, metas, coords, first_host

    @staticmethod
    def _time_zero_index(times):
        z = np.nonzero(times == 0)[0]
        if len(z) == 0:
            raise KeyError(0)      # msd_all.xs(0, 0) in the reference (:213)
        return int(z[0])

    def _com_series(self, filename, num_mols, num_atoms_per_mol, mass):
        """Unwrapped molecule centres of mass of every frame: (times[T], com device [T,3,M], mol_mass [M], layout)."""
        times, _, coords, h0 = self._load_unwrapped(filename, extra_cols=["type"], masses=not mass)
        layout = MoleculeLayout(num_mols, num_atoms_per_mol, mass)
        layout.check(coords.shape[2])                 # before segment_com, which reads seg_off unchecked
        com, mol_mass, _ = ops.segment_com(coords, layout.masses(h0["type"], h0.get("mass"), coords.device), layout.seg_d)
        return times, com, mol_mass, layout

    def get_msd_from_dump(self, filename, msd_type="com", num_mols=None, num_atoms_per_mol=None, mass=None, com_drift=False,
                          avg_interval=False, tao_coeff=4):
        """See the reference docstring (:112-171).  Returns (msd, msd_all[, msd_int]) DataFrames."""
        if msd_type not in ("allatom", "com"):
            raise ValueError("msd_type must be 'allatom' or 'com'.")
        conv = constants.DISTANCE_CONVERSION[self.units]
        disps = ["dx2", "dy2", "dz2"]
        if msd_type == "allatom":
            times, metas, coords, h0 = self._load_unwrapped(filename)
            ids = h0["id"].astype(np.int64)
            T, _, N = coords.shape
            t0 = self._time_zero_index(times)
            # atoms split over ranks; per-frame sums all-reduced (fp64)
            lo, hi = dist.shard_range(N)
            w = dist.world_size()
            if w > 1:
                local = coords[:, :, lo:hi].contiguous()
                sums, per_atom = ops.msd_single_origin(local, local[t0].contiguous(), conv, per_atom=True)
                dist.all_reduce_sum_(sums)
                full = torch.zeros((T, 4, N), dtype=torch.float64, device=coords.device)
                full[:, :, lo:hi] = per_atom
                dist.all_reduce_sum_(full)
                per_atom = full
            else:
                sums, per_atom = ops.msd_single_origin(coords, coords[t0].contiguous(), conv, per_atom=True)
            mean = (sums[:, 0, :] / N).cpu().numpy()                      # groupby(Time).mean() (:218)
            msd = pd.DataFrame(mean, columns=disps + ["msd"])
            msd.insert(0, "Time (s)", times)
            pa = per_atom.permute(0, 2, 1).reshape(T * N, 4).cpu().numpy()
            msd_all = pd.DataFrame(pa, columns=disps + ["msd"])
            msd_all.insert(0, "id", np.tile(ids, T))
            msd_all.insert(0, "Time (s)", np.repeat(times, N))
            if avg_interval:
                sel = coords[::tao_coeff].contiguous()                   # times[::tao_coeff] (:226-228)
                mi = ops.msd_interval(sel, conv, 1).cpu().numpy()
                msd_int = pd.DataFrame(mi.T, columns=disps + ["msd"])
                msd_int.insert(0, "id", ids)
                return msd, msd_all, msd_int
            return msd, msd_all

        # ---- centre-of-mass MSD per molecule type -------------------------------------------------
        times, com, mol_mass, layout = self._com_series(filename, num_mols, num_atoms_per_mol, mass)   # com [T,3,M]
        T, _, M = com.shape
        dev = com.device
        com = com * conv                                                  # SI before anything else (:201-203)
        mol_mass = mol_mass * constants.MASS_CONVERSION[self.units]       # (:193)
        ntypes = len(num_mols)
        t0 = self._time_zero_index(times)
        if com_drift:
            # _modify_dump_coordinates (:91-96): subtract the drift of each type's centre of mass
            tcom, _, _ = ops.segment_com(com, mol_mass, torch.from_numpy(layout.type_off.astype(np.int32)).to(dev))  # [T,3,G]
            drift = tcom - tcom[t0:t0 + 1]
            tidx = torch.from_numpy(np.repeat(np.arange(ntypes), num_mols)).to(dev)
            com = (com - drift.index_select(2, tidx)).contiguous()
        sums, per_mol = ops.msd_single_origin(com, com[t0].contiguous(), 1.0, group_off=layout.type_off, per_atom=True)
        counts = torch.tensor(np.asarray(num_mols, dtype=np.float64), device=dev)
        mean = (sums / counts[None, :, None]).cpu().numpy()              # [T, ntypes, 4]
        cols, data = [], []
        for ti in range(ntypes):                                           # pivot + sort by type (:219-222)
            for k, name in enumerate(disps + ["msd"]):
                cols.append(f"{name}{ti + 1}")
                data.append(mean[:, ti, k])
        msd = pd.DataFrame(np.stack(data, axis=1), columns=cols)
        msd.insert(0, "Time (s)", times)
        pm = per_mol.permute(0, 2, 1).reshape(T * M, 4).cpu().numpy()
        msd_all = pd.DataFrame(pm, columns=disps + ["msd"])
        msd_all.insert(0, "mol_id", np.tile(layout.mol_id, T))
        msd_all.insert(0, "type", np.tile(layout.mol_type, T))
        msd_all.insert(0, "Time (s)", np.repeat(times, M))
        if avg_interval:
            mi = ops.msd_interval(com[::tao_coeff].contiguous(), 1.0, 1).cpu().numpy()
            msd_int = pd.DataFrame(mi.T, columns=disps + ["msd"])
            msd_int.insert(0, "mol_id", layout.mol_id)
            msd_int.insert(0, "type", layout.mol_type)
            return msd, msd_all, msd_int
        return msd, msd_all

    # ------------------------------------------------------------------------------------------
    def get_msd_from_arrays(self, positions, timesteps, batch_frames=64):
        """Array front end of the all-atom MSD for trajectories already in memory (the single-origin arithmetic
        of :207-218 without building the T*N-row ``msd_all`` frame, which cannot exist at 10^10 atom-frames).

        positions float64 [T, 3, N] host array (numpy or pinned torch tensor) of UNWRAPPED coordinates in id order,
        timesteps [T] LAMMPS step numbers (the frame with step 0 is the origin, :213).  Frames stream through the
        device in batches (copy of batch k+1 overlaps the reduction of batch k).  Returns the ``msd`` DataFrame.
        """
        pos = positions if isinstance(positions, torch.Tensor) else torch.from_numpy(
            np.ascontiguousarray(positions, dtype=np.float64))
        T, _, N = pos.shape
        conv = constants.DISTANCE_CONVERSION[self.units]
        times = np.asarray(timesteps) * self.timestep * constants.TIME_CONVERSION[self.units]
        t0 = self._time_zero_index(times)
        dev = torch.device("cuda", torch.cuda.current_device())
        ref = pos[t0].to(dev)
        sums = torch.empty((T, 1, 4), dtype=torch.float64, device=dev)
        for f0, f1, x in ArrayBatches(pos, batch_frames, dev):   # copy of batch k+1 overlaps the reduction of batch k
            s, _ = ops.msd_single_origin(x, ref, conv)
            sums[f0:f1] = s
        mean = (sums[:, 0, :] / N).cpu().numpy()
        msd = pd.DataFrame(mean, columns=["dx2", "dy2", "dz2", "msd"])
        msd.insert(0, "Time (s)", times)
        return msd

    def get_msd_all_origins(self, filename, max_lag=None, msd_type="allatom", num_mols=None, num_atoms_per_mol=None,
                            mass=None):
        """North-star extension (no reference counterpart): MSD averaged over ALL time origins,
        msd(lag) = < |r_i(t0 + lag) - r_i(t0)|^2 >_{i, t0}, for lag < max_lag.  Returns a DataFrame with the lag
        time and dx2/dy2/dz2/msd (per molecule type for ``com``)."""
        conv = constants.DISTANCE_CONVERSION[self.units]
        if msd_type == "allatom":
            times, metas, coords, h0 = self._load_unwrapped(filename)
            group_off, counts, labels = None, np.array([coords.shape[2]], dtype=np.float64), [""]
        else:
            times, coords, _, layout = self._com_series(filename, num_mols, num_atoms_per_mol, mass)
            group_off, counts = layout.type_off, np.asarray(num_mols, dtype=np.float64)
            labels = [str(k + 1) for k in range(len(num_mols))]
        T, _, N = coords.shape
        max_lag = T if max_lag is None else min(int(max_lag), T)
        lo, hi = dist.shard_range(N) if group_off is None else (0, N)
        local = coords[:, :, lo:hi].contiguous() if (lo, hi) != (0, N) else coords
        sums = ops.msd_all_origins(local, max_lag, conv, group_off=group_off)
        if group_off is None:
            dist.all_reduce_sum_(sums)
        norig = torch.arange(T, T - max_lag, -1, dtype=torch.float64, device=sums.device)
        mean = (sums / (norig[:, None, None] * torch.tensor(counts, device=sums.device)[None, :, None])).cpu().numpy()
        out = pd.DataFrame({"Time (s)": times[:max_lag] - times[0]})
        for g, lab in enumerate(labels):
            for k, name in enumerate(["dx2", "dy2", "dz2", "msd"]):
                out[f"{name}{lab}"] = mean[:, g, k]
        return out

    # ------------------------------------------------------------------------------------------
    def calc_diff(self, msd, initial_time=None, final_time=None, dimension=3, diff_names=None, save=False, plot=False):
        """Einstein relation: least-squares slope THROUGH THE ORIGIN of every ``msd*`` column against time
        (``sm.OLS(y, t).fit()``, :323), D = slope / (2 dim), std = bse / (2 dim), uncentred R^2 (:325-329).
        The three sums are reduced on the device (mdp_ols_sums); slope/bse/R^2 follow in closed form."""
        if initial_time is None:
            initial_time = {}
        if final_time is None:
            final_time = {}
        min_t = min(msd["Time (s)"])
        max_t = max(msd["Time (s)"])
        msd_col_names = [col for col in msd.columns if "msd" in col.lower()]
        diff = np.zeros((len(msd_col_names), 3))
        tvals = msd["Time (s)"].to_numpy(dtype=np.float64)
        summaries = []
        for ind, col in enumerate(msd_col_names):
            mask = (tvals >= initial_time.get(ind, min_t)) & (tvals <= final_time.get(ind, max_t))
            t = torch.from_numpy(np.ascontiguousarray(tvals[mask])).cuda()
            y = torch.from_numpy(np.ascontiguousarray(msd[col].to_numpy(dtype=np.float64)[mask])).cuda()
            stt, sty, syy = ops.ols_sums(t, y.reshape(1, -1))[0].cpu().tolist()
            n = int(mask.sum())
            slope = sty / stt
            ssr = syy - 2.0 * slope * sty + slope * slope * stt
            ssr = max(ssr, 0.0)
            bse = float(np.sqrt(ssr / (n - 1) / stt))
            r2 = 1.0 - ssr / syy
            diff[ind] = [slope / (2 * dimension), bse / (2 * dimension), r2]
            summaries.append((col, n, slope, bse, r2))
            if save:
                name = diff_names[ind] if diff_names else ind + 1
                with open(f"{self.diff_dir}/diff_{name}.txt", "w") as f:
                    f.write("OLS regression through the origin (no intercept)\n")
                    f.write(f"dep. variable: {col}\nobservations: {n}\nslope: {slope!r}\nstd err: {bse!r}\n"
                            f"R-squared (uncentered): {r2!r}\n")
        ind_names = diff_names or [i + 1 for i in range(len(msd_col_names))]
        diffusion = pd.DataFrame(diff, columns=["diffusion (m2/s)", "std", "R2"], index=ind_names)
        if plot:
            self._plot(msd, msd_col_names, summaries, ind_names)
        diffusion.to_csv(f"{self.diff_dir}/diffusion.csv")
        return diffusion

    def _plot(self, msd, cols, summaries, names):
        try:
            import matplotlib
            matplotlib.use("Agg")
            import matplotlib.pyplot as plt
        except ImportError as exc:  # plotting is outside the hot path; matplotlib is optional
            raise ImportError("plot=True needs matplotlib") from exc
        t = msd["Time (s)"] * 10 ** 9
        for fname, logscale in (("msd.png", False), ("msd_log.png", True)):
            ncols = 2
            nrows = int(np.ceil(len(cols) / ncols))
            fig, axes = plt.subplots(nrows, ncols, figsize=(12, 8), squeeze=False)
            for ax, col, (_, _, slope, _, _), name in zip(axes.flatten(), cols, summaries, names):
                ax.plot(t, msd[col], linewidth=2, label=name)
                ax.plot(t, slope * msd["Time (s)"], color="k", ls="--", linewidth=2)
                if logscale:
                    ax.set(xscale="log", yscale="log")
                ax.legend(frameon=False)
                ax.set_xlabel("Time, 10^9 (s)")
                ax.set_ylabel("MSD (m^2)")
            fig.tight_layout()
            fig.savefig(f"{self.diff_dir}/{fname}", bbox_inches="tight", pad_inches=0.1)
            plt.close(fig)

    def get_msd_from_log(self, log_pattern):
        """MSD columns of LAMMPS thermo logs converted to SI (:241-265)."""
        full_log = concat_log(log_pattern, step=None, working_dir=self.outputs_dir)
        msd = full_log.filter(regex="msd").copy()
        for col in msd:
            msd.loc[:, col] = msd[col] * constants.DISTANCE_CONVERSION[self.units] ** 2
        msd["Time (s)"] = full_log["Step"] * self.timestep * constants.TIME_CONVERSION[self.units]
        return msd

    def get_diff_dist(self, msd_int, dump_freq, dimension=3, tao_coeff=4, plot=False, diff_names=None):
        """Distribution of per-atom / per-molecule diffusion coefficients from the interval-averaged MSD ``msd_int`` of
        ``get_msd_from_dump(avg_interval=True)`` (:410-516): adds the column
        ``diff = msd / (2 * dimension * tao_coeff * dump_freq * timestep * TIME_CONVERSION)`` in place and returns the frame.
        With ``plot`` the histograms (one panel per molecule type when a ``type`` column is present) go to
        ``<diff_dir>/diff_dist.png``; matplotlib is imported only then."""
        delta = dump_freq * self.timestep * constants.TIME_CONVERSION[self.units]
        msd_int["diff"] = msd_int["msd"] / (2 * dimension * tao_coeff * delta)
        if plot:
            try:
                import matplotlib
                matplotlib.use("Agg")
                import matplotlib.pyplot as plt
            except ImportError as exc:
                raise ImportError("plot=True needs matplotlib") from exc
            if "type" in msd_int.columns:
                groups = msd_int.groupby("type")
                ind = diff_names or [i + 1 for i in range(len(groups))]
                ncols = 2
                nrows = int(np.ceil(groups.ngroups / ncols))
                fig, axes = plt.subplots(nrows, ncols, figsize=(12, 8), squeeze=False)
                for ax, (key, grp) in zip(axes.flatten(), groups):
                    ax.hist(grp["diff"] * 10 ** 9, bins=max(1, int(np.sqrt(len(grp)))), density=True, edgecolor="k",
                            label=str(ind[key - 1]))
                    ax.legend(frameon=False)
                    ax.set_xlabel("Diffusivity, 10^-9 (m^2/s)")
                    ax.set_ylabel("Frequency")
                if len(groups) % 2 != 0:
                    fig.delaxes(ax=axes.flatten()[-1])
            else:
                fig, ax = plt.subplots(figsize=(8, 6))
                ax.hist(msd_int["diff"] * 10 ** 9, bins=max(1, int(np.sqrt(len(msd_int)))), density=True, edgecolor="k")
                ax.set_xlabel("Diffusivity, 10^-9 (m^2/s)")
                ax.set_ylabel("Frequency")
            fig.tight_layout()
            fig.savefig(f"{self.diff_dir}/diff_dist.png", bbox_inches="tight", pad_inches=0.1)
            plt.close(fig)
        return msd_int

    # ------------------------------------------------------------------------------------------
    def get_vacf(self, filename, max_lag=None, vacf_type="allatom", num_mols=None, num_atoms_per_mol=None, mass=None):
        """Velocity autocorrelation over all time origins, C(lag) = < v_i(t0 + lag) . v_i(t0) >_{i, t0}, in m^2/s^2 for
        lags 0 .. max_lag - 1 (default T // 2) of evenly spaced frames with ``vx vy vz`` columns.

        ``allatom``: one group per atom type (ascending type id; the types must not change between frames), columns
        ``vxvx{t} vyvy{t} vzvz{t} vacf{t}`` (means over the type's atoms) and ``vacf``, the mean over all atoms.
        ``com``: mass-weighted centre-of-mass velocities of the molecules (``num_mols``, ``num_atoms_per_mol``; masses from
        ``mass`` by type, else the dump's ``mass`` column), one group per molecule type labelled 1..ntypes.
        The first column is ``Time (s)``, the lag times from 0.  Velocities are not centred: a drift is part of C.
        All (type, axis) groups go through one mdp_group_acf_fft call.  Multi-GPU: every rank parses every frame and
        keeps a contiguous block of each group's atoms (or molecules); the sums are merged with one fp64 all-reduce."""
        if vacf_type not in ("allatom", "com"):
            raise ValueError("vacf_type must be 'allatom' or 'com'.")
        if max_lag is not None and int(max_lag) < 1:
            raise ValueError(f"max_lag must be at least 1, got {max_lag}")
        pattern = f"{self.outputs_dir}/{filename}"
        plan = DumpColumns(pattern)
        if not {"vx", "vy", "vz"} <= set(plan.available):
            raise ValueError(f"the velocity autocorrelation needs the dump columns vx vy vz "
                             f"({pattern!r} has {sorted(plan.available)})")
        com = vacf_type == "com"
        want = plan.select(["id", "type", "vx", "vy", "vz"], masses=com and not mass)
        dev = torch.device("cuda", torch.cuda.current_device())
        vs = constants.VELOCITY_CONVERSION[self.units]
        types0 = sel_d = md = layout = None
        pieces, steps = [], []
        for batch in FrameBatches(pattern, want):
            d = batch.wait()
            host = batch.host.numpy()
            if types0 is None:
                types0 = host[0, 1].copy()
                if com:
                    layout = MoleculeLayout(num_mols, num_atoms_per_mol, mass)
                    layout.check(len(types0))
                    md = layout.masses(types0, None if mass else host[0, batch.col("mass")], dev)
                    labels = [str(k + 1) for k in range(len(num_mols))]
                    members = layout.type_members()
                else:
                    tids = np.unique(types0)
                    labels = [str(int(t)) for t in tids]
                    members = [np.nonzero(types0 == t)[0] for t in tids]
                sel_d, nloc = rank_blocks(members, dev)
                counts = np.array([len(idx) for idx in members], dtype=np.float64)
            if not (host[:, 1] == types0).all():
                raise ValueError("atom types must be the same in every frame for the velocity autocorrelation")
            vel = d[:, 2:5, :]
            if com:
                vel, _, _ = ops.segment_com(vel.contiguous(), md, layout.seg_d)       # [F, 3, M]
            pieces.append(vel.index_select(2, sel_d) * vs)                               # [F, 3, local]
            steps += [m.timestep for m in batch.metas]
        times = even_times(steps, self.units, self.timestep, repr(pattern), who="the velocity autocorrelation needs")
        T = len(steps)
        max_lag = lag_count(max_lag, T)
        v = torch.cat(pieces, dim=0) if len(pieces) > 1 else pieces[0]                   # [T, 3, local]
        del pieces
        # channels [group][axis][atom] (groups are (type, axis)), one row per series
        G = len(nloc)
        goff = np.concatenate(([0], np.cumsum(np.repeat(nloc, 3)))).astype(np.int64)
        chans = torch.empty((int(goff[-1]), T), dtype=torch.float64, device=dev)
        s0 = 0
        for g in range(G):
            chans[3 * s0:3 * (s0 + nloc[g])].view(3, nloc[g], T).copy_(v[:, :, s0:s0 + nloc[g]].permute(1, 2, 0))
            s0 += nloc[g]
        del v
        sums = all_reduce_groups(lambda c: ops.group_acf_fft(c, goff, max_lag), chans, 3 * G, max_lag)   # [3 G, max_lag]
        del chans
        sums = sums.cpu().numpy().reshape(G, 3, max_lag)
        out = {"Time (s)": times[:max_lag] - times[0]}
        for g, lab in enumerate(labels):
            for k, name in enumerate(["vxvx", "vyvy", "vzvz"]):
                out[f"{name}{lab}"] = sums[g, k] / counts[g]
            out[f"vacf{lab}"] = sums[g].sum(axis=0) / counts[g]
        if not com:
            out["vacf"] = sums.sum(axis=(0, 1)) / counts.sum()
        return pd.DataFrame(out)

    def calc_diff_green_kubo(self, vacf, initial_time=None, final_time=None, dimension=3, diff_names=None, save=False):
        """Green-Kubo self-diffusion D = (1/dimension) integral of the VACF, for every ``vacf*`` column of ``get_vacf``.
        The running integral (trapezoid, leading zero) is formed on the device; D is its mean over the fit window divided
        by ``dimension`` and ``std`` its standard deviation (ddof 0) over the window divided by ``dimension``.  The window of
        column ``ind`` runs from ``initial_time[ind]`` to ``final_time[ind]`` (dicts keyed by column index, as in
        ``calc_diff``), by default over the lags max(1, L // 10) to L - 1.  ``save`` writes vacf_integral.csv and
        diffusion_gk.csv into ``diff_dir``."""
        initial_time = initial_time or {}
        final_time = final_time or {}
        names = [col for col in vacf.columns if "vacf" in col.lower()]
        t = vacf["Time (s)"].to_numpy(dtype=np.float64)
        if len(t) < 2:
            raise ValueError(f"the Green-Kubo integral needs at least 2 lag times, got {len(t)}")
        y = torch.from_numpy(np.array(vacf[names].to_numpy(dtype=np.float64).T, order="C")).cuda()
        integral = ops.cumtrapz(y, float(t[1] - t[0]), 1.0, leading_zero=True).cpu().numpy()     # [columns, L]
        diff = np.zeros((len(names), 2))
        for ind, row in enumerate(integral):
            win = row[fit_window(t, initial_time.get(ind), final_time.get(ind))]
            diff[ind] = [win.mean() / dimension, win.std() / dimension]
        diffusion = pd.DataFrame(diff, columns=["diffusion (m2/s)", "std"],
                                 index=diff_names or [i + 1 for i in range(len(names))])
        if save and dist.rank() == 0:
            run = pd.DataFrame(integral.T, columns=names)
            run.insert(0, "Time (s)", t)
            run.to_csv(f"{self.diff_dir}/vacf_integral.csv", index=False)
            diffusion.to_csv(f"{self.diff_dir}/diffusion_gk.csv")
        return diffusion

    def get_vdos(self, vacf, window="hann", save=False):
        """Vibrational density of states of every ``vacf*`` column of ``get_vacf``: ``vdos*`` = S(nu) of
        ``vdos_transform`` (normalised to unit area over nu), with ``Frequency (Hz)`` and ``Wavenumber (cm^-1)`` columns.
        ValueError for fewer than 2 lags or a column with C(0) = 0.  ``save`` writes vdos.csv into ``diff_dir``."""
        names = [col for col in vacf.columns if "vacf" in col.lower()]
        t = vacf["Time (s)"].to_numpy(dtype=np.float64)
        dt = float(t[1] - t[0]) if len(t) > 1 else 0.0
        dev = torch.device("cuda", torch.cuda.current_device())
        out = {}
        for col in names:
            c = vacf[col].to_numpy(dtype=np.float64)
            if len(c) < 2 or c[0] == 0:
                raise ValueError(f"the VDOS of {col!r} needs at least 2 lags and a nonzero C(0) "
                                 f"({len(c)} lags, C(0) = {c[0] if len(c) else None})")
            nu, S = vdos_transform(torch.from_numpy(np.ascontiguousarray(c)).to(dev), dt, window)
            if not out:
                nu = nu.cpu().numpy()
                out["Frequency (Hz)"] = nu
                out["Wavenumber (cm^-1)"] = nu / constants.LIGHT_SPEED / 100
            out["vdos" + col[len("vacf"):]] = S.cpu().numpy()
        vdos = pd.DataFrame(out)
        if save and dist.rank() == 0:
            vdos.to_csv(f"{self.diff_dir}/vdos.csv", index=False)
        return vdos
