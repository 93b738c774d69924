"""Tensor-level wrappers over the C ABI (one function per entry point of include/mdprop_b200.h).

Inputs are CUDA torch tensors (torch is only the device-memory / stream plumbing); every function enqueues
work on the current torch stream.  Nothing here has a CPU path.
"""
from __future__ import annotations

import ctypes
from ctypes import c_double, c_int, c_int32, c_int64

import numpy as np
import torch

from . import _lib
from ._lib import Context, check, lib, ptr, stream_ptr


def _f64(t: torch.Tensor, name: str) -> torch.Tensor:
    if not (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()):
        raise ValueError(f"{name} must be a contiguous float64 CUDA tensor")
    return t


def _i32(t, name: str):
    if t is None:
        return None
    if not (t.is_cuda and t.dtype == torch.int32 and t.is_contiguous()):
        raise ValueError(f"{name} must be a contiguous int32 CUDA tensor")
    return t


def _host_i64(a):
    if a is None:
        return None, None
    arr = np.ascontiguousarray(a, dtype=np.int64)
    return arr, arr.ctypes.data_as(ctypes.POINTER(c_int64))


def sym_rows(ncls: int) -> int:
    return ncls * (ncls + 1) // 2


def sym_row(ci: int, cj: int, ncls: int) -> int:
    a, b = (ci, cj) if ci <= cj else (cj, ci)
    return a * ncls - a * (a - 1) // 2 + (b - a)


def _host_box(box, F, flags):
    """[F,3] box lengths, or [F,6] = (lx, ly, lz, xy, xz, yz) when the triclinic image is requested."""
    box = np.asarray(box, dtype=np.float64)
    w = 6 if flags & _lib.PAIR_TRICLINIC else 3
    if box.size != F * w:
        raise ValueError(f"box must hold {w} values per frame ({F} frames), got shape {box.shape}")
    return np.ascontiguousarray(box.reshape(F, w))


def pair_hist(xyz_a, cls_a, ncls_a, box, rcut2, edges, uniform_ddr, xyz_b=None, cls_b=None, ncls_b=1, out=None,
              flags=0):
    """mdp_pair_hist.  xyz_* float64 [F,3,N]; cls_* int32 [N] or [F,N] or None; box array-like [F,3] (host), or
    [F,6] = (lx, ly, lz, xy, xz, yz) with ``flags & PAIR_TRICLINIC``.

    Returns uint64 counts as an int64 tensor [F, rows, nbins] (accumulated into ``out`` when given).
    """
    xyz_a = _f64(xyz_a, "xyz_a")
    F, _, na = xyz_a.shape
    ctx = Context.get(xyz_a.device.index)
    box = _host_box(box, F, flags)
    edges = np.ascontiguousarray(edges, dtype=np.float64)
    nbins = edges.shape[0] - 1
    symm = xyz_b is None
    rows = sym_rows(ncls_a) if symm else ncls_a * ncls_b
    if out is None:
        out = torch.zeros((F, rows, nbins), dtype=torch.int64, device=xyz_a.device)
    cls_a = _i32(cls_a, "cls_a")
    sa = 0 if cls_a is None or cls_a.dim() == 1 else na
    nb_ = 0
    sb = 0
    if not symm:
        xyz_b = _f64(xyz_b, "xyz_b")
        nb_ = xyz_b.shape[2]
        cls_b = _i32(cls_b, "cls_b")
        sb = 0 if cls_b is None or cls_b.dim() == 1 else nb_
    check(lib().mdp_pair_hist(ctx.handle, F, na, ptr(xyz_a), ptr(cls_a), sa, int(ncls_a),
                              nb_, ptr(xyz_b), ptr(cls_b), sb, int(ncls_b),
                              _lib.dptr(box), float(rcut2), _lib.dptr(edges), int(nbins), float(uniform_ddr),
                              ptr(out), int(flags), stream_ptr()), "mdp_pair_hist")
    return out


def hist_reduce(hist, weights, cumulative=False):
    """mdp_hist_reduce: hist int64 [F, rows, nbins], weights int array [nout, rows] -> int64 [F, nout, nbins]."""
    F, rows, nbins = hist.shape
    w = np.ascontiguousarray(weights, dtype=np.int32).reshape(-1, rows)
    nout = w.shape[0]
    ctx = Context.get(hist.device.index)
    out = torch.empty((F, nout, nbins), dtype=torch.int64, device=hist.device)
    check(lib().mdp_hist_reduce(ctx.handle, F, rows, nbins, ptr(hist), nout, w.ctypes.data_as(ctypes.POINTER(c_int32)),
                                1 if cumulative else 0, ptr(out), stream_ptr()), "mdp_hist_reduce")
    return out


def pair_list(xyz_a, xyz_b, box, r_in2, r_out2, shell_mode, exclude_same_index=False, capacity=None, want_rsq=False,
              flags=0):
    """mdp_pair_list -> (list int32 [M,3] = (frame, ia, ib), rsq float64 [M] or None); grows capacity as needed."""
    xyz_a = _f64(xyz_a, "xyz_a")
    xyz_b = _f64(xyz_b, "xyz_b")
    F, _, na = xyz_a.shape
    nb_ = xyz_b.shape[2]
    ctx = Context.get(xyz_a.device.index)
    box = _host_box(box, F, flags)
    cap = int(capacity or max(1 << 16, 64 * na * F))
    if shell_grid_enabled() and not want_rsq and flags == 0 and na <= 4096 and 8 * na <= nb_:
        # small set A against a large set B through a cell grid over A (csrc/shell.cu); answers 1 when it does not apply
        while True:
            lst = torch.empty((cap, 3), dtype=torch.int32, device=xyz_a.device)
            cnt = torch.zeros((1,), dtype=torch.int64, device=xyz_a.device)
            rc = lib().mdp_shell_search(ctx.handle, F, na, ptr(xyz_a), nb_, ptr(xyz_b), _lib.dptr(box), float(r_in2), float(r_out2),
                                        int(shell_mode), 1 if exclude_same_index else 0, ptr(lst), cap, ptr(cnt), stream_ptr())
            if rc == 1:
                break                      # the grid does not apply (radius above a third of the box): general engine below
            check(rc, "mdp_shell_search")
            m = int(cnt.item())
            if m <= cap:
                return lst[:m], None
            cap = int(m * 1.1) + 1024
    while True:
        lst = torch.empty((cap, 3), dtype=torch.int32, device=xyz_a.device)
        rsq = torch.empty((cap,), dtype=torch.float64, device=xyz_a.device) if want_rsq else None
        cnt = torch.zeros((1,), dtype=torch.int64, device=xyz_a.device)
        check(lib().mdp_pair_list(ctx.handle, F, na, ptr(xyz_a), nb_, ptr(xyz_b), _lib.dptr(box), float(r_in2),
                                  float(r_out2), int(shell_mode), 1 if exclude_same_index else 0, ptr(lst), ptr(rsq),
                                  cap, ptr(cnt), int(flags), stream_ptr()), "mdp_pair_list")
        m = int(cnt.item())
        if m <= cap:
            return lst[:m], (rsq[:m] if want_rsq else None)
        cap = int(m * 1.1) + 1024


def list_group(lst, n_a, nframes, key=None):
    """mdp_list_group: neighbour list int32 [M,3] -> (seg_off int64 [nframes*n_a+1], key_out int32-as-uint32 [M], perm int64 [M]):
    entries grouped by (frame, ia) and sorted by key (default ib) inside a group."""
    lst = _i32(lst.contiguous(), "lst")
    M = lst.shape[0]
    ctx = Context.get(lst.device.index)
    seg_off = torch.empty((nframes * n_a + 1,), dtype=torch.int64, device=lst.device)
    okey = torch.empty((max(M, 1),), dtype=torch.int32, device=lst.device)
    perm = torch.empty((max(M, 1),), dtype=torch.int64, device=lst.device)
    check(lib().mdp_list_group(ctx.handle, int(nframes), int(n_a), int(M), ptr(lst), ptr(key), ptr(seg_off), ptr(okey), ptr(perm),
                               stream_ptr()), "mdp_list_group")
    return seg_off, okey[:M], perm[:M]


def hydration_count(lst, xyz_cat, xyz_o, xyz_h1, xyz_h2, box, threshold=-0.72):
    """mdp_hydration_count: -> (cos float64 [M] in (frame, cation, water) order, seg_off int64 [F*ncat+1],
    counts int32 [F, ncat, 2] = (waters in range, waters with cos < threshold))."""
    xyz_cat, xyz_o, xyz_h1, xyz_h2 = (_f64(t, "xyz") for t in (xyz_cat, xyz_o, xyz_h1, xyz_h2))
    lst = _i32(lst.contiguous(), "lst")
    F, _, ncat = xyz_cat.shape
    nw = xyz_o.shape[2]
    M = lst.shape[0]
    ctx = Context.get(lst.device.index)
    box = np.ascontiguousarray(np.asarray(box, dtype=np.float64).reshape(F, 3))
    cos = torch.empty((max(M, 1),), dtype=torch.float64, device=lst.device)
    seg_off = torch.empty((F * ncat + 1,), dtype=torch.int64, device=lst.device)
    counts = torch.empty((F, ncat, 2), dtype=torch.int32, device=lst.device)
    check(lib().mdp_hydration_count(ctx.handle, F, ncat, ptr(xyz_cat), nw, ptr(xyz_o), ptr(xyz_h1), ptr(xyz_h2), _lib.dptr(box), M,
                                    ptr(lst), float(threshold), ptr(cos), ptr(seg_off), ptr(counts), stream_ptr()),
          "mdp_hydration_count")
    return cos[:M], seg_off, counts


def cluster_members(lst, n_central, force, mol_seg_off, mol_of_atom, force_constant, max_force):
    """mdp_cluster_members: -> (seg_off int64 [F*n_central+1], mols int32 [M], mol_count int32 [F*n_central]); the kept
    molecules of segment s are mols[seg_off[s] : seg_off[s] + mol_count[s]] (sorted, unique)."""
    force = _f64(force, "force")
    lst = _i32(lst.contiguous(), "lst")
    F, _, n = force.shape
    M = lst.shape[0]
    nmol = mol_seg_off.shape[0] - 1
    ctx = Context.get(lst.device.index)
    seg_off = torch.empty((F * n_central + 1,), dtype=torch.int64, device=lst.device)
    mols = torch.empty((max(M, 1),), dtype=torch.int32, device=lst.device)
    cnt = torch.empty((F * n_central,), dtype=torch.int32, device=lst.device)
    check(lib().mdp_cluster_members(ctx.handle, F, int(n_central), n, ptr(force), nmol, ptr(_i32(mol_seg_off, "mol_seg_off")),
                                    ptr(_i32(mol_of_atom, "mol_of_atom")), float(force_constant), float(max_force), M, ptr(lst),
                                    ptr(seg_off), ptr(mols), ptr(cnt), stream_ptr()), "mdp_cluster_members")
    return seg_off, mols[:M], cnt


def segment_com(attr, w, seg_off, extra=None):
    """mdp_segment_com: attr [F,C,N], w [N], seg_off int32 [S+1] -> (out [F,C,S], wsum [S], extra_sum [S] or None)."""
    attr = _f64(attr, "attr")
    w = _f64(w, "w")
    seg_off = _i32(seg_off, "seg_off")
    F, C, n = attr.shape
    S = seg_off.shape[0] - 1
    ctx = Context.get(attr.device.index)
    out = torch.empty((F, C, S), dtype=torch.float64, device=attr.device)
    wsum = torch.empty((S,), dtype=torch.float64, device=attr.device)
    esum = torch.empty((S,), dtype=torch.float64, device=attr.device) if extra is not None else None
    if extra is not None:
        extra = _f64(extra, "extra")
    check(lib().mdp_segment_com(ctx.handle, F, C, n, ptr(attr), ptr(w), S, ptr(seg_off), ptr(out), ptr(wsum), ptr(extra),
                                ptr(esum), stream_ptr()), "mdp_segment_com")
    return out, wsum, esum


def msd_single_origin(traj, ref, scale=1.0, group_off=None, per_atom=False):
    """mdp_msd_single_origin: traj [F,3,N], ref [3,N] -> (sums [F,G,4], per_atom [F,4,N] or None)."""
    traj = _f64(traj, "traj")
    ref = _f64(ref, "ref")
    F, _, n = traj.shape
    ctx = Context.get(traj.device.index)
    garr, gptr = _host_i64(group_off)
    G = 1 if garr is None else len(garr) - 1
    sums = torch.empty((F, G, 4), dtype=torch.float64, device=traj.device)
    pa = torch.empty((F, 4, n), dtype=torch.float64, device=traj.device) if per_atom else None
    done = 0
    while done < F:   # the ABI takes at most 65535 frames per call
        k = min(F - done, 32768)
        check(lib().mdp_msd_single_origin(ctx.handle, k, n, ptr(traj[done:]), ptr(ref), float(scale), gptr, G,
                                          ptr(sums[done:]), ptr(pa[done:]) if per_atom else None, stream_ptr()),
              "mdp_msd_single_origin")
        done += k
    return sums, pa


def msd_interval(traj, scale, stride):
    traj = _f64(traj, "traj")
    F, _, n = traj.shape
    ctx = Context.get(traj.device.index)
    out = torch.empty((4, n), dtype=torch.float64, device=traj.device)
    check(lib().mdp_msd_interval(ctx.handle, F, n, ptr(traj), float(scale), int(stride), ptr(out), stream_ptr()),
          "mdp_msd_interval")
    return out


def msd_all_origins(traj, max_lag, scale=1.0, group_off=None, out=None):
    traj = _f64(traj, "traj")
    F, _, n = traj.shape
    ctx = Context.get(traj.device.index)
    garr, gptr = _host_i64(group_off)
    G = 1 if garr is None else len(garr) - 1
    if out is None:
        out = torch.zeros((max_lag, G, 4), dtype=torch.float64, device=traj.device)
    check(lib().mdp_msd_all_origins(ctx.handle, F, n, ptr(traj), float(scale), gptr, G, int(max_lag), ptr(out),
                                    stream_ptr()), "mdp_msd_all_origins")
    return out


def charge_flux(vel, mass, q, seg_off, group_seg_off, vel_scale, q_scale, out=None, frame0=0):
    """mdp_charge_flux: vel [F,3,N] -> J [3, G, F] (or written into ``out`` [3,G,Ttot] at column frame0)."""
    vel = _f64(vel, "vel")
    F, _, n = vel.shape
    ctx = Context.get(vel.device.index)
    garr, gptr = _host_i64(group_seg_off)
    G = len(garr) - 1
    S = seg_off.shape[0] - 1
    if out is None:
        out = torch.zeros((3, G, F), dtype=torch.float64, device=vel.device)
    check(lib().mdp_charge_flux(ctx.handle, F, n, ptr(vel), ptr(_f64(mass, "mass")), ptr(_f64(q, "q")), S,
                                ptr(_i32(seg_off, "seg_off")), gptr, G, float(vel_scale), float(q_scale), ptr(out),
                                out.shape[2], int(frame0), stream_ptr()), "mdp_charge_flux")
    return out


def xcorr_unbiased(a, b, nlags=None):
    """mdp_xcorr_unbiased: a, b [C,T] -> [C,nlags]."""
    a = _f64(a, "a")
    b = _f64(b, "b")
    C, T = a.shape
    nlags = T if nlags is None else int(nlags)
    ctx = Context.get(a.device.index)
    out = torch.empty((C, nlags), dtype=torch.float64, device=a.device)
    if xcorr_fft_enabled(T):
        # N log N through the fp64 Stockham FFT (csrc/fftcorr.cu); the direct O(T^2) kernel serves short series
        check(lib().mdp_xcorr_fft(ctx.handle, C, T, ptr(a), ptr(b), nlags, ptr(out), stream_ptr()), "mdp_xcorr_fft")
        return out
    check(lib().mdp_xcorr_unbiased(ctx.handle, C, T, ptr(a), ptr(b), nlags, ptr(out), stream_ptr()), "mdp_xcorr_unbiased")
    return out


def cross_msd_fft(a, b, group_off, nlags):
    """mdp_cross_msd_fft: a, b [C,T] (b None: the self case, b = a), group_off host ints [G+1] ->
    out [G, nlags] = sum over the group's channels of the all-origins mean of (a(t+tau) - a(t)) * (b(t+tau) - b(t))."""
    a = _f64(a, "a")
    C, T = a.shape
    if b is not None:
        b = _f64(b, "b")
        if b.shape != a.shape:
            raise ValueError(f"b must have the shape of a {tuple(a.shape)}, got {tuple(b.shape)}")
    garr, gptr = _host_i64(group_off)
    G = len(garr) - 1
    ctx = Context.get(a.device.index)
    out = torch.empty((max(G, 0), max(int(nlags), 0)), dtype=torch.float64, device=a.device)
    check(lib().mdp_cross_msd_fft(ctx.handle, C, T, ptr(a), ptr(b), G, gptr, int(nlags), ptr(out), stream_ptr()),
          "mdp_cross_msd_fft")
    return out


def group_acf_fft(a, group_off, nlags):
    """mdp_group_acf_fft: a [C,T], group_off host ints [G+1] -> out [G, nlags] = sum over the group's channels of the
    all-origins mean of a(t+tau) * a(t) (not centred)."""
    a = _f64(a, "a")
    C, T = a.shape
    garr, gptr = _host_i64(group_off)
    G = len(garr) - 1
    ctx = Context.get(a.device.index)
    out = torch.empty((max(G, 0), max(int(nlags), 0)), dtype=torch.float64, device=a.device)
    check(lib().mdp_group_acf_fft(ctx.handle, C, T, ptr(a), G, gptr, int(nlags), ptr(out), stream_ptr()), "mdp_group_acf_fft")
    return out


def structure_factor(xyz, cls, ncls, cell, miller, bin_off, nbins):
    """mdp_structure_factor: xyz float64 [F,3,N]; cls int32 [N] or [F,N] or None (one class); cell host (lx, ly, lz, xy, xz,
    yz) shared by the F frames; miller host ints [nk,3] sorted by bin; bin_off host ints [nbins+1] ->
    float64 [F, ncls(ncls+1)/2, nbins]: per class-pair row (ops.sym_row) the sum over each bin's k-vectors of
    Re(rho_a(k) conj(rho_b(k)))."""
    xyz = _f64(xyz, "xyz")
    F, _, n = xyz.shape
    cell = np.ascontiguousarray(cell, dtype=np.float64).reshape(-1)
    if cell.size != 6:
        raise ValueError(f"cell must hold 6 values (lx, ly, lz, xy, xz, yz), got {cell.size}")
    miller = np.ascontiguousarray(miller, dtype=np.int32).reshape(-1, 3)
    boff, bptr = _host_i64(bin_off)
    if boff.shape != (int(nbins) + 1,):
        raise ValueError(f"bin_off must hold nbins + 1 = {int(nbins) + 1} offsets, got shape {boff.shape}")
    cls = _i32(cls, "cls")
    stride = 0 if cls is None or cls.dim() == 1 else n
    ctx = Context.get(xyz.device.index)
    out = torch.empty((F, sym_rows(int(ncls)), int(nbins)), dtype=torch.float64, device=xyz.device)
    check(lib().mdp_structure_factor(ctx.handle, F, n, ptr(xyz), ptr(cls), stride, int(ncls), _lib.dptr(cell), miller.shape[0],
                                     miller.ctypes.data_as(ctypes.POINTER(c_int32)), int(nbins), bptr, ptr(out), stream_ptr()),
          "mdp_structure_factor")
    return out


def sk_rho(xyz, cls, ncls, cell, miller, out=None, frame0=0):
    """mdp_sk_rho: xyz float64 [F,3,N]; cls, cell, miller as for ``structure_factor`` -> complex128 [C >= ncls, nk, T]:
    rho_c(k) of frame f at column frame0 + f of ``out`` for c < ncls (a new [ncls, nk, F] series when None; other columns
    and channels untouched)."""
    xyz = _f64(xyz, "xyz")
    F, _, n = xyz.shape
    cell = np.ascontiguousarray(cell, dtype=np.float64).reshape(-1)
    if cell.size != 6:
        raise ValueError(f"cell must hold 6 values (lx, ly, lz, xy, xz, yz), got {cell.size}")
    miller = np.ascontiguousarray(miller, dtype=np.int32).reshape(-1, 3)
    nk = miller.shape[0]
    if out is None:
        out = torch.zeros((int(ncls), nk, F), dtype=torch.complex128, device=xyz.device)
    if not (out.is_cuda and out.dtype == torch.complex128 and out.is_contiguous() and out.dim() == 3
            and out.shape[0] >= int(ncls) and out.shape[1] == nk):
        raise ValueError(f"out must be a contiguous complex128 CUDA tensor [>= {int(ncls)}, {nk}, T]")
    cls = _i32(cls, "cls")
    stride = 0 if cls is None or cls.dim() == 1 else n
    ctx = Context.get(xyz.device.index)
    check(lib().mdp_sk_rho(ctx.handle, F, n, ptr(xyz), ptr(cls), stride, int(ncls), _lib.dptr(cell), nk,
                           miller.ctypes.data_as(ctypes.POINTER(c_int32)), ptr(out), out.shape[2], int(frame0), stream_ptr()),
          "mdp_sk_rho")
    return out


def isf_fft(rho, pairs, bin_off, nlags):
    """mdp_isf_fft: rho complex128 [nchan, nk, T]; pairs host ints [npairs, 2] of channels; bin_off host ints [nbins+1] ->
    float64 [npairs, nbins, nlags]: per pair and bin the sum over the bin's k-vectors of the symmetrised all-origins
    correlation 1/2 Re<z_a(t+tau) z_b(t)* + z_b(t+tau) z_a(t)*>."""
    if not (rho.is_cuda and rho.dtype == torch.complex128 and rho.is_contiguous() and rho.dim() == 3):
        raise ValueError("rho must be a contiguous complex128 CUDA tensor [nchan, nk, T]")
    nchan, nk, T = rho.shape
    pr = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
    boff, bptr = _host_i64(bin_off)
    nbins = boff.shape[0] - 1
    ctx = Context.get(rho.device.index)
    out = torch.empty((pr.shape[0], max(nbins, 0), max(int(nlags), 0)), dtype=torch.float64, device=rho.device)
    check(lib().mdp_isf_fft(ctx.handle, nchan, nk, T, ptr(rho), pr.shape[0], pr.ctypes.data_as(ctypes.POINTER(c_int32)), nbins, bptr,
                            int(nlags), ptr(out), stream_ptr()), "mdp_isf_fft")
    return out


def orient_series(xyz, cells, kind, atoms, out, frame0=0):
    """mdp_orient_series: xyz float64 [F,3,N]; cells host [F,6] = (lx, ly, lz, xy, xz, yz) per frame; kind 0 (bond), 1
    (bisector) or 2 (normal); atoms host ints [nvec,3] (rows of xyz; the third is ignored for a bond); out float64
    [8, nvec, T] -> out, with the channels of frame f at column frame0 + f (other columns untouched)."""
    xyz = _f64(xyz, "xyz")
    F, _, n = xyz.shape
    cells = np.ascontiguousarray(cells, dtype=np.float64).reshape(-1)
    if cells.size != 6 * F:
        raise ValueError(f"cells must hold 6 values (lx, ly, lz, xy, xz, yz) per frame ({F} frames), got {cells.size}")
    atoms = np.ascontiguousarray(atoms, dtype=np.int32).reshape(-1, 3)
    out = _f64(out, "out")
    if out.dim() != 3 or out.shape[0] != 8 or out.shape[1] != atoms.shape[0]:
        raise ValueError(f"out must be [8, {atoms.shape[0]}, T], got {tuple(out.shape)}")
    ctx = Context.get(xyz.device.index)
    check(lib().mdp_orient_series(ctx.handle, F, n, ptr(xyz), _lib.dptr(cells), int(kind), atoms.shape[0],
                                  atoms.ctypes.data_as(ctypes.POINTER(c_int32)), ptr(out), out.shape[2], int(frame0),
                                  stream_ptr()), "mdp_orient_series")
    return out


def cumtrapz(y, dx, scale=1.0, leading_zero=True):
    y = _f64(y, "y")
    R, T = y.shape
    ctx = Context.get(y.device.index)
    out = torch.empty((R, T if leading_zero else T - 1), dtype=torch.float64, device=y.device)
    check(lib().mdp_cumtrapz(ctx.handle, R, T, ptr(y), float(dx), float(scale), 1 if leading_zero else 0, ptr(out),
                             stream_ptr()), "mdp_cumtrapz")
    return out


XCORR_FFT_MIN_T = 2048


def xcorr_fft_enabled(T: int = XCORR_FFT_MIN_T) -> bool:
    """The FFT route is the default for series of at least XCORR_FFT_MIN_T steps (validated on hardware in round 2:
    30 x 100 000 steps in 1.56 ms against 12.7 ms for the direct sum); MDP_XCORR_FFT=0 forces the direct kernel,
    MDP_XCORR_FFT=1 forces the FFT for every length."""
    import os

    v = os.environ.get("MDP_XCORR_FFT", "")
    if v == "":
        return T >= XCORR_FFT_MIN_T
    return v != "0"


def shell_grid_enabled() -> bool:
    """The small-set shell search (csrc/shell.cu) is the default for n_a <= 4096 central points against a set at least 8
    times larger (round 2 on hardware, C5: 13.6 ms against 47 ms for the general engine's list mode, same entries);
    MDP_SHELL_GRID=0 selects the general engine."""
    import os

    return os.environ.get("MDP_SHELL_GRID", "1") not in ("", "0")


def survival_runs_enabled() -> bool:
    """Run-based survival counts (csrc/survival.cu) are the default (validated on hardware in round 2: C5 correlation
    48 ms -> 7 ms with the same integers); MDP_SURVIVAL_RUNS=0 selects the AND-shift-popcount kernel."""
    import os

    return os.environ.get("MDP_SURVIVAL_RUNS", "1") not in ("", "0")


def unique_pair_keys(lst, n_a, n_b):
    """mdp_unique_pair_keys: the distinct (ia, ib) of a neighbour list as sorted int64 keys ia * n_b + ib."""
    lst = _i32(lst.contiguous(), "lst")
    M = lst.shape[0]
    ctx = Context.get(lst.device.index)
    cap = max(M, 1)
    keys = torch.empty((cap,), dtype=torch.int64, device=lst.device)
    cnt = torch.zeros((1,), dtype=torch.int64, device=lst.device)
    check(lib().mdp_unique_pair_keys(ctx.handle, M, ptr(lst), int(n_a), int(n_b), ptr(keys), cap, ptr(cnt), stream_ptr()),
          "mdp_unique_pair_keys")
    return keys[: int(cnt.item())]


def bitmask_autocorr_from_list(lst, n_b, T, n_a=None):
    """Neighbour list (frame, ia, ib) -> integer survival counts cnt[tau] (int64 [T]) and the number of ever-neighbour pairs."""
    ctx = Context.get(lst.device.index)
    cnt = torch.zeros((T,), dtype=torch.int64, device=lst.device)
    if lst.shape[0] == 0:
        return cnt, 0
    lst = lst.contiguous()
    n_a = int(n_a) if n_a is not None else int(lst[:, 1].max().item()) + 1
    ukeys = unique_pair_keys(lst, n_a, int(n_b))                # sorted distinct (ia, ib) keys: bitmap + popcount scan, no sort
    P = int(ukeys.shape[0])
    W = (T + 63) // 64
    masks = torch.zeros((P, W), dtype=torch.int64, device=lst.device)
    lst = lst.contiguous()
    check(lib().mdp_bitmask_fill(ctx.handle, lst.shape[0], ptr(lst), int(n_b), ptr(ukeys), P, W, ptr(masks),
                                 stream_ptr()), "mdp_bitmask_fill")
    if survival_runs_enabled() and T * 8 + 32768 <= 200 * 1024:
        # the same integers from the runs of each mask (csrc/survival.cu); series too long for its shared-memory
        # second-difference array take the popcount kernel below
        check(lib().mdp_survival_runs(ctx.handle, P, W, T, ptr(masks), ptr(cnt), stream_ptr()), "mdp_survival_runs")
        return cnt, P
    step = 65535 * 64
    for p0 in range(0, P, step):
        m = masks[p0:p0 + step]
        check(lib().mdp_bitmask_autocorr(ctx.handle, m.shape[0], W, T, ptr(m), ptr(cnt), stream_ptr()),
              "mdp_bitmask_autocorr")
    return cnt, P


def ols_sums(t, y, i0=0, i1=None):
    t = _f64(t, "t")
    y = _f64(y, "y")
    C, T = y.shape
    i1 = T if i1 is None else int(i1)
    ctx = Context.get(t.device.index)
    out = torch.empty((C, 3), dtype=torch.float64, device=t.device)
    check(lib().mdp_ols_sums(ctx.handle, C, T, ptr(t), ptr(y), int(i0), i1, ptr(out), stream_ptr()), "mdp_ols_sums")
    return out


def axis_density(coord, key, surface_key, target_keys, dist_from_interface, bin_size, nbins):
    """mdp_axis_density: coord, key float64 [F, N] -> (counts int64 [F, ntargets, nbins], minmax float64 [F, 2])."""
    coord = _f64(coord, "coord")
    key = _f64(key, "key")
    F, n = coord.shape
    tk = np.ascontiguousarray(target_keys, dtype=np.float64)
    ctx = Context.get(coord.device.index)
    counts = torch.empty((F, len(tk), nbins), dtype=torch.int64, device=coord.device)
    mm = torch.empty((F, 2), dtype=torch.float64, device=coord.device)
    check(lib().mdp_axis_density(ctx.handle, F, n, ptr(coord), ptr(key), float(surface_key), len(tk), _lib.dptr(tk),
                                 float(dist_from_interface), float(bin_size), int(nbins), ptr(counts), ptr(mm), stream_ptr()),
          "mdp_axis_density")
    return counts, mm


def dump_parse_device(text, begin, end, longest, natoms, ncols, colsel, id_col, out, seen, status, stream=None):
    """mdp_dump_parse_device (the file pipeline's parser, io/pipeline.py): text uint8 [bytes], begin/end int64 [F] byte offsets of each frame's
    rows, out float64 [F, nwant, N], seen int32 [F, ceil(N/32)] scratch, status int64 [F, 2] = (rows parsed, flags) --
    all on the device.  Enqueued on ``stream`` (default: the current stream); the caller checks ``status``."""
    F, nwant, stride = out.shape
    cs = (c_int * int(ncols))(*[int(v) for v in colsel])
    ctx = Context.get(out.device.index)
    sp = stream_ptr() if stream is None else ctypes.c_void_p(stream.cuda_stream)
    check(lib().mdp_dump_parse_device(ctx.handle, F, ptr(text), ptr(begin), ptr(end), int(longest), int(natoms), int(ncols), cs,
                                      int(id_col), nwant, ptr(out), nwant * stride, stride, ptr(seen), ptr(status), sp),
          "mdp_dump_parse_device")
