#!/usr/bin/env python
"""bench.py -- headline benchmark of the mdproptools hot path on B200 (see DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (N>1: launched by torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference algorithm on the host CPU
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # + the last step's histograms as DIR/*.npy

The inputs are generated from fixed seeds, so two builds run with the same arguments can be compared output for output.

Workload (BASELINE.json configs[1], "C2", at its full size): synthetic LJ-like fluid, 100 000 atoms per frame,
1 000 frames, triclinic cell (lx=ly=lz=167.19 A, xy=0.2lx, xz=0.1lx, yz=-0.15ly), all-pair RDF with r_cut = 20 A,
bin = 0.05 A (400 bins), minimum image as the reference applies it (orthogonal wrap with the lattice lengths).
One *step* is one pass of the RDF hot path over the WHOLE trajectory, resident in HBM (2.4 GB of coordinates, far
larger than the 126 MB L2, so no L2 flush is needed between steps); with N GPUs the frames are split in contiguous
blocks (STRONG scaling: the job is the same 1 000 frames at every N) and the per-frame integer histograms are
all-gathered.  The headline metric is RDF pair-evaluations per second, counted NOMINALLY as frames x N(N-1)/2 (what
the reference's loop evaluates); the kernel actually evaluates only the pairs that survive the bounding-box tests,
that number is reported beside it and is what the roofline fraction is computed from.  The run checks itself: the GPU
histogram of frame 0 must equal the oracle's brute-force histogram bit for bit (`parity_frame0`), at N > 1 rank 0
recomputes frames of the other ranks' blocks (`nrank_equals_1rank`), and `hist_sha256` of all 1 000 per-frame
histograms is the same string at every N.  The same JSON line carries the second half of the BASELINE metric, MSD
atom-frames/s (config C3), and the C4/C5 legs, each with its own roofline.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

# OpenMP workers (the oracle's CPU legs, torch's CPU ops) must SLEEP when they have nothing to do: with the default
# spin-waiting the idle workers of an earlier parallel region keep every core busy while the file pipeline's reader
# threads need them -- measured on the 16-core B200 host: rdf_from_files 1.0 ms/frame with spinning workers, 0.28 ms/frame
# without (MDP_PIPELINE_TRACE timelines of the leg).  Must be set before the OpenMP runtimes load, i.e. before numpy / torch.
for _k, _v in (("OMP_WAIT_POLICY", "PASSIVE"), ("GOMP_SPINCOUNT", "0"), ("KMP_BLOCKTIME", "0")):
    os.environ.setdefault(_k, _v)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
_emit = print
sys.path.insert(0, ROOT)

N_ATOMS = 100_000
LBOX = 167.19
TILT = (0.20 * LBOX, 0.10 * LBOX, -0.15 * LBOX)
R_CUT = 20
BIN = 0.05
NBINS = 400
FRAMES_TOTAL = 1000            # C2 as BASELINE.json states it: 100k atoms x 1k frames
SEED = 20261017
FLOPS_PER_PAIR = 11            # SURVEY 8(d): 3 sub, 3 minimum-image add, 3 mul, 2 add, unfused
MSD_ATOMS = 1_000_000
MSD_FRAMES = 10_000            # C3 as BASELINE.json states it: 1M atoms x 10k frames (240 GB; walked in resident 30 GB chunks)
MSD_BYTES_PER_ATOM_FRAME = 24  # SURVEY 8(d)


def lattice_lengths():
    xy, xz, yz = TILT
    return (LBOX, float(np.sqrt(xy * xy + LBOX * LBOX)), float(np.sqrt(xz * xz + yz * yz + LBOX * LBOX)))


def make_frames(nframes, seed, xp, keep=None):
    """C2 generator (SURVEY 8d): simple-cubic lattice sites (first N of 47^3) in fractional coordinates, jitter,
    per-frame Gaussian steps of 0.05 A, wrapped into the triclinic cell.  xp = "cuda" (device) or "cpu" (host).
    The trajectory is one random walk, so a rank that owns frames keep=[lo, hi) walks frames 0..hi-1 and keeps its block
    (same seed on every rank: the union over the ranks is the one 1000-frame trajectory whatever the rank count)."""
    import torch
    g = torch.Generator(device="cuda" if xp == "cuda" else "cpu")
    g.manual_seed(seed)
    dev = "cuda" if xp == "cuda" else "cpu"
    m = 47
    idx = torch.arange(N_ATOMS, device=dev)
    frac = torch.stack([(idx // (m * m)) % m, (idx // m) % m, idx % m]).to(torch.float64) / m
    cell = torch.tensor([[LBOX, 0.0, 0.0], [TILT[0], LBOX, 0.0], [TILT[1], TILT[2], LBOX]], dtype=torch.float64, device=dev)
    inv = torch.linalg.inv(cell)
    cart = cell.T @ frac                                           # r = sx a + sy b + sz c
    cart = cart + (torch.rand((3, N_ATOMS), generator=g, dtype=torch.float64, device=dev) - 0.5) * 2 * 0.3 * 3.405
    lo, hi = keep if keep is not None else (0, nframes)
    out = torch.empty((hi - lo, 3, N_ATOMS), dtype=torch.float64, device=dev)
    for f in range(hi):
        cart = cart + torch.randn((3, N_ATOMS), generator=g, dtype=torch.float64, device=dev) * 0.05
        s = inv.T @ cart
        s = s - torch.floor(s)
        cart = cell.T @ s
        if f >= lo:
            out[f - lo] = cart
    return out


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
            except ValueError:
                continue
            for nm, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    """Driver-written MEASURED_PEAKS.json (HBM, bf16) + this repo's own FP64 micro-benchmark (tools/peaks.cu,
    result committed as profiles/peaks_b200.json)."""
    p = {}
    for f in (os.path.join(ROOT, "profiles", "peaks_b200.json"), os.path.join(ROOT, "MEASURED_PEAKS.json")):
        if os.path.exists(f):
            try:
                p.update(json.load(open(f)))
            except Exception:
                pass
    return p


def ncu_traffic(name, scale=1.0):
    """DRAM bytes (read + write) of one launch of kernel `name` from the committed ncu --set full summary
    (the newest profiles/rNNx_k_<name>.txt, written by tools/ncu_summary.py), times `scale` when the bench launch is that much larger
    than the captured one (traffic is linear in the number of frames for every kernel here).  None when absent."""
    import glob as _g
    cands = sorted(_g.glob(os.path.join(ROOT, "profiles", f"r*_k_{name}.txt")))   # newest round last (r01a < r01b < ...)
    if not cands:
        return None
    path = cands[-1]
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    total = 0.0
    for ln in open(path):
        p = ln.split()
        if len(p) >= 3 and p[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            total += float(p[1]) * unit.get(p[2], 1.0)
    return total * scale if total else None


# ------------------------------------------------------------------------------------------------
# CPU legs (oracle port; the only place bench.py touches oracle/)
# ------------------------------------------------------------------------------------------------
def host_threads():
    """Threads the CPU legs use: every core this process may run on.  Passed to the oracle explicitly -- torchrun
    exports OMP_NUM_THREADS=1 to its workers, which made the round-1 reference arm single-threaded at N > 1."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_rdf_frame0(host_frame):
    """The exact oracle histogram of one whole C2 frame (reference wrap with the lattice lengths): int64 [NBINS] = rdf_full
    of rdf_cn.py:85-86 (2 per in-cutoff pair).  ~2 s on 16 threads; bench.py compares the GPU histogram of the same frame
    with it bit for bit (`parity_frame0`)."""
    from oracle import oracle as O
    x, y, z = host_frame
    full, _ = O.rdf_loop(np.ones(N_ATOMS), x, y, z, np.array([[1, 1]]), lattice_lengths(), R_CUT, BIN, NBINS,
                         nthreads=host_threads())
    return np.asarray(full).astype(np.int64)


def cpu_rdf_frame0_triclinic(host_frame):
    from oracle import oracle as O
    x, y, z = host_frame
    full, _ = O.rdf_loop_tri(np.ones(N_ATOMS), x, y, z, np.array([[1, 1]]), (LBOX, LBOX, LBOX) + TILT, R_CUT, BIN, NBINS,
                             nthreads=host_threads())
    return np.asarray(full).astype(np.int64)


def cpu_rdf_sample(target_seconds, host_frame=None):
    """The reference's pair loop (oracle/oracle.c restatement of rdf_cn.py:35-97) on a bounded sample of the C2
    workload: the first n_sub atoms of one frame against all N atoms (n_sub x N pair evaluations, same
    arithmetic per pair), all host threads.  Returns (pair_evals_per_s, cores, description)."""
    from oracle import oracle as O
    if host_frame is None:
        host_frame = make_frames(1, SEED, "cpu")[0].numpy()
    L = lattice_lengths()
    x, y, z = host_frame
    ones = np.ones(N_ATOMS)
    cores = host_threads()
    rel = np.array([[1, 1]])

    def run(n_sub):
        t = time.perf_counter()
        O.rdf_rect(ones[:n_sub], x[:n_sub], y[:n_sub], z[:n_sub], ones, x, y, z, rel, L, R_CUT, BIN, NBINS, nthreads=cores)
        return time.perf_counter() - t

    run(64)                                            # warm-up (thread pool, page faults)
    n_probe = 512
    rate = n_probe * N_ATOMS / run(n_probe)
    n_sub = int(min(N_ATOMS, max(n_probe, rate * target_seconds / N_ATOMS)))
    dt = run(n_sub)
    return n_sub * N_ATOMS / dt, cores, f"{n_sub} of {N_ATOMS} outer atoms x all atoms of one C2 frame ({dt:.1f} s)"


def _ref_worker(args):
    """One process of the reference arm: the UNMODIFIED reference's numba loop `_rdf_loop` (rdf_cn.py:72-97) on a slice of the
    frame's atoms taken as a system of its own (same box, same cutoff, same bins)."""
    lo, hi = args
    from mdproptools.structural import rdf_cn as R            # the installed reference (baseline/_ref), via the harness
    data = _REF_STATE["data"][lo:hi]
    full = np.zeros(NBINS)
    part = np.zeros((1, NBINS))
    t = time.perf_counter()
    R._rdf_loop(np.asfortranarray(data), _REF_STATE["rel"], 1, _REF_STATE["L"], R_CUT, BIN, full, part)
    return time.perf_counter() - t, float(full.sum())


_REF_STATE = {}


def reference_numba_sample(host_frame, n_sub=8000):
    """The unmodified reference (pip-installed into baseline/_ref, imported through oracle/ref_harness.py: pymatgen stand-in
    and plotting mocks only, every numerical line is the reference's) on a bounded sample of the C2 frame: every host core
    runs the stock `_rdf_loop` on its own slice of n_sub atoms.  Returns (pair_evals_per_s, cores, one-core rate, sample) or
    None when the reference or numba is not importable on this box."""
    ref_root = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_root, "mdproptools")):
        return None
    try:
        os.environ["MDPROP_REFERENCE_ROOT"] = ref_root
        from oracle import ref_harness as H
        H.install()
        from mdproptools.structural import rdf_cn as R
    except Exception as exc:  # noqa: BLE001 - reported, the port stands in
        sys.stderr.write(f"reference arm: cannot import the installed reference ({exc}); using the port\n")
        return None
    import multiprocessing as mp
    cores = host_threads()
    n_sub = min(n_sub, N_ATOMS // max(cores, 1))            # one disjoint slice per core
    x, y, z = host_frame
    data = np.column_stack([np.ones(N_ATOMS), x, y, z])
    _REF_STATE.update(data=data, rel=np.array([[1, 1]], dtype=np.int64), L=tuple(lattice_lengths()))
    # JIT compile once in the parent (excluded from the timing, ~15 s); the forked workers inherit the compiled loop
    tj = time.perf_counter()
    R._rdf_loop(np.asfortranarray(data[:64]), _REF_STATE["rel"], 1, _REF_STATE["L"], R_CUT, BIN, np.zeros(NBINS), np.zeros((1, NBINS)))
    jit_s = time.perf_counter() - tj
    slices = [(k * n_sub, (k + 1) * n_sub) for k in range(min(cores, N_ATOMS // n_sub))]
    ctx = mp.get_context("fork")
    t = time.perf_counter()
    with ctx.Pool(len(slices)) as pool:
        res = pool.map(_ref_worker, slices)
    wall = time.perf_counter() - t
    pairs = len(slices) * n_sub * (n_sub - 1) // 2
    one_core = (n_sub * (n_sub - 1) // 2) / float(np.mean([r[0] for r in res]))
    return (pairs / wall, len(slices), one_core,
            f"unmodified reference _rdf_loop (numba, as shipped: serial) on {len(slices)} processes x {n_sub}-atom slices of one C2 "
            f"frame ({wall:.1f} s; JIT {jit_s:.0f} s excluded; {one_core:.3g} pair-evals/s per core)")


def cpu_msd_sample(target_seconds):
    from oracle import oracle as O
    n, T = 100_000, 100                                 # BASELINE.md plan: 100k atoms x 100 frames
    rng = np.random.default_rng(SEED + 1)
    traj = np.cumsum(rng.normal(0, 0.1, (T, 3, n)), axis=0)
    t = time.perf_counter()
    reps = 0
    while reps == 0 or (time.perf_counter() - t < target_seconds and reps < 50):
        O.msd_single_origin(traj, 0, 1e-10)
        reps += 1
    dt = (time.perf_counter() - t) / reps
    return n * T / dt, 1, f"numpy restatement of diffusion.py:207-218 on {n} atoms x {T} frames ({dt:.2f} s/pass)"


WORKLOAD = "C2: LJ fluid 100k atoms/frame x 1000 frames, triclinic cell, all-pair RDF r_cut=20 bin=0.05 (400 bins)"


def headline_config(world, T_total):
    """The `config` object of BOTH arms (the driver compares them key by key)."""
    return {"workload": WORKLOAD, "frames_total": T_total, "atoms_per_frame": N_ATOMS,
            "mic": "reference (orthogonal wrap with lattice lengths)",
            "pair_evals": "nominal: frames*N(N-1)/2, what the reference's loop evaluates",
            "l2_policy": "inputs larger than L2 (2.4 MB of coordinates per frame, every frame read once per step)",
            "parallelism": f"frames x{world}"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # the reference arm: bounded samples of the same C2 workload on all host cores.  `value` = the UNMODIFIED reference
    # (baseline/_ref, numba loop as shipped, one process per core) when it is importable on this box; the C port of the same loop
    # (oracle/oracle.c, OpenMP, ~30x faster per core) is timed beside it and stands in when it is not.
    host_frame = make_frames(1, SEED, "cpu")[0].numpy()
    ref = None if args.port_only else reference_numba_sample(host_frame)
    for _ in range(args.warmup):
        cpu_rdf_sample(0.5, host_frame)
    rates, descr, cores = [], "", 1
    t0 = time.perf_counter()
    ref_rates = []
    for _ in range(args.steps):
        r, cores, descr = cpu_rdf_sample(3.0, host_frame)
        rates.append(r)
        if ref is not None:
            rr = reference_numba_sample(host_frame)
            ref_rates.append(rr[0])
            ref = rr
    wall = time.perf_counter() - t0
    port_value = float(np.mean(rates))
    if ref is not None:
        value, kind, rcores, sample = float(np.mean(ref_rates)), "reference", ref[1], ref[3]
    else:
        value, kind, rcores, sample = port_value, "port", cores, descr
    out = {
        "impl": "reference", "metric": "rdf_pair_evals_per_s", "value": value, "unit": "pair-evals/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": headline_config(args.gpus, args.frames),
        "note": "each step is a bounded sample of one frame of the same trajectory (per-unit throughput); the reference cannot "
                "finish one C2 frame per core in less than ~8 minutes",
        "cpu_baseline": {"value": value, "unit": "pair-evals/s", "cores": rcores, "kind": kind, "sample": sample},
        "port": {"value": port_value, "unit": "pair-evals/s", "cores": cores, "kind": "port",
                 "sample": "oracle/oracle.c restatement of rdf_cn.py:35-97, OpenMP: " + descr},
        "e2e": {"value": value, "unit": "pair-evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    _emit(json.dumps(out))
    return 0


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from mdproptools_b200 import ops
    from mdproptools_b200._lib import Context, bin_edges
    from mdproptools_b200.dynamical.diffusion import Diffusion
    from mdproptools_b200.structural import rdf_cn

    from mdproptools_b200 import dist as mdist
    dev = torch.device("cuda", local)
    ctx = Context.get(local)
    # STRONG scaling: the whole C2 trajectory (T_total frames, default 1000) is one job; rank r owns the contiguous block
    # shard_range(T_total) of its frames.  One step = one pass of the RDF hot path over all T_total frames.
    T_total = args.frames
    lo, hi = mdist.shard_range(T_total, rank, world)
    F = hi - lo
    L = lattice_lengths()
    boxes = np.tile(np.asarray(L), (F, 1))
    edges = bin_edges(BIN, NBINS)
    rcut2 = float(R_CUT ** 2)
    weights = np.array([[2], [2]], dtype=np.int32)            # g_full and the single like relation 1-1
    frames = make_frames(T_total, SEED, "cuda", keep=(lo, hi))   # resident in HBM before the timed region

    def step():
        hist = ops.pair_hist(frames, None, 1, boxes, rcut2, edges, BIN)
        red = ops.hist_reduce(hist, weights)
        return mdist.all_gather_blocks(red, T_total)             # [T_total, 2, NBINS] on every rank (exact integers)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        out = step()
    barrier()
    stats = ctx.pair_stats()
    st = torch.tensor([stats["pair_evals"], stats.get("exact_path_pairs", 0)], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(st)
    evaluated_per_step, exact_per_step = int(st[0].item()), int(st[1].item())
    nominal_per_step = T_total * N_ATOMS * (N_ATOMS - 1) // 2
    in_cut = int(out[0, 0].sum().item()) // 2
    import hashlib
    hist_sha = hashlib.sha256(out.cpu().numpy().astype(np.int64).tobytes()).hexdigest()   # same at every N: N-rank == 1-rank

    # ---- parity at headline scale: frame 0 of the trajectory against the exact oracle histogram (brute force on the host
    # cores), bit for bit; and, at N > 1, rank 0 recomputes the first frame of every other rank's block from its own walk
    parity = {"parity_frame0": None}
    src = frames[0:1]
    if rank == 0 and not args.skip_cpu:
        f0_host = frames[0].cpu().numpy()                       # frame 0 of the benchmarked trajectory itself (rank 0 owns it)
        want = cpu_rdf_frame0(f0_host)
        parity = {"parity_frame0": bool(np.array_equal(out[0, 0].cpu().numpy(), want)),
                  "parity_frame0_pairs_in_cutoff": int(want.sum()) // 2,
                  "parity_frame0_note": "per-frame histogram 0 of the timed step's own output == oracle/oracle.c brute force over all "
                                        "N(N-1)/2 pairs of that frame, all 400 bins, bit for bit"}
    if world > 1:
        # N-rank == 1-rank on hardware: rank 0 walks the trajectory itself up to the first frame of each other block
        firsts = sorted({mdist.shard_range(T_total, r, world)[0] for r in range(1, world)})
        ok = True
        if rank == 0:
            for fidx in firsts[: args.nrank_checks]:
                fr = make_frames(T_total, SEED, "cuda", keep=(fidx, fidx + 1))
                mine = ops.hist_reduce(ops.pair_hist(fr, None, 1, boxes[:1], rcut2, edges, BIN), weights)[0]
                ok = ok and bool(torch.equal(mine, out[fidx]))
            parity["nrank_equals_1rank_frames"] = firsts[: args.nrank_checks]
            parity["nrank_equals_1rank"] = ok

    ctx.timing(True)
    ctx.timing_read(0), ctx.timing_read(1)
    launches0 = ctx.launch_count()
    clocks = ClockSampler(local)
    clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        last = step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clk = clocks.stop()
    launches = ctx.launch_count() - launches0
    pair_ms, pair_n = ctx.timing_read(0)
    prep_ms, _ = ctx.timing_read(1)
    ctx.timing(False)
    if args.dump_outputs and rank == 0:
        dump_output(args.dump_outputs, "rdf_counts", last.cpu().numpy())
    del last
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = nominal_per_step * args.steps / (ms * 1e-3)
    evaluated_local = stats["pair_evals"]

    # ---- the same workload with the general triclinic image (mic="triclinic": true nearest image in the tilted cell;
    # an extension, the reference wraps tilted cells as if they were orthogonal)
    tric = None
    if not args.skip_triclinic:
        from mdproptools_b200._lib import PAIR_TRICLINIC
        cells = np.tile(np.asarray((LBOX, LBOX, LBOX) + TILT), (F, 1))

        def step_tri():
            hist = ops.pair_hist(frames, None, 1, cells, rcut2, edges, BIN, flags=PAIR_TRICLINIC)
            return ops.hist_reduce(hist, weights)

        for _ in range(3):
            out_t = step_tri()
        barrier()
        ev_t = ctx.pair_stats()["pair_evals"]
        in_cut_t = int(out_t[0, 0].sum().item()) // 2
        if rank == 0 and parity.get("parity_frame0") is not None:
            gt = ops.hist_reduce(ops.pair_hist(src.contiguous(), None, 1, cells[:1], rcut2, edges, BIN, flags=PAIR_TRICLINIC),
                                 weights)[0, 0].cpu().numpy()
            parity["parity_frame0_triclinic"] = bool(np.array_equal(gt, cpu_rdf_frame0_triclinic(f0_host)))
        ctx.timing(True)
        ctx.timing_read(0), ctx.timing_read(1)
        t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0e.record()
        for _ in range(args.steps):
            step_tri()
        t1e.record()
        barrier()
        ms_t = t0e.elapsed_time(t1e)
        pair_ms_t, pair_n_t = ctx.timing_read(0)
        ctx.timing_read(1)
        ctx.timing(False)
        tt = torch.tensor([ms_t], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_t = float(tt.item())
        tric = {"value": nominal_per_step * args.steps / (ms_t * 1e-3), "unit": "pair-evals/s",
                "ms_per_step": ms_t / args.steps, "pair_kernel_ms_per_step": pair_ms_t / args.steps,
                "evaluated_pair_evals_per_step_rank0": ev_t, "pairs_in_cutoff_frame0": in_cut_t,
                "achieved_tflops_11_per_pair": ev_t * FLOPS_PER_PAIR * args.steps / (pair_ms_t * 1e-3) / 1e12,
                "mic": "triclinic (sequential z,y,x single shift of the restricted triclinic cell; oracle-defined extension)"}

    # ---- end to end through the public array API: pinned host frames -> H2D -> kernels -> D2H -> normalised g(r)
    # (every rank streams ITS block of the trajectory from its own pinned buffer; the integer histograms are all-gathered and
    # every rank normalises all T_total frames, as a user of the API on N GPUs would get it)
    host = torch.empty((F, 3, N_ATOMS), dtype=torch.float64, pin_memory=True)
    host.copy_(frames)
    rel = [[1], [1]]
    types = np.ones(N_ATOMS)
    for _ in range(2):
        rdf_cn.calc_atomic_rdf_from_arrays(host, types, L, R_CUT, BIN, rel, batch_frames=128, frame_range=(lo, hi, T_total))
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(3, min(args.steps, 6))
    for _ in range(e2e_steps):
        df_e2e = rdf_cn.calc_atomic_rdf_from_arrays(host, types, L, R_CUT, BIN, rel, batch_frames=128, frame_range=(lo, hi, T_total))
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = nominal_per_step * e2e_steps / float(te.item())
    del host

    # ---- MSD (second half of the BASELINE metric), C3 shape: 1M atoms, resident chunk of frames
    msd = None
    if not args.skip_msd:
        msd = bench_msd(args, torch, dist, ops, ctx, dev, world, rank)

    gk = None if args.skip_gk else bench_green_kubo(args, torch, dist, ops, ctx, dev, world, rank)
    res = None if args.skip_residence else bench_residence(args, torch, dist, ops, ctx, dev, world, rank)
    c5s = None if args.skip_clusters else bench_clusters_hydration(args, torch, dist, ops, ctx, dev, world, rank)

    # --files-leg at N > 1: the file-based entry points run HERE, under the process group, on every rank (each rank writes
    # the same files into a directory of its own; the reads are sharded over the ranks and the per-frame histograms
    # all-gathered) -- what tests/test_gpu_parity.py::test_nrank_equals_1rank_under_nccl compares with the 1-rank result
    files_early = None
    if world > 1 and args.files_leg:
        files_early = (bench_rdf_from_files(torch, make_frames(32, SEED, "cuda"), N_ATOMS * (N_ATOMS - 1) // 2,
                                            copies=args.files_copies), bench_c1(torch))
    # every rank leaves the process group here: what follows on rank 0 (CPU baselines, host parser, the file-based leg)
    # is single-process work and must not meet a collective whose peers are gone
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return 0

    peaks = measured_peaks()
    fp64_peak = peaks.get("fp64_unfused_tflops_sustained") or peaks.get("fp64_unfused_tflops_burst")
    peak_src = "measured (tools/peaks.cu on this pool's B200, profiles/peaks_b200.json)"
    if not fp64_peak:
        fp64_peak = 148 * 64 * 1.965e9 / 1e12            # nominal: 64 DP lanes/SM, unfused = 1 flop/lane/clk
        peak_src = "nominal 148 SMs x 64 FP64 lanes x 1965 MHz, unfused (no measured FP64 peak on file yet)"
    # roofline of the dominant kernel on rank 0: its evaluated pairs x 11 flops over its CUDA-event kernel time (all launches
    # of the timed region: a 1000-frame call is cut into sub-batches that fit the scratch arena)
    achieved = evaluated_local * FLOPS_PER_PAIR * args.steps / (pair_ms * 1e-3) / 1e12
    nominal_tflops = (F * N_ATOMS * (N_ATOMS - 1) // 2) * FLOPS_PER_PAIR * args.steps / (pair_ms * 1e-3) / 1e12
    frames_per_launch = F * args.steps / max(pair_n, 1)
    # what actually bounds k_pair_fast: instruction issue.  Warp instructions per 32 evaluated pairs from the committed ncu
    # capture (profiles/r*_k_pair_fast_meta.json) x this run's evaluated pairs / its kernel time, against 4 schedulers x
    # 148 SMs x 1 instruction per clock
    issue = None
    try:
        import glob
        meta_path = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_k_pair_fast_meta.json")))[-1]      # the newest capture
        meta = json.load(open(meta_path))
        wi = meta["warp_instr_per_32_pairs"] if not os.environ.get("MDP_PAIR_F64") else meta["all_fp64_kernel"]["warp_instr_per_32_pairs"]
        ips = evaluated_local / 32.0 * wi * args.steps / (pair_ms * 1e-3)
        ipk = 148 * 4 * (clk.get("sm_mhz") or 1965.0) * 1e6
        issue = {"bound": "issue slots", "achieved": ips, "peak": ipk, "unit": "warp-instr/s", "frac": ips / ipk,
                 "warp_instr_per_32_pairs": wi, "source": f"instruction count per evaluated pair from profiles/{os.path.basename(meta_path)} "
                 f"(smsp__inst_executed.sum of the committed ncu capture; issue slots {meta.get('issue_active_pct', 83.7)} % busy "
                 "under ncu), scaled to this run"}
    except Exception:
        pass
    cpu_rate, cores, sample = cpu_rdf_sample(10.0) if not args.skip_cpu else (None, None, "skipped")
    out = {
        "metric": "rdf_pair_evals_per_s", "value": value, "unit": "pair-evals/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": headline_config(world, T_total),
        "frames_per_gpu": F, "hist_sha256": hist_sha, **parity,
        "evaluated_pair_evals_per_step": evaluated_per_step, "nominal_pair_evals_per_step": nominal_per_step,
        "exact_path_pairs_per_step": exact_per_step,
        "pairs_in_cutoff_frame0": in_cut,
        "gpu_launches": launches,
        "kernel_share": {"pair_kernel_ms_per_step": pair_ms / args.steps, "prep_ms_per_step": prep_ms / args.steps,
                         "step_ms": ms / args.steps},
        "roofline": {"bound": "fp64", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s", "frac": achieved / fp64_peak,
                     "traffic": ncu_traffic("pair_fast", frames_per_launch / 16.0), "peak_source": peak_src,
                     "traffic_note": "dram bytes of the 16-frame launch captured in the newest profiles/r*_k_pair_fast.txt (56 MB = the "
                                     "sorted records read once), scaled to this launch's frames; irrelevant to an issue-bound kernel",
                     "kernel": "k_pair_fast" if not os.environ.get("MDP_PAIR_F64") else "k_pair (all fp64)",
                     "issue": issue,
                     "note": f"pair kernel only; achieved = evaluated pair-evals x {FLOPS_PER_PAIR} unfused fp64 flops (the ALGORITHMIC "
                             f"cost of a pair in the reference, SURVEY 8d) / CUDA-event kernel time, against the measured unfused FP64 "
                             f"rate.  k_pair_fast does that arithmetic in fp32 (6 FP32-pipe instructions per pair, fp64 only for the "
                             f"{exact_per_step / max(evaluated_per_step, 1):.2%} of pairs within the proven error bound of a bin edge), so "
                             f"the fraction says how fast the kernel is relative to an ideal all-fp64 one, not how busy the FP64 pipe is; "
                             f"what bounds it is instruction issue (`issue`).  Nominal-pair equivalent = {nominal_tflops:.1f} TFLOP/s "
                             f"({nominal_tflops / fp64_peak:.2f} of peak) because culling skips work the reference does"},
        "e2e": {"value": e2e_value, "unit": "pair-evals/s", "h2d_bytes_per_step": T_total * 3 * N_ATOMS * 8,
                "d2h_bytes_per_step": world * T_total * 2 * NBINS * 8, "g_full_max": float(df_e2e["g_full(r)"].max()),
                "api": "rdf_cn.calc_atomic_rdf_from_arrays (pinned host frames, frame blocks over the ranks)"},
        "clocks": clk,
        "cpu_baseline": {"value": cpu_rate, "unit": "pair-evals/s", "cores": cores, "kind": "port", "sample": sample},
    }
    if tric:
        tric["roofline_frac"] = tric["achieved_tflops_11_per_pair"] / fp64_peak
        out["rdf_triclinic"] = tric
    if msd:
        out["msd"] = msd
    if gk:
        out["green_kubo"] = gk
    if res:
        out["residence"] = res
    if c5s:
        out["clusters_hydration"] = c5s
    if not args.skip_cpu:
        out["dump_parse"] = bench_dump_parse()
    if not args.skip_cpu or args.files_leg:
        # the first 32 frames of the walk on EVERY rank (not the rank's block): all ranks then see the same files, the file
        # reads are sharded over them, and the DataFrame (df_sha256) must not depend on the number of ranks
        del frames
        if files_early is not None:
            out["rdf_from_files"], c1 = files_early
            out["rdf_from_files"]["ranks"] = world
        else:
            out["rdf_from_files"] = bench_rdf_from_files(torch, make_frames(32, SEED, "cuda"), N_ATOMS * (N_ATOMS - 1) // 2,
                                                         copies=args.files_copies)
            c1 = bench_c1(torch)
        if c1:
            out["c1"] = c1
            parity["c1_sha256"] = out["c1_sha256"] = all(c1["sha256_equals_reference"].values())
    _emit(json.dumps(out))
    bad = [k for k in ("parity_frame0", "parity_frame0_triclinic", "nrank_equals_1rank", "c1_sha256")
           if parity.get(k) is False]
    if bad:
        sys.stderr.write(f"PARITY FAILURE: {bad}\n")
        return 1
    return 0


def bench_msd(args, torch, dist, ops, ctx, dev, world, rank):
    """C3 at its full size, STRONG scaling: 1 000 000 atoms x 10 000 frames of unwrapped fp64 coordinates (240 GB), single-origin
    MSD (diffusion.py:207-218).  Atoms are split over the ranks; a rank walks its atoms in resident chunks of <= 125 000 atoms
    x all frames (30 GB: one chunk per GPU at N = 8, eight chunks one after the other at N = 1, which cannot hold 240 GB).  A
    chunk is generated on the device (untimed), then `steps` passes of the kernel over it are timed with CUDA events; the job
    time is the sum over the rank's chunks, max over ranks.  The per-frame sums [T, 1, 4] are all-reduced (fp64)."""
    n, T = args.msd_atoms, args.msd_frames
    nchunks = 8 * ((world + 7) // 8)
    if nchunks % world:
        nchunks = world
    ca = (n + nchunks - 1) // nchunks                       # atoms per chunk
    mine = range(rank * nchunks // world, (rank + 1) * nchunks // world)
    steps = max(args.steps, 4)
    total = torch.zeros((T, 1, 4), dtype=torch.float64, device=dev)
    ms_sum, kms_sum, kn_sum = 0.0, 0.0, 0
    traj = None
    for c in mine:
        a0, a1 = c * ca, min(n, (c + 1) * ca)
        nc = a1 - a0
        del traj
        g = torch.Generator(device="cuda")
        g.manual_seed(SEED + 100 + c)                       # chunk c holds the same atoms whatever the rank count
        traj = torch.empty((T, 3, nc), dtype=torch.float64, device=dev)
        cur = torch.rand((3, nc), generator=g, dtype=torch.float64, device=dev) * 215.0
        TB = 250
        for f0 in range(0, T, TB):
            k = min(TB, T - f0)
            blk = torch.randn((k, 3, nc), generator=g, dtype=torch.float64, device=dev).mul_(0.1).cumsum_(0).add_(cur)
            traj[f0:f0 + k] = blk
            cur = blk[-1].clone()
            del blk
        ref = traj[0].contiguous()
        for _ in range(2):
            sums, _ = ops.msd_single_origin(traj, ref, 1e-10)
        torch.cuda.synchronize()
        ctx.timing(True)
        ctx.timing_read(2)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            sums, _ = ops.msd_single_origin(traj, ref, 1e-10)
        e1.record()
        torch.cuda.synchronize()
        ms_sum += e0.elapsed_time(e1)
        kms, kn = ctx.timing_read(2)
        ctx.timing(False)
        kms_sum += kms
        kn_sum += kn
        total += sums
    if world > 1:
        dist.all_reduce(total)                              # atoms are split over ranks: fp64 all-reduce of [T,1,4]
    msd_last = float(total[-1, 0, 0].item()) / n
    ms = ms_sum
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = n * T * steps / (ms * 1e-3)
    kms, kn = kms_sum, kn_sum
    n_local = sum(min(n, (c + 1) * ca) - c * ca for c in mine)
    nfull = n
    n = nc                                                  # the legs below run on the last resident chunk
    # ---- windowed MSD over all time origins (north-star extension): FP64-pipe bound, 2 pipe slots (DADD + DFMA) per
    # (atom, axis, origin, lag); same C3-shaped random walk re-cut as n/4 atoms x 4T frames so that a long window fits
    allo = None
    if not args.skip_msd_window:
        nw, Tw = n, min(T, 1024)
        W = min(args.msd_window, Tw)
        trajw = traj[:Tw]                                         # the first Tw frames of the resident chunk
        outw = torch.zeros((W, 1, 4), dtype=torch.float64, device=dev)
        for _ in range(2):
            ops.msd_all_origins(trajw, W, 1e-10, out=outw)
        torch.cuda.synchronize()
        ctx.timing(True)
        ctx.timing_read(5)
        reps = 3
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record()
        for _ in range(reps):
            ops.msd_all_origins(trajw, W, 1e-10, out=outw)
        w1.record()
        torch.cuda.synchronize()
        msw = w0.elapsed_time(w1) / reps
        kmsw, knw = ctx.timing_read(5)
        ctx.timing(False)
        triples = nw * (W * Tw - W * (W - 1) // 2)                # (atom, origin, lag) with origin + lag < T
        slots = triples * 3 * 2
        peaks_ = measured_peaks()
        pk = peaks_.get("fp64_unfused_tflops_sustained") or 148 * 64 * 1.965e9 / 1e12
        ach = slots / (kmsw / reps * 1e-3) / 1e12
        allo = {"metric": "msd_all_origins_lag_pairs_per_s", "value": world * triples / (msw * 1e-3), "unit": "(atom,origin,lag)/s",
                "config": {"workload": f"{nw} atoms x {Tw} frames resident ({nw * Tw * 24 / 1e9:.1f} GB), window {W} lags"},
                "ms_per_step": msw, "launches_per_step": knw // reps,
                "roofline": {"bound": "fp64", "achieved": ach, "peak": pk, "unit": "T fp64-instr/s", "frac": ach / pk,
                             "traffic": None,
                             "note": "k_msd_window only; 6 FP64 pipe slots (3 DADD + 3 DFMA) per (atom, origin, lag); peak = measured "
                                     "DADD/DMUL issue rate (tools/peaks.cu), which is also the DFMA issue rate"}}
    # end to end: pinned host frames through Diffusion.get_msd_from_arrays
    from mdproptools_b200.dynamical.diffusion import Diffusion
    Te = min(T, 512)
    host = torch.empty((Te, 3, n), dtype=torch.float64, pin_memory=True)
    host.copy_(traj[:Te])
    d = Diffusion(timestep=1, units="real")
    steps_e = np.arange(Te) * 1000
    d.get_msd_from_arrays(host, steps_e, batch_frames=16)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e_reps = 3
    for _ in range(e_reps):
        d.get_msd_from_arrays(host, steps_e, batch_frames=16)
    torch.cuda.synchronize()
    e2e = world * n * Te * e_reps / (time.perf_counter() - t0)        # each rank streams its own atoms: PCIe lanes in parallel
    peaks = measured_peaks()
    hbm = peaks.get("hbm_gbs", 6650.0)
    src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    achieved = n_local * T * steps * MSD_BYTES_PER_ATOM_FRAME / (kms * 1e-3) / 1e9   # this rank's bytes over its kernel time
    cpu = cpu_msd_sample(5.0) if (rank == 0 and not args.skip_cpu) else (None, None, "skipped")
    return {
        "metric": "msd_atom_frames_per_s", "value": value, "unit": "atom-frames/s", "scaling": "strong",
        "config": {"workload": f"C3: {nfull} atoms x {T} frames ({nfull * T * 24 / 1e9:.0f} GB of fp64 coordinates), single-origin MSD "
                               f"(diffusion.py:207-218); resident chunks of {ca} atoms x {T} frames ({ca * T * 24 / 1e9:.1f} GB, "
                               f"generated on the device, {len(mine)} per GPU)", "parallelism": f"atoms x{world}"},
        "ms_per_step": ms / steps, "steps": steps, "msd_last_frame": msd_last, "kernel_launches": kn,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm,
                     "traffic": ncu_traffic("msd_single", n_local * T * steps / max(kn, 1) / (1_000_000 * 64.0)),
                     "peak_source": src, "note": "k_msd_single only; 24 algorithmic bytes per atom-frame; traffic = dram bytes of "
                                                 "the 64-frame launch in profiles/r01e_k_msd_single.txt (1.545 GB for 1.536 GB "
                                                 "algorithmic) scaled to this launch"},
        "e2e": {"value": e2e, "unit": "atom-frames/s", "h2d_bytes_per_step": Te * 3 * n * 8, "d2h_bytes_per_step": Te * 32,
                "api": f"Diffusion.get_msd_from_arrays (pinned host frames; {n} atoms x {Te} frames per rank)"},
        "cpu_baseline": {"value": cpu[0], "unit": "atom-frames/s", "cores": cpu[1], "kind": "port", "sample": cpu[2]},
        "all_origins": allo,
    }


def _timed(ctx, torch, tag, fn, reps):
    """Run fn reps times; return (ms per rep by CUDA events on the current stream, kernel ms per rep from the library's own
    event pairs around kernel `tag`, launches of that kernel per rep)."""
    fn()
    torch.cuda.synchronize()
    ctx.timing(True)
    ctx.timing_read(tag)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    kms, kn = ctx.timing_read(tag)
    ctx.timing(False)
    return e0.elapsed_time(e1) / reps, kms / reps, kn // reps


def bench_green_kubo(args, torch, dist, ops, ctx, dev, world, rank):
    """C4 shape (SURVEY 8d): ionic liquid, 50 000 atoms = 2 500 cations + 2 500 anions of 10 atoms.  (i) charge-flux
    reduction over a resident chunk of velocity frames (HBM-bound, 24 B per atom-frame); (ii) the unbiased time
    correlations of a 100 000-step series: 27 conductivity channels (3 axes x 9 ordered type pairs incl. totals) + 3
    pressure-tensor channels = 30 channels, direct sum in fp64 FMA (FP64-pipe bound: T(T+1)/2 FMAs per channel).
    Channels are split over the ranks."""
    from mdproptools_b200 import dist as mdist
    n, nmol, per = 50_000, 5_000, 10
    Tf_total = args.gk_flux_frames                      # C4: 100 000 frames of velocities = 120 GB, frames split over ranks
    f_lo, f_hi = mdist.shard_range(Tf_total, rank, world)
    CH = 8192                                           # resident chunk: 8192 frames = 9.8 GB, generated on the device
    g = torch.Generator(device="cuda")
    masses = torch.tensor([12.01, 1.008, 14.01, 16.0, 19.0, 32.06, 12.01, 1.008, 16.0, 19.0], dtype=torch.float64, device=dev).repeat(nmol)
    q = torch.cat([torch.full((n // 2,), 0.1, dtype=torch.float64, device=dev), torch.full((n // 2,), -0.1, dtype=torch.float64, device=dev)])
    seg_off = torch.arange(0, n + 1, per, dtype=torch.int32, device=dev)
    type_off = np.array([0, nmol // 2, nmol], dtype=np.int64)
    ms_f = kms_f = 0.0
    kn_f = 0
    reps_f = 3
    vel = None
    flux_sum = 0.0
    for c0f in range(f_lo, f_hi, CH):
        k = min(CH, f_hi - c0f)
        del vel
        vel = torch.empty((k, 3, n), dtype=torch.float64, device=dev)
        GB = 128                                        # the trajectory is defined in blocks of 128 frames seeded by the block
        for b in range(c0f // GB, (c0f + k - 1) // GB + 1):   # index, so it is the same trajectory at every rank count
            g.manual_seed(SEED + 200 + b)
            blk = torch.randn((GB, 3, n), generator=g, dtype=torch.float64, device=dev).mul_(1e-3)
            a0, a1 = max(b * GB, c0f), min((b + 1) * GB, c0f + k)
            vel[a0 - c0f:a1 - c0f] = blk[a0 - b * GB:a1 - b * GB]
            del blk
        out = torch.zeros((3, 2, k), dtype=torch.float64, device=dev)
        # the ABI takes <= 65535 frames per call
        a_, b_, c_ = _timed(ctx, torch, 4, lambda: ops.charge_flux(vel, masses, q, seg_off, type_off, 1e5, 1.602e-19, out=out), reps_f)
        ms_f += a_
        kms_f += b_
        kn_f += c_
        flux_sum += float(out.abs().sum().item())
    del vel
    tf = torch.tensor([ms_f, flux_sum], dtype=torch.float64, device=dev)
    if world > 1:
        tm = tf.clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(tf, op=dist.ReduceOp.SUM)
        ms_f_max, flux_sum = float(tm[0].item()), float(tf[1].item())
    else:
        ms_f_max = ms_f
    peaks = measured_peaks()
    hbm = peaks.get("hbm_gbs", 6650.0)
    Tf = f_hi - f_lo
    flux_gbs = n * Tf * 24 / (kms_f * 1e-3) / 1e9 if kms_f > 0 else 0.0
    T = args.gk_steps
    C_all = 30
    c0, c1 = (rank * C_all) // world, ((rank + 1) * C_all) // world
    C = max(1, c1 - c0)
    a = torch.randn((C, T), generator=g, dtype=torch.float64, device=dev)
    b = torch.randn((C, T), generator=g, dtype=torch.float64, device=dev)
    ms_x, kms_x, kn_x = _timed(ctx, torch, 3, lambda: ops.xcorr_unbiased(a, b), 3)
    t = torch.tensor([ms_x], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_x_max = float(t.item())
    fma = C * T * (T + 1) // 2
    fma_peak = peaks.get("fp64_fma_tflops_burst", 2 * 148 * 64 * 1.965e9 / 1e12)
    ach = 2 * fma / (kms_x * 1e-3) / 1e12
    use_fft = ops.xcorr_fft_enabled(T)
    if use_fft:
        # FFT route (the default at this length): HBM-bound.  Algorithmic bytes = the two input series read once and the
        # correlation written once (24 B per channel-step); the Stockham passes (three stages each) move more: per point of
        # the padded transform 32 B per inner pass, which is what `traffic` states
        p2 = 1
        while (1 << p2) < 2 * T:
            p2 += 1
        passes = -(-p2 // 3)
        alg = C * T * 24
        npts = C * (1 << p2)
        # transform 1: first pass reads the series (16 B per step) and writes 16 B per point, the others 32 B; cross
        # spectrum 48 B (two reads, one write); transform 2: 32 B per pass, the last one reads 16 B and writes the lags
        moved = C * T * 16 + npts * 16 + npts * 32 * (passes - 1) + npts * 48 + npts * 32 * (passes - 1) + npts * 16 + C * T * 8
        gbs = alg / (kms_x * 1e-3) / 1e9
        roof_x = {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm, "traffic": moved,
                  "note": f"mdp_xcorr_fft (all its launches: twiddles, 2 x {passes} passes of three radix-2 stages, cross spectrum); "
                          f"algorithmic bytes = 24 B per channel-step; traffic = bytes the {2 * passes + 1} passes move (computed, "
                          f"not measured: {moved / 1e9:.2f} GB -> {moved / (kms_x * 1e-3) / 1e9:.0f} GB/s); the same job as a direct "
                          f"sum costs {fma:.3g} FMAs ({ach:.0f} TFLOP/s-equivalent at this time)"}
    else:
        roof_x = {"bound": "fp64", "achieved": ach, "peak": fma_peak, "unit": "TFLOP/s", "frac": ach / fma_peak, "traffic": None,
                  "note": "k_xcorr only; 2 flops per fp64 FMA, T(T+1)/2 FMAs per channel; peak = measured DFMA rate "
                          "(tools/peaks.cu); inputs are a few MB, HBM bandwidth is not a meaningful bound here"}
    # the integral on device as well (conductivity.py:231)
    corr = ops.xcorr_unbiased(a, b)
    ms_c, _, _ = _timed(ctx, torch, 7, lambda: ops.cumtrapz(corr, 1.0, 1.0, True), 3)
    return {
        "metric": "acf_lag_products_per_s", "value": C_all * T * (T + 1) // 2 / (ms_x_max * 1e-3), "unit": "fp64 FMA/s",
        "method": "fft (Stockham, three radix-2 stages per pass, fp64)" if use_fft else "direct sum",
        "config": {"workload": f"C4 shape: {C_all} channels x {T} steps, unbiased correlation at every lag, "
                               f"channels x{world}; charge flux on {n} atoms x {Tf_total} frames ({n * Tf_total * 24 / 1e9:.0f} GB, frames "
                               f"x{world}, resident chunks of {CH} frames generated on the device)"},
        "ms_per_step": ms_x_max, "cumtrapz_ms": ms_c,
        "roofline": roof_x,
        "charge_flux": {"value": n * Tf_total / (ms_f_max * 1e-3), "unit": "atom-frames/s", "ms_per_step": ms_f_max, "scaling": "strong",
                        "abs_flux_sum": flux_sum,
                        "roofline": {"bound": "hbm", "achieved": flux_gbs, "peak": hbm, "unit": "GB/s", "frac": flux_gbs / hbm,
                                     "traffic": None, "note": "k_charge_flux only (two molecule types = two launches, each reads "
                                                              "its own molecules); 24 B per atom-frame in total"}},
    }


def bench_residence(args, torch, dist, ops, ctx, dev, world, rank):
    """C5 shape (SURVEY 8d): 2 000 cations and 62 666 water oxygens in a 126 A cubic box, T frames of a random walk;
    residence shell r <= 3.0 A.  (i) neighbour search mdp_pair_list (cations x oxygens per frame, the pair engine in list
    mode) on this rank's block of FRAMES, (ii) the entries are routed to the rank owning the central atom
    (dist.exchange_rows: all-to-all over NVLink), (iii) time bitmasks of the ever-neighbour pairs and survival counts
    cnt[tau] = sum_p popc(m_p & m_p >> tau) for this rank's CENTRAL ATOMS, (iv) int64 all-reduce of cnt."""
    from mdproptools_b200 import dist as mdist
    ncat, nox, L = 2_000, 62_666, 126.0
    T = args.res_frames
    t0, t1 = (rank * T) // world, ((rank + 1) * T) // world
    Tl = t1 - t0
    g = torch.Generator(device="cuda")
    g.manual_seed(SEED + 300)
    cat = torch.empty((Tl, 3, ncat), dtype=torch.float64, device=dev)
    ox = torch.empty((Tl, 3, nox), dtype=torch.float64, device=dev)
    pc = torch.rand((3, ncat), generator=g, dtype=torch.float64, device=dev) * L
    po = torch.rand((3, nox), generator=g, dtype=torch.float64, device=dev) * L
    CH = 250
    for f0 in range(0, T, CH):          # random walk, sigma = 0.15 A per frame, wrapped; every rank walks all T frames
        k = min(CH, T - f0)             # (same seed) and keeps its own block
        sc = torch.randn((k, 3, ncat), generator=g, dtype=torch.float64, device=dev).mul_(0.15).cumsum_(0)
        so = torch.randn((k, 3, nox), generator=g, dtype=torch.float64, device=dev).mul_(0.15).cumsum_(0)
        a0, a1 = max(f0, t0), min(f0 + k, t1)
        if a1 > a0:
            cat[a0 - t0:a1 - t0] = torch.remainder(pc + sc[a0 - f0:a1 - f0], L)
            ox[a0 - t0:a1 - t0] = torch.remainder(po + so[a0 - f0:a1 - f0], L)
        pc, po = pc + sc[-1], po + so[-1]
        del sc, so
    boxes = np.tile(np.array([L, L, L]), (Tl, 1))
    FB = 500                              # frames per search call

    def search():
        parts = []
        for f0 in range(0, Tl, FB):
            lst, _ = ops.pair_list(cat[f0:f0 + FB], ox[f0:f0 + FB], boxes[f0:f0 + FB], 0.0, 9.0, 1, capacity=16 * ncat * FB)
            lst[:, 0] += t0 + f0
            parts.append(lst)
        return torch.cat(parts) if parts else torch.zeros((0, 3), dtype=torch.int32, device=dev)

    holder = {}

    def step():
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record()
        lst = search()
        e[1].record()
        if world > 1:
            lst = mdist.exchange_rows(lst, mdist.owner_of_rows(lst[:, 1], ncat, world))
        e[2].record()
        holder["cnt"], holder["P"] = ops.bitmask_autocorr_from_list(lst.contiguous(), nox, T, n_a=ncat)
        if world > 1:
            dist.all_reduce(holder["cnt"], op=dist.ReduceOp.SUM)
        e[3].record()
        torch.cuda.synchronize()
        holder["entries"] = int(lst.shape[0])
        return [e[i].elapsed_time(e[i + 1]) for i in range(3)]

    step()
    ms_search, ms_x, ms_c = step()
    lst = None
    holder2 = {}
    ent = torch.tensor([holder["entries"], holder["P"]], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(ent, op=dist.ReduceOp.SUM)
    entries_all, P_all = int(ent[0].item()), int(ent[1].item())

    # kernel time of the popcount correlation alone (this rank's central atoms), for the roofline
    lst_local = search()
    if world > 1:
        lst_local = mdist.exchange_rows(lst_local, mdist.owner_of_rows(lst_local[:, 1], ncat, world))
    lst_local = lst_local.contiguous()

    def corr():
        holder2["cnt"], holder2["P"] = ops.bitmask_autocorr_from_list(lst_local, nox, T, n_a=ncat)

    _, kms_c, kn_c = _timed(ctx, torch, 6, corr, 3)
    P = holder2["P"]
    cnt = holder["cnt"]
    W = (T + 63) // 64
    runs = ops.survival_runs_enabled() and T * 8 + 32768 <= 200 * 1024
    if runs:
        # run-based survival counts (csrc/survival.cu): every mask word is read once; the work after that is a few integer
        # updates per pair of runs.  Bound: HBM, algorithmic bytes = the masks (P x W x 8 B)
        alg = P * W * 8
        gbs = alg / (kms_c * 1e-3) / 1e9 if kms_c > 0 else 0.0
        hbm = measured_peaks().get("hbm_gbs", 6650.0)
        roof_r = {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm, "traffic": None,
                  "note": f"k_survival_runs (+ its prefix-sum kernel) only, {kms_c:.3f} ms for this rank's {P} ever-neighbour pairs; "
                          "algorithmic bytes = the time bitmasks read once; the kernel is latency/atomic bound at this size (a few "
                          "hundred thousand pairs), the figure of merit is the time: the AND-shift-popcount kernel it replaces "
                          "needed 48 ms for the same integers"}
    else:
        words = P * sum(W - (tau >> 6) for tau in range(T))            # 64-bit AND+POPC per (pair, lag, word)
        gpop = words / (kms_c * 1e-3) / 1e9
        peak = 148 * 16 * 1.965 / 2                                     # POPC runs at 16 lanes/clk/SM; popcll = 2 POPC
        roof_r = {"bound": "int", "achieved": gpop, "peak": peak, "unit": "G popc64/s", "frac": gpop / peak, "traffic": None,
                  "note": "k_bitmask_autocorr only (this rank's central atoms); one 64-bit AND + POPC per (pair, lag, word); "
                          "peak = nominal XU rate 16 POPC/clk/SM x 148 SMs x 1965 MHz / 2 (popcll = 2 POPC)"}
    # the neighbour search alone (this rank's frames): HBM-bound by design, both coordinate sets read once
    roof_s = None
    if ops.shell_grid_enabled():
        _, kms_s, kn_s = _timed(ctx, torch, 0, search, 2)
        alg_s = Tl * (ncat + nox) * 24
        hbm = measured_peaks().get("hbm_gbs", 6650.0)
        gbs_s = alg_s / (kms_s * 1e-3) / 1e9 if kms_s > 0 else 0.0
        roof_s = {"bound": "hbm", "achieved": gbs_s, "peak": hbm, "unit": "GB/s", "frac": gbs_s / hbm, "traffic": None,
                  "note": f"k_shell_grid only ({kn_s} launches of {FB} frames, {kms_s:.3f} ms for this rank's {Tl} frames); algorithmic "
                          "bytes = 24 B per atom and frame of both sets; the kernel is issue-bound (cell walk + exact fp64 test per "
                          "candidate: profiles/*_k_shell_grid.txt), HBM is the floor it is compared with"}
    t = torch.tensor([ms_search + ms_x + ms_c, ms_search, ms_x, ms_c], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, ms_search, ms_x, ms_c = (float(v) for v in t.tolist())
    return {
        "search_roofline": roof_s,
        "metric": "residence_pair_evals_per_s", "value": ncat * nox * T / (total_ms * 1e-3), "unit": "pair-evals/s",
        "config": {"workload": f"C5 shape: {ncat} cations x {nox} water O x {T} frames, shell r <= 3.0 A, search + bitmask "
                               f"survival correlation at all {T} lags; search: frames x{world}, correlation: central atoms x{world}"},
        "ms_per_step": total_ms, "search_ms": ms_search, "exchange_ms": ms_x, "correlation_ms": ms_c,
        "neighbour_entries": entries_all, "ever_neighbour_pairs": P_all, "cnt0": int(cnt[0].item()),
        "cnt_sha256": __import__("hashlib").sha256(cnt.cpu().numpy().astype(np.int64).tobytes()).hexdigest(),
        "correlation_kernel_ms": kms_c, "correlation_method": "runs (second-difference updates)" if runs else "AND-shift-popcount",
        "roofline": roof_r,
    }


def bench_clusters_hydration(args, torch, dist, ops, ctx, dev, world, rank):
    """C5 (SURVEY 8d), the structural half: 200 000 atoms = 2 000 cations (1 atom) + 2 000 anions (5 atoms) + 62 666 three-site
    waters (O, H, H) in a 126 A cubic box, T frames (default 5 000), molecule centres on a random walk (sigma 0.15 A per frame,
    rigid translation).  Per frame (i) hydration: cation x water-O search inside 3.0 A + the cosine / counter epilogue
    (mdp_hydration_count); (ii) clusters: cation x all-atom search inside 3.0 A + molecule completion and force filter
    (mdp_cluster_members).  STRONG scaling: frames are split over the ranks; a rank walks its frames in resident chunks
    generated on the device (coordinates + forces of 250 frames = 2.4 GB)."""
    from mdproptools_b200 import dist as mdist
    ncat, nan, nwat, L = 2_000, 2_000, 62_666, 126.0
    n = ncat + 5 * nan + 3 * nwat
    nmol = ncat + nan + nwat
    T = args.c5_frames
    t_lo, t_hi = mdist.shard_range(T, rank, world)
    sizes = np.concatenate([np.full(ncat, 1), np.full(nan, 5), np.full(nwat, 3)])
    seg_off = np.concatenate(([0], np.cumsum(sizes))).astype(np.int32)
    mol_of_atom = np.repeat(np.arange(nmol), sizes).astype(np.int32)
    seg_d, moa_d = torch.from_numpy(seg_off).to(dev), torch.from_numpy(mol_of_atom).to(dev)
    moa_l = moa_d.to(torch.int64)
    g = torch.Generator(device="cuda")
    g.manual_seed(SEED + 600)
    centre0 = torch.rand((3, nmol), generator=g, dtype=torch.float64, device=dev) * L
    intra = torch.randn((3, n), generator=g, dtype=torch.float64, device=dev) * 0.55       # fixed offsets inside a molecule
    first = torch.from_numpy(seg_off[:-1].astype(np.int64)).to(dev)
    intra[:, first] = 0.0                                                                   # first atom = molecule centre (O, cation)
    cat_rows = torch.arange(ncat, device=dev)
    o_rows = first[ncat + nan:]
    CH = 250
    GB = 50                                    # the walk is defined in blocks of 50 frames seeded by the block index
    rc2 = 9.0
    ms = {"hyd_search": 0.0, "hyd_epilogue": 0.0, "cl_search": 0.0, "cl_epilogue": 0.0}
    tot = {"hyd_entries": 0, "oriented": 0, "cl_entries": 0, "cl_members": 0, "evaluated": 0}

    def block_steps(b):
        g.manual_seed(SEED + 700 + b)
        return torch.randn((GB, 3, nmol), generator=g, dtype=torch.float64, device=dev).mul_(0.15).cumsum_(0)

    # centre position at the start of this rank's first frame: sum of the whole blocks before it (cheap: one block at a time)
    cur = centre0.clone()
    for b in range(t_lo // GB):
        cur += block_steps(b)[-1]
    for c0 in range(t_lo, t_hi, CH):
        k = min(CH, t_hi - c0)
        cen = torch.empty((k, 3, nmol), dtype=torch.float64, device=dev)
        for b in range(c0 // GB, (c0 + k - 1) // GB + 1):
            st = block_steps(b)
            a0, a1 = max(b * GB, c0), min((b + 1) * GB, c0 + k)
            cen[a0 - c0:a1 - c0] = cur + st[a0 - b * GB:a1 - b * GB]
            if a1 == (b + 1) * GB:
                cur = cur + st[-1]
            del st
        xyz = torch.remainder(cen.index_select(2, moa_l) + intra, L)                      # [k, 3, n] wrapped atom coordinates
        del cen
        g.manual_seed(SEED + 800 + c0)
        force = torch.randn((k, 3, n), generator=g, dtype=torch.float64, device=dev) * 60.0
        boxes = np.tile(np.array([L, L, L]), (k, 1))
        xa = xyz.index_select(2, cat_rows).contiguous()
        xo = xyz.index_select(2, o_rows).contiguous()
        xh1 = xyz.index_select(2, o_rows + 1).contiguous()
        xh2 = xyz.index_select(2, o_rows + 2).contiguous()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        for rep in range(2):                   # first pass warms the arena, second is timed
            ev[0].record()
            lst_h, _ = ops.pair_list(xa, xo, boxes, 0.0, rc2, 0, capacity=8 * ncat * k)
            ev[1].record()
            cos, so_h, cnt_h = ops.hydration_count(lst_h, xa, xo, xh1, xh2, boxes, -0.72)
            ev[2].record()
            lst_c, _ = ops.pair_list(xa, xyz, boxes, 0.0, rc2, 0, capacity=24 * ncat * k)
            ev[3].record()
            so_c, mols, cnt_c = ops.cluster_members(lst_c, ncat, force, seg_d, moa_d, 0.043363 / 16, 0.75)
            ev[4].record()
        torch.cuda.synchronize()
        evs = ctx.pair_stats()["pair_evals"]                      # of the last pair call = the cation x all-atom search
        for name, a, b_ in (("hyd_search", 0, 1), ("hyd_epilogue", 1, 2), ("cl_search", 2, 3), ("cl_epilogue", 3, 4)):
            ms[name] += ev[a].elapsed_time(ev[b_])
        tot["hyd_entries"] += int(lst_h.shape[0])
        tot["oriented"] += int(cnt_h[:, :, 1].sum().item())
        tot["cl_entries"] += int(lst_c.shape[0])
        tot["cl_members"] += int(cnt_c.sum().item())
        tot["evaluated"] += evs
        del xyz, force, xa, xo, xh1, xh2, lst_h, lst_c
    t = torch.tensor([sum(ms.values())] + [ms[k_] for k_ in ("hyd_search", "hyd_epilogue", "cl_search", "cl_epilogue")], dtype=torch.float64,
                     device=dev)
    c = torch.tensor([tot[k_] for k_ in ("hyd_entries", "oriented", "cl_entries", "cl_members", "evaluated")], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(c)
    total_ms, hs, he, cs, ce = (float(v) for v in t.tolist())
    hyd_entries, oriented, cl_entries, cl_members, evaluated = (int(v) for v in c.tolist())
    nominal = T * ncat * (n + nwat)
    peaks = measured_peaks()
    if ops.shell_grid_enabled():
        # both searches run in k_shell_grid (csrc/shell.cu): every coordinate of both sets is read once per frame
        hbm = peaks.get("hbm_gbs", 6650.0)
        alg = T * ((ncat + nwat) + (ncat + n)) * 24 / world
        gbs = alg / ((hs + cs) * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm, "traffic": None,
                "note": "the two neighbour searches (cation x water O, cation x all atoms; k_shell_grid + list allocation) only, "
                        "per GPU: algorithmic bytes = 24 B per atom and frame of both sets over their CUDA-event time; the kernel "
                        "is issue-bound (cell walk + exact fp64 test per candidate), HBM is the floor it is compared with"}
    else:
        pk = peaks.get("fp64_unfused_tflops_sustained") or 148 * 64 * 1.965e9 / 1e12
        ach = evaluated * FLOPS_PER_PAIR / (cs * 1e-3) / 1e12 * (1.0 if world == 1 else 1.0 / world)
        roof = {"bound": "fp64", "achieved": ach, "peak": pk, "unit": "TFLOP/s", "frac": ach / pk, "traffic": None,
                "note": "the cation x all-atom search (k_pair in list mode, all-fp64) only: evaluated pairs x 11 unfused flops over "
                        "its time; the search of 2 000 points against 200 000 is dominated by sorting and culling the large set, "
                        "not by pair arithmetic -- the figure of merit is the time per frame"}
    return {
        "metric": "cluster_hydration_pair_evals_per_s", "value": nominal / (total_ms * 1e-3), "unit": "pair-evals/s", "scaling": "strong",
        "config": {"workload": f"C5: {n} atoms ({ncat} cations, {nan} anions x 5, {nwat} waters x 3) x {T} frames, 126 A box; per frame "
                               f"hydration (cation x water O inside 3.0 A + cosine/counter epilogue) and clusters (cation x all atoms "
                               f"inside 3.0 A + molecule completion + force filter); frames x{world}, resident chunks of {CH} frames"},
        "ms_per_step": total_ms, "hydration_search_ms": hs, "hydration_epilogue_ms": he, "cluster_search_ms": cs,
        "cluster_epilogue_ms": ce, "hydration_entries": hyd_entries, "oriented_waters": oriented, "cluster_entries": cl_entries,
        "cluster_member_molecules": cl_members,
        "roofline": roof,
    }


def bench_c1(torch):
    """Config C1 (SURVEY 8d / BASELINE.md section 2): the reference's own example trajectory, all 101 frames of 10 479 atoms,
    through the reference's entry points calc_atomic_rdf (486 s on one core there) and calc_atomic_cn (534 s).  The frames
    are the git-ignored fixture tests/golden_large/c1_frames.tar.gz (oracle/make_c1_fixture.py); absent -> no leg.  The
    DataFrames are checked against the survey's sha256 known answers of the unmodified reference."""
    import hashlib
    import shutil
    import tarfile
    import tempfile
    from mdproptools_b200.structural import rdf_cn
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "tests", "golden_large", "c1_frames.tar.gz")
    if not os.path.exists(path):
        sys.stderr.write("c1 leg skipped: tests/golden_large/c1_frames.tar.gz is absent (oracle/make_c1_fixture.py)\n")
        return None
    d = tempfile.mkdtemp(prefix="mdp_c1_")
    try:
        with tarfile.open(path) as tf:
            tf.extractall(d)
        pat = os.path.join(d, "dump.nvt.*.dump")
        mass = [16.0, 12.01, 1.008, 14.01, 32.06, 16.0, 12.01, 19.0, 24.305]
        rel = [[9, 9, 9, 9], [1, 4, 6, 9]]
        sha = lambda df: hashlib.sha256(np.ascontiguousarray(df.values, dtype=np.float64).tobytes()).hexdigest()

        def best(fn):
            fn()
            torch.cuda.synchronize()
            ts = []
            for _ in range(3):
                t = time.perf_counter()
                df = fn()
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t)
            return min(ts), df

        t_rdf, df_rdf = best(lambda: rdf_cn.calc_atomic_rdf(20, 0.05, 9, mass, rel, pat, save_mode=False))
        t_cn, df_cn = best(lambda: rdf_cn.calc_atomic_cn([2.325, 4.375, 2.375, 13.0], 0.05, 9, mass, rel, pat, save_mode=False))
        ok_rdf = sha(df_rdf) == "b418f238f5e58393edbe59e8419c8afe1053dada1af6959fa589ce88cfa9ccfc"
        ok_cn = sha(df_cn) == "0ad5461c6508bf07e42aeb21004303b189fbf2a1ed756a2a01fc4ce1b488bb1e"
        return {"metric": "c1_wall_seconds", "unit": "s", "higher_is_better": False, "frames": 101, "atoms": 10479,
                "calc_atomic_rdf_s": t_rdf, "calc_atomic_cn_s": t_cn,
                "published_reference_s": {"calc_atomic_rdf": 486.0, "calc_atomic_cn": 534.0,
                                          "source": "BASELINE.md section 2: one core, numba, other hardware, incl. ~20 s JIT"},
                "vs_published": {"calc_atomic_rdf": 486.0 / t_rdf, "calc_atomic_cn": 534.0 / t_cn},
                "sha256_equals_reference": {"calc_atomic_rdf": ok_rdf, "calc_atomic_cn": ok_cn},
                "api": "rdf_cn.calc_atomic_rdf / calc_atomic_cn(filename=<101 dump files>), warm (best of 3 after one pass)"}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def bench_rdf_from_files(torch, frames, nominal_pairs_per_frame, nfiles=32, copies=8):
    """The call a user of the reference makes: calc_atomic_rdf on LAMMPS dump FILES (C2 frames written as text with
    LAMMPS' default %g, ids shuffled) -> page cache -> pinned TEXT (reader threads) -> H2D on the copy stream -> device
    parser (k_dump_rows) -> pair engine -> D2H -> per-frame normalisation -> DataFrame.  (MDP_DEVICE_PARSE=0: the host
    parser, a batch of frames per call, one frame per host thread -> pinned SoA -> H2D.)"""
    import shutil
    import tempfile
    from mdproptools_b200.structural import rdf_cn
    d = tempfile.mkdtemp(prefix="mdp_bench_dumps_")
    try:
        rng = np.random.default_rng(SEED + 500)
        host = frames[:nfiles].cpu().numpy()
        xy, xz, yz = TILT
        nbytes = 0
        for f in range(host.shape[0]):
            ids = rng.permutation(N_ATOMS) + 1
            x, y, z = host[f][:, ids - 1]
            body = "\n".join(["%d 1 %g %g %g" % t for t in zip(ids.tolist(), x.tolist(), y.tolist(), z.tolist())])
            xlo, xhi = min(0.0, xy, xz, xy + xz), LBOX + max(0.0, xy, xz, xy + xz)
            ylo, yhi = min(0.0, yz), LBOX + max(0.0, yz)
            txt = (f"ITEM: TIMESTEP\n{f * 1000}\nITEM: NUMBER OF ATOMS\n{N_ATOMS}\nITEM: BOX BOUNDS xy xz yz pp pp pp\n"
                   f"{xlo!r} {xhi!r} {xy!r}\n{ylo!r} {yhi!r} {xz!r}\n0.0 {LBOX!r} {yz!r}\nITEM: ATOMS id type x y z\n" + body + "\n")
            nbytes += len(txt)
            with open(os.path.join(d, f"dump.c2.{f * 1000}.dump"), "w") as fh:
                fh.write(txt)
        # 256 files: the 32 generated frames, copied (not linked) 8 times under later timestep names -- formatting 25 million
        # numbers as text in Python is what limits the number of distinct frames, the reader sees 800 MB of text either way
        for c in range(1, copies):
            for f in range(host.shape[0]):
                shutil.copy(os.path.join(d, f"dump.c2.{f * 1000}.dump"), os.path.join(d, f"dump.c2.{(c * host.shape[0] + f) * 1000}.dump"))
        nbytes *= copies
        pat = os.path.join(d, "dump.c2.*.dump")
        # the files were written a moment ago: let the kernel finish writing them back before anything is timed (reads
        # of pages under writeback stall: passes of 0.5 s next to passes of 0.08 s were measured without this), then one
        # untimed pass (pinned buffers, page cache) and the best of three timed ones; the mean is reported beside it
        os.sync()
        rdf_cn.calc_atomic_rdf(R_CUT, BIN, 1, [39.948], [[1], [1]], pat, save_mode=False)
        torch.cuda.synchronize()
        times = []
        for _ in range(3):
            t = time.perf_counter()
            df = rdf_cn.calc_atomic_rdf(R_CUT, BIN, 1, [39.948], [[1], [1]], pat, save_mode=False)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t)
        dt = min(times)
        T = host.shape[0] * copies
        return {"metric": "rdf_pair_evals_per_s", "value": nominal_pairs_per_frame * T / dt, "unit": "pair-evals/s",
                "frames": T, "ms_per_frame": dt / T * 1e3, "ms_per_frame_mean_of_3": sum(times) / 3 / T * 1e3,
                "text_MB_per_s": nbytes / dt / 1e6, "text_bytes": nbytes,
                "g_full_max": float(df["g_full(r)"].max()),
                "df_sha256": __import__("hashlib").sha256(np.ascontiguousarray(df.values, dtype=np.float64).tobytes()).hexdigest(),
                "api": "rdf_cn.calc_atomic_rdf(filename=<dump files>) -- the reference's own entry point (rdf_cn.py:385)",
                "parser": "device (k_dump_rows)" if os.environ.get("MDP_DEVICE_PARSE", "1") not in ("", "0") else "host",
                "note": "text is %g (6 significant digits) as LAMMPS writes by default; files are read from the page cache"}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def bench_dump_parse(reps=3, batch=32):
    """SURVEY 8(f1): the native LAMMPS dump reader (csrc/dump_parse.cpp) on C2-sized frames of text (100 000 atoms,
    columns id type x y z, ids shuffled), all host threads, into id-sorted SoA float64 buffers.  `value` is the pipeline's
    mode: a batch of frames per native call (one frame per thread), numbers written as LAMMPS writes them by default (%g);
    the single-frame call (rows of one frame split over the threads) and 17-digit text (every token misses the exact
    fast path and goes to std::from_chars) are reported beside it."""
    from mdproptools_b200.io import dump as D
    rng = np.random.default_rng(SEED + 400)
    n = N_ATOMS
    ids = rng.permutation(n) + 1
    xyz = rng.uniform(0.0, LBOX, (n, 3))
    head = ["ITEM: TIMESTEP", "1000", "ITEM: NUMBER OF ATOMS", str(n), "ITEM: BOX BOUNDS pp pp pp",
            f"0.0 {LBOX!r}", f"0.0 {LBOX!r}", f"0.0 {LBOX!r}", "ITEM: ATOMS id type x y z"]
    want = ["id", "type", "x", "y", "z"]
    order = np.argsort(ids)

    def text(fmt):
        return ("\n".join(head + [("%d 1 " + fmt + " " + fmt + " " + fmt) % (i, x, y, z)
                                  for i, (x, y, z) in zip(ids.tolist(), xyz.tolist())]) + "\n").encode()

    res = {}
    ok = True
    for name, fmt in (("g", "%g"), ("repr17", "%.17g")):
        buf = text(fmt)
        expect = np.array([float(fmt % v) for v in xyz[order, 0]])
        out = np.empty((batch, 5, n), dtype=np.float64)
        D.parse_frames([buf] * batch, want, out, 0)
        ok = ok and bool(np.array_equal(out[0, 2], expect) and np.array_equal(out[batch - 1, 2], expect))
        t = time.perf_counter()
        for _ in range(reps):
            D.parse_frames([buf] * batch, want, out, 0)
        dt_b = (time.perf_counter() - t) / (reps * batch)
        D.parse_frame(buf, want, 0, out[0])
        ok = ok and bool(np.array_equal(out[0, 2], expect))
        t = time.perf_counter()
        for _ in range(reps):
            D.parse_frame(buf, want, 0, out[0])
        dt_s = (time.perf_counter() - t) / reps
        res[name] = (len(buf), dt_b, dt_s)
    nb, dt_b, dt_s = res["g"]
    nb17, dt_b17, dt_s17 = res["repr17"]
    return {"metric": "dump_parse_MB_per_s", "value": nb / dt_b / 1e6, "unit": "MB/s", "atoms_per_s": n / dt_b,
            "ms_per_frame": dt_b * 1e3, "bytes_per_frame": nb, "frames_per_call": batch, "threads": os.cpu_count(),
            "single_frame_MB_per_s": nb / dt_s / 1e6, "single_frame_atoms_per_s": n / dt_s,
            "repr17_MB_per_s": nb17 / dt_b17 / 1e6, "repr17_atoms_per_s": n / dt_b17, "repr17_bytes_per_frame": nb17,
            "round_trip_exact": ok,
            "note": "host-side parser (text -> id-sorted SoA fp64, correctly rounded = strtod/float()); the reference reads the same "
                    "text through pandas.read_csv + sort_values at ~24 MB/s (SURVEY 8f)"}


DUMP_BYTES_MAX = 64 << 20


def dump_output(d, name, arr):
    """Write `arr` (leading axis = frames) as d/<name>.npy in float64, so that two builds can be compared output for
    output.  Beyond DUMP_BYTES_MAX a fixed, seeded sample of frames is written instead, with the frame indices in
    d/<name>_frames.npy."""
    os.makedirs(d, exist_ok=True)
    a = np.asarray(arr, dtype=np.float64)
    idx = os.path.join(d, f"{name}_frames.npy")
    if os.path.exists(idx):                                        # from an earlier, sampled run into the same DIR
        os.remove(idx)
    if a.nbytes > DUMP_BYTES_MAX:
        k = (DUMP_BYTES_MAX - 4096) // (a[0].nbytes + 8)         # a frame and its index; 4 KB for the two .npy headers
        keep = np.sort(np.random.default_rng(SEED).choice(len(a), k, replace=False))
        np.save(idx, keep.astype(np.float64))
        a = a[keep]
    np.save(os.path.join(d, f"{name}.npy"), a)


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1")
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=8, help="timed steps of the headline RDF loop (passes of the hot path over all frames); the "
                    "secondary legs set their own counts from it (end to end: 3..6, MSD: at least 4)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the per-frame integer RDF histograms of the last step [frames, 2, bins] "
                         "(g_full and the 1-1 relation, 2 per pair as the reference counts) as DIR/rdf_counts.npy, float64")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--port-only", action="store_true", help="reference arm: time only the C port (skip the installed reference)")
    ap.add_argument("--frames", "--frames-per-step", dest="frames", type=int, default=FRAMES_TOTAL,
                    help="frames of the C2 trajectory (the whole job; split over the GPUs)")
    ap.add_argument("--nrank-checks", type=int, default=3, help="N>1: how many other ranks' first frames rank 0 recomputes")
    ap.add_argument("--msd-atoms", type=int, default=MSD_ATOMS)
    ap.add_argument("--msd-frames", type=int, default=MSD_FRAMES)
    ap.add_argument("--skip-msd", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--files-leg", action="store_true", help="run the file-based legs (rdf_from_files, c1) even with --skip-cpu")
    ap.add_argument("--files-copies", type=int, default=8, help="rdf_from_files reads 32 x this many dump files")
    ap.add_argument("--skip-triclinic", action="store_true")
    ap.add_argument("--skip-msd-window", action="store_true")
    ap.add_argument("--msd-window", type=int, default=512)
    ap.add_argument("--skip-gk", action="store_true")
    ap.add_argument("--skip-residence", action="store_true")
    ap.add_argument("--gk-steps", type=int, default=100_000)
    ap.add_argument("--gk-flux-frames", type=int, default=100_000)
    ap.add_argument("--res-frames", type=int, default=5000)
    ap.add_argument("--c5-frames", type=int, default=5000)
    ap.add_argument("--skip-clusters", action="store_true")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's histograms; the reference arm times samples and has none")
    # stdout carries exactly one JSON line (rank 0): anything a library prints there while the bench runs (NCCL's
    # version banner, for one) is sent to stderr instead
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    global _emit
    _emit = lambda line: os.write(real_stdout, (line + "\n").encode())
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
