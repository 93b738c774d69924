"""Einstein / Nernst-Einstein conductivity at the C4 shape: times of its three device stages, with achieved HBM rates.

    python tools/einstein_bench.py [--out profiles/einstein_b200.json] [--frames 100000] [--per-type 2500] [--no-direct]

The trajectory is generated on the device from a fixed seed: 2 x 2500 ten-atom ions (charges +1 and -1 per molecule), T
frames; each molecule's centre moves with an Ornstein-Uhlenbeck velocity, its atoms at fixed offsets around it.  Positions
are integrated chunk by chunk, so the [T][3][50 000] trajectory (120 GB at 10^5 frames) never exists at once.  Timed:

  * dipole   the translational dipole (k_charge_flux on positions, what Conductivity.get_translational_dipole runs),
             from the library's kernel timer; bytes = 24 per atom-frame (positions) + 24 per molecule-frame.
  * einstein_msd   correlate_translational_dipole's call: mdp_cross_msd_fft on 3 (ntypes + 1) = 9 cross channels,
             max_lag = T/2; CUDA events.
  * nernst_msd     the Nernst-Einstein MSD: mdp_cross_msd_fft on [M][3] = 15 000 self channels grouped by type,
             max_lag = T/2 (CUDA events), against mdp_msd_all_origins on the same centres (CUDA events), results compared
             to the accuracy contract (1e-10 of the maximum); in a separate torch.profiler pass the kernel time of the
             FFT passes (k_msd_fft_pass) and their rate at 32 B per point and pass.

Achieved GB/s are bytes computed here over measured time; the card's name and power limit are read in the same run.
Writes nothing unless --out is given.  Needs a GPU: there is no CPU path.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        pl, clk = r.stdout.strip().split(",")[:2]
        info["power_limit_w"], info["sm_max_mhz"] = float(pl), float(clk)
    except Exception as exc:  # noqa: BLE001
        info["power_limit_w"] = f"not read ({exc})"
    return info


def events_ms(fn, reps):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = None
    times = []
    for _ in range(reps):
        e0.record()
        out = fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return out, times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=100_000)
    ap.add_argument("--per-type", type=int, default=2500)
    ap.add_argument("--atoms", type=int, default=10)
    ap.add_argument("--chunk", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--no-direct", action="store_true", help="skip mdp_msd_all_origins (about 10 s at the default shape)")
    ap.add_argument("--out")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("einstein_bench: no CUDA device (there is no CPU path)")
    from mdproptools_b200 import ops
    from mdproptools_b200._lib import Context
    from mdproptools_b200.common import constants as K

    dev = torch.device("cuda", torch.cuda.current_device())
    T, P, A, F = args.frames, args.per_type, args.atoms, args.chunk
    M, N = 2 * P, 2 * P * A
    type_off = np.array([0, P, 2 * P], dtype=np.int64)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234)
    offsets = torch.randn((3, A), generator=gen, device=dev, dtype=torch.float64)
    offsets -= offsets.mean(dim=1, keepdim=True)                        # equal masses: the centre is the molecule's COM
    mol_of_atom = torch.arange(N, device=dev) // A
    atom_off = offsets.repeat(1, M)                                     # [3, N]
    mass = torch.full((N,), 12.0, dtype=torch.float64, device=dev)
    q = torch.full((N,), 0.1, dtype=torch.float64, device=dev)
    q[P * A:] = -0.1                                                    # +1 and -1 per molecule
    seg = torch.arange(0, N + 1, A, dtype=torch.int32, device=dev)
    phi, sig = float(np.exp(-1.0 / 50.0)), 0.02                         # OU velocity: 50-step memory, 0.02 A per step
    x = torch.rand((3, M), generator=gen, device=dev, dtype=torch.float64) * 100.0
    v = torch.randn((3, M), generator=gen, device=dev, dtype=torch.float64) * sig
    com = torch.empty((M, 3, T), dtype=torch.float64, device=dev)      # Nernst-Einstein channels [M][3][T]
    dip = torch.zeros((3, 2, T), dtype=torch.float64, device=dev)
    ctx = Context.get()
    ctx.timing(True)
    ctx.timing_read(4)
    t0 = time.time()
    for f0 in range(0, T, F):
        f1 = min(T, f0 + F)
        noise = torch.randn((f1 - f0, 3, M), generator=gen, device=dev, dtype=torch.float64)
        chunk = torch.empty((f1 - f0, 3, M), dtype=torch.float64, device=dev)
        for k in range(f1 - f0):
            v.mul_(phi).add_(noise[k], alpha=sig * float(np.sqrt(1 - phi * phi)))
            x.add_(v)
            chunk[k] = x
        com[:, :, f0:f1] = chunk.permute(2, 1, 0)
        pos = (chunk[:, :, mol_of_atom] + atom_off[None]).contiguous()  # [F, 3, N]
        ops.charge_flux(pos, mass, q, seg, type_off, K.DISTANCE_CONVERSION["real"], K.CHARGE_CONVERSION["real"], out=dip,
                        frame0=f0)
    torch.cuda.synchronize()
    dip_ms, dip_launches = ctx.timing_read(4)
    gen_s = time.time() - t0
    res = {"card": card(), "shape": {"frames": T, "molecules": M, "atoms": N, "lags": T // 2},
           "generate_s": round(gen_s, 1)}
    dip_bytes = 24.0 * N * T + 24.0 * M * T
    res["dipole"] = {"kernel_ms": dip_ms, "launches": dip_launches, "bytes": dip_bytes, "gbs": dip_bytes / dip_ms / 1e6}

    def fft_bytes(units, groups, nchan, self_case):
        """HBM bytes of one mdp_cross_msd_fft call: (forward passes) 32 B per point and pass over the units' transforms,
        16 B per point of the spectrum accumulation, the inverse transforms (ceil(groups/2), 32 B per point and pass), and
        the reads of the series for the means and the p sums (8 B per point and series)."""
        p = int(np.ceil(np.log2(T + T // 2)))
        n, passes = 1 << p, -(-p // 3)
        fwd = 32.0 * n * units * passes
        return fwd + 16.0 * n * units + 32.0 * n * passes * ((groups + 1) // 2) + \
            8.0 * T * nchan * (1 if self_case else 2) * 2, fwd

    # Einstein: correlate_translational_dipole's 9 channels
    tot = dip[:, 0] + dip[:, 1]
    rows = torch.cat([dip.permute(1, 0, 2), tot[None]], dim=0)         # [3, 3, T]
    a9 = rows.reshape(9, T).contiguous()
    b9 = tot[None].expand(3, 3, T).reshape(9, T).contiguous()
    g9 = np.array([0, 3, 6, 9])
    ops.cross_msd_fft(a9, b9, g9, T // 2)
    _, ms = events_ms(lambda: ops.cross_msd_fft(a9, b9, g9, T // 2), args.reps)
    eb, _ = fft_bytes(9, 3, 9, False)
    res["einstein_msd"] = {"ms": ms, "bytes": eb, "gbs": eb / min(ms) / 1e6}

    # Nernst-Einstein: 15 000 self channels grouped by type
    chans = com.reshape(3 * M, T)
    goff = 3 * type_off
    ops.cross_msd_fft(chans, None, goff, T // 2)
    fft_out, ms = events_ms(lambda: ops.cross_msd_fft(chans, None, goff, T // 2), args.reps)
    nb, fwd = fft_bytes(3 * M // 2, 2, 3 * M, True)
    res["nernst_msd"] = {"fft_ms": ms, "fft_bytes": nb, "fft_gbs": nb / min(ms) / 1e6}
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ops.cross_msd_fft(chans, None, goff, T // 2)
        torch.cuda.synchronize()
    kt = {}
    for e in prof.key_averages():
        m = re.search(r"(k_msd_\w+)", e.key)
        if m:
            kt[m.group(1)] = kt.get(m.group(1), 0.0) + e.device_time_total / 1e3
    res["nernst_msd"]["kernel_ms"] = kt
    if "k_msd_fft_pass" in kt:
        peak = json.load(open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                           "peaks_b200.json")))["stream_read_gbs"]
        p = int(np.ceil(np.log2(T + T // 2)))
        inv = 32.0 * (1 << p) * (-(-p // 3)) * 1                        # one inverse transform (two groups)
        g = (fwd + inv) / kt["k_msd_fft_pass"] / 1e6
        res["nernst_msd"]["fft_pass_gbs"] = g
        res["nernst_msd"]["fft_pass_share_of_stream_read"] = g / peak
        res["nernst_msd"]["stream_read_gbs"] = peak
    if args.no_direct:
        res["nernst_msd"]["direct"] = "not measured"
    else:
        traj = com.permute(2, 1, 0).contiguous()                        # [T, 3, M]
        del com
        sums, ms_d = events_ms(lambda: ops.msd_all_origins(traj, T // 2, 1.0, group_off=type_off), 1)
        direct = (sums[:, :, 3].T / torch.arange(T, T - T // 2, -1, dtype=torch.float64, device=dev)[None]).cpu().numpy()
        got = fft_out.cpu().numpy()
        err = max(float(np.abs(got[g] - direct[g]).max() / np.abs(direct[g]).max()) for g in range(2))
        res["nernst_msd"].update({"direct_ms": ms_d, "speedup": ms_d[0] / min(ms), "max_err_over_max": err,
                                  "within_contract": err < 1e-10})
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
