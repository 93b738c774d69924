"""Velocity autocorrelation at a user's shape: the grouped FFT autocorrelation, the gather and transpose before it, and
accuracy.

    python tools/vacf_bench.py [--out profiles/vacf_b200.json] [--atoms 100000] [--frames 10000] [--reps 3]

The velocities are generated on the device from a fixed seed: 10^5 atoms in 3 types (every third atom), T frames of
Ornstein-Uhlenbeck velocities (20-frame memory), nlags = T/2, so 3 * 10^5 channels in 9 (type, axis) groups and
transforms of N = 2^14 points at the default shape.  Timed:

  * gather     what Diffusion.get_vacf does to the parsed velocities: the index_select of the atoms into group order
               ([T][3][N]) and the transpose into [3 N][T] channels; CUDA events.
  * acf        one mdp_group_acf_fft call, warmed up: the library's kernel timer (tag 10) and CUDA events; in a separate
               torch.profiler pass the time of the FFT passes (k_fft_pass), their bytes (32 per point and pass of the forward
               and inverse transforms) over that time, and that rate as a share of the read stream measured in the same run
               (a torch sum over 4 GiB, best of 5).
  * accuracy   the first lags of a few groups against an fp64 direct sum on the device, over out[g][0].

The card's name and power limit are read in the same run.  Writes nothing unless --out is given.  Needs a GPU.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.einstein_bench import card, events_ms  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--atoms", type=int, default=100_000)
    ap.add_argument("--frames", type=int, default=10_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("vacf_bench: no CUDA device (there is no CPU path)")
    from mdproptools_b200 import ops
    from mdproptools_b200._lib import Context

    dev = torch.device("cuda", torch.cuda.current_device())
    N, T = args.atoms, args.frames
    L = T // 2
    gen = torch.Generator(device=dev)
    gen.manual_seed(4321)
    phi, sig = float(np.exp(-1.0 / 20.0)), 1e-2
    vel = torch.empty((T, 3, N), dtype=torch.float64, device=dev)        # as the parser leaves it: [T][3][N], id order
    vel[0] = torch.randn((3, N), generator=gen, device=dev, dtype=torch.float64) * sig
    for t in range(1, T):
        vel[t] = vel[t - 1] * phi + torch.randn((3, N), generator=gen, device=dev, dtype=torch.float64) * (sig * np.sqrt(1 - phi * phi))
    types = np.arange(N) % 3
    members = [np.nonzero(types == k)[0] for k in range(3)]
    sel = torch.from_numpy(np.concatenate(members)).to(dev)
    nloc = [len(m) for m in members]
    goff = np.concatenate(([0], np.cumsum(np.repeat(nloc, 3)))).astype(np.int64)
    res = {"card": card(), "shape": {"atoms": N, "types": 3, "frames": T, "lags": L, "channels": 3 * N, "groups": 9}}

    def gather():
        v = vel.index_select(2, sel)
        chans = torch.empty((3 * N, T), dtype=torch.float64, device=dev)
        s0 = 0
        for n in nloc:
            chans[3 * s0:3 * (s0 + n)].view(3, n, T).copy_(v[:, :, s0:s0 + n].permute(1, 2, 0))
            s0 += n
        return chans

    gather()
    chans, ms = events_ms(gather, args.reps)
    gbytes = 8.0 * T * 3 * N * 4                                           # read + write of the gather and of the transpose
    res["gather"] = {"ms": ms, "bytes": gbytes, "gbs": gbytes / min(ms) / 1e6}
    del vel
    torch.cuda.empty_cache()

    ctx = Context.get()
    ctx.timing(True)
    ops.group_acf_fft(chans, goff, L)
    torch.cuda.synchronize()
    ctx.timing_read(10)
    out, ms = events_ms(lambda: ops.group_acf_fft(chans, goff, L), args.reps)
    tag_ms, tag_n = ctx.timing_read(10)
    ctx.timing(False)
    p = int(np.ceil(np.log2(T + L)))
    n, passes = 1 << p, -(-p // 3)
    units = sum((c + 1) // 2 for c in np.repeat(nloc, 3))
    pass_bytes = 32.0 * n * passes * (units + (9 + 1) // 2)
    total = pass_bytes + 16.0 * n * units
    res["acf"] = {"N": n, "passes_per_transform": passes, "forward_transforms": int(units), "event_ms": ms,
                  "tag10_ms_per_call": tag_ms / max(tag_n, 1), "bytes": total, "gbs": total / min(ms) / 1e6}
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ops.group_acf_fft(chans, goff, L)
        torch.cuda.synchronize()
    kt = {}
    for e in prof.key_averages():
        m = re.search(r"(k_(?:msd|fft)_\w+)", e.key)
        if m:
            kt[m.group(1)] = kt.get(m.group(1), 0.0) + e.device_time_total / 1e3
    res["acf"]["kernel_ms"] = kt
    buf = torch.ones((1 << 29,), dtype=torch.float64, device=dev)        # 4 GiB
    buf.sum()
    _, rms = events_ms(lambda: buf.sum(), 5)
    stream = buf.numel() * 8 / min(rms) / 1e6
    del buf
    res["stream_read_gbs"] = stream
    if "k_fft_pass" in kt:
        g = pass_bytes / kt["k_fft_pass"] / 1e6
        res["acf"]["fft_pass_gbs"] = g
        res["acf"]["fft_pass_share_of_stream_read"] = g / stream

    # accuracy: the first 64 lags of groups 0, 4 and 8 against an fp64 direct sum on the device
    errs = {}
    for g in (0, 4, 8):
        a = chans[goff[g]:goff[g + 1]]
        want = torch.stack([(a[:, k:] * a[:, :T - k]).sum() / (T - k) for k in range(64)]).cpu().numpy()
        got = out[g, :64].cpu().numpy()
        errs[str(g)] = float(np.abs(got - want).max() / abs(out[g, 0].item()))
    res["accuracy"] = {"lags": 64, "max_err_over_out0": errs, "within_contract": max(errs.values()) < 1e-10}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
