"""Coherent intermediate scattering function at a user's shape: the rho stage (mdp_sk_rho, tag 8) and the FFT stage
(mdp_isf_fft, tag 9) timed separately, with the deviation from a direct sum on a few bins.

    python tools/isf_bench.py [--out profiles/isf_b200.json] [--frames 2000] [--reps 3]

A trajectory is generated on the device from a fixed seed: 20 000 atoms in 3 classes (N/2, 3N/10, N/5) in a triclinic cell at
the density of SURVEY 8d's C2 (L = 97.8 A, xy = 0.2 L, xz = 0.1 L, yz = -0.15 L), each atom a random walk of 0.05 A per
axis and frame.  k_max = 3 / A, bin_size = 0.02, max_k_per_bin = 64, T frames (default 2000), max_lag = T / 2; pairs: the
total with itself and the three class pairs (0,0), (0,1), (1,2) -- the shape of calc_intermediate_scattering with three
relations.

  rho stage   mdp_sk_rho over all frames, in chunks of 250 frames, straight into the [4, nk, T] series: terms/s =
              T * N * nk / time, next to mdp_structure_factor's measured 1.9e12 (profiles/sk_b200.json);
  FFT stage   mdp_isf_fft: bytes moved by the passes = 32 B per point and pass * ceil(p/3) passes * (forward transforms
              nk * 4 + inverse transforms nbins * ceil(4/2)), over time, next to the data sheet's 7.7 TB/s HBM read stream
              (a comparison of scale, not a share of a measured peak);
  accuracy    on a few bins, every pair against an fp64 direct sum (torch) of the same rho: the largest deviation over
              max_tau |direct sum| per (pair, bin), against the contract's 1e-10.
Times from the library's timer tags and from CUDA events around each stage, over warmed repeats; the card's name and power
limit are read in the same run.  Needs a GPU.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.einstein_bench import card, events_ms  # noqa: E402

SK_TERMS_PER_S = 1.9e12
HBM_BYTES_PER_S = 7.7e12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--atoms", type=int, default=20_000)
    ap.add_argument("--frames", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("isf_bench: no CUDA device (there is no CPU path)")
    from mdproptools_b200 import ops
    from mdproptools_b200._lib import Context
    from mdproptools_b200.structural.structure_factor import kset

    dev = torch.device("cuda", torch.cuda.current_device())
    gen = torch.Generator(device=dev)
    gen.manual_seed(20262)
    n, T = args.atoms, args.frames
    L = 167.19 * (n / 100_000) ** (1 / 3)
    cell = (L, L, L, 0.2 * L, 0.1 * L, -0.15 * L)
    H = torch.tensor([[cell[0], cell[3], cell[4]], [0, cell[1], cell[5]], [0, 0, cell[2]]], dtype=torch.float64, device=dev)
    x0 = torch.rand((n, 3), generator=gen, device=dev, dtype=torch.float64) @ H.T
    steps = torch.randn((T, n, 3), generator=gen, device=dev, dtype=torch.float64) * 0.05
    xyz = (x0[None] + torch.cumsum(steps, dim=0)).permute(0, 2, 1).contiguous()            # [T, 3, n]
    del steps
    cls = torch.zeros(n, dtype=torch.int32, device=dev)
    cls[n // 2:] = 1
    cls[n // 2 + 3 * n // 10:] = 2
    ncls = 3
    t0 = time.time()
    miller, bin_off = kset(cell, 3.0, 0.02, max_k_per_bin=64)
    kset_s = time.time() - t0
    nk, nbins = int(bin_off[-1]), len(bin_off) - 1
    nlags = T // 2
    pairs = [(3, 3), (0, 0), (0, 1), (1, 2)]
    ctx = Context.get()
    rho = torch.empty((ncls + 1, nk, T), dtype=torch.complex128, device=dev)

    def rho_stage():
        for f0 in range(0, T, 250):
            ops.sk_rho(xyz[f0:f0 + 250], cls, ncls, cell, miller, out=rho, frame0=f0)
        rho[ncls] = rho[0] + rho[1] + rho[2]
        return rho

    def fft_stage():
        return ops.isf_fft(rho, pairs, bin_off, nlags)

    rho_stage()
    out = fft_stage()
    torch.cuda.synchronize()
    ctx.timing(True)
    for tag in (8, 9):
        ctx.timing_read(tag)
    _, ev_rho = events_ms(rho_stage, args.reps)
    tag8_ms, tag8_n = ctx.timing_read(8)
    out, ev_fft = events_ms(fft_stage, args.reps)
    tag9_ms, tag9_n = ctx.timing_read(9)
    ctx.timing(False)

    terms = float(T) * n * nk
    rho_ms = tag8_ms / args.reps                      # the sk_rho calls of one stage (the total-channel sum excluded)
    p = max(1, math.ceil(math.log2(T + nlags)))
    N = 1 << p
    passes = math.ceil(p / 3)
    transforms = nk * 4 + nbins * math.ceil(len(pairs) / 2)
    fft_bytes = 32.0 * N * passes * transforms
    fft_ms = tag9_ms / max(tag9_n, 1)
    res = {"card": card(), "atoms": n, "frames": T, "cell": cell, "classes": ncls, "k_max": 3.0, "bin_size": 0.02,
           "max_k_per_bin": 64, "nk": nk, "nbins": nbins, "nlags": nlags, "pairs": pairs, "kset_host_s": round(kset_s, 3),
           "rho_stage": {"event_ms": ev_rho, "tag8_ms_per_stage": rho_ms, "tag8_calls": tag8_n, "terms": terms,
                         "terms_per_s": terms / rho_ms * 1e3, "sk_kernel_terms_per_s_measured": SK_TERMS_PER_S},
           "fft_stage": {"event_ms": ev_fft, "tag9_ms_mean": fft_ms, "tag9_calls": tag9_n, "N": N, "passes_per_transform": passes,
                         "transforms": transforms, "pass_bytes": fft_bytes, "pass_bytes_per_s": fft_bytes / fft_ms * 1e3,
                         "hbm_read_stream_bytes_per_s_datasheet": HBM_BYTES_PER_S,
                         "note": "pass bytes only; the spectrum accumulation and loads are extra traffic"}}
    # accuracy: a few bins, every pair, against an fp64 direct sum of the same rho
    got = out.cpu().numpy()
    worst = 0.0
    checked = [b for b in (5, 40, 100, nbins - 1) if 0 <= b < nbins and bin_off[b + 1] > bin_off[b]]
    for b in checked:
        z = rho[:, bin_off[b]:bin_off[b + 1]]
        for q, (a, c) in enumerate(pairs):
            want = torch.empty(nlags, dtype=torch.float64, device=dev)
            for tau in range(nlags):
                m = T - tau
                s = (z[a, :, tau:] * z[c, :, :m].conj()).real.sum() + (z[c, :, tau:] * z[a, :, :m].conj()).real.sum()
                want[tau] = 0.5 * s / m
            w = want.cpu().numpy()
            worst = max(worst, float(np.abs(got[q, b] - w).max() / np.abs(w).max()))
    res["accuracy"] = {"bins_checked": checked, "max_dev_over_max_abs": worst, "contract": 1e-10, "within_contract": worst <= 1e-10}
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
