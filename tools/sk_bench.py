"""Static structure factor (mdp_structure_factor) at the C2 shape: kernel time, terms/s, SASS instructions per term, accuracy.

    python tools/sk_bench.py [--out profiles/sk_b200.json] [--frames 16] [--reps 5]

Frames are generated on the device from a fixed seed: uniform positions in the C2 cell (SURVEY 8d: lx = ly = lz = 167.19 A,
xy = 0.2 lx, xz = 0.1 lx, yz = -0.15 ly), two classes (half the atoms each).  Runs:

  (a) 100 000 atoms, k_max = 3 / A, bin_size = 0.02, max_k_per_bin = 256: the user's case;
  (b) 20 000 atoms in the cell scaled to the same density (97.8 A), every k-vector up to k_max = 2 / A: a long run.

Per run: the k-set's host time, the kernel time from the library's timer (tag 8, the whole call: k_sk_sort, k_sk_rho,
k_sk_bins) and from CUDA events around the call, over warmed repeats; terms/s = frames * N * nk / time; terms per SM and
cycle at the card's maximum SM clock (a lower bound of the per-cycle rate when the clock runs below it).  The static SASS
of k_sk_rho (cuobjdump, when the toolkit is on the PATH) gives the instructions per term: the hot loop holds one
MUFU.SIN and one MUFU.COS per term, which bound it at the guide's 16 MUFU results per clock and SM (8 terms per clock and
SM); the achieved share of that rate is "not measured" (no micro-benchmark of the MUFU rate on this card here).  Accuracy:
on the first frame and a subset of bins, the pair sums against an fp64 direct sum (torch), as the largest ratio of the
deviation to the contract's bound.  The card's name and power limit are read in the same run.  Needs a GPU.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.einstein_bench import card, events_ms  # noqa: E402

C2_L = 167.19


def c2_cell(L):
    return (L, L, L, 0.2 * L, 0.1 * L, -0.15 * L)


def sass_counts():
    """opcode counts of k_sk_rho's static SASS, or None without cuobjdump"""
    from mdproptools_b200 import _lib
    exe = shutil.which("cuobjdump") or ("/usr/local/cuda/bin/cuobjdump" if os.path.exists("/usr/local/cuda/bin/cuobjdump") else None)
    if exe is None:
        return None
    txt = subprocess.run([exe, "-sass", _lib.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
    out, inside = {}, False
    for line in txt.splitlines():
        if "Function :" in line:
            inside = "k_sk_rho" in line
            continue
        m = re.match(r"\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)", line)
        if inside and m:
            out[m.group(1)] = out.get(m.group(1), 0) + 1
    return out


def per_term(ops_count):
    """instructions of the term body per MUFU.SIN (one per term): the phase IMADs, the mantissa LEA.HI, the FADD/FMUL of the
    angle, the range FMUL.RZ, the two MUFUs and the two accumulating FADDs, plus the LDS.128 per atom."""
    if not ops_count or not ops_count.get("MUFU.SIN"):
        return "not measured"
    t = ops_count["MUFU.SIN"]
    body = {k: v for k, v in ops_count.items() if k.split(".")[0] in ("IMAD", "LEA", "FADD", "FMUL", "MUFU", "IADD3", "LDS")}
    return {"terms_in_code": t, "per_term": {k: round(v / t, 3) for k, v in sorted(body.items())},
            "total_per_term": round(sum(body.values()) / t, 2), "mufu_per_term": round((ops_count.get("MUFU.SIN", 0) +
                                                                                         ops_count.get("MUFU.COS", 0)) / t, 2)}


def run(ops, Context, torch, name, n, L, F, k_max, bin_size, max_k, reps, gen, check_bins):
    from mdproptools_b200.structural.structure_factor import kset
    dev = torch.device("cuda", torch.cuda.current_device())
    cell = c2_cell(L)
    H = torch.tensor([[cell[0], cell[3], cell[4]], [0, cell[1], cell[5]], [0, 0, cell[2]]], dtype=torch.float64, device=dev)
    s = torch.rand((F, n, 3), generator=gen, device=dev, dtype=torch.float64)
    xyz = (s @ H.T).permute(0, 2, 1).contiguous()                         # [F, 3, n]
    cls = (torch.arange(n, device=dev) % 2).to(torch.int32)
    t0 = time.time()
    miller, bin_off = kset(cell, k_max, bin_size, max_k_per_bin=max_k)
    kset_s = time.time() - t0
    nbins = len(bin_off) - 1
    nk = int(bin_off[-1])
    ctx = Context.get()
    ctx.timing(True)

    def call():
        return ops.structure_factor(xyz, cls, 2, cell, miller, bin_off, nbins)
    call()
    torch.cuda.synchronize()
    ctx.timing_read(8)
    out, ev = events_ms(call, reps)
    tag_ms, tag_n = ctx.timing_read(8)
    ctx.timing(False)
    terms = float(F) * n * nk
    best = min(ev)
    res = {"atoms": n, "frames": F, "cell": cell, "k_max": k_max, "bin_size": bin_size, "max_k_per_bin": max_k, "nk": nk,
           "kset_host_s": round(kset_s, 3), "event_ms": ev, "tag8_ms_mean": tag_ms / max(tag_n, 1), "tag8_calls": tag_n,
           "terms_per_call": terms, "terms_per_s": terms / best * 1e3}
    # accuracy: first frame, a subset of bins, against an fp64 direct sum
    got = out[0].cpu().numpy()
    K = 2 * np.pi * np.linalg.inv(H.cpu().numpy()).T
    bins = [b for b in check_bins if b < nbins]
    worst, worst_rel = 0.0, 0.0
    x0 = xyz[0].T                                                          # [n, 3]
    for b in bins:
        m = miller[bin_off[b]:bin_off[b + 1]]
        if len(m) == 0:
            continue
        kv = torch.from_numpy(m.astype(np.float64) @ K.T).to(dev)          # [nb, 3]
        re = torch.zeros((2, len(m)), dtype=torch.float64, device=dev)
        im = torch.zeros_like(re)
        for c in range(2):
            ph = kv @ x0[cls == c].T                                       # [nb, n_c]
            re[c], im[c] = torch.cos(ph).sum(1), torch.sin(ph).sum(1)
        amp = torch.hypot(re, im)
        for row, (a, bb) in enumerate([(0, 0), (0, 1), (1, 1)]):
            want = float((re[a] * re[bb] + im[a] * im[bb]).sum())
            na, nb_ = float((cls == a).sum()), float((cls == bb).sum())
            bound = float((1e-5 * (na * amp[bb] + nb_ * amp[a]) + 1e-10 * na * nb_).sum())
            d = abs(got[row, b] - want)
            worst = max(worst, d / bound)
            worst_rel = max(worst_rel, d / max(abs(want), 1e-300))
    res["accuracy"] = {"bins_checked": bins, "max_dev_over_contract_bound": float(worst), "max_rel_dev": float(worst_rel),
                       "within_contract": bool(worst <= 1.0)}
    print(name, json.dumps(res)[:400], flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--frames-b", type=int, default=32)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sk_bench: no CUDA device (there is no CPU path)")
    from mdproptools_b200 import ops
    from mdproptools_b200._lib import Context

    dev = torch.device("cuda", torch.cuda.current_device())
    gen = torch.Generator(device=dev)
    gen.manual_seed(20261)
    info = card()
    props = torch.cuda.get_device_properties(dev)
    res = {"card": info, "sms": props.multi_processor_count}
    res["a_user_case"] = run(ops, Context, torch, "a", 100_000, C2_L, args.frames, 3.0, 0.02, 256, args.reps, gen,
                             [5, 6, 40, 149])
    L_b = C2_L * (20_000 / 100_000) ** (1 / 3)
    res["b_full_kset"] = run(ops, Context, torch, "b", 20_000, L_b, args.frames_b, 2.0, 0.02, None, max(2, args.reps), gen,
                             [5, 50, 99])
    ops_count = sass_counts()
    res["sass_k_sk_rho"] = per_term(ops_count)
    res["bound"] = ("two MUFU results per term (MUFU.SIN, MUFU.COS); at the CUDA guide's 16 per clock and SM that is at most "
                    "8 terms per clock and SM; share of the card's MUFU rate: not measured")
    clk = info.get("sm_max_mhz")
    for key in ("a_user_case", "b_full_kset"):
        r = res[key]
        r["terms_per_sm_clock_at_max_clock"] = (r["terms_per_s"] / (res["sms"] * clk * 1e6)) if isinstance(clk, float) else "not measured"
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
