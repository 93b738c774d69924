"""Reorientation at a user's shape: the channel kernel (mdp_orient_series), the grouped FFT autocorrelation after it, and
accuracy.

    python tools/reorient_bench.py [--out profiles/reorient_b200.json] [--waters 20000] [--frames 10000] [--batch 500]

The trajectory is generated on the device from a fixed seed: rigid three-site waters (O-H 0.9572 A, H-O-H 104.52 deg) in
a triclinic cell, each spinning about its own random axis at its own rate (0.01-0.2 rad per frame) with its centre fixed,
wrapped into the cell.  Three definitions (O-H bond, H-O-H bisector, plane normal) give 3 x 8 x M channels of T frames
(4.8e5 x 1e4 x 8 B = 38 GB at the default shape); the positions are generated and consumed batch by batch, as the file
pipeline delivers them, and not kept.  Timed:

  * orient     every batch's three mdp_orient_series calls, warmed up: the library's kernel timer (tag 11) and CUDA events
               around the whole stream; bytes = per vector and frame 24 B per atom read (2 for a bond, 3 otherwise) and
               64 B written, over the tag-11 time, and that rate as a share of a device-to-device copy (read + write of
               4 GiB, best of 5) measured in the same run.
  * acf        one mdp_group_acf_fft call over the whole buffer with the (3 M, 5 M) groups of each definition, T/2 lags:
               tag 10 and CUDA events.
  * accuracy   the first 16 lags of C1 and C2 of a 512-molecule subset of each definition from the FFT against a direct
               fp64 sum of P_l(u(t).u(t+tau)) over every origin, from the same channels (which checks the channel identity
               and the correlator); and every lag of the whole result against the closed form of a rigid rotor,
               C1 = <cos^2 th + sin^2 th cos(w tau)>, C2 = <P2(that)>.

The card's name and power limit are read in the same run.  Writes nothing unless --out is given.  Needs a GPU.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.einstein_bench import card, events_ms  # noqa: E402

CELL = (84.0, 83.0, 82.0, 2.0, 1.0, 0.5)
DEFS = (("bond", 0, (0, 1, 0)), ("bisector", 1, (0, 1, 2)), ("normal", 2, (0, 1, 2)))


def rodrigues(axis, ang):
    """rotation matrices [..., 3, 3]; axis [..., 3] unit, ang [...]"""
    import torch
    K = torch.zeros(axis.shape[:-1] + (3, 3), dtype=axis.dtype, device=axis.device)
    K[..., 0, 1], K[..., 0, 2], K[..., 1, 2] = -axis[..., 2], axis[..., 1], -axis[..., 0]
    K = K - K.transpose(-1, -2)
    s, c = torch.sin(ang)[..., None, None], torch.cos(ang)[..., None, None]
    return torch.eye(3, dtype=axis.dtype, device=axis.device) + s * K + (1 - c) * K @ K


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--waters", type=int, default=20_000)
    ap.add_argument("--frames", type=int, default=10_000)
    ap.add_argument("--batch", type=int, default=500)
    ap.add_argument("--out")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("reorient_bench: no CUDA device (there is no CPU path)")
    from mdproptools_b200 import ops
    from mdproptools_b200._lib import Context

    dev = torch.device("cuda", torch.cuda.current_device())
    M, T, B = args.waters, args.frames, args.batch
    L = T // 2
    f64 = dict(dtype=torch.float64, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(2024)
    lx, ly, lz, xy, xz, yz = CELL
    H = torch.tensor([[lx, xy, xz], [0.0, ly, yz], [0.0, 0.0, lz]], **f64)
    Hinv = torch.linalg.inv(H)
    centre = torch.rand((M, 3), generator=gen, **f64) @ H.T
    axis = torch.randn((M, 3), generator=gen, **f64)
    axis /= axis.norm(dim=1, keepdim=True)
    omega = 0.01 + 0.19 * torch.rand((M,), generator=gen, **f64)
    half = math.radians(104.52) / 2
    body = torch.tensor([[0.0, 0.0, 0.0], [0.9572 * math.sin(half), 0.0, 0.9572 * math.cos(half)],
                         [-0.9572 * math.sin(half), 0.0, 0.9572 * math.cos(half)]], **f64)
    q0 = rodrigues(torch.nn.functional.normalize(torch.randn((M, 3), generator=gen, **f64), dim=1),
                   2 * math.pi * torch.rand((M,), generator=gen, **f64))
    body = torch.einsum("mij,sj->msi", q0, body)                                  # [M, 3 sites, 3]

    def frames(f0, f1):
        """[f1 - f0, 3, 3 M] wrapped positions, atom id order (molecule-major)"""
        t = torch.arange(f0, f1, **f64)
        R = rodrigues(axis[None], omega[None] * t[:, None])                        # [F, M, 3, 3]
        r = torch.einsum("fmij,msj->fmsi", R, body) + centre[None, :, None, :]
        s = r @ Hinv.T
        r = (s - torch.floor(s)) @ H.T
        return r.reshape(f1 - f0, 3 * M, 3).permute(0, 2, 1).contiguous()

    rows = [np.ascontiguousarray(3 * np.arange(M)[:, None] + np.array(a)[None, :], dtype=np.int32) for _, _, a in DEFS]
    res = {"card": card(), "shape": {"waters": M, "atoms": 3 * M, "frames": T, "lags": L, "definitions": len(DEFS),
                                     "channels": 8 * M * len(DEFS), "batch_frames": B}}
    buf = torch.empty((8 * M * len(DEFS), T), **f64)
    res["shape"]["channel_buffer_gb"] = buf.numel() * 8 / 1e9
    cells = np.tile(np.array(CELL), (T, 1))

    def orient(x, f0):
        for d, (_, kind, _) in enumerate(DEFS):
            ops.orient_series(x, cells[f0:f0 + x.shape[0]], kind, rows[d], buf[8 * M * d:8 * M * (d + 1)].view(8, M, T), f0)

    ctx = Context.get()
    orient(frames(0, B), 0)                                                          # warm-up
    torch.cuda.synchronize()
    ctx.timing(True)
    ctx.timing_read(11)
    ev_ms = 0.0
    for f0 in range(0, T, B):
        x = frames(f0, min(T, f0 + B))
        _, ms = events_ms(lambda: orient(x, f0), 1)
        ev_ms += ms[0]
        del x
    tag_ms, tag_n = ctx.timing_read(11)
    nbytes = float(T) * M * sum(24 * (2 if kind == 0 else 3) + 64 for _, kind, _ in DEFS)
    src = torch.ones((1 << 29,), **f64)                                              # 4 GiB
    dst = torch.empty_like(src)
    dst.copy_(src)
    _, cms = events_ms(lambda: dst.copy_(src), 5)
    copy_gbs = 2 * src.numel() * 8 / min(cms) / 1e6
    del src, dst
    torch.cuda.empty_cache()
    res["orient"] = {"tag11_ms": tag_ms, "tag11_launches": tag_n, "event_ms": ev_ms, "bytes": nbytes,
                     "gbs": nbytes / tag_ms / 1e6, "copy_gbs": copy_gbs, "share_of_copy": nbytes / tag_ms / 1e6 / copy_gbs}

    goff = np.concatenate(([0], np.cumsum([k * M for _ in DEFS for k in (3, 5)]))).astype(np.int64)
    ops.group_acf_fft(buf[:8], [0, 3, 8], L)                                          # module load, off the timed call
    torch.cuda.synchronize()
    ctx.timing_read(10)
    sums, ams = events_ms(lambda: ops.group_acf_fft(buf, goff, L), 2)
    t10_ms, t10_n = ctx.timing_read(10)
    ctx.timing(False)
    res["acf"] = {"event_ms": ams, "tag10_ms_per_call": t10_ms / max(t10_n, 1), "lags": L}
    sums = sums.cpu().numpy()

    # accuracy: a 512-molecule subset, FFT against the direct sum of P_l over every origin (first 16 lags)
    S, K = 512, 16
    acc = {}
    for d, (name, _, _) in enumerate(DEFS):
        blk = buf[8 * M * d:8 * M * (d + 1)].view(8, M, T)[:, :S]
        sub = ops.group_acf_fft(blk.contiguous().view(8 * S, T), [0, 3 * S, 8 * S], K).cpu().numpy()
        u = blk[:3]
        x = [(u[:, :, k:] * u[:, :, :T - k]).sum(dim=0) for k in range(K)]
        c1 = torch.stack([xx.mean() for xx in x]).cpu().numpy()
        c2 = torch.stack([(1.5 * xx * xx - 0.5).mean() for xx in x]).cpu().numpy()
        acc[name] = {"c1_fft_vs_direct": float(np.abs(sub[0] / S - c1).max()),
                     "c2_fft_vs_direct": float(np.abs(1.5 * sub[1] / S - c2).max())}
    # the whole result against the rigid-rotor closed form
    tau = torch.arange(L, **f64)
    w0 = {"bond": body[:, 1] - body[:, 0], "bisector": (body[:, 1] + body[:, 2]) / 2 - body[:, 0],
          "normal": torch.linalg.cross(body[:, 1] - body[:, 0], body[:, 2] - body[:, 0])}
    for d, (name, _, _) in enumerate(DEFS):
        c = (w0[name] * axis).sum(dim=1) / w0[name].norm(dim=1)
        xx = c[:, None] ** 2 + (1 - c[:, None] ** 2) * torch.cos(omega[:, None] * tau[None, :])      # [M, L]
        e1 = np.abs(sums[2 * d] / M - xx.mean(dim=0).cpu().numpy()).max()
        e2 = np.abs(1.5 * sums[2 * d + 1] / M - (1.5 * xx * xx - 0.5).mean(dim=0).cpu().numpy()).max()
        acc[name].update({"c1_vs_closed_form_all_lags": float(e1), "c2_vs_closed_form_all_lags": float(e2)})
    worst = max(v for a in acc.values() for v in a.values())
    res["accuracy"] = {"subset_molecules": S, "direct_lags": K, "max_abs_err": acc, "within_1e-10": worst < 1e-10}
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
