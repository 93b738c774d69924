"""CPU-only tests (no GPU): the C-ABI library loads and exports every declared symbol, the host-side logic
(dump parser, bin-edge table, type remapping, class weights, normalisation, sharding) agrees with the oracle
and with golden outputs of the reference.  No compute entry point is called."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as O
from tests.conftest import MASS, NUM_ATOMS, NUM_MOLS, ROOT


def test_abi_exports_every_declared_symbol():
    from mdproptools_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "mdprop_b200.h")).read()
    declared = set(re.findall(r"\b(mdp_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.EXPORTED_SYMBOLS)
    lib = _lib.lib()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.mdp_version() == 100


def test_product_never_imports_the_oracle():
    bad = []
    for dirpath, _, files in os.walk(os.path.join(ROOT, "mdproptools_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                if re.search(r"^\s*(from|import)\s+oracle\b", txt, re.M) or "liboracle" in txt:
                    bad.append(f)
    assert not bad, bad


def test_no_cuda_means_loud_failure():
    import torch
    if torch.cuda.is_available():
        # the same check in a process that sees no device
        code = ("import pytest\nfrom mdproptools_b200._lib import Context, MdpropError\n"
                "with pytest.raises(MdpropError, match='no CPU fallback'):\n    Context.get()\n")
        r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""},
                           capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        return
    from mdproptools_b200._lib import Context, MdpropError
    with pytest.raises(MdpropError, match="no CPU fallback"):
        Context.get()


def test_bin_edges_define_the_reference_bin_function():
    from mdproptools_b200._lib import bin_edges
    rng = np.random.default_rng(1)
    for ddr, nb in [(0.05, 400), (0.07, 104), (0.1, 3), (0.05, 46), (0.3, 7)]:
        e = bin_edges(ddr, nb)
        assert e[0] == 0 and np.all(np.diff(e) > 0)
        rsq = np.concatenate([rng.uniform(0, (nb * ddr) ** 2 * 1.02, 100000), e[1:], np.nextafter(e[1:], 0),
                              np.nextafter(e[1:], np.inf)])
        ref = np.minimum((np.sqrt(rsq) / ddr).astype(np.int64), nb)       # rdf_cn.py:68,85
        assert np.array_equal(np.searchsorted(e[1:], rsq, side="right"), ref)


def test_native_parser_matches_oracle_reader(sample_dir, mini_dir):
    from mdproptools_b200.io import dump as D
    for pat, cols in ((os.path.join(sample_dir, "dump.nvt.*.dump"), ["id", "type", "x", "y", "z", "fx", "q", "iz"]),
                      (os.path.join(mini_dir, "dump.mini.*.dump"), ["id", "xu", "yu", "zu", "vx", "mass"])):
        got = list(D.read_dumps(pat, cols, nthreads=3))
        ref = list(O.read_dumps(pat))
        assert [g.timestep for g in got] == [r.timestep for r in ref]
        for g, r in zip(got, ref):
            c = r.sorted_by_id()
            assert g.natoms == r.natoms
            assert g.box.lattice_lengths() == r.lattice_lengths and g.box.bound_lengths() == r.bound_lengths
            for k in cols:
                assert np.array_equal(g.data[k], c[k]), k


def test_batch_parser_equals_single_frame_parser(sample_dir):
    """mdp_dump_parse_batch (one frame per thread, rows written straight to id - 1) against mdp_dump_parse, which the
    previous test pins to the oracle reader: real sample frames, sizes around the store pipeline depth, ids that are not
    a permutation of 1..N (ranking path), blank lines, number spellings on and off the exact fast path, and errors."""
    from mdproptools_b200.io import dump as D
    want = ["id", "type", "x", "y", "z"]
    bufs = [open(os.path.join(sample_dir, f), "rb").read() for f in sorted(os.listdir(sample_dir)) if f.endswith(".dump")]
    n = D.parse_frame(bufs[0], want).natoms
    out = np.full((len(bufs) * 6, len(want), n), np.nan)
    frames = D.parse_frames(bufs * 6, want, out, nthreads=4)          # 12 frames >= threads / 2: frame-parallel mode
    for k, fr in enumerate(frames):
        ref = D.parse_frame(bufs[k % len(bufs)], want, nthreads=1)
        assert fr.timestep == ref.timestep and fr.box.lattice_lengths() == ref.box.lattice_lengths()
        for c in want:
            assert np.array_equal(fr.data[c], ref.data[c]), (k, c)
    rng = np.random.default_rng(2)
    spell = [lambda v: repr(float(v)), lambda v: "%g" % v, lambda v: "%.17g" % v, lambda v: "%+.3e" % v, lambda v: "%.12f" % v,
             lambda v: ("%f" % v).rstrip("0"), lambda v: "%.25f" % v, lambda v: "%dE0" % int(v)]
    for nn, shift, blank in [(1, 0, False), (15, 0, False), (16, 0, True), (17, 0, False), (33, 0, False), (64, 5, False),
                             (200, 0, True)]:
        ids = rng.permutation(nn) + 1 + shift
        xyz = rng.normal(0, 30, (nn, 3))
        rows = ["%d %d %s %s %s" % (i, 1 + i % 3, spell[i % 8](x), spell[(i + 3) % 8](y), spell[(i + 5) % 8](z))
                for i, (x, y, z) in zip(ids.tolist(), xyz.tolist())]
        if blank:
            rows.insert(len(rows) // 2, "   ")
        txt = ("ITEM: TIMESTEP\n7\nITEM: NUMBER OF ATOMS\n%d\nITEM: BOX BOUNDS pp pp pp\n0 9\n0 9\n0 9\nITEM: ATOMS id type x y z\n"
               % nn + "\n".join(rows) + "\n").encode()
        ref = D.parse_frame(txt, want, nthreads=1)
        py = np.array([[float(t) for t in r.split()] for r in rows if r.strip()])
        py = py[np.argsort(py[:, 0], kind="stable")]
        out = np.full((8, 5, nn), np.nan)
        for fr in D.parse_frames([txt] * 8, want, out, nthreads=4):
            for k, c in enumerate(want):
                assert np.array_equal(fr.data[c], ref.data[c]) and np.array_equal(fr.data[c], py[:, k]), (nn, c)
    bad = txt.replace(b" 1 ", b" x ", 1)
    with pytest.raises(RuntimeError):
        D.parse_frames([txt, bad] * 4, want, np.empty((8, 5, nn)), nthreads=4)
    short = txt[: txt.rstrip().rfind(b"\n") + 1]
    with pytest.raises(RuntimeError):
        D.parse_frames([short] * 8, want, np.empty((8, 5, nn)), nthreads=4)


def test_parser_numbers_equal_python_float():
    """Every spelling the parser accepts must give the double Python's float() gives (correctly rounded): random decimal
    strings around the limits of the exact fast path -- 1 to 25 digits, the point anywhere, exponents from -30 to 30,
    signs, leading zeros -- through both entry points (rows of one frame split over threads / one frame per thread)."""
    from mdproptools_b200.io import dump as D
    rng = np.random.default_rng(77)
    toks = []
    for _ in range(30000):
        nd = int(rng.integers(1, 26))
        digits = "".join(rng.choice(list("0123456789"), nd))
        pos = int(rng.integers(0, nd + 1))
        body = digits[:pos] + ("." if rng.uniform() < 0.8 else "") + digits[pos:] if pos < nd or rng.uniform() < 0.5 else digits + "."
        if body in (".", ""):
            body = "0."
        if body.startswith(".") and rng.uniform() < 0.3:
            body = "0" + body
        if rng.uniform() < 0.35:
            body += rng.choice(["e", "E"]) + rng.choice(["", "+", "-"]) + str(int(rng.integers(0, 31)))
        toks.append(rng.choice(["", "-", "+"]) + ("000" if rng.uniform() < 0.05 else "") + body)
    toks += ["0", "-0", "-0.0", "9007199254740992", "9007199254740993", "9007199254740993.", "0.000000000000000000000001",
             "1e22", "1e23", "1e-22", "1e-23", "123456789012345678901234567890", "4.9e-324", "1.7976931348623157e308"]
    n = len(toks)
    want = np.array([float(t) for t in toks])
    txt = ("ITEM: TIMESTEP\n0\nITEM: NUMBER OF ATOMS\n%d\nITEM: BOX BOUNDS pp pp pp\n0 1\n0 1\n0 1\nITEM: ATOMS id x\n" % n
           + "\n".join("%d %s" % (i + 1, t) for i, t in enumerate(toks)) + "\n").encode()
    for nthreads in (1, 3):
        got = D.parse_frame(txt, ["id", "x"], nthreads=nthreads).data["x"]
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), toks[int(np.flatnonzero(got.view(np.uint64) != want.view(np.uint64))[0])]
    out = np.empty((8, 2, n))
    for fr in D.parse_frames([txt] * 8, ["id", "x"], out, nthreads=4):
        assert np.array_equal(fr.data["x"].view(np.uint64), want.view(np.uint64))


def test_frame_batches_pipeline_on_host(tmp_path):
    """FrameBatches without a device: batching by atom count and by the frame cap, frame_select (rank sharding), global
    frame indices, total_frames, and the pinned-buffer ring -- more batches than ring slots, with a deliberately slow
    consumer, must still hand every batch over intact."""
    import time as _t
    from mdproptools_b200.io import dump as D
    from mdproptools_b200.io.pipeline import FrameBatches
    rng = np.random.default_rng(4)
    sizes = [7] * 9 + [5] * 3 + [7] * 11
    p = tmp_path / "traj.dump"
    with open(p, "w") as f:
        for t, n in enumerate(sizes):
            ids = rng.permutation(n) + 1
            xyz = rng.normal(0, 5, (n, 3))
            f.write(f"ITEM: TIMESTEP\n{t * 5}\nITEM: NUMBER OF ATOMS\n{n}\nITEM: BOX BOUNDS pp pp pp\n0 9\n0 9\n0 9\n")
            f.write("ITEM: ATOMS id type x y z\n")
            for i, (x, y, z) in zip(ids, xyz):
                f.write(f"{i} {1 + i % 2} {x:.6g} {y:.6g} {z:.6g}\n")
    want = ["id", "type", "x", "y", "z"]
    ref = list(D.read_dumps(str(p), want, nthreads=1))
    assert len(ref) == len(sizes)
    for sel in (None, lambda i: i % 2 == 1):
        fb = FrameBatches(str(p), want, max_batch_frames=2, to_device=False, frame_select=sel, prefetch=2)
        seen = []
        for batch in fb:
            assert batch.dev is None and batch.ready is None
            n = batch.metas[0].natoms
            assert all(m.natoms == n for m in batch.metas) and len(batch.metas) <= 2
            _t.sleep(0.01)                               # the producer runs ahead and cycles through its ring meanwhile
            host = batch.host.numpy()
            assert host.shape == (len(batch.metas), len(want), n)
            for k, m in enumerate(batch.metas):
                assert m.timestep == ref[m.index].timestep
                for c, name in enumerate(want):
                    assert np.array_equal(host[k, c], ref[m.index].data[name]), (m.index, name)
                seen.append(m.index)
        assert fb.total_frames == len(sizes)
        assert seen == [i for i in range(len(sizes)) if sel is None or sel(i)]


def _atoms_section(buf: bytes):
    a = buf.index(b"ITEM: ATOMS")
    return buf.index(b"\n", a) + 1


def test_device_parser_body_on_host(sample_dir, tmp_path):
    """The body of the device dump parser, mdp_parse_chunk of csrc/dump_rows.h, run on the host for every
    (frame, chunk) in both orders against the host parser: real sample frames (20 columns, 8 wanted), generated frames
    with row lengths around the 64-byte chunk size, CRLF and blank lines; and its refusals -- tokens off the exact fast
    path, short rows, duplicate / out-of-range ids, a wrong row count -- which the caller answers with the host parser."""
    import ctypes
    from mdproptools_b200.io import dump as D
    so = tmp_path / "dump_rows_host.so"
    src = os.path.join(ROOT, "tests", "native", "dump_rows_host.cpp")
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-fno-fast-math", "-o", str(so), src], check=True)
    emu = ctypes.CDLL(str(so)).emulate_dump_rows
    LL, I = ctypes.c_longlong, ctypes.c_int

    def run(bufs, want, reverse):
        cols = D.frame_columns(bufs[0])
        n = int(bufs[0].split(b"\n")[3])                            # the line after ITEM: NUMBER OF ATOMS
        text = b"".join(bufs)
        begin, end, off = [], [], 0
        for b in bufs:
            begin.append(off + _atoms_section(b))
            end.append(off + len(b))
            off += len(b)
        colsel = [want.index(c) if c in want else -1 for c in cols]
        F = len(bufs)
        out = np.full((F, len(want), n), np.nan)
        seen = np.zeros((F, (n + 31) // 32), dtype=np.uint32)
        status = np.zeros((F, 2), dtype=np.uint64)
        rc = emu(I(F), text, (LL * F)(*begin), (LL * F)(*end), LL(n), I(len(cols)), (I * len(cols))(*colsel), I(cols.index("id")),
                 I(len(want)), out.ctypes.data_as(ctypes.c_void_p), LL(len(want) * n), LL(n), seen.ctypes.data_as(ctypes.c_void_p),
                 status.ctypes.data_as(ctypes.c_void_p), I(1 if reverse else 0))
        assert rc == 0
        return out, status, n

    want = ["id", "type", "x", "y", "z", "fx", "q", "iz"]
    bufs = [open(os.path.join(sample_dir, f), "rb").read() for f in sorted(os.listdir(sample_dir)) if f.endswith(".dump")]
    for reverse in (False, True):
        out, status, n = run(bufs, want, reverse)
        assert status[:, 0].tolist() == [n] * len(bufs) and status[:, 1].tolist() == [0] * len(bufs)
        for f, b in enumerate(bufs):
            ref = D.parse_frame(b, want, nthreads=1)
            for k, c in enumerate(want):
                assert np.array_equal(out[f, k], ref.data[c]), (f, c)

    rng = np.random.default_rng(8)
    head = "ITEM: TIMESTEP\n3\nITEM: NUMBER OF ATOMS\n%d\nITEM: BOX BOUNDS pp pp pp\n0 9\n0 9\n0 9\nITEM: ATOMS id type x y z extra\n"
    fmts = ["%.3f", "%.6g", "%.10f", "%.12f", "%d.", "%.1f"]
    for nn, eol, pad in [(1, "\n", 0), (3, "\n", 40), (50, "\r\n", 0), (200, "\n", 17), (333, "\n", 64), (64, "\n", 128)]:
        ids = rng.permutation(nn) + 1
        xyz = rng.normal(0, 40, (nn, 3))
        rows = []
        for i, (x, y, z) in zip(ids.tolist(), xyz.tolist()):
            f1, f2, f3 = fmts[i % 6], fmts[(i + 2) % 6], fmts[(i + 4) % 6]
            rows.append(" " * (i % 3) + "%d %d %s %s  %s %s" % (i, 1 + i % 4, f1 % x, f2 % y, f3 % z, "p" * (pad + 1 + i % 5)))
        rows.insert(nn // 2, "  ")                                   # a blank line
        buf = ((head % nn).replace("\n", eol) + eol.join(rows) + eol).encode()
        if nn == 3:
            buf = buf.rstrip()                                        # last row without a line end
        want5 = ["x", "id", "z", "type", "y"]
        ref = D.parse_frame(buf, want5, nthreads=1)
        for reverse in (False, True):
            out, status, n = run([buf, buf], want5, reverse)
            assert status.tolist() == [[nn, 0], [nn, 0]], (nn, status)
            for k, c in enumerate(want5):
                assert np.array_equal(out[0, k], ref.data[c]) and np.array_equal(out[1, k], ref.data[c]), (nn, c)

    good = ((head % 4) + "1 1 0.5 1.5 2.5 a\n2 1 0.25 1 2 a\n3 2 7 8 9 a\n4 2 1 1 1 a\n").encode()
    cases = {
        "exponent beyond 10^22": (good.replace(b"0.25", b"2.5e-30"), 1),   # DPF_SLOW_TOKEN
        "digits": (good.replace(b"0.25", b"0.12345678901234567890123"), 1),
        "nan": (good.replace(b"0.25", b"nan"), 1),
        "short row": (good.replace(b"3 2 7 8 9 a", b"3 2 7"), 2),      # DPF_BAD_ROW
        "duplicate id": (good.replace(b"4 2 1 1 1", b"3 2 1 1 1"), 4),  # DPF_BAD_ID
        "id out of range": (good.replace(b"4 2 1 1 1", b"9 2 1 1 1"), 4),
    }
    # exponents inside the exact range stay on the device (%g writes them for |x| < 1e-4)
    out, status, _ = run([good.replace(b"0.25", b"2.5e-1"), good.replace(b"0.25", b"-1.25E-05")], ["id", "x", "y", "z"], False)
    assert status.tolist() == [[4, 0], [4, 0]] and out[0, 1, 1] == 0.25 and out[1, 1, 1] == float("-1.25E-05")
    for name, (buf, flag) in cases.items():
        _, status, _ = run([good, buf], ["id", "x", "y", "z"], False)
        assert status[0].tolist() == [4, 0], name
        assert int(status[1, 1]) & flag, (name, status)
    fewer = good[: good.rstrip().rfind(b"\n") + 1]                    # 3 rows where the header announces 4
    _, status, _ = run([fewer], ["id", "x"], False)
    assert status[0].tolist() == [3, 0]                              # rows != natoms: the caller rejects the frame


def test_survival_counts_from_runs_on_host(tmp_path):
    """The run-based survival correlation (csrc/survival_runs.h: run extraction from the time bitmask + four
    second-difference updates per run pair + two prefix sums) against the oracle's direct sum: random indicators of
    every density, runs touching both ends, trajectories that are / are not a multiple of 64 frames, empty and full
    masks.  Integer counts, equal bit for bit."""
    import ctypes
    so = tmp_path / "survival_runs_host.so"
    src = os.path.join(ROOT, "tests", "native", "survival_runs_host.cpp")
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", str(so), src], check=True)
    emu = ctypes.CDLL(str(so)).emulate_survival_runs
    emu.restype = ctypes.c_int
    rng = np.random.default_rng(12)

    def check(h, cap=None):
        T, P = h.shape
        W = (T + 63) // 64
        bits = np.zeros((P, W * 64), dtype=np.uint8)
        bits[:, :T] = h.T
        masks = np.packbits(bits.reshape(P, W, 64), axis=2, bitorder="little").view(np.uint64).reshape(P, W)
        masks = np.ascontiguousarray(masks)
        cnt = np.zeros(T, dtype=np.int64)
        k = emu(masks.ctypes.data_as(ctypes.c_void_p), ctypes.c_longlong(P), ctypes.c_int(W), ctypes.c_longlong(T),
                ctypes.c_int(cap or T // 2 + 2), cnt.ctypes.data_as(ctypes.c_void_p))
        assert np.array_equal(cnt, O.survival_counts(h)), (T, P)
        return k

    for T in (1, 2, 63, 64, 65, 127, 128, 200, 321, 1023, 1025, 2500):
        for dens in (0.02, 0.3, 0.5, 0.9):
            check((rng.uniform(size=(T, 7)) < dens).astype(np.uint8))
        # persistent neighbours: long runs with a few flips, as a residence shell produces them
        walk = np.cumsum(rng.normal(0, 0.4, (T, 9)), axis=0) + rng.normal(0, 1, 9)
        check((np.abs(walk) < 1.0).astype(np.uint8))
        check(np.zeros((T, 2), dtype=np.uint8))
        check(np.ones((T, 3), dtype=np.uint8))
        edge = np.zeros((T, 4), dtype=np.uint8)
        edge[0, 0] = 1; edge[T - 1, 1] = 1; edge[0, 2] = edge[T - 1, 2] = 1; edge[T // 2:, 3] = 1
        check(edge)
    assert check((np.arange(300)[:, None] % 2 == 0).astype(np.uint8)) == 150      # alternating bits: T/2 runs
    # a run buffer that is too small for some pairs: those take the word route (AND-shift-popcount), the sum is the same
    for T in (64, 129, 500):
        assert check((rng.uniform(size=(T, 11)) < 0.5).astype(np.uint8), cap=8) > 8


def test_shell_grid_search_on_host(tmp_path):
    """The small-set neighbour search (csrc/shell_grid.h: periodic cell grid over A as a conservative filter, the
    reference's own rsq arithmetic as the test) against the oracle's all-pairs shell mask: wrapped and unwrapped
    coordinates, points on the box faces, pairs planted exactly on the shell radii, radii close to a third of the box,
    both shell modes, same-set exclusion.  Every pair is found exactly once."""
    import ctypes
    so = tmp_path / "shell_grid_host.so"
    src = os.path.join(ROOT, "tests", "native", "shell_grid_host.cpp")
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-o", str(so), src], check=True)
    emu = ctypes.CDLL(str(so)).emulate_shell_grid
    emu.restype = ctypes.c_int
    D = ctypes.c_double
    dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    rng = np.random.default_rng(31)

    def check(A, B, L, r_in, r_out, mode, same):
        A = [np.ascontiguousarray(v, dtype=np.float64) for v in A]
        B = [np.ascontiguousarray(v, dtype=np.float64) for v in B]
        na, nb = len(A[0]), len(B[0])
        out = np.zeros((na, nb), dtype=np.uint8)
        Lc = np.asarray(L, dtype=np.float64)
        rc = emu(dp(A[0]), dp(A[1]), dp(A[2]), na, dp(B[0]), dp(B[1]), dp(B[2]), nb, dp(Lc), D(O.rcut_sq(r_in)), D(O.rcut_sq(r_out)),
                 mode, 1 if same else 0, out.ctypes.data_as(ctypes.c_void_p))
        if rc != 0:
            return False
        if mode:
            want = O.shell_mask(A[0], A[1], A[2], B[0], B[1], B[2], L, r_in, r_out, same)
        else:
            rsq = np.stack([O.calc_rsq([A[0][i], A[1][i], A[2][i]], B[0], B[1], B[2], L) for i in range(na)])
            want = (rsq < O.rcut_sq(r_out)).astype(np.uint8)
            if same:
                want[np.arange(min(na, nb)), np.arange(min(na, nb))] = 0
        assert np.array_equal(out, want), (na, nb, L, r_out, mode)
        return True

    L = (21.0, 19.5, 23.25)
    for na, nb in [(1, 50), (40, 900), (300, 300), (7, 5000)]:
        a = rng.uniform(0, 1, (3, na)) * np.asarray(L)[:, None]
        b = rng.uniform(0, 1, (3, nb)) * np.asarray(L)[:, None]
        for r_in, r_out in [(0.0, 3.0), (1.5, 4.0), (0.0, 6.4)]:              # 6.4: three cells on the short axis
            assert check(a, b, L, r_in, r_out, 1, False)
            assert check(a, b, L, r_in, r_out, 0, False)
        # unwrapped coordinates (several box lengths away, both signs) and a shifted origin
        shift_a = rng.integers(-3, 4, (3, na)) * np.asarray(L)[:, None]
        shift_b = rng.integers(-3, 4, (3, nb)) * np.asarray(L)[:, None]
        assert check(a + shift_a + 100.0, b + shift_b + 100.0, L, 0.0, 3.0, 1, False)
    # same set, self pairs excluded (residence_time.py:103-104)
    a = rng.uniform(0, 1, (3, 400)) * np.asarray(L)[:, None]
    assert check(a, a, L, 0.0, 3.5, 1, True) and check(a, a, L, 0.0, 3.5, 0, True)
    # points on the faces and pairs planted exactly at the radii (<= r_out counts in shell mode, < r_out does not in mode 0)
    a = np.array([[0.0, 21.0, 10.5, 0.0], [0.0, 0.0, 19.5, 9.75], [0.0, 23.25, 0.0, 23.25]])
    b = np.concatenate([a + np.array([[3.0], [0.0], [0.0]]), a - np.array([[0.0], [3.0], [0.0]]),
                        a + np.array([[0.0], [0.0], [1.5]]), a + 1e-13, rng.uniform(0, 20, (3, 50))], axis=1)
    assert check(a, b, L, 1.5, 3.0, 1, False) and check(a, b, L, 0.0, 3.0, 0, False)
    # a radius beyond a third of the shortest box length: the grid does not apply
    assert not check(a, b, L, 0.0, 7.0, 1, False)


def test_fft_correlation_on_host(tmp_path):
    """The FFT route of the unbiased correlation (csrc/fft_corr.h: Stockham butterflies, three stages per pass, both spectra from one
    transform of a + i*b, second transform of the conjugated cross spectrum) against the oracle's long-double direct sum
    and the reference's numpy-FFT form: cross- and auto-correlation, lengths around powers of two, fewer lags than
    steps.  Tolerance: the north star's 1e-10 of max|C| (observed ~1e-15)."""
    import ctypes
    so = tmp_path / "fft_corr_host.so"
    src = os.path.join(ROOT, "tests", "native", "fft_corr_host.cpp")
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-o", str(so), src], check=True)
    lib = ctypes.CDLL(str(so))
    emu = lib.emulate_fft_xcorr
    emu.restype = ctypes.c_int
    dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    rng = np.random.default_rng(51)
    # three stages per pass (mdp_fft_radix_pass) are, bit for bit, three radix-2 stages: every log2 size up to 2^13,
    # which covers every mix of radix-8, radix-4 and radix-2 passes
    lib.fft_fused_vs_radix2.restype = ctypes.c_longlong
    for p in range(1, 14):
        re, im = rng.normal(0, 1, 1 << p), rng.normal(0, 1, 1 << p)
        assert lib.fft_fused_vs_radix2(dp(re), dp(im), ctypes.c_int(p)) == 0, p
    worst = 0.0
    for T in (1, 2, 3, 7, 8, 9, 100, 255, 256, 257, 1000, 4097):
        for same in (False, True):
            a = np.cumsum(rng.normal(0, 1, T)) * 0.1 + rng.normal(0, 1, T)
            b = a if same else rng.normal(0, 2, T) + 0.5
            for nlags in sorted({T, max(1, T // 3)}):
                out = np.empty(nlags)
                emu(dp(a), dp(b), ctypes.c_longlong(T), ctypes.c_longlong(nlags), dp(out))
                want = O.xcorr_direct(a, b)[:nlags]
                scale = np.abs(want).max() + 1e-300
                err = np.abs(out - want).max() / scale
                worst = max(worst, err)
                assert err < 1e-10, (T, same, nlags, err)
                if T > 1:
                    assert np.abs(out - O.correlate_fft(a, b)[:nlags]).max() / scale < 1e-10
    assert worst < 1e-12


def test_parser_multiframe_triclinic_and_ragged(tmp_path):
    from mdproptools_b200.io import dump as D
    rng = np.random.default_rng(0)
    p = tmp_path / "traj.dump"
    frames = []
    with open(p, "w") as f:
        for t, n in enumerate([5, 9, 1]):
            ids = rng.permutation(n) + 1 + (10 if t == 1 else 0)         # frame 1: ids not contiguous from 1
            xyz = rng.normal(0, 5, (n, 3))
            f.write(f"ITEM: TIMESTEP\n{t * 10}\nITEM: NUMBER OF ATOMS\n{n}\n")
            f.write("ITEM: BOX BOUNDS xy xz yz pp pp pp\n-1.0 11.5 2.0\n0.0 10.0 1.0\n0.5 9.5 -1.5\n")
            f.write("ITEM: ATOMS id type x y z\n")
            for i, (x, y, z) in zip(ids, xyz):
                f.write(f"{i} {1 + i % 2} {float(x)!r} {y:.9e} {z:+.5f}\n")
            frames.append((ids, xyz))
    got = list(D.read_dumps(str(p), ["id", "x", "y", "z"]))
    ref = list(O.read_dumps(str(p)))
    assert len(got) == 3
    for g, r, (ids, xyz) in zip(got, ref, frames):
        c = r.sorted_by_id()
        for k in ("id", "x", "y", "z"):
            assert np.array_equal(g.data[k], c[k])
        assert np.array_equal(g.data["id"], np.sort(ids))
        assert g.box.tilt == [2.0, 1.0, -1.5]
        # pymatgen's tilt correction of the bounds and the row norms of the cell matrix
        assert np.allclose(np.array(g.box.bounds), r.bounds, rtol=0, atol=0)
        assert g.box.lattice_lengths() == r.lattice_lengths
    with pytest.raises(KeyError):
        list(D.read_dumps(str(p), ["id", "vx"]))


def test_parser_errors(tmp_path):
    from mdproptools_b200 import _lib
    from mdproptools_b200.io import dump as D
    p = tmp_path / "bad.dump"
    p.write_text("ITEM: TIMESTEP\n0\nITEM: NUMBER OF ATOMS\n3\nITEM: BOX BOUNDS pp pp pp\n0 1\n0 1\n0 1\n"
                 "ITEM: ATOMS id x\n1 0.5\n2 abc\n3 0.1\n")
    with pytest.raises(_lib.MdpropError, match="cannot parse"):
        list(D.read_dumps(str(p), ["id", "x"]))
    q = tmp_path / "short.dump"
    q.write_text("ITEM: TIMESTEP\n0\nITEM: NUMBER OF ATOMS\n3\nITEM: BOX BOUNDS pp pp pp\n0 1\n0 1\n0 1\n"
                 "ITEM: ATOMS id x\n1 0.5\n")
    with pytest.raises(_lib.MdpropError, match="announces 3 atoms"):
        list(D.read_dumps(str(q), ["id", "x"]))


def test_frame_batches_host_only(sample_dir):
    from mdproptools_b200.io.pipeline import FrameBatches
    fb = FrameBatches(os.path.join(sample_dir, "dump.nvt.*.dump"), ["id", "x"], to_device=False, max_batch_frames=1)
    batches = list(fb)
    assert fb.total_frames == 2 and len(batches) == 2
    assert [b.metas[0].timestep for b in batches] == [0, 2500000]
    assert batches[0].host.shape == (1, 2, 10479)
    only_second = list(FrameBatches(os.path.join(sample_dir, "dump.nvt.*.dump"), ["id"], to_device=False,
                                    frame_select=lambda i: i == 1))
    assert len(only_second) == 1 and only_second[0].metas[0].index == 1


def test_calc_atom_type_ids_matches_oracle():
    from mdproptools_b200.structural.rdf_cn import calc_atom_type_ids
    n = sum(a * b for a, b in zip(NUM_MOLS, NUM_ATOMS))
    ids = np.arange(1, n + 6, dtype=np.float64)          # a few ids beyond the last block stay untouched
    assert np.array_equal(calc_atom_type_ids(ids, NUM_MOLS, NUM_ATOMS), O.calc_atom_type(ids, NUM_MOLS, NUM_ATOMS))


def test_class_maps_and_weights_reproduce_reference_counting():
    """Derive full/partial histograms from a class-pair histogram built on the CPU and compare with _rdf_loop."""
    from mdproptools_b200 import ops
    from mdproptools_b200.structural.rdf_cn import _ClassMap, _sym_weights
    rng = np.random.default_rng(3)
    n, L = 400, (12.0, 13.0, 11.0)
    pos = rng.uniform(0, 1, (3, n)) * np.asarray(L)[:, None]
    typ = rng.integers(1, 6, n).astype(np.float64)
    rel = [[5, 5, 2, 1], [1, 5, 2, 3]]
    relm = np.asarray(rel).T
    nb, ddr, rc = 50, 0.1, 5.0
    full, part = O.rdf_loop(typ, pos[0], pos[1], pos[2], relm, L, rc, ddr, nb)
    cmap = _ClassMap(rel[0] + rel[1])
    cls = cmap.classes_of(typ)
    assert cmap.ncls == 5 and set(cls[typ == 4]) == {cmap.other}
    rows = ops.sym_rows(cmap.ncls)
    H = np.zeros((rows, nb), dtype=np.int64)
    for c1 in range(cmap.ncls):
        for c2 in range(c1, cmap.ncls):
            a, b = cls == c1, cls == c2
            if c1 == c2:
                f, _ = O.rdf_loop(np.ones(a.sum()), pos[0][a], pos[1][a], pos[2][a], [[1, 1]], L, rc, ddr, nb)
                H[ops.sym_row(c1, c2, cmap.ncls)] = f // 2
            else:
                p = O.rdf_rect(np.ones(a.sum()), pos[0][a], pos[1][a], pos[2][a], np.ones(b.sum()), pos[0][b], pos[1][b],
                               pos[2][b], [[1, 1]], L, rc, ddr, nb)
                H[ops.sym_row(c1, c2, cmap.ncls)] = p[0]
    w = _sym_weights(cmap, relm, with_full=True)
    red = w @ H
    assert np.array_equal(red[0], full) and np.array_equal(red[1:], part)


def test_host_normalisation_is_bit_identical_to_reference(sample_dir, gold_structural):
    """Feed the reference's own raw counts through the product's host normalisation."""
    from mdproptools_b200.io import dump as D
    from mdproptools_b200.structural import rdf_cn as R
    fr = next(D.read_dumps(os.path.join(sample_dir, "dump.nvt.0.dump"), ["id", "type"]))
    rel = [[9, 9, 9, 9], [1, 4, 6, 9]]
    at = R._value_counts(fr.data["type"])
    L = fr.box.lattice_lengths()
    rho, rho_pairs = R._calc_props(L, fr.natoms, at, at, 9, MASS, rel, "type")
    full, part = R._normalize_rdf(0.05, rho_pairs, at, rel, 4, 400, gold_structural["rdf_raw_part_f0"].astype(np.float64),
                                  gold_structural["rdf_raw_full_f0"].astype(np.float64), fr.natoms, rho)
    df = R._save_rdf((np.arange(400) + 0.5) * 0.05, np.asarray(rel).T, None, False, part / 1, rdf_full_sum=full / 1)
    assert list(df.columns) == list(gold_structural["atomic_rdf_columns"])
    assert np.array_equal(df.values, gold_structural["atomic_rdf_f0"])
    with pytest.raises(ValueError, match="Consistency check failed"):
        R._calc_props(L, fr.natoms, at, at, 8, MASS, rel, "type")


def test_cn_edges_table():
    from mdproptools_b200.structural.rdf_cn import _cn_edges
    edges, rmax, upto = _cn_edges([2.325, 4.375, 2.375, 13.0, 4.375])
    assert rmax == 169.0 and len(edges) == 5 and edges[0] == 0
    assert upto.tolist() == [0, 2, 1, 3, 2]
    assert edges[1] == 2.325 * 2.325


def test_thermo_log_parser(visc_dir):
    from mdproptools_b200.io.log import concat_log, parse_lammps_log
    logs = parse_lammps_log(os.path.join(visc_dir, "log.visc_1"))
    assert len(logs) == 1 and list(logs[0].columns) == ["Step", "Temp", "Pxy", "Pxz", "Pyz"]
    assert len(logs[0]) == 4001 and logs[0]["Step"].iloc[-1] == 20000
    full = concat_log("log.visc_*", working_dir=visc_dir)
    assert len(full) == 4000 + 4001


def test_unique_configurations_reproduce_reference(tmp_path):
    """get_unique_configurations (cluster_analysis.py:238-457) on the 33 frame-50 clusters the reference's own test uses
    (tests/structural/test_cluster_analysis.py:62-100).  Golden = the unmodified reference run by oracle/gen_golden.py,
    whose five conf_*.xyz files were byte-identical to the reference's committed goldens and whose counts are the
    notebook's 20/8/3/1/1 (60.6/24.2/9.1/3.0/3.0 %)."""
    import io
    import json
    import pandas as pd
    from mdproptools_b200.structural.cluster_analysis import get_unique_configurations
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_unique_conf.json")))
    assert g["conf_identical_to_reference_goldens"] == 5 and g["counts"] == [20, 8, 3, 1, 1]
    for name, text in g["cluster_files"].items():
        (tmp_path / name).write_text(text)
    df, df1 = get_unique_configurations(cluster_pattern="Cluster_*.xyz", r_cut=2.3, molecules=g["species"], mol_num=2,
                                        type_coord_atoms=["O", "N", "Mg"], working_dir=str(tmp_path), find_top=True,
                                        perc=None, cum_perc=100, mol_names=["dme", "tfsi", "mg"], zip=False)
    assert df1["count"].tolist() == g["counts"]
    assert np.allclose(df1["%"].values, g["percent"], rtol=0, atol=0)
    for name, text in g["conf_files"].items():
        assert (tmp_path / name).read_text() == text, name
    for key, fname in (("clusters_csv", "clusters.csv"), ("configurations_csv", "configurations.csv"), ("top_conf_csv", "top_conf.csv")):
        ours = pd.read_csv(tmp_path / fname).fillna("")
        ref = pd.read_csv(io.StringIO(g[key])).fillna("")
        pd.testing.assert_frame_equal(ours, ref, check_dtype=False)
    ref_clusters = pd.read_csv(io.StringIO(g["clusters_csv"])).fillna("")
    pd.testing.assert_frame_equal(df.fillna(""), ref_clusters, check_dtype=False)
    # zip=True moves the cluster files into Clusters.zip
    for name in g["conf_files"]:
        os.remove(tmp_path / name)
    get_unique_configurations("Cluster_*.xyz", 2.3, g["species"], 2, ["O", "N", "Mg"], str(tmp_path), find_top=False, zip=True)
    assert (tmp_path / "Clusters.zip").exists() and not list(tmp_path.glob("Cluster_*.xyz"))


def test_shard_ranges_cover_everything():
    from mdproptools_b200 import dist
    for n in (0, 1, 7, 8, 101, 1000):
        for w in (1, 2, 3, 8):
            r = [dist.shard_range(n, k, w) for k in range(w)]
            assert r[0][0] == 0 and r[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(r, r[1:]))
            assert max(hi - lo for lo, hi in r) - min(hi - lo for lo, hi in r) <= 1


def test_read_text_frames_offsets_and_headers(tmp_path):
    """The reader-thread body of the text pipeline (io/dump.py: read_text_frames): a file is read into the middle of a
    staging buffer; frame starts, first-row offsets, ends, headers (orthogonal and triclinic, LF and CRLF) and column
    lists of a multi-frame file must describe exactly the text the host parser would be given."""
    from mdproptools_b200.io import dump as D
    rng = np.random.default_rng(3)
    for eol in ("\n", "\r\n"):
        p = tmp_path / ("t%d.dump" % len(eol))
        frames = []
        with open(p, "w", newline="") as f:
            for k, (n, tri) in enumerate([(5, False), (9, True), (1, False)]):
                head = f"ITEM: TIMESTEP{eol}{k * 7}{eol}ITEM: NUMBER OF ATOMS{eol}{n}{eol}"
                head += (f"ITEM: BOX BOUNDS xy xz yz pp pp pp{eol}0 10 1.5{eol}0 11 -0.5{eol}0 12 0.25{eol}" if tri else
                         f"ITEM: BOX BOUNDS pp pp pp{eol}0 10{eol}-1 11{eol}0.5 12{eol}")
                head += f"ITEM: ATOMS id type x y z{eol}"
                rows = "".join("%d 1 %g %g %g%s" % (i + 1, *rng.uniform(0, 9, 3), eol) for i in rng.permutation(n))
                f.write(head + rows)
                frames.append((head, rows, n, k * 7, tri))
        size = os.path.getsize(p)
        buf = np.zeros(size + 100, dtype=np.uint8)
        got, frs = D.read_text_frames(str(p), memoryview(buf), buf.ctypes.data, 37, size)
        assert got == size and len(frs) == 3
        text = bytes(buf[37:37 + size])
        assert text == open(p, "rb").read()
        off = 37
        for fr, (head, rows, n, ts, tri) in zip(frs, frames):
            assert (fr.begin, fr.rows, fr.end) == (off, off + len(head), off + len(head) + len(rows))
            assert (fr.timestep, fr.natoms, fr.columns) == (ts, n, ["id", "type", "x", "y", "z"])
            assert (fr.box.tilt is not None) == tri
            ref = D.parse_frame(bytes(buf[fr.begin:fr.end]), ["id", "x"])
            assert ref.natoms == n and ref.box.bounds == fr.box.bounds and ref.box.tilt == fr.box.tilt
            off = fr.end


def test_text_pipeline_file_groups():
    from mdproptools_b200.io.pipeline import _file_groups
    rng = np.random.default_rng(1)
    for _ in range(200):
        sizes = rng.integers(0, 100, int(rng.integers(0, 40))).tolist()
        mf, mb = int(rng.integers(1, 9)), int(rng.integers(1, 300))
        g = _file_groups(sizes, mf, mb)
        assert [k for grp in g for k in grp] == list(range(len(sizes)))             # every file once, in order
        for grp in g:
            assert 1 <= len(grp) <= mf
            assert len(grp) == 1 or sum(sizes[k] for k in grp) <= mb                # only a single oversized file may exceed
        for a, b in zip(g, g[1:]):                                                  # greedy: the next file did not fit
            assert len(a) == mf or sum(sizes[k] for k in a) + sizes[b[0]] > mb


def test_gpu_side_test_tools_compile():
    """The randomised cross-checks (tests/fuzz/) and the NCCL worker only run on a GPU box; a syntax error in them should
    not wait for one."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "tests", "fuzz", "*.py"))) + [os.path.join(ROOT, "tests", "nccl_api_worker.py")]
    assert len(files) == 5
    for f in files:
        compile(open(f).read(), f, "exec")


def test_owner_of_rows_agrees_with_shard_range():
    """The rank a central atom's rows are sent to (dist.owner_of_rows, int32 and int64 indices) is the rank whose
    shard_range block holds it -- the residence-time exchange relies on it."""
    import torch
    from mdproptools_b200 import dist
    for n in (1, 7, 8, 16, 101, 2000):
        for w in (1, 2, 3, 8):
            want = np.empty(n, dtype=np.int64)
            for k in range(w):
                lo, hi = dist.shard_range(n, k, w)
                want[lo:hi] = k
            for dt in (torch.int32, torch.int64):
                got = dist.owner_of_rows(torch.arange(n, dtype=dt), n, w)
                assert got.tolist() == want.tolist(), (n, w, dt)


def test_per_frame_host_caches():
    """The caches that keep the consumer thread of the file pipeline off the critical path: _same_values (memcmp of
    contiguous arrays, element comparison otherwise), _TypeCache (recompute only when the column changes; an identical
    object needs no comparison), _PropsCache (box / density work once per kind of frame, consistency error on the first)."""
    from mdproptools_b200.io.dump import Box
    from mdproptools_b200.io.pipeline import FrameMeta
    from mdproptools_b200.structural import rdf_cn as R
    a = np.arange(10, dtype=np.float64)
    assert R._same_values(a, a.copy()) and not R._same_values(a, a + 1) and not R._same_values(a, a[:5])
    assert R._same_values(a[::2], a[::2].copy()) and not R._same_values(a[::2], a[1::2])       # non-contiguous: element-wise
    calls = []
    tc = R._TypeCache()
    make = lambda col: (calls.append(1), col.sum())[1]
    buf = np.stack([a, a, a + 1])
    assert tc.get(buf[0], make) == 45 and tc.get(buf[1], make) == 45 and len(calls) == 1     # equal rows of a staging buffer
    assert tc.get(buf[2], make) == 55 and len(calls) == 2
    obj = a.copy()
    assert tc.get(obj, make) == 45 and tc.get(obj, make) == 45 and len(calls) == 3           # the same object again: no compare
    at = {1: 6, 2: 4}
    box = Box([[0.0, 10.0], [0.0, 10.0], [0.0, 10.0]], None)
    pc = R._PropsCache(0, 2, [1.0, 2.0], [[1], [2]], "type", None)
    row, rho, rho_pairs = pc.get(FrameMeta(0, 0, 10, box), at)
    want_rho, want_pairs = R._calc_props((10.0, 10.0, 10.0), 10, at, at, 2, [1.0, 2.0], [[1], [2]], "type", None)
    assert row == (10.0, 10.0, 10.0) and rho == want_rho and np.array_equal(rho_pairs, want_pairs)
    assert pc.get(FrameMeta(1, 5, 10, Box([[0.0, 10.0], [0.0, 10.0], [0.0, 10.0]], None)), at)[1] == rho      # same kind of frame
    row2, rho2, _ = pc.get(FrameMeta(2, 9, 10, Box([[0.0, 20.0], [0.0, 10.0], [0.0, 10.0]], None)), at)
    assert row2 == (20.0, 10.0, 10.0) and rho2 == rho / 2
    with pytest.raises(ValueError, match="Consistency check failed"):
        R._PropsCache(0, 3, [1.0, 2.0, 3.0], [[1], [2]], "type", None).get(FrameMeta(0, 0, 10, box), at)


@pytest.mark.gpu
def test_pinned_pool_reuses_buffers():
    from mdproptools_b200.io.pipeline import _PinnedPool
    import torch
    pool = _PinnedPool(cap=64 << 20)
    b = pool.take(1000)
    assert b.numel() == _PinnedPool.GRAIN and b.is_pinned()
    pool.give(b)
    assert pool.take(5 << 20) is b                       # reused: large enough and not wastefully large
    pool.give(b)
    c = pool.take(40 << 20)
    assert c is not b and c.numel() == 48 << 20
    pool.give(c)
    pool.give(torch.empty(1))                            # beyond the cap nothing more is kept
    assert sum(x.numel() for x in pool.free) <= 64 << 20


_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as d
d.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=2)
from mdproptools_b200 import dist
from mdproptools_b200.structural.rdf_cn import _merge_frames, _gather_props
r = dist.rank()
assert dist.world_size() == 2
# frames round-robin: rank r owns frames r, r+2, ...; integer histograms merge exactly
T = 5
mine = {{i: torch.full((2, 3), i + 1, dtype=torch.int64) for i in range(T) if i % 2 == r}}
allc = _merge_frames(mine, T, (2, 3), torch.device("cpu"))
assert allc[:, 0, 0].tolist() == [1, 2, 3, 4, 5]
props = _gather_props({{i: ("p", i) for i in mine}}, T)
assert sorted(props) == list(range(T))
lo, hi = dist.shard_range(11)
x = torch.zeros(11, dtype=torch.float64); x[lo:hi] = 1.0
dist.all_reduce_sum_(x)
assert x.sum().item() == 11
# residence time: (frame, central, neighbour) entries found on a rank's frames go to the owner of the central atom
n_cent = 7
rng = np.random.default_rng(5)
full = np.stack([rng.integers(0, 9, 40), rng.integers(0, n_cent, 40), rng.integers(0, 30, 40)], axis=1).astype(np.int32)
mine_rows = torch.from_numpy(full[full[:, 0] % 2 == r])
got = dist.exchange_rows(mine_rows, dist.owner_of_rows(mine_rows[:, 1], n_cent, 2))
lo, hi = dist.shard_range(n_cent)
want = full[(full[:, 1] >= lo) & (full[:, 1] < hi)]
assert sorted(map(tuple, got.tolist())) == sorted(map(tuple, want.tolist()))
assert all(dist.owner_of(i, n_cent, 2) == int(dist.owner_of_rows(torch.tensor([i]), n_cent, 2)) for i in range(n_cent))
empty = dist.exchange_rows(torch.zeros((0, 3), dtype=torch.int32), torch.zeros((0,), dtype=torch.int64))
assert empty.shape == (0, 3)
# strong-scaling merge: contiguous frame blocks are all-gathered (uneven split: 7 frames over 2 ranks)
lo, hi = dist.shard_range(7)
blk = torch.arange(lo, hi, dtype=torch.int64).reshape(-1, 1, 1).expand(-1, 2, 3).contiguous()
whole = dist.all_gather_blocks(blk, 7)
assert whole.shape == (7, 2, 3) and whole[:, 1, 2].tolist() == list(range(7))
# sharded file reads: every rank reads only its files; frame index = file index; total = number of files
from mdproptools_b200.io.pipeline import FrameBatches
from mdproptools_b200.structural.rdf_cn import _agree_sharding, _RetryUnsharded
def write(path, step, n=4):
    rows = "\n".join("%d 1 %g %g %g" % (i + 1, 0.5 * i + step, 1.0 * i, 2.0 * i) for i in range(n))
    return "ITEM: TIMESTEP\n%d\nITEM: NUMBER OF ATOMS\n%d\nITEM: BOX BOUNDS pp pp pp\n0 9\n0 9\n0 9\nITEM: ATOMS id type x y z\n%s\n" % (step, n, rows)
base = {tmp!r}
if r == 0:
    os.makedirs(base + "/one", exist_ok=True); os.makedirs(base + "/multi", exist_ok=True)
    for k in range(5):
        open(base + "/one/dump.t.%d.dump" % (k * 10), "w").write(write(None, k * 10))
    for k in range(3):
        open(base + "/multi/dump.t.%d.dump" % (k * 10), "w").write(write(None, k * 10) + (write(None, k * 10 + 5) if k == 1 else ""))
d.barrier()
fb = FrameBatches(base + "/one/dump.t.*.dump", ["id", "x"], to_device=False, file_shard=(r, 2))
seen = {{m.index: (m.timestep, float(b.host[k, 1, 0])) for b in fb for k, m in enumerate(b.metas)}}
assert sorted(seen) == list(range(r, 5, 2)) and fb.total_frames == 5 and not fb.multi_frame_seen
assert all(seen[i] == (i * 10, float(i * 10)) for i in seen)
_agree_sharding(fb, torch.device("cpu"))
fb = FrameBatches(base + "/multi/dump.t.*.dump", ["id", "x"], to_device=False, file_shard=(r, 2))
list(fb)
assert fb.multi_frame_seen == (r == 1)          # file 1 holds two frames; only the rank that read it knows ...
try:
    _agree_sharding(fb, torch.device("cpu"))
    raise SystemExit("no retry")
except _RetryUnsharded:
    pass                                         # ... and both ranks learn it
fb = FrameBatches(base + "/multi/dump.t.*.dump", ["id", "x"], to_device=False, frame_select=lambda i: i % 2 == r)
seen = sorted(m.index for b in fb for m in b.metas)
assert seen == list(range(r, 4, 2)) and fb.total_frames == 4
d.destroy_process_group()
print("rank", r, "ok")
"""


def test_two_rank_gloo_merge(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT, tmp=str(tmp_path)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29611", str(script)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout + res.stderr
    assert res.stdout.count("ok") == 2


def test_utilities_mirror_reference_import_paths(tmp_path):
    """mdproptools.utilities.{log,fluctuations,plots} resolve under the same names; the fluctuation statistics are
    pandas describe()'s mean / std (fluctuations.py:43)."""
    import pandas as pd

    from mdproptools_b200.io import log as io_log
    from mdproptools_b200.utilities import fluctuations, log, plots

    assert log.concat_log is io_log.concat_log and callable(plots.set_axis)
    rng = np.random.default_rng(3)
    df = pd.DataFrame({"Step": np.arange(50) * 100, "Press": rng.normal(1.0, 40.0, 50)})
    want = df["Press"].describe().loc[["mean", "std"]].to_dict()
    got = fluctuations.fluctuation_stats(df, "Press")
    assert got["mean"] == pytest.approx(want["mean"], rel=1e-14) and got["std"] == pytest.approx(want["std"], rel=1e-14)
    try:
        import matplotlib  # noqa: F401
    except ImportError:
        return
    mean, std = fluctuations.plot_fluctuations(df, "Press", "P", "press.png", working_dir=str(tmp_path))
    assert (tmp_path / "press.png").exists() and mean == got["mean"] and std == got["std"]


def test_frame_batches_producer_stops_when_the_consumer_leaves(tmp_path):
    """A consumer that raises (or drops the generator) mid-iteration must not leave the producer thread blocked in q.put()
    with its pinned buffers: FrameBatches.__iter__ stops and joins it."""
    import threading
    from mdproptools_b200.io.pipeline import FrameBatches
    rows = "\n".join("%d 1 %g %g %g" % (i + 1, 0.5 * i, 1.0 * i, 2.0 * i) for i in range(50))
    for k in range(40):
        (tmp_path / f"dump.s.{k}.dump").write_text(
            f"ITEM: TIMESTEP\n{k}\nITEM: NUMBER OF ATOMS\n50\nITEM: BOX BOUNDS pp pp pp\n0 9\n0 9\n0 9\nITEM: ATOMS id type x y z\n{rows}\n")
    before = threading.active_count()
    fb = FrameBatches(str(tmp_path / "dump.s.*.dump"), ["id", "x"], to_device=False, max_batch_frames=2, prefetch=1)
    with pytest.raises(RuntimeError):
        for n, batch in enumerate(fb):
            if n == 2:
                raise RuntimeError("consumer gives up")
    it = iter(FrameBatches(str(tmp_path / "dump.s.*.dump"), ["id", "x"], to_device=False, max_batch_frames=2, prefetch=1))
    next(it)
    it.close()                                           # generator dropped after one batch
    assert threading.active_count() <= before            # both producer threads were joined
    assert sum(len(b.metas) for b in FrameBatches(str(tmp_path / "dump.s.*.dump"), ["id", "x"], to_device=False)) == 40
