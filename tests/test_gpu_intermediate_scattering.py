"""Coherent intermediate scattering function on the device: mdp_sk_rho (csrc/sk.cu) against the rho that
mdp_structure_factor bins, mdp_isf_fft (csrc/isffft.cu) against the oracle's long-double direct sum (tests/isf_oracle.py),
its bit-level guarantees (pair order, scratch limits, bin sub-ranges) and argument errors; calc_intermediate_scattering end
to end against the oracle and against calc_structure_factor at t = 0, on a rigidly translating triclinic configuration, its
ValueErrors, and N ranks against one."""
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from tests import isf_oracle as IO  # noqa: E402
from tests import sk_oracle as SO  # noqa: E402
from tests.test_gpu_einstein import fresh_ctx  # noqa: E402,F401
from tests.test_gpu_structure_factor import _write_dump  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = 1e-5
CONTRACT = 1e-10
CELL = (25.0, 21.0, 18.0, 5.0, -2.5, 3.15)


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mdproptools_b200 import ops as _ops
    return _ops


def _dev(a, dtype=torch.float64):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dtype).cuda()


# ------------------------------------------------------------------------------------------------
# mdp_sk_rho
# ------------------------------------------------------------------------------------------------
def test_sk_rho_is_what_structure_factor_bins(ops):
    """Per-frame classes with an empty class (1 of 4), nk no multiple of the k-block (512), frames placed at column
    frame0 + f of a longer series: a sequential host sum of x.re y.re + x.im y.im in k order over mdp_sk_rho's values gives
    mdp_structure_factor's sums bit for bit, and the other columns are untouched."""
    rng = np.random.default_rng(1)
    F, n, ncls = 3, 1537, 4
    pos = rng.uniform(-1, 2, (F, n, 3)) @ SO.cell_matrix(CELL).T
    cls = rng.choice([0, 2, 3], (F, n)).astype(np.int32)
    miller, bin_off, _ = SO.kset_brute(CELL, 2.0, 0.1)
    nk, nb = len(miller), len(bin_off) - 1
    assert nk % 512 and nk > 512
    xyz = _dev(pos.transpose(0, 2, 1))
    cls_d = _dev(cls, torch.int32)
    sums = ops.structure_factor(xyz, cls_d, ncls, CELL, miller, bin_off, nb).cpu().numpy()
    out = torch.full((ncls, nk, 7), 7 + 7j, dtype=torch.complex128, device="cuda")
    ops.sk_rho(xyz, cls_d, ncls, CELL, miller, out=out, frame0=2)
    rho = out.cpu().numpy()
    assert np.all(rho[:, :, [0, 1, 5, 6]] == 7 + 7j)
    assert not np.any(rho[1, :, 2:5])
    re, im = rho.real, rho.imag
    rows = [(a, b) for a in range(ncls) for b in range(a, ncls)]
    ia = np.array([a for a, _ in rows])
    ib = np.array([b for _, b in rows])
    for f in range(F):
        want = np.zeros((len(rows), nb))
        for q in range(nb):
            s = np.zeros(len(rows))
            for k in range(bin_off[q], bin_off[q + 1]):
                x_re, x_im = re[ia, k, 2 + f], im[ia, k, 2 + f]
                y_re, y_im = re[ib, k, 2 + f], im[ib, k, 2 + f]
                s = s + (x_re * y_re + x_im * y_im)
            want[:, q] = s
        assert np.array_equal(want, sums[f]), f
    # a fresh series: the same values
    fresh = ops.sk_rho(xyz, cls_d, ncls, CELL, miller).cpu().numpy()
    assert np.array_equal(fresh, rho[:, :, 2:5])


def test_sk_rho_bad_arguments(ops):
    from mdproptools_b200._lib import MdpropError
    xyz = _dev(np.ones((2, 3, 10)))
    m = np.array([[1, 0, 0], [0, 1, 0]])
    out = torch.zeros((1, 2, 3), dtype=torch.complex128, device="cuda")
    for kw in (dict(frame0=2), dict(frame0=-1)):
        with pytest.raises(MdpropError, match="rc=-2"):
            ops.sk_rho(xyz, None, 1, (10.0, 10.0, 10.0, 0, 0, 0), m, out=out, **kw)
    with pytest.raises(MdpropError, match="rc=-2"):
        ops.sk_rho(xyz, None, 1, (10.0, 0.0, 10.0, 0, 0, 0), m)


# ------------------------------------------------------------------------------------------------
# mdp_isf_fft
# ------------------------------------------------------------------------------------------------
PAIRS = [(3, 3), (0, 1), (2, 2), (1, 0), (0, 2)]


def _series(rng, nchan, nk, T):
    t = np.arange(T)
    base = rng.normal(0, 3, (nchan, nk, 1)) + 1j * rng.normal(0, 3, (nchan, nk, 1))
    wave = np.exp(1j * rng.uniform(0, 0.3, (nchan, nk, 1)) * t)
    return base + wave + 0.5 * (rng.normal(0, 1, (nchan, nk, T)) + 1j * rng.normal(0, 1, (nchan, nk, T)))


def _contract_error(got, want):
    worst = 0.0
    for q in range(want.shape[0]):
        for b in range(want.shape[1]):
            scale = float(np.abs(want[q, b]).max())
            if scale == 0.0:
                assert not np.any(got[q, b]), (q, b)
                continue
            worst = max(worst, float(np.abs(got[q, b] - want[q, b]).max()) / scale)
    return worst


@pytest.mark.parametrize("T,nlags", [(2, 1), (300, 150), (257, 257), (1500, 700)])
def test_isf_fft_matches_direct_sum(ops, T, nlags):
    """Self and cross pairs, an odd number of pairs, empty bins first, in the middle and last: within 1e-10 of max_tau of
    the long-double direct sum per (pair, bin), empty bins exactly zero; every pair swapped gives the same bits."""
    rng = np.random.default_rng(T)
    bin_off = np.array([0, 0, 3, 3, 4, 11, 11])
    z = _series(rng, 4, int(bin_off[-1]), T)
    rho = _dev(z, torch.complex128)
    got = ops.isf_fft(rho, PAIRS, bin_off, nlags).cpu().numpy()
    want = IO.direct_corr(z.real, z.imag, PAIRS, bin_off, nlags).astype(np.float64)
    assert not np.any(got[:, [0, 2, 5]])
    assert _contract_error(got, want) < CONTRACT
    swapped = ops.isf_fft(rho, [(b, a) for a, b in PAIRS], bin_off, nlags).cpu().numpy()
    assert np.array_equal(got, swapped)
    assert np.array_equal(got, ops.isf_fft(rho, PAIRS, bin_off, nlags).cpu().numpy())


def test_isf_fft_empty_k_set_and_arguments(ops, fresh_ctx):  # noqa: F811
    from mdproptools_b200 import _lib
    from mdproptools_b200._lib import MdpropError
    z0 = torch.zeros((2, 0, 40), dtype=torch.complex128, device="cuda")
    e = ops.isf_fft(z0, [(0, 1), (1, 1)], [0, 0, 0], 20)
    assert e.shape == (2, 2, 20) and not torch.any(e)
    rho = _dev(_series(np.random.default_rng(3), 2, 4, 40), torch.complex128)
    bad = [dict(pairs=[(0, 2)]), dict(pairs=[(-1, 0)]), dict(bin_off=[1, 4]), dict(bin_off=[0, 3]),
           dict(bin_off=[0, 3, 2, 4]), dict(nlags=0), dict(nlags=41)]
    for c in bad:
        a = dict(pairs=[(0, 1)], bin_off=[0, 4], nlags=20)
        a.update(c)
        with pytest.raises(MdpropError, match="rc=-2"):
            ops.isf_fft(rho, a["pairs"], a["bin_off"], a["nlags"])
    fresh_ctx(1 << 16)                      # 2 pairs x 500 bins over 64 points: 264 kB of accumulators
    with pytest.raises(MdpropError, match="exceed the context limit"):
        ops.isf_fft(rho, [(0, 1), (1, 1)], [0] + [4] * 500, 20)
    ctx = _lib.Context.get()
    bo = np.array([0, 4], dtype=np.int64)
    pr = np.array([0, 1], dtype=np.int32)
    out = torch.empty((1, 1, 20), dtype=torch.float64, device="cuda")
    rc = _lib.lib().mdp_isf_fft(ctx.handle, 2, 4, 1 << 31, _lib.ptr(rho), 1, pr.ctypes.data_as(_lib.POINTER(_lib.c_int32)), 1,
                                bo.ctypes.data_as(_lib.POINTER(_lib.c_int64)), 1 << 30, _lib.ptr(out), _lib.stream_ptr())
    assert rc == -2                                                          # p > 30


def test_isf_fft_scratch_limits_and_bin_subranges(ops, fresh_ctx):  # noqa: F811
    """Scratch limits from below the smallest that admits the call to one sub-batch: every admitted limit gives the bits
    of the unlimited call (launch counts fall as the sub-batches grow); a call on a sub-range of the bins gives those
    bins' bits unchanged."""
    from mdproptools_b200._lib import MdpropError
    rng = np.random.default_rng(8)
    T, nlags = 600, 300
    bin_off = np.array([0, 5, 5, 9, 17, 30, 31, 40])
    z = _series(rng, 3, int(bin_off[-1]), T)
    rho = _dev(z, torch.complex128)
    pairs = [(2, 2), (0, 1), (1, 1)]
    ref = ops.isf_fft(rho, pairs, bin_off, nlags)
    for lo, hi in ((0, 1), (1, 4), (3, 7), (6, 7), (2, 3)):
        sub = rho[:, bin_off[lo]:bin_off[hi]].contiguous()
        got = ops.isf_fft(sub, pairs, bin_off[lo:hi + 1] - bin_off[lo], nlags)
        assert torch.equal(got, ref[:, lo:hi]), (lo, hi)
    n, nb = 1024, len(bin_off) - 1
    H = n // 2 + 1
    fixed = 16 * (n // 2) + 8 * len(pairs) * nb * H + 4 * len(pairs) * nb
    per_k = 2 * 3 * n * 16
    seen = {}
    for lim in sorted({fixed + per_k * m + d for m in (1, 2, 3, 7, 40) for d in (-8192, 0, 8192, 16384)}):
        ctx = fresh_ctx(lim)
        try:
            seen[lim] = (ops.isf_fft(rho, pairs, bin_off, nlags), ctx.launch_count())
        except MdpropError as e:
            seen[lim] = str(e)
    ok = sorted(l for l, v in seen.items() if not isinstance(v, str))
    bad = sorted(l for l, v in seen.items() if isinstance(v, str))
    assert ok and bad, (ok, bad)
    for l in bad:
        assert "exceed" in seen[l] and l < ok[0], seen[l]
    launches = [seen[l][1] for l in ok]
    assert all(x >= y for x, y in zip(launches, launches[1:])) and launches[0] > launches[-1], launches
    for l in ok:
        assert torch.equal(seen[l][0], ref), l


# ------------------------------------------------------------------------------------------------
# calc_intermediate_scattering end to end
# ------------------------------------------------------------------------------------------------
def _read(pattern):
    from mdproptools_b200.io.dump import read_dumps
    fr = list(read_dumps(pattern, ["id", "type", "x", "y", "z"]))
    b = fr[0].box
    cell = tuple(b.bound_lengths()) + (tuple(b.tilt) if b.tilt is not None else (0.0, 0.0, 0.0))
    return cell, [np.stack([f.data[c] for c in "xyz"], axis=1) for f in fr], fr[0].data["type"]


def _bound(cell, frames_pos, types, k_max, bin_size, relations, L, max_k=None):
    """per (pair, bin, lag), normalised: the S(k) contract (|rho_c error| <= eps N_c) carried through the products
    z_a(t+tau) z_b(t)*, plus the FFT contract on the largest value of the (pair, bin)"""
    named = sorted(set(int(t) for pair in relations for t in pair))
    cls = np.array([named.index(t) if t in named else len(named) for t in np.asarray(types).astype(np.int64)])
    ncls = len(named) + 1
    miller, bin_off, nbins = SO.kset_brute(cell, k_max, bin_size, None, max_k)
    re, im = IO.series(cell, frames_pos, cls, ncls, miller)
    amp = np.hypot(np.concatenate([re, re.sum(0, keepdims=True)]), np.concatenate([im, im.sum(0, keepdims=True)])).max(axis=2)
    counts = np.append(np.bincount(cls, minlength=ncls), len(cls)).astype(np.float64)
    rel = [(ncls, ncls)] + [(named.index(int(a)), named.index(int(b))) for a, b in relations]
    nk = np.diff(bin_off).astype(np.float64)
    out = []
    for a, b in rel:
        e = EPS * (counts[a] * amp[b] + counts[b] * amp[a]) + EPS * EPS * counts[a] * counts[b]
        s = np.array([e[bin_off[q]:bin_off[q + 1]].sum() for q in range(nbins)])
        norm = counts[a] if a == b == ncls else np.sqrt(counts[a] * counts[b])
        with np.errstate(invalid="ignore", divide="ignore"):
            out.append(np.repeat((s / (nk * norm))[:, None], L, axis=1))
    return np.stack(out)


def _compare(df, want, bound, relations, L):
    k, F, Fab, nk = want
    nbins = len(k)
    got = df.to_numpy().reshape(nbins, L, -1)
    assert list(df.columns) == ["k ($\\AA^{-1}$)", "t (s)", "F(k,t)"] + [f"F_{a}-{b}" for a, b in np.asarray(relations).T] + ["n_k"]
    assert np.array_equal(got[:, 0, 0], k) and np.array_equal(got[:, 0, -1], nk)
    vals = np.concatenate([F[None], Fab])
    mine = np.moveaxis(got[:, :, 2:2 + vals.shape[0]], 2, 0)
    assert np.array_equal(np.isnan(mine), np.isnan(vals))
    ok = ~np.isnan(vals)
    assert ok.sum() > 3 * L
    tol = bound + CONTRACT * np.nan_to_num(np.abs(vals).max(axis=2, keepdims=True)) + 1e-13
    assert np.all(np.abs(mine - vals)[ok] <= tol[ok]), np.max((np.abs(mine - vals) - tol)[ok])


def test_calc_intermediate_scattering_on_mini_traj(ops, mini_dir, tmp_path):
    """26 evenly spaced frames: against the oracle within the S(k) contract carried through the products plus the FFT
    contract; at t = 0, calc_structure_factor's S and S_ab on the same files to 1e-12 relative; the time axis."""
    from mdproptools_b200.common import constants as K
    from mdproptools_b200.dynamical.intermediate_scattering import calc_intermediate_scattering
    from mdproptools_b200.structural.structure_factor import calc_structure_factor
    pat = os.path.join(mini_dir, "dump.mini.*.dump")
    rel = [[3, 1, 8], [3, 2, 6]]
    out = tmp_path / "isf.csv"
    df = calc_intermediate_scattering(2.0, 0.1, rel, pat, timestep=2, max_k_per_bin=30, path_or_buff=str(out))
    assert out.stat().st_size > 0
    L = 13
    cell, frames, types = _read(pat)
    want = IO.isf(cell, frames, types, 2.0, 0.1, list(zip(*rel)), max_k_per_bin=30)
    _compare(df, want, _bound(cell, frames, types, 2.0, 0.1, list(zip(*rel)), L, 30), rel, L)
    got = df.to_numpy().reshape(20, L, -1)
    assert np.array_equal(got[0, :, 1], np.arange(L) * (200000.0 * 2 * K.TIME_CONVERSION["real"]))
    sk = calc_structure_factor(2.0, 0.1, rel, pat, max_k_per_bin=30, save_mode=False).to_numpy()
    ok = ~np.isnan(sk[:, 1])
    assert ok.sum() > 10
    np.testing.assert_allclose(got[ok, 0, 2:-1], sk[ok, 1:-1], rtol=1e-12, atol=1e-14)


def test_rigid_translation_matches_closed_form(ops, tmp_path):
    """A triclinic configuration translated by v per frame: F_ab(k, tau) = sum_k Re(rho_a rho_b*)(0) cos(k.v tau) / norm
    within the contract."""
    from mdproptools_b200.dynamical.intermediate_scattering import calc_intermediate_scattering
    rng = np.random.default_rng(31)
    cell = (26.0, 22.0, 19.0, 4.0, -2.0, 3.0)
    n, T = 900, 20
    types = rng.integers(1, 4, n)
    pos0 = rng.uniform(0, 1, (n, 3)) @ SO.cell_matrix(cell).T
    v = np.array([0.31, -0.17, 0.23])
    path = tmp_path / "dump.rigid.lammpstrj"
    _write_dump(path, [(50 * t, cell, pos0 + v * t, types) for t in range(T)])
    rel = [[1, 2], [3, 2]]
    df = calc_intermediate_scattering(1.5, 0.1, rel, str(path), max_lag=T, save_mode=False)
    cls = types - 1                                   # types 1, 2, 3 -> classes 0, 1, 2; channel 3 the total
    miller, bin_off, nbins = SO.kset_brute(cell, 1.5, 0.1)
    pairs = [(3, 3)] + [(int(a) - 1, int(b) - 1) for a, b in zip(*rel)]          # relations (1, 3) and (2, 2)
    C = IO.rigid_translation(cell, pos0, cls, 3, miller, v, pairs, bin_off, T)
    counts = np.append(np.bincount(cls, minlength=3), n).astype(np.float64)
    nk = np.diff(bin_off).astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        F = C[0] / (nk[:, None] * n)
        Fab = np.stack([C[q] / (nk[:, None] * np.sqrt(counts[a] * counts[b])) for q, (a, b) in enumerate(pairs) if q])
    F[nk == 0] = np.nan
    Fab[:, nk == 0] = np.nan
    frames = [pos0 + v * t for t in range(T)]
    _compare(df, ((np.arange(nbins) + 0.5) * 0.1, F, Fab, nk), _bound(cell, frames, types, 1.5, 0.1, list(zip(*rel)), T), rel, T)


def test_value_errors(ops, tmp_path):
    from mdproptools_b200.dynamical import intermediate_scattering as M
    rng = np.random.default_rng(32)
    c0, c1 = (18.0, 18.0, 18.0, 0.0, 0.0, 0.0), (18.5, 18.0, 18.0, 0.0, 0.0, 0.0)
    types = rng.integers(1, 3, 200)

    def dump(name, steps, cells, ns=None):
        frames = []
        for i, (s, c) in enumerate(zip(steps, cells)):
            m = 200 if ns is None else ns[i]
            frames.append((s, c, rng.uniform(0, 1, (m, 3)) @ SO.cell_matrix(c).T, types[:m]))
        _write_dump(tmp_path / name, frames)
        return str(tmp_path / name)

    cases = [(dump("cell.lammpstrj", [0, 10, 20], [c0, c0, c1]), "one cell"),
             (dump("uneven.lammpstrj", [0, 10, 30], [c0] * 3), "evenly spaced"),
             (dump("count.lammpstrj", [0, 10, 20], [c0] * 3, [200, 200, 150]), "atom count"),
             (dump("one.lammpstrj", [0], [c0]), "at least 2 frames")]
    for path, msg in cases:
        with pytest.raises(ValueError, match=msg):
            M.calc_intermediate_scattering(1.0, 0.1, [[1], [2]], path, save_mode=False)
    good = dump("good.lammpstrj", [0, 10, 20], [c0] * 3)
    for L in (0, 4):
        with pytest.raises(ValueError, match="max_lag"):
            M.calc_intermediate_scattering(1.0, 0.1, [[1], [2]], good, max_lag=L, save_mode=False)
    with pytest.raises(ValueError, match="no atom of type 5"):
        M.calc_intermediate_scattering(1.0, 0.1, [[1], [5]], good, save_mode=False)
    real = torch.cuda.mem_get_info
    try:
        torch.cuda.mem_get_info = lambda *a: (1024, 1 << 30)
        with pytest.raises(ValueError, match="max_k_per_bin"):
            M.calc_intermediate_scattering(1.0, 0.1, [[1], [2]], good, save_mode=False)
    finally:
        torch.cuda.mem_get_info = real


# ------------------------------------------------------------------------------------------------
# N ranks against one
# ------------------------------------------------------------------------------------------------
WORKER = '''
import os, sys
import numpy as np
sys.path.insert(0, sys.argv[3])
import torch
import torch.distributed as dist
world = int(os.environ.get("WORLD_SIZE", "1"))
torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
if world > 1:
    dist.init_process_group("nccl")
from mdproptools_b200.dynamical.intermediate_scattering import calc_intermediate_scattering
df = calc_intermediate_scattering(2.0, 0.1, [[3, 1], [3, 2]], sys.argv[2], max_k_per_bin=40, save_mode=False)
if int(os.environ.get("RANK", "0")) == 0:
    np.save(sys.argv[1], df.to_numpy())
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
'''


def test_intermediate_scattering_nrank_equals_1rank(ops, mini_dir, tmp_path):
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs at least 2 GPUs")
    worker = tmp_path / "isf_worker.py"
    worker.write_text(WORKER)
    res = {}
    for n in sorted({1, 2, min(ngpu, 4)}):
        out = tmp_path / f"n{n}.npy"
        cmd = ([sys.executable] if n == 1 else
               [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
                "127.0.0.1", "--master-port", str(29791 + n)])
        r = subprocess.run(cmd + [str(worker), str(out), os.path.join(mini_dir, "dump.mini.*.dump"), ROOT], cwd=ROOT,
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        res[n] = np.load(out)
    for n in res:
        assert np.array_equal(res[1], res[n], equal_nan=True), n
