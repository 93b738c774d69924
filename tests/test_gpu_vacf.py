"""Velocity autocorrelation on the device: mdp_group_acf_fft (csrc/msdfft.cu) against the long-double direct sum and against
per-channel correlations, its determinism and its scratch-limited sub-batches; Diffusion.get_vacf / calc_diff_green_kubo /
get_vdos end to end against the oracle's restatements, exact constructions and the Einstein route; the errors they raise;
N ranks against one."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from tests import vacf_oracle as VO  # noqa: E402
from tests.conftest import MASS, NUM_ATOMS  # noqa: E402
from tests.test_gpu_einstein import LIMIT_MAX, fresh_ctx  # noqa: E402,F401
from tests.test_host_einstein import GROUPINGS  # noqa: E402
from tests.test_host_vacf import CONTRACT, acf_error, velocity_series, write_vel_dump  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mdproptools_b200 import ops as _ops
    return _ops


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _acf(ops, a, off, nlags):
    return ops.group_acf_fft(_dev(a), off, nlags).cpu().numpy()


# ------------------------------------------------------------------------------------------------
# the kernel
# ------------------------------------------------------------------------------------------------
def test_group_acf_fft_matches_direct_sum(ops):
    """Lengths around powers of two, nlags = T and T // 3, odd channel counts, empty groups, series offset by 10^3: within
    1e-10 of max_tau |out[g]| of the long-double direct sum; empty groups exactly zero."""
    rng = np.random.default_rng(61)
    for T in (1, 2, 3, 7, 2047, 2048, 2049, 4097):
        for name, counts in GROUPINGS.items():
            off = np.concatenate(([0], np.cumsum(counts))).astype(np.int64)
            a = velocity_series(rng, int(off[-1]), T)
            for nlags in sorted({T, max(1, T // 3)}):
                err = acf_error(_acf(ops, a, off, nlags), VO.acf_direct(a, off, nlags), counts)
                assert err < CONTRACT, (T, name, nlags, err)


def test_group_acf_fft_long_series(ops):
    """T = 10^5 (a 2^18-point transform with nlags = T/2), groups of 1, 2 and 3 channels offset by 10^3: the first 300 lags
    against the direct sum, to the contract."""
    rng = np.random.default_rng(62)
    T = 100_000
    off = np.array([0, 1, 3, 6])
    a = velocity_series(rng, 6, T)
    got = _acf(ops, a, off, T // 2)
    want = VO.acf_direct(a, off, 300)
    for g in range(3):
        assert np.abs(got[g, :300] - want[g]).max() < CONTRACT * np.abs(got[g]).max(), g


def test_group_acf_fft_equals_summed_xcorr(ops):
    """the per-group sum of ops.xcorr_unbiased(a, a) over the group's channels, to the contract"""
    rng = np.random.default_rng(63)
    T, nlags = 3000, 1200
    off = np.array([0, 3, 3, 8, 9])
    a = _dev(velocity_series(rng, 9, T, offset=-20.0))
    got = ops.group_acf_fft(a, off, nlags).cpu().numpy()
    xc = ops.xcorr_unbiased(a, a, nlags).cpu().numpy()
    for g in range(4):
        want = xc[off[g]:off[g + 1]].sum(axis=0)
        if off[g + 1] == off[g]:
            assert not np.any(got[g])
            continue
        assert np.abs(got[g] - want).max() < CONTRACT * np.abs(want).max(), g


def test_group_acf_fft_is_deterministic(ops):
    rng = np.random.default_rng(64)
    a = _dev(velocity_series(rng, 11, 5000))
    off = [0, 4, 4, 11]
    assert torch.equal(ops.group_acf_fft(a, off, 2500), ops.group_acf_fft(a, off, 2500))


def test_group_acf_fft_bad_arguments(ops, fresh_ctx):
    from mdproptools_b200 import _lib
    from mdproptools_b200._lib import MdpropError
    a = _dev(np.ones((4, 100)))
    for off, nlags in (([0, 4], 101), ([0, 4], 0), ([1, 4], 10), ([0, 3], 10), ([0, 5], 10), ([0, 3, 2, 4], 10), ([0], 10)):
        with pytest.raises(MdpropError, match="rc=-2"):
            ops.group_acf_fft(a, off, nlags)
    with pytest.raises(MdpropError, match="rc=-2"):
        ops.group_acf_fft(a, [0] + [4] * 65536, 10)
    ctx = _lib.Context.get()
    go = np.array([0, 4], dtype=np.int64)
    rc = _lib.lib().mdp_group_acf_fft(ctx.handle, 4, 1 << 30, _lib.ptr(a), 1, go.ctypes.data_as(_lib.POINTER(_lib.c_int64)), 10,
                                      _lib.ptr(a), _lib.stream_ptr())
    assert rc == -2 and "2^31" in _lib.last_error()
    rc = _lib.lib().mdp_group_acf_fft(ctx.handle, 4, 100, None, 1, go.ctypes.data_as(_lib.POINTER(_lib.c_int64)), 10,
                                      _lib.ptr(a), _lib.stream_ptr())
    assert rc == -2 and "NULL" in _lib.last_error()
    fresh_ctx(1 << 20)                                  # 200 group accumulators of 8193 values: over 1 MB
    with pytest.raises(MdpropError, match="rc=-2.*accumulators"):
        ops.group_acf_fft(_dev(np.ones((200, 4097))), np.arange(201), 4097)


def test_group_acf_fft_subbatches_under_scratch_limits(ops, fresh_ctx):
    """Groups of 9, 0 and 6 channels of 4097 steps, 1500 lags, swept over scratch limits on fresh contexts from the smallest
    that works up to 64 MB: every working limit gives the bits of the unlimited call (the group accumulators carry across
    sub-batches in unit order), within the contract; calls never fail above the smallest working limit; the number of
    launches never grows with the limit and the sweep sees groups split over several sub-batches."""
    from mdproptools_b200._lib import MdpropError
    rng = np.random.default_rng(65)
    T, nlags, off = 4097, 1500, np.array([0, 9, 9, 15])
    a = velocity_series(rng, 15, T)
    a_d = _dev(a)
    ref = ops.group_acf_fft(a_d, off, nlags)
    assert acf_error(ref.cpu().numpy(), VO.acf_direct(a, off, nlags), [9, 0, 6]) < CONTRACT
    seen = {}

    def attempt(limit):
        if limit not in seen:
            ctx = fresh_ctx(limit)
            try:
                seen[limit] = (ops.group_acf_fft(a_d, off, nlags), ctx.launch_count())
            except MdpropError as e:
                seen[limit] = str(e)
        return not isinstance(seen[limit], str)

    assert attempt(LIMIT_MAX), seen[LIMIT_MAX]
    lo, hi = 0, LIMIT_MAX
    while hi - lo > 256:
        mid = (lo + hi) // 2
        if attempt(mid):
            hi = mid
        else:
            lo = mid
    for k in range(-16, 48):
        if hi + k * (16 << 10) > 0:
            attempt(hi + k * (16 << 10))
    lim = hi + (1 << 20)
    while lim < LIMIT_MAX:
        attempt(lim)
        lim = int(lim * 1.5)
    ok = sorted(l for l, v in seen.items() if not isinstance(v, str))
    bad = sorted(l for l, v in seen.items() if isinstance(v, str))
    for l in bad:
        assert "exceeds the context limit" in seen[l] or "exceed the context limit" in seen[l], (l, seen[l])
    assert not [l for l in bad if l > ok[0]], (ok[0], [l for l in bad if l > ok[0]][:8])
    launches = [seen[l][1] for l in ok]
    assert all(x >= y for x, y in zip(launches, launches[1:])), list(zip(ok, launches))
    assert len(set(launches)) >= 3, sorted(set(launches))          # from one unit per sub-batch to all in one
    for l in ok:
        assert torch.equal(seen[l][0], ref), l


# ------------------------------------------------------------------------------------------------
# Diffusion.get_vacf / calc_diff_green_kubo / get_vdos end to end
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mini_mols():
    from tests.conftest import GOLDEN
    return np.load(os.path.join(GOLDEN, "ref_dynamical.npz"))["mini_num_mols"].tolist()


def _diff(d):
    from mdproptools_b200.dynamical.diffusion import Diffusion
    return Diffusion(timestep=1, units="real", outputs_dir=d, diff_dir=d)


def _assert_frame_close(got, want, rel=1e-12):
    assert list(got.columns) == list(want), (list(got.columns), list(want))
    for col, w in want.items():
        g = got[col].to_numpy()
        assert g.shape == w.shape, col
        assert np.abs(g - w).max() <= rel * np.abs(w).max(), col


@pytest.mark.parametrize("vacf_type", ["allatom", "com"])
def test_get_vacf_on_mini_traj(ops, mini_dir, mini_mols, tmp_path, vacf_type):
    """values, column names and lag times against the oracle within 1e-12 of each column's maximum; the Green-Kubo and VDOS
    steps against the oracle's; the files they save"""
    from mdproptools_b200.common import constants as K
    d = str(tmp_path / "mini")
    shutil.copytree(mini_dir, d)
    kw = dict(num_mols=mini_mols, num_atoms_per_mol=NUM_ATOMS, mass=MASS) if vacf_type == "com" else {}
    df = _diff(d)
    got = df.get_vacf("dump.mini.*.dump", vacf_type=vacf_type, **kw)
    want = VO.get_vacf(os.path.join(d, "dump.mini.*.dump"), K.TIME_CONVERSION["real"], K.VELOCITY_CONVERSION["real"],
                       vacf_type=vacf_type, **kw)
    assert len(got) == 13 and got["Time (s)"].iloc[0] == 0.0
    _assert_frame_close(got, want)
    gk = df.calc_diff_green_kubo(got, save=True)
    names = [c for c in want if c.startswith("vacf")]
    assert list(gk.columns) == ["diffusion (m2/s)", "std"] and list(gk.index) == list(range(1, len(names) + 1))
    t = want["Time (s)"]
    for i, c in enumerate(names):
        D, std, _ = VO.green_kubo(t, want[c])
        assert gk["diffusion (m2/s)"].iloc[i] == pytest.approx(D, rel=1e-11, abs=1e-12 * abs(D))
        assert gk["std"].iloc[i] == pytest.approx(std, rel=1e-9, abs=1e-9 * abs(D))
    vd = df.get_vdos(got, save=True)
    assert list(vd.columns) == ["Frequency (Hz)", "Wavenumber (cm^-1)"] + ["vdos" + c[4:] for c in names]
    for c in names:
        nu, S = VO.vdos(want[c], t[1] - t[0])
        np.testing.assert_allclose(vd["Frequency (Hz)"], nu, rtol=1e-14)
        assert np.abs(vd["vdos" + c[4:]].to_numpy() - S).max() <= 1e-11 * np.abs(S).max(), c
    for f in ("vacf_integral.csv", "diffusion_gk.csv", "vdos.csv"):
        assert os.path.getsize(os.path.join(d, f)) > 0, f


def test_constant_velocities(ops, tmp_path):
    """vacf = mean |v|^2 at every lag, the running integral is linear in t, and the VDOS identities hold on the device"""
    from mdproptools_b200.common import constants as K
    rng = np.random.default_rng(66)
    T, N = 40, 6
    v0 = rng.normal(0, 0.01, (3, N))
    vel = np.repeat(v0[None], T, axis=0)
    write_vel_dump(tmp_path / "dump.c.lammpstrj", np.arange(T) * 5, vel, np.array([1, 1, 2, 2, 2, 1]), np.ones(N))
    df = _diff(str(tmp_path))
    vac = df.get_vacf("dump.c.lammpstrj", max_lag=30)
    want = (v0 * K.VELOCITY_CONVERSION["real"]) ** 2
    assert np.abs(vac["vacf"] - want.sum() / N).max() <= 1e-12 * want.sum() / N
    assert np.abs(vac["vacf2"] - want[:, 2:5].sum() / 3).max() <= 1e-12 * want[:, 2:5].sum() / 3
    gk = df.calc_diff_green_kubo(vac, save=True)
    run = np.loadtxt(os.path.join(str(tmp_path), "vacf_integral.csv"), delimiter=",", skiprows=1)
    t = run[:, 0]
    for k in range(1, run.shape[1]):
        slope = run[-1, k] / t[-1]
        assert np.abs(run[:, k] - slope * t).max() <= 1e-12 * abs(run[-1, k]), k
    # zero frequency of the unwindowed VDOS: S(0) C_0 / 4 = the last value of the running integral (times dimension is D)
    vd = df.get_vdos(vac, window="none")
    c0 = vac["vacf"].iloc[0]
    assert vd["vdos"].iloc[0] * c0 / 4 == pytest.approx(run[-1, -1], rel=1e-12)
    assert gk["diffusion (m2/s)"].iloc[-1] > 0


def test_vdos_units_and_peak(ops, tmp_path):
    """a cosine VACF at a grid frequency peaks there, and the Hz and cm^-1 columns describe the same frequency"""
    from mdproptools_b200.common import constants as K
    from mdproptools_b200.dynamical.diffusion import Diffusion
    import pandas as pd
    L, dt, k0 = 301, 2e-15, 40
    nu0 = k0 / (2 * (L - 1) * dt)
    vac = pd.DataFrame({"Time (s)": np.arange(L) * dt, "vacf": np.cos(2 * np.pi * nu0 * np.arange(L) * dt)})
    vd = Diffusion(diff_dir=str(tmp_path)).get_vdos(vac)
    k = int(np.argmax(vd["vdos"].to_numpy()))
    assert k == k0
    assert vd["Frequency (Hz)"].iloc[k] == pytest.approx(nu0, rel=1e-14)
    assert vd["Wavenumber (cm^-1)"].iloc[k] == pytest.approx(nu0 / K.LIGHT_SPEED / 100, rel=1e-14)
    assert np.trapezoid(vd["vdos"], vd["Frequency (Hz)"]) == pytest.approx(1.0, abs=1e-12)


def ou_trajectory(seed, N=64, T=4000, tau=1.0, sig=0.01, every=10):
    """Ornstein-Uhlenbeck velocities (memory tau frames, Angstrom/fs) and unwrapped positions integrated from them by the
    trapezoid rule over the frame spacing of ``every`` fs"""
    rng = np.random.default_rng(seed)
    phi = np.exp(-1 / tau)
    v = np.empty((T, 3, N))
    v[0] = rng.normal(0, sig, (3, N))
    kick = rng.normal(0, sig * np.sqrt(1 - phi * phi), (T, 3, N))
    for t in range(1, T):
        v[t] = phi * v[t - 1] + kick[t]
    pos = np.empty_like(v)
    pos[0] = rng.uniform(0, 30, (3, N))
    for t in range(1, T):
        pos[t] = pos[t - 1] + 0.5 * (v[t] + v[t - 1]) * every
    return v, pos, np.arange(T) * every


def test_green_kubo_agrees_with_einstein(ops, tmp_path):
    """64 atoms (two types), 4000 frames of Ornstein-Uhlenbeck velocities with a one-frame memory, positions integrated from
    them: the Green-Kubo D of the all-atom VACF (200 lags) against calc_diff of the all-origins MSD (200 lags).  A host run
    of the oracle on this trajectory gives a deviation of +0.16 % (+0.39 % and -0.07 % per type; the spread over five
    seeds is -1.6 % to +3.2 %, the through-origin fit's bias included); the tolerance is 1 %."""
    v, pos, steps = ou_trajectory(53)
    write_vel_dump(tmp_path / "dump.ou.lammpstrj", steps, v, np.repeat([1, 2], 32), np.ones(64), pos=pos, L=30.0)
    df = _diff(str(tmp_path))
    gk = df.calc_diff_green_kubo(df.get_vacf("dump.ou.lammpstrj", max_lag=200))
    ein = df.calc_diff(df.get_msd_all_origins("dump.ou.lammpstrj", max_lag=200))
    d_gk, d_e = gk["diffusion (m2/s)"].iloc[-1], ein["diffusion (m2/s)"].iloc[0]
    assert abs(d_gk / d_e - 1) < 0.01, (d_gk, d_e)


def test_vacf_errors(ops, tmp_path):
    """ValueError for a dump without velocities, uneven frames, varying types, max_lag < 1 and fewer than 2 lags"""
    import pandas as pd
    rng = np.random.default_rng(67)
    T, N = 10, 4
    vel = rng.normal(0, 0.01, (T, 3, N))
    types = np.array([1, 1, 2, 2])
    cases = {}
    for key, steps, tp in (("ok", np.arange(T) * 5, types), ("uneven", np.r_[np.arange(T - 1) * 5, 5 * T + 3], types),
                           ("types", np.arange(T) * 5, np.array([types] * (T - 1) + [[1, 2, 1, 2]]))):
        d = tmp_path / key
        d.mkdir()
        write_vel_dump(d / "dump.lammpstrj", steps, vel, tp, np.ones(N))
        cases[key] = str(d)
    d = tmp_path / "novel"
    d.mkdir()
    (d / "dump.lammpstrj").write_text((tmp_path / "ok" / "dump.lammpstrj").read_text().replace("vx vy vz", "xu yu zu"))
    cases["novel"] = str(d)
    assert np.all(np.isfinite(_diff(cases["ok"]).get_vacf("dump.lammpstrj")["vacf"]))
    for key in ("uneven", "types", "novel"):
        with pytest.raises(ValueError):
            _diff(cases[key]).get_vacf("dump.lammpstrj")
    with pytest.raises(ValueError):
        _diff(cases["ok"]).get_vacf("dump.lammpstrj", max_lag=0)
    one = pd.DataFrame({"Time (s)": [0.0], "vacf": [1.0]})
    with pytest.raises(ValueError, match="vacf"):
        _diff(cases["ok"]).get_vdos(one)
    with pytest.raises(ValueError, match="vacf"):
        _diff(cases["ok"]).get_vdos(pd.DataFrame({"Time (s)": [0.0, 1.0], "vacf": [0.0, 1.0]}))


def test_com_msd_all_origins_checks_molecule_atom_count(ops, mini_dir, mini_mols):
    """Molecules that claim more or fewer atoms than the dump holds: the ValueError of get_msd_from_dump, raised on the host
    before the centre-of-mass reduction would read past the arrays or drop atoms."""
    df = _diff(mini_dir)
    for extra in (1, -1):
        mols = mini_mols[:-1] + [mini_mols[-1] + extra]
        for call in (df.get_msd_all_origins, df.get_msd_from_dump):
            with pytest.raises(ValueError, match="does not match length of index"):
                call("dump.mini.*.dump", msd_type="com", num_mols=mols, num_atoms_per_mol=NUM_ATOMS, mass=MASS)


# ------------------------------------------------------------------------------------------------
# N ranks against one
# ------------------------------------------------------------------------------------------------
WORKER = '''
import os, sys
import numpy as np
sys.path.insert(0, sys.argv[3])
import torch
import torch.distributed as dist
from tests.conftest import MASS, NUM_ATOMS
from mdproptools_b200.dynamical.diffusion import Diffusion
world = int(os.environ.get("WORLD_SIZE", "1"))
torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
if world > 1:
    dist.init_process_group("nccl")
num_mols = [int(v) for v in sys.argv[4].split(",")]
df = Diffusion(timestep=1, units="real", outputs_dir=sys.argv[2], diff_dir=sys.argv[2])
res = {}
for kind, kw in (("allatom", {}), ("com", dict(num_mols=num_mols, num_atoms_per_mol=NUM_ATOMS, mass=MASS))):
    v = df.get_vacf("dump.mini.*.dump", vacf_type=kind, **kw)
    res["vacf_" + kind] = v.to_numpy()
    res["gk_" + kind] = df.calc_diff_green_kubo(v).to_numpy()
    res["vdos_" + kind] = df.get_vdos(v).to_numpy()
if int(os.environ.get("RANK", "0")) == 0:
    np.savez(sys.argv[1], **res)
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
'''


def test_vacf_nrank_equals_1rank(ops, mini_dir, mini_mols, tmp_path):
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs at least 2 GPUs")
    worker = tmp_path / "vacf_worker.py"
    worker.write_text(WORKER)
    res = {}
    for n in sorted({1, 2, min(ngpu, 4)}):
        out = tmp_path / f"n{n}.npz"
        cmd = ([sys.executable] if n == 1 else
               [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
                "127.0.0.1", "--master-port", str(29671 + n)])
        r = subprocess.run(cmd + [str(worker), str(out), mini_dir, ROOT, ",".join(map(str, mini_mols))], cwd=ROOT,
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        res[n] = np.load(out)
    for n in res:
        for k in res[1].files:
            a, b = res[1][k], res[n][k]
            assert a.shape == b.shape, (n, k)
            assert np.abs(a - b).max() <= 1e-12 * np.abs(a).max(), (n, k)
