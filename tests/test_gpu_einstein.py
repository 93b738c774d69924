"""Einstein and Nernst-Einstein conductivity on the device: mdp_cross_msd_fft (csrc/msdfft.cu) against the oracle's
long-double direct sum and against mdp_msd_all_origins, its determinism and its scratch-limited sub-batches;
Conductivity.einstein / nernst end to end against the oracle's restatements and against two exact constructions; the
errors they raise; N ranks against one."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from tests import einstein_oracle as EO  # noqa: E402
from tests.conftest import MASS, NUM_ATOMS  # noqa: E402
from tests.test_host_einstein import CONTRACT, GROUPINGS, _series, contract_error, write_dump  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MINI_VOLUME = 49.182348836183905 ** 3


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mdproptools_b200 import ops as _ops
    return _ops


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _fft(ops, a, b, off, nlags):
    return ops.cross_msd_fft(_dev(a), None if b is None else _dev(b), off, nlags).cpu().numpy()


# ------------------------------------------------------------------------------------------------
# the kernel
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["self", "cross"])
def test_cross_msd_fft_matches_direct_sum(ops, case):
    """Lengths around powers of two, nlags < T and = T, odd channel counts, empty groups: within 1e-10 of max_tau |out[g]|
    of the long-double direct sum; empty groups are exactly zero."""
    rng = np.random.default_rng(31)
    for T in (1, 2, 3, 7, 2047, 2048, 2049, 4097):
        for name, counts in GROUPINGS.items():
            off = np.concatenate(([0], np.cumsum(counts))).astype(np.int64)
            C = int(off[-1])
            a = _series(rng, C, T)
            b = None if case == "self" else _series(rng, C, T) - 2.0
            for nlags in sorted({T, max(1, T // 3)}):
                got = _fft(ops, a, b, off, nlags)
                for g in range(len(counts)):
                    if counts[g] == 0:
                        assert not np.any(got[g]), (T, name, nlags, g)
                floor = np.var(a, axis=1).sum() + (0.0 if b is None else np.var(b, axis=1).sum())
                err = contract_error(got, EO.cross_msd_direct(a, b, off, nlags), floor)
                assert err < CONTRACT, (T, name, nlags, err)


@pytest.mark.parametrize("case", ["self", "cross"])
def test_cross_msd_fft_long_series(ops, case):
    """T = 10^5 (a 2^18-point transform with nlags = T/2), groups of 1, 2 and 3 channels, series offset by 1e8 steps: the
    first 1000 lags against the direct sum, to the contract (max over all T/2 lags from the FFT's own result is an upper
    bound of the direct maximum's scale, so the direct maximum over the checked lags is used)."""
    rng = np.random.default_rng(32)
    T, step = 100_000, 0.02
    off = np.array([0, 1, 3, 6])
    a = np.cumsum(rng.normal(0, step, (6, T)), axis=1) + 1e8 * step
    b = None if case == "self" else np.cumsum(rng.normal(0, step, (6, T)), axis=1) - 1e8 * step
    got = _fft(ops, a, b, off, T // 2)
    want = EO.cross_msd_direct(a, b, off, 1000)
    for g in range(3):
        scale = max(np.abs(got[g]).max(), np.abs(want[g]).max())
        assert np.abs(got[g, :1000] - want[g]).max() < CONTRACT * scale, g


def test_cross_msd_fft_self_case_equals_windowed_msd_kernel(ops):
    """[3N][T] channels in one group against the [.., 3] sums of mdp_msd_all_origins on the same coordinates (divided by
    T - lag), and a per-type grouping against its per-group sums."""
    rng = np.random.default_rng(33)
    T, N, max_lag = 3000, 40, 1000
    traj = np.cumsum(rng.normal(0, 0.2, (T, 3, N)), axis=0) + rng.uniform(0, 50, (1, 3, N))
    gtraj = np.array([0, 15, 40])
    sums = ops.msd_all_origins(_dev(traj), max_lag, 1.0, group_off=gtraj).cpu().numpy()      # [max_lag, G, 4]
    direct = sums[:, :, 3].T / (T - np.arange(max_lag))[None]
    chans = traj.transpose(2, 1, 0).reshape(-1, T)
    got = _fft(ops, chans, None, 3 * gtraj, max_lag)
    for g in range(2):
        assert np.abs(got[g] - direct[g]).max() < CONTRACT * np.abs(direct[g]).max(), g
    one = _fft(ops, chans, None, [0, 3 * N], max_lag)[0]
    assert np.abs(one - direct.sum(axis=0)).max() < CONTRACT * np.abs(one).max()


def test_cross_msd_fft_is_deterministic(ops):
    rng = np.random.default_rng(34)
    a, b = _dev(_series(rng, 11, 5000)), _dev(_series(rng, 11, 5000))
    off = [0, 4, 4, 11]
    for bb in (None, b):
        r1 = ops.cross_msd_fft(a, bb, off, 2500)
        r2 = ops.cross_msd_fft(a, bb, off, 2500)
        assert torch.equal(r1, r2)


def test_cross_msd_fft_bad_arguments(ops, fresh_ctx):
    from mdproptools_b200 import _lib
    from mdproptools_b200._lib import MdpropError
    a = _dev(np.ones((4, 100)))
    for off, nlags in (([0, 4], 101), ([0, 4], 0), ([1, 4], 10), ([0, 3], 10), ([0, 5], 10), ([0, 3, 2, 4], 10), ([0], 10)):
        with pytest.raises(MdpropError, match="rc=-2"):
            ops.cross_msd_fft(a, None, off, nlags)
    with pytest.raises(MdpropError, match="rc=-2"):
        ops.cross_msd_fft(a, None, [0] + [4] * 65536, 10)
    ctx = _lib.Context.get()
    go = np.array([0, 4], dtype=np.int64)
    rc = _lib.lib().mdp_cross_msd_fft(ctx.handle, 4, 1 << 30, _lib.ptr(a), None, 1,
                                      go.ctypes.data_as(_lib.POINTER(_lib.c_int64)), 10, _lib.ptr(a), _lib.stream_ptr())
    assert rc == -2 and "2^31" in _lib.last_error()
    fresh_ctx(1 << 20)                                  # 200 group accumulators of 8193 + 3 x 4097 values: over 1 MB
    with pytest.raises(MdpropError, match="rc=-2.*accumulators"):
        ops.cross_msd_fft(_dev(np.ones((200, 4097))), None, np.arange(201), 4097)


# scratch-limited sub-batches, on fresh contexts (the pattern of tests/test_gpu_batching.py)
LIMIT_MAX = 64 << 20


@pytest.fixture
def fresh_ctx(ops, monkeypatch):
    """install(limit) -> a new library context with that scratch limit, which every ops.* call on the current device uses
    until the next install or the end of the test (a context whose slab has never grown)."""
    from mdproptools_b200 import _lib
    dev = torch.cuda.current_device()
    old = _lib.Context._instances.get(dev)
    made = []

    def release():
        while made:
            ctx = made.pop()
            for tag in range(10):
                ctx.timing_read(tag)
            _lib.lib().mdp_ctx_destroy(ctx.handle)

    def install(limit):
        ctx = _lib.Context(dev)
        _lib.check(_lib.lib().mdp_ctx_set_scratch_limit(ctx.handle, int(limit)), "mdp_ctx_set_scratch_limit")
        ctx.timing(True)
        monkeypatch.setitem(_lib.Context._instances, dev, ctx)
        release()
        made.append(ctx)
        return ctx

    yield install
    if old is None:
        _lib.Context._instances.pop(dev, None)
    else:
        _lib.Context._instances[dev] = old
    release()


@pytest.mark.parametrize("case", ["self", "cross"])
def test_cross_msd_fft_subbatches_under_scratch_limits(ops, fresh_ctx, case):
    """Groups of 9, 0 and 6 channels of 4097 steps, 1500 lags, swept over scratch limits on fresh contexts from the
    smallest that works up to 64 MB: every working limit gives the bits of the unlimited call (the group accumulators carry
    across sub-batches in unit order), within the contract of the direct sum; calls never fail above the smallest working
    limit; the number of launches (sub-batches) never grows with the limit and the sweep sees groups split over several
    sub-batches."""
    from mdproptools_b200._lib import MdpropError
    rng = np.random.default_rng(35)
    T, nlags, off = 4097, 1500, np.array([0, 9, 9, 15])
    a = _series(rng, 15, T) + 1e5
    b = None if case == "self" else _series(rng, 15, T)
    a_d, b_d = _dev(a), (None if b is None else _dev(b))
    ref = ops.cross_msd_fft(a_d, b_d, off, nlags)
    assert contract_error(ref.cpu().numpy(), EO.cross_msd_direct(a, b, off, nlags)) < CONTRACT
    seen = {}

    def attempt(limit):
        if limit not in seen:
            ctx = fresh_ctx(limit)
            try:
                seen[limit] = (ops.cross_msd_fft(a_d, b_d, off, nlags), ctx.launch_count())
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
# Conductivity.einstein / nernst end to end
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mini_mols():
    from tests.conftest import GOLDEN
    return np.load(os.path.join(GOLDEN, "ref_dynamical.npz"))["mini_num_mols"].tolist()


def _mini_cond(d, num_mols, **kw):
    from mdproptools_b200.dynamical.conductivity import Conductivity
    return Conductivity("dump.mini.*.dump", num_mols, NUM_ATOMS, volume=MINI_VOLUME, mass=MASS, temp=298.15, timestep=1,
                        units="real", working_dir=d, **kw)


def _oracle_args(d, num_mols, dt_si):
    from mdproptools_b200.common import constants as K
    return (os.path.join(d, "dump.mini.*.dump"), num_mols, NUM_ATOMS, MINI_VOLUME * 1e-30, 298.15, dt_si, MASS,
            K.DISTANCE_CONVERSION["real"], K.CHARGE_CONVERSION["real"], K.BOLTZMANN)


def test_einstein_and_nernst_on_mini_traj(ops, mini_dir, mini_mols, tmp_path):
    d = str(tmp_path / "mini")
    shutil.copytree(mini_dir, d)
    c = _mini_cond(d, mini_mols)
    M = c.get_translational_dipole()
    ntypes, T = len(mini_mols), 26
    assert M.shape == (3, ntypes, T)
    dt = c.time[1] - c.time[0]
    assert dt == pytest.approx(200000 * 1e-15) and len(c.time) == T
    msd = c.correlate_translational_dipole(M)
    assert msd.shape == (ntypes + 1, T // 2) and np.abs(msd[:, 0]).max() < 1e-12 * np.abs(msd).max()
    sig_e = c.einstein(save=True)
    sig_ne = c.nernst(save=True)
    assert sig_e.shape == (ntypes + 1,) and sig_ne.shape == (ntypes + 1,)
    want_e, want_msd = EO.einstein_conductivity(*_oracle_args(d, mini_mols, dt))
    want_ne, _ = EO.nernst_einstein(*_oracle_args(d, mini_mols, dt))
    np.testing.assert_allclose(msd, want_msd, rtol=1e-9, atol=1e-9 * np.abs(want_msd).max())
    np.testing.assert_allclose(sig_e, want_e, rtol=1e-9, atol=1e-12 * np.abs(want_e).max())
    np.testing.assert_allclose(sig_ne, want_ne, rtol=1e-9)
    assert np.all(sig_ne[:ntypes] >= 0) and sig_ne[-1] == pytest.approx(sig_ne[:ntypes].sum(), rel=1e-15)
    for f in ("dipole_msd.csv", "einstein_conductivity.csv", "nernst_einstein.csv"):
        assert os.path.getsize(os.path.join(d, f)) > 0, f
    with open(os.path.join(d, "dipole_msd.csv")) as f:
        assert f.readline().strip() == "t," + ",".join(str(i + 1) for i in range(ntypes)) + ",tot"
    e = np.loadtxt(os.path.join(d, "einstein_conductivity.csv"), delimiter=",", skiprows=1)
    np.testing.assert_array_equal(e[:, 2], sig_e)
    # an explicit window and lag count against the oracle with the same ones
    kw = dict(max_lag=20, initial_time=3 * dt, final_time=15 * dt)
    np.testing.assert_allclose(c.einstein(**kw), EO.einstein_conductivity(*_oracle_args(d, mini_mols, dt), **kw)[0],
                               rtol=1e-9, atol=1e-12 * np.abs(want_e).max())
    np.testing.assert_allclose(c.nernst(**kw), EO.nernst_einstein(*_oracle_args(d, mini_mols, dt), **kw)[0], rtol=1e-9)
    with pytest.raises(ValueError):
        c.einstein(initial_time=5 * dt, final_time=5.5 * dt)


def test_einstein_and_nernst_from_image_flags(ops, mini_dir, mini_mols, tmp_path):
    """A copy of the fixture without xu yu zu: x + ix (xhi - xlo) against the oracle's restatement of that unwrapping."""
    d = tmp_path / "wrapped"
    d.mkdir()
    for name in os.listdir(mini_dir):
        with open(os.path.join(mini_dir, name)) as f:
            lines = f.read().splitlines()
        i = next(k for k, l in enumerate(lines) if l.startswith("ITEM: ATOMS"))
        cols = lines[i].split()[2:]
        keep = [k for k, cname in enumerate(cols) if cname not in ("xu", "yu", "zu")]
        out = lines[:i] + ["ITEM: ATOMS " + " ".join(cols[k] for k in keep)]
        out += [" ".join(l.split()[k] for k in keep) for l in lines[i + 1:] if l.strip()]
        (d / name).write_text("\n".join(out) + "\n")
    c = _mini_cond(str(d), mini_mols)
    sig_e, sig_ne = c.einstein(), c.nernst()
    dt = c.time[1] - c.time[0]
    want_e, _ = EO.einstein_conductivity(*_oracle_args(str(d), mini_mols, dt), unwrap="image")
    want_ne, _ = EO.nernst_einstein(*_oracle_args(str(d), mini_mols, dt), unwrap="image")
    np.testing.assert_allclose(sig_e, want_e, rtol=1e-9, atol=1e-12 * np.abs(want_e).max())
    np.testing.assert_allclose(sig_ne, want_ne, rtol=1e-9)


def _rigid_system(tmp_path, kind, T=3000):
    """A generated dump: (a) one charged two-atom molecule alone in type 1, three neutral two-atom molecules (internal
    charges +-0.3) in type 2; (b) a cation and an anion (types 1 and 2) rigidly bound, plus two neutral molecules (type 3).
    Returns the Conductivity object."""
    from mdproptools_b200.dynamical.conductivity import Conductivity
    rng = np.random.default_rng(36 if kind == "a" else 37)
    if kind == "a":
        num_mols, num_atoms = [1, 3], [2, 2]
        q = np.array([0.6, 0.4, 0.3, -0.3, 0.3, -0.3, 0.3, -0.3])
        walks = np.cumsum(rng.normal(0, 0.3, (T, 3, 4)), axis=0)
        centre = np.repeat(walks, 2, axis=2)
    else:
        num_mols, num_atoms = [1, 1, 2], [1, 1, 2]
        q = np.array([1.0, -1.0, 0.2, -0.2, 0.2, -0.2])
        walks = np.cumsum(rng.normal(0, 0.3, (T, 3, 3)), axis=0)
        centre = walks[:, :, [0, 0, 1, 1, 2, 2]]
    n = len(q)
    pos = centre + rng.uniform(-1, 1, (1, 3, n)) + 20.0
    mass = np.array([12.0, 16.0] * (n // 2))
    types = np.arange(1, n + 1)
    write_dump(tmp_path / "dump.rigid.lammpstrj", np.arange(T) * 10, pos, None, q, mass, types, 40.0)
    return Conductivity("dump.rigid.lammpstrj", num_mols, num_atoms, volume=40.0 ** 3, temp=300.0, timestep=2, units="real",
                        working_dir=str(tmp_path))


def test_single_charged_molecule_einstein_equals_nernst(ops, tmp_path):
    c = _rigid_system(tmp_path, "a")
    sig_e, sig_ne = c.einstein(), c.nernst()
    assert sig_ne[-1] > 0 and sig_ne[1] == 0.0
    assert abs(sig_e[-1] - sig_ne[-1]) <= 1e-9 * sig_ne[-1], (sig_e, sig_ne)


def test_bound_ion_pair_has_no_einstein_conductivity(ops, tmp_path):
    c = _rigid_system(tmp_path, "b")
    sig_e, sig_ne = c.einstein(), c.nernst()
    assert sig_ne[-1] > 0
    assert abs(sig_e[-1]) <= 1e-6 * sig_ne[-1], (sig_e, sig_ne)


def test_einstein_rejects_varying_charges_missing_positions_and_uneven_frames(ops, tmp_path):
    from mdproptools_b200.dynamical.conductivity import Conductivity
    rng = np.random.default_rng(38)
    T, n = 12, 4
    pos = np.cumsum(rng.normal(0, 0.3, (T, 3, n)), axis=0) + 5.0
    q = np.array([0.5, -0.5, 0.5, -0.5])
    mass = np.ones(n)
    types = np.array([1, 1, 2, 2])
    cases = {}
    d = tmp_path / "even"
    d.mkdir()
    write_dump(d / "dump.lammpstrj", np.arange(T) * 5, pos, None, q, mass, types, 20.0)
    cases["ok"] = d
    d = tmp_path / "uneven"
    d.mkdir()
    write_dump(d / "dump.lammpstrj", np.r_[np.arange(T - 1) * 5, 5 * T + 3], pos, None, q, mass, types, 20.0)
    cases["uneven"] = d
    d = tmp_path / "charges"
    d.mkdir()
    write_dump(d / "dump.lammpstrj", np.arange(T) * 5, pos, None, q, mass, types, 20.0)
    text = (d / "dump.lammpstrj").read_text().splitlines()
    last = max(k for k, l in enumerate(text) if l.startswith("ITEM: ATOMS")) + 1
    row = text[last].split()
    row[3] = repr(float(row[3]) + 0.1)
    text[last] = " ".join(row)
    (d / "dump.lammpstrj").write_text("\n".join(text) + "\n")
    cases["charges"] = d
    d = tmp_path / "nopos"
    d.mkdir()
    text = (cases["ok"] / "dump.lammpstrj").read_text().replace("id type mass q xu yu zu", "id type mass q vx vy vz")
    (d / "dump.lammpstrj").write_text(text)
    cases["nopos"] = d

    def cond(key):
        return Conductivity("dump.lammpstrj", [1, 1], [2, 2], volume=20.0 ** 3, working_dir=str(cases[key]))
    assert np.all(np.isfinite(cond("ok").einstein())) and np.all(np.isfinite(cond("ok").nernst()))
    for key in ("uneven", "charges", "nopos"):
        for method in ("einstein", "nernst", "get_translational_dipole"):
            with pytest.raises(ValueError):
                getattr(cond(key), method)()


def test_max_lag_below_one_is_rejected(ops, mini_dir, mini_mols, tmp_path):
    """nernst, einstein and correlate_translational_dipole share the lag rule: max_lag = 0 names itself in the error."""
    c = _mini_cond(mini_dir, mini_mols)
    for call in (lambda: c.nernst(max_lag=0), lambda: c.einstein(max_lag=0),
                 lambda: c.correlate_translational_dipole(c.get_translational_dipole(), max_lag=0)):
        with pytest.raises(ValueError, match=r"max_lag must be at least 1 \(26 frames\)"):
            call()


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
from mdproptools_b200.dynamical.conductivity import Conductivity
world = int(os.environ.get("WORLD_SIZE", "1"))
torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
if world > 1:
    dist.init_process_group("nccl")
num_mols = [int(v) for v in sys.argv[4].split(",")]
c = Conductivity("dump.mini.*.dump", num_mols, NUM_ATOMS, volume=49.182348836183905 ** 3, mass=MASS, temp=298.15,
                 timestep=1, units="real", working_dir=sys.argv[2])
M = c.get_translational_dipole()
res = dict(dipole=M, dipole_msd=c.correlate_translational_dipole(M), einstein=c.einstein(), nernst=c.nernst())
if int(os.environ.get("RANK", "0")) == 0:
    np.savez(sys.argv[1], **res)
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
'''


def test_einstein_nrank_equals_1rank(ops, mini_dir, mini_mols, tmp_path):
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs at least 2 GPUs")
    worker = tmp_path / "einstein_worker.py"
    worker.write_text(WORKER)
    res = {}
    for n in sorted({1, 2, min(ngpu, 4)}):
        out = tmp_path / f"n{n}.npz"
        cmd = ([sys.executable] if n == 1 else
               [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
                "127.0.0.1", "--master-port", str(29661 + n)])
        r = subprocess.run(cmd + [str(worker), str(out), mini_dir, ROOT, ",".join(map(str, mini_mols))], cwd=ROOT,
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        res[n] = np.load(out)
    for n in res:
        for k in res[1].files:
            a, b = res[1][k], res[n][k]
            assert a.shape == b.shape, (n, k)
            assert np.abs(a - b).max() <= 1e-12 * np.abs(a).max(), (n, k)
