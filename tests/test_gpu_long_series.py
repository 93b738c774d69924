"""The time-correlation kernels at every lag of long series, against exact integer-valued references.

On integer series whose sums stay below 2^53 (tests/exact_series.py) the direct kernels are exact: k_xcorr and
k_msd_window are pinned bit for bit to the host's int64 sums at sampled lags, and then serve as full-lag references for
the FFT calls, which must agree to their contract of 1e-10 of max_tau |out| at every lag, the last ones (where T - tau
is smallest) included.  The survival counts are integers and are compared exactly at the two boundaries of their
routes.  Each FFT comparison prints its worst error (in units of max_tau |out|) and the lag where it occurs.
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import oracle as O  # noqa: E402
from tests import exact_series as ES  # noqa: E402
from tests.test_host_einstein import CONTRACT, GROUPINGS  # noqa: E402


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mdproptools_b200 import ops as _ops
    return _ops


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _direct(ops, monkeypatch, a, b, nlags):
    monkeypatch.setenv("MDP_XCORR_FFT", "0")
    return ops.xcorr_unbiased(a, b, nlags).cpu().numpy()


def _fft(ops, monkeypatch, a, b, nlags):
    monkeypatch.setenv("MDP_XCORR_FFT", "1")
    return ops.xcorr_unbiased(a, b, nlags).cpu().numpy()


def _worst(what, got, want):
    """worst |got - want| / max_tau |want| over the rows, and where; asserts the contract, reports the figure"""
    got = got.reshape(-1, got.shape[-1])
    want = want.reshape(-1, want.shape[-1])
    worst, at = 0.0, (0, 0)
    for r in range(want.shape[0]):
        scale = np.abs(want[r]).max()
        if scale == 0.0:                              # an empty group or bin is written as exact zeros
            assert not np.any(got[r]), (what, r)
            continue
        err = np.abs(got[r] - want[r]) / scale
        k = int(np.argmax(err))
        if err[k] > worst:
            worst, at = float(err[k]), (r, k)
    print(f"\n[long-series] {what}: worst {worst:.2e} of max|out| at row {at[0]} lag {at[1]} of {want.shape[1]}")
    assert worst <= CONTRACT, (what, worst, at)
    return worst


def _series_pair(rng, C, T):
    """C channels of integer OU series; channel 0 correlates a series with itself, the others two different ones"""
    a = ES.ou_series(rng, C, T)
    b = ES.ou_series(rng, C, T, offset=7)
    b[0] = a[0]
    return a, b


# ----------------------------------------------------------------------------------------------------------------------
# direct kernels: bit for bit against int64 sums
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [10 ** 5, 10 ** 6])
def test_xcorr_direct_bit_exact(ops, monkeypatch, T):
    """k_xcorr with nlags = T: the first, the last and random lags equal fl(X(tau) / (T - tau)) exactly"""
    rng = np.random.default_rng(T)
    a, b = _series_pair(rng, 2, T)
    got = _direct(ops, monkeypatch, _dev(a), _dev(b), T)
    lags = ES.sample_lags(T, T, rng)
    for c in range(2):
        assert np.array_equal(got[c, lags], ES.xcorr_lags(a[c], b[c], lags)), c


def test_msd_window_bit_exact(ops):
    """k_msd_window at T = 10^5 over every lag (98 launches of MW_WCAP = 1024 lags) on walks offset by up to 10^6,
    groups of 1, 5 and 7 atoms: per axis and total, the sums equal the int64 sums at sampled lags"""
    rng = np.random.default_rng(71)
    T, N = 10 ** 5, 13
    off = np.array([0, 1, 6, 13])
    chans = ES.walk_series(rng, 3 * N, T)                      # channel 3 i + c is axis c of atom i
    ES.assert_exact_msd(chans)
    traj = chans.reshape(N, 3, T).transpose(2, 1, 0)
    sums = ops.msd_all_origins(_dev(traj), T, 1.0, group_off=off).cpu().numpy()     # [T, G, 4]
    lags = ES.sample_lags(T, T, rng)
    for g in range(3):
        gch = chans[3 * off[g]:3 * off[g + 1]]
        for c in range(3):
            assert np.array_equal(sums[lags, g, c], ES.msd_sums(gch[c::3], lags).astype(np.float64)), (g, c)
        assert np.array_equal(sums[lags, g, 3], ES.msd_sums(gch, lags).astype(np.float64)), g


# ----------------------------------------------------------------------------------------------------------------------
# mdp_xcorr_fft at every lag
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T,C", [(10 ** 5, 4), (10 ** 6, 3)])
def test_xcorr_fft_every_lag(ops, monkeypatch, T, C):
    rng = np.random.default_rng(T + 1)
    a, b = _series_pair(rng, C, T)
    ES.assert_exact_xcorr(a, b)
    a_d, b_d = _dev(a), _dev(b)
    ref = _direct(ops, monkeypatch, a_d, b_d, T)
    _worst(f"mdp_xcorr_fft T={T} nlags=T", _fft(ops, monkeypatch, a_d, b_d, T), ref)
    half = _fft(ops, monkeypatch, a_d, b_d, T // 2)
    _worst(f"mdp_xcorr_fft T={T} nlags=T/2", half, ref[:, :T // 2])


def test_xcorr_fft_ten_million_steps(ops, monkeypatch):
    """T = 10^7, nlags = T: N = 2^25, where the 2 GiB group budget holds one channel, so two channels take two groups.
    Every lag against k_xcorr, which is itself pinned to the int64 sums at the first 64, random and the last 1000 lags."""
    from mdproptools_b200._lib import Context
    rng = np.random.default_rng(10 ** 7)
    T = 10 ** 7
    a, b = _series_pair(rng, 2, T)
    ES.assert_exact_xcorr(a, b)
    a_d, b_d = _dev(a), _dev(b)
    ctx = Context.get(a_d.device.index)
    n0 = ctx.launch_count()
    _fft(ops, monkeypatch, a_d[:1], b_d[:1], T)
    n1 = ctx.launch_count()
    got = _fft(ops, monkeypatch, a_d, b_d, T)
    n2 = ctx.launch_count()
    assert n2 - n1 > n1 - n0, "two channels at N = 2^25 should run as two groups"
    ref = _direct(ops, monkeypatch, a_d, b_d, T)
    lags = np.union1d(ES.sample_lags(T, T, rng), np.arange(T - 1000, T))
    for c in range(2):
        assert np.array_equal(ref[c, lags], ES.xcorr_lags(a[c], b[c], lags)), c
    _worst("mdp_xcorr_fft T=1e7 nlags=T", got, ref)


# ----------------------------------------------------------------------------------------------------------------------
# the MSD, ACF and ISF calls at every lag
# ----------------------------------------------------------------------------------------------------------------------
def _channel_msd(ops, chans, T):
    """[T, C] exact per-channel all-origins sums of squared displacements from k_msd_window (scale 1)"""
    C = chans.shape[0]
    A = (C + 2) // 3
    pad = np.zeros((3 * A, T), dtype=np.int64)
    pad[:C] = chans
    traj = pad.reshape(A, 3, T).transpose(2, 1, 0)
    sums = ops.msd_all_origins(_dev(traj), T, 1.0, group_off=np.arange(A + 1)).cpu().numpy()   # [T, A, 4]
    return sums[:, :, :3].reshape(T, 3 * A)[:, :C]


@pytest.mark.parametrize("case", ["self", "cross"])
def test_cross_msd_fft_every_lag(ops, case):
    """T = 10^5, nlags = T/2 and T, integer walks offset by up to 10^6, the GROUPINGS layouts.  Reference: k_msd_window
    (self), or for the cross case (|d(a+b)|^2 - |d(a-b)|^2) / 4 of two exact self sums."""
    rng = np.random.default_rng(72 if case == "self" else 73)
    T = 10 ** 5
    Cmax = max(sum(c) for c in GROUPINGS.values())
    a = ES.walk_series(rng, Cmax, T)
    b = None
    if case == "self":
        ES.assert_exact_msd(a)
        per_chan = _channel_msd(ops, a, T)
    else:
        b = a // 2 + ES.walk_series(rng, Cmax, T)                  # correlated with a, far from it
        ES.assert_exact_msd(np.concatenate((a + b, a - b)))
        per_chan = (_channel_msd(ops, a + b, T) - _channel_msd(ops, a - b, T)) / 4.0
    norm = (T - np.arange(T)).astype(np.float64)
    for name, counts in GROUPINGS.items():
        off = np.concatenate(([0], np.cumsum(counts))).astype(np.int64)
        C = int(off[-1])
        want = np.stack([per_chan[:, off[g]:off[g + 1]].sum(axis=1) / norm for g in range(len(counts))])
        for nlags in (T // 2, T):
            got = ops.cross_msd_fft(_dev(a[:C]), None if b is None else _dev(b[:C]), off, nlags).cpu().numpy()
            _worst(f"mdp_cross_msd_fft {case} {name} T=1e5 nlags={nlags}", got, want[:, :nlags])


def test_group_acf_fft_every_lag(ops, monkeypatch):
    """T = 10^5, nlags = T, series offset by 10^3 (the ACF is not centred), an empty group: the per-group sum of k_xcorr"""
    rng = np.random.default_rng(74)
    T = 10 ** 5
    off = np.array([0, 1, 3, 3, 6])
    a = ES.ou_series(rng, 6, T, offset=1000)
    ES.assert_exact_xcorr(a, a)
    a_d = _dev(a)
    xc = _direct(ops, monkeypatch, a_d, a_d, T)
    want = np.stack([xc[off[g]:off[g + 1]].sum(axis=0) for g in range(4)])
    got = ops.group_acf_fft(a_d, off, T).cpu().numpy()
    _worst("mdp_group_acf_fft T=1e5 nlags=T", got, want)


def test_isf_fft_every_lag(ops, monkeypatch):
    """T = 10^5 (N = 2^18), self and cross pairs, three bins (the middle one empty), every lag.  Reference per k-vector:
    1/2 (xc(ar, br) + xc(ai, bi) + xc(br, ar) + xc(bi, ai)) from k_xcorr, summed over the bin."""
    rng = np.random.default_rng(75)
    T, nk = 10 ** 5, 5
    rho = ES.complex_rho(rng, 2, nk, T)
    ES.assert_exact_xcorr(rho.real, rho.real, terms=4 * nk)
    ES.assert_exact_xcorr(rho.imag, rho.imag, terms=4 * nk)
    pairs = np.array([[0, 0], [0, 1], [1, 1]])
    bin_off = np.array([0, 2, 2, 5])
    rho_d = torch.from_numpy(rho).cuda()
    got = ops.isf_fft(rho_d, pairs, bin_off, T).cpu().numpy()             # [npairs, nbins, T]
    want = np.zeros_like(got)
    for p, (i, j) in enumerate(pairs):
        ra, ia, rb, ib = rho[i].real, rho[i].imag, rho[j].real, rho[j].imag
        xa = _dev(np.concatenate((ra, ia, rb, ib)))
        xb = _dev(np.concatenate((rb, ib, ra, ia)))
        four = _direct(ops, monkeypatch, xa, xb, T).reshape(4, nk, T)
        per_k = 0.5 * four.sum(axis=0)
        for q in range(len(bin_off) - 1):
            want[p, q] = per_k[bin_off[q]:bin_off[q + 1]].sum(axis=0)
    _worst("mdp_isf_fft T=1e5 nlags=T", got, want)


# ----------------------------------------------------------------------------------------------------------------------
# Viscosity end to end
# ----------------------------------------------------------------------------------------------------------------------
def _write_log(path, steps, p):
    rows = np.column_stack((steps, np.full(len(steps), 298), p.T))
    with open(path, "w") as f:
        f.write("LAMMPS (synthetic)\nunits real\nPer MPI rank memory allocation (min/avg/max) = 1 | 1 | 1 Mbytes\n")
        f.write("Step Temp Pxy Pxz Pyz\n")
        np.savetxt(f, rows, fmt="%d")
        f.write("Loop time of 1.0 on 1 procs for 1 steps with 1 atoms\n")


def test_viscosity_end_to_end(ops, monkeypatch, tmp_path):
    """Three replicate logs of 150 001 thermo rows with integer Pxy, Pxz, Pyz: calc_avg_visc's ACFs and running
    integrals against the exact ACF (k_xcorr, pinned to the int64 sums at sampled lags) carried through the same
    constants, with a long-double running trapezoid, to 1e-10 of max"""
    import mdproptools_b200.dynamical.viscosity as vmod
    from mdproptools_b200.common import constants
    rng = np.random.default_rng(76)
    T, R = 150_001, 3
    steps = np.arange(T, dtype=np.int64) * 5
    press = [ES.ou_series(rng, 3, T, tau=200.0, sigma=400.0) for _ in range(R)]
    for r in range(R):
        _write_log(tmp_path / f"log.visc_{r}", steps, press[r])
    real = vmod.glob.glob
    monkeypatch.setattr(vmod.glob, "glob", lambda p: sorted(real(p)))
    monkeypatch.delenv("MDP_XCORR_FFT", raising=False)                    # the default route: the FFT from 2048 steps
    v = vmod.Viscosity("log.visc_*", cutoff_time=0, volume=40.0 ** 3, temp=298.15, timestep=1, units="real",
                       working_dir=str(tmp_path))
    _, visc_data, acf_data, _ = v.calc_avg_visc(output_all_data=True)
    conv2 = constants.PRESSURE_CONVERSION["real"] ** 2
    step_to_s = v.step_to_s
    dt = np.longdouble(steps[1] * step_to_s - steps[0] * step_to_s)
    factor = np.longdouble(v.volume / (constants.BOLTZMANN * v.temp))
    lags = ES.sample_lags(T, T, rng)
    for r in range(R):
        p = press[r]
        ES.assert_exact_xcorr(p, p)
        exact = _direct(ops, monkeypatch, _dev(p), _dev(p), T)
        for c in range(3):
            assert np.array_equal(exact[c, lags], ES.xcorr_lags(p[c], p[c], lags)), (r, c)
        acf = exact.astype(np.longdouble) * np.longdouble(conv2)
        integ = factor * np.cumsum(dt * (acf[:, 1:] + acf[:, :-1]) / 2, axis=1)
        _worst(f"Viscosity ACF replicate {r}", np.asarray(acf_data[r]), acf.astype(np.float64))
        _worst(f"Viscosity running integral replicate {r}", np.asarray(visc_data[r]), integ.astype(np.float64))


# ----------------------------------------------------------------------------------------------------------------------
# survival counts at the boundaries of their routes
# ----------------------------------------------------------------------------------------------------------------------
RUNS_LAST_T = 21_504            # ops.bitmask_autocorr_from_list: T * 8 + 32768 <= 200 KiB takes mdp_survival_runs
POPCOUNT_LAST_T = 28_992        # mdp_bitmask_autocorr: 64 pairs x (T/64 + 1) words of shared memory <= 227 KB


def _indicators(rng, T):
    """h [T, 2, 4]: every frame, alternating (T/2 runs, past the run buffer), period 3, long runs, random, one run open
    at the end, first and last frame only, never"""
    t = np.arange(T)
    h = np.zeros((T, 8), dtype=np.uint8)
    h[:, 0] = 1
    h[:, 1] = t % 2 == 0
    h[:, 2] = t % 3 != 2
    edges = np.cumsum(rng.integers(500, 3000, T // 500 + 2))
    h[:, 3] = np.searchsorted(edges, t, side="right") % 2
    h[:, 4] = rng.uniform(size=T) < 0.5
    h[T // 3:, 5] = 1
    h[[0, T - 1], 6] = 1
    return h.reshape(T, 2, 4)


def _survival(ops, monkeypatch, h, runs):
    """ops.bitmask_autocorr_from_list on the list of h -> (counts, pairs, the counting entry points it called)"""
    T = h.shape[0]
    f, ia, ib = np.nonzero(h)
    lst = torch.from_numpy(np.stack([f, ia, ib], axis=1).astype(np.int32)).cuda()
    monkeypatch.setenv("MDP_SURVIVAL_RUNS", runs)
    real, called = ops.lib(), []

    class Spy:
        def __getattr__(self, name):
            called.append(name)
            return getattr(real, name)

    with monkeypatch.context() as m:
        m.setattr(ops, "lib", lambda: Spy())
        cnt, P = ops.bitmask_autocorr_from_list(lst, h.shape[2], T)
    routes = [c for c in called if c in ("mdp_survival_runs", "mdp_bitmask_autocorr")]
    return cnt.cpu().numpy(), P, routes


@pytest.mark.parametrize("T", [RUNS_LAST_T, RUNS_LAST_T + 1, POPCOUNT_LAST_T])
def test_survival_counts_at_route_boundaries(ops, monkeypatch, T):
    """the last length on the runs route (a multiple of 64: a run is still open in the last word), the first on the
    popcount route and the last one admitted: the oracle's integers; at the runs route's last length both routes"""
    if torch.cuda.get_device_properties(0).shared_memory_per_block_optin != 227 * 1024:
        pytest.skip("the popcount route's limit is stated for parts with 227 KB of opt-in shared memory")
    rng = np.random.default_rng(T)
    h = _indicators(rng, T)
    ref = O.survival_counts(h.reshape(T, -1))
    cnt, P, routes = _survival(ops, monkeypatch, h, "1")
    assert P == 7 and np.array_equal(cnt, ref), T
    assert routes == ["mdp_survival_runs" if T <= RUNS_LAST_T else "mdp_bitmask_autocorr"], (T, routes)
    if T == RUNS_LAST_T:
        cnt0, P0, routes0 = _survival(ops, monkeypatch, h, "0")
        assert P0 == 7 and routes0 == ["mdp_bitmask_autocorr"] and np.array_equal(cnt0, ref)


def test_survival_counts_refuse_past_the_popcount_limit(ops, monkeypatch):
    """one frame more than the popcount kernel's shared memory admits: a clean MdpropError from the host-side check"""
    from mdproptools_b200._lib import MdpropError
    if torch.cuda.get_device_properties(0).shared_memory_per_block_optin != 227 * 1024:
        pytest.skip("the popcount route's limit is stated for parts with 227 KB of opt-in shared memory")
    h = _indicators(np.random.default_rng(1), POPCOUNT_LAST_T + 1)
    with pytest.raises(MdpropError, match="exceed shared memory"):
        _survival(ops, monkeypatch, h, "1")
