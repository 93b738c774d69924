"""Paths of the CUDA kernels that only large inputs or a small scratch limit reach, checked against references:

  * mdp_charge_flux past one tile, one chunk and one frame per CTA (the double-buffered bulk-copy pipeline of
    k_charge_flux, its frame walk, the chunk sum of k_flux_finish, out/frame0) -- bit for bit on inputs for which
    every operation is exact, and to a stated rounding bound on realistic ones;
  * the frame sub-batches of the pair engine and the channel groups of the FFT correlation, on fresh contexts whose
    scratch limit is swept from the smallest one that works up to 64 MB: every limit that works gives the unlimited
    result, and a larger limit never fails.
"""
import math
from fractions import Fraction

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import oracle as O  # noqa: E402
from tests.conftest import MASS  # noqa: E402

FLUX_B, FLUX_TILE = 128, 1408          # molecules per chunk and atoms per tile of k_charge_flux (csrc/reduce.cu)


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mdproptools_b200 import ops as _ops
    return _ops


def _dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


@pytest.fixture
def fresh_ctx(ops, monkeypatch):
    """install(limit) -> a new library context with that scratch limit (and kernel timing on), which every ops.* call
    on the current device uses until the next install or the end of the test.  Each install is a context whose slab has
    never grown: once it has, arena_reserve serves smaller requests without looking at the limit again."""
    from mdproptools_b200 import _lib
    dev = torch.cuda.current_device()
    old = _lib.Context._instances.get(dev)
    made = []

    def release():
        while made:
            ctx = made.pop()
            for tag in range(10):                  # frees the timing events the calls recorded
                ctx.timing_read(tag)
            _lib.lib().mdp_ctx_destroy(ctx.handle)

    def install(limit):
        # the previous context is still the installed one until the new one replaces it
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


# ------------------------------------------------------------------------------------------------
# charge flux on exact inputs: bit for bit against the oracle
# ------------------------------------------------------------------------------------------------
VS_EXACT, QS_EXACT = 0.125, 2.0        # powers of two: scaling is exact


def _dyadic_molecule(rng, k):
    """k small integer masses whose sum is a power of two (the division by the molecule's mass is then exact)"""
    if k == 1:
        return [float(2 ** int(rng.integers(0, 5)))]
    m = rng.integers(1, 4, k - 1).tolist()
    s = sum(m)
    return [float(v) for v in m] + [float((1 << s.bit_length()) - s)]


def _exact_system(rng, types, nframes):
    """types = list over molecule types of the list of molecule sizes -> (vel [F,3,N], mass, q, seg_off, type_off).
    Velocities a * 2^-8 with a nonzero integer |a| <= 200, charges b * 2^-4 with |b| <= 24."""
    mass, sizes = [], []
    for mols in types:
        for k in mols:
            mass += _dyadic_molecule(rng, k)
            sizes.append(k)
    n = len(mass)
    a = rng.integers(1, 201, (nframes, 3, n)) * rng.choice([-1, 1], (nframes, 3, n))
    q = rng.integers(-24, 25, n) / 16.0
    seg_off = np.concatenate(([0], np.cumsum(sizes))).astype(np.int64)
    type_off = np.concatenate(([0], np.cumsum([len(m) for m in types]))).astype(np.int64)
    return a / 256.0, np.asarray(mass), q, seg_off, type_off


def _assert_exactly_representable(vel, mass, q, seg_off, type_off):
    """Every J[c, g, t] is a sum of terms S * Q * 2^(wmax - w) in units of 2^-(12 + wmax) * vs * qs, with S = sum m*a and
    Q = sum b of a molecule of mass 2^w, integers.  When the sum of their magnitudes stays below 2^53, every partial sum
    in every order is an exactly representable double, so the kernel and the oracle must agree bit for bit."""
    a = np.rint(vel * 256.0).astype(np.int64)
    m = mass.astype(np.int64)
    b = np.rint(q * 16.0).astype(np.int64)
    assert np.array_equal(a / 256.0, vel) and np.array_equal(m.astype(np.float64), mass) and np.array_equal(b / 16.0, q)
    seg = seg_off[:-1]
    W = np.add.reduceat(m, seg)
    w = np.log2(W).astype(np.int64)
    assert np.array_equal(1 << w, W)
    Q = np.abs(np.add.reduceat(b, seg))
    S = np.abs(np.add.reduceat(np.abs(a) * m, seg, axis=2))          # [F, 3, M], bounds |S| of every partial sum
    for g in range(len(type_off) - 1):
        s, e = type_off[g], type_off[g + 1]
        shift = w[s:e].max() - w[s:e]
        worst = max(sum(int(x) * int(y) << int(z) for x, y, z in zip(S[f, c, s:e], Q[s:e], shift))
                    for f in range(S.shape[0]) for c in range(3))
        assert worst < 2 ** 53, (g, worst.bit_length())


def _flux_exact_case(ops, rng, types, nframes, calls=None):
    """Build an exact system, check the precondition, run ops.charge_flux over the whole trajectory and compare with
    the oracle bit for bit."""
    vel, mass, q, seg_off, type_off = _exact_system(rng, types, nframes)
    _assert_exactly_representable(vel, mass, q, seg_off, type_off)
    want = O.charge_flux(vel, mass, q, seg_off, type_off, VS_EXACT, QS_EXACT)
    seg_d = _dev(seg_off, torch.int32)
    got = ops.charge_flux(_dev(vel), _dev(mass), _dev(q), seg_d, type_off, VS_EXACT, QS_EXACT).cpu().numpy()
    assert np.array_equal(got, want)
    assert np.count_nonzero(want) > 0.9 * want.size
    return vel, mass, q, seg_off, type_off, want


def _slots():
    return 2 * torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _lanes(nframes, nchunks):
    """frame lanes of one molecule type (mdp_charge_flux, csrc/reduce.cu)"""
    slots = _slots()
    return max(1, min(nframes, slots // max(1, min(nchunks, slots))))


def test_charge_flux_tiles_cross_molecules_exactly(ops):
    """Chunks of 2048 and 4905 atoms (2 and 4 tiles): a molecule starting exactly at A0 + 1408, one straddling that
    offset, one of 3000 atoms spanning three tiles; one frame per CTA, so both stages and both barrier parities turn
    over inside a frame."""
    rng = np.random.default_rng(101)
    big = [15] * 100 + [3000] + [15] * 99           # molecule 93 straddles 1408; molecule 100 is larger than a tile
    types = [[16] * 300, big]                        # 16 * 88 = 1408: molecules 88 and 216 start on a tile boundary
    assert 16 * 88 == FLUX_TILE and 15 * 93 < FLUX_TILE < 15 * 94 and 3000 > 2 * FLUX_TILE
    _flux_exact_case(ops, rng, types, 5)


def test_charge_flux_frame_walk_exactly(ops):
    """Eight chunks of two tiles each and F = 3 * lanes + 1 frames: every CTA walks at least three frames, reusing
    both stages and waiting on both parities several times, with the copies of its next frame in flight."""
    rng = np.random.default_rng(102)
    nchunks = 8
    lanes = _lanes(10 ** 6, nchunks)
    F = 3 * lanes + 1
    assert _lanes(F, nchunks) == lanes and lanes < F
    _flux_exact_case(ops, rng, [[16] * (FLUX_B * nchunks - 5)], F)


def test_charge_flux_many_chunks_exactly(ops):
    """More chunks than resident CTA slots (one frame lane) with single-atom molecules and a partial last chunk; a
    type of exactly one full chunk; a type of one molecule."""
    rng = np.random.default_rng(103)
    nmol = FLUX_B * (_slots() + 1) + 37
    assert _lanes(3, -(-nmol // FLUX_B)) == 1
    _flux_exact_case(ops, rng, [[1] * nmol, [3] * FLUX_B, [5]], 3)


def test_charge_flux_unaligned_rows_exactly(ops):
    """Molecule types starting at odd atom offsets, an odd atom count, velocities passed as one-frame views whose base
    is 8 mod 16 for odd frames, and masses and charges as views at an odd element offset: every row of a tile is
    copied with a shift of 0 and of 1."""
    rng = np.random.default_rng(104)
    types = [[7] * 3, [2] * 5, [3] * 130, [1], [5, 4]]          # first atoms 0, 21, 31, 421, 422; chunk 2 of type 3 at 415
    F = 6
    vel, mass, q, seg_off, type_off, want = _flux_exact_case(ops, rng, types, F)
    n = len(mass)
    assert n % 2 == 1
    vel_d = _dev(vel)
    buf = torch.zeros((2, n + 1), dtype=torch.float64, device="cuda")
    buf[0, 1:] = _dev(mass)
    buf[1, 1:] = _dev(q)
    mass_v, q_v = buf[0, 1:], buf[1, 1:]
    assert mass_v.data_ptr() % 16 == 8 and q_v.data_ptr() % 16 == 8
    seg_d = _dev(seg_off, torch.int32)
    got = ops.charge_flux(vel_d, mass_v, q_v, seg_d, type_off, VS_EXACT, QS_EXACT).cpu().numpy()
    assert np.array_equal(got, want)
    for k in range(F):
        v = vel_d[k:k + 1]
        assert v.data_ptr() % 16 == (8 if k % 2 else 0)
        for m_, q_ in ((mass_v, q_v), (_dev(mass), _dev(q))):
            got = ops.charge_flux(v, m_, q_, seg_d, type_off, VS_EXACT, QS_EXACT).cpu().numpy()
            assert np.array_equal(got[:, :, 0], want[:, :, k]), k


def test_charge_flux_out_and_frame0_exactly(ops):
    """Into a NaN-filled [3, G, Ttot] at frame0 > 0: the frames land in their columns, the other columns stay NaN, and
    two calls on disjoint frame ranges equal one call."""
    rng = np.random.default_rng(105)
    F, T0, Ttot = 9, 3, 16
    vel, mass, q, seg_off, type_off, want = _flux_exact_case(ops, rng, [[16] * 200, [1] * 50, [3] * 7], F)
    G = len(type_off) - 1
    args = (_dev(mass), _dev(q), _dev(seg_off, torch.int32), type_off, VS_EXACT, QS_EXACT)
    vel_d = _dev(vel)
    one = torch.full((3, G, Ttot), float("nan"), dtype=torch.float64, device="cuda")
    ops.charge_flux(vel_d, *args, out=one, frame0=T0)
    two = torch.full((3, G, Ttot), float("nan"), dtype=torch.float64, device="cuda")
    ops.charge_flux(vel_d[:4], *args, out=two, frame0=T0)
    ops.charge_flux(vel_d[4:], *args, out=two, frame0=T0 + 4)
    one, two = one.cpu().numpy(), two.cpu().numpy()
    assert np.array_equal(one[:, :, T0:T0 + F], want)
    assert np.isnan(one[:, :, :T0]).all() and np.isnan(one[:, :, T0 + F:]).all()
    assert np.array_equal(one, two, equal_nan=True)


def test_charge_flux_scratch_limit_is_a_clean_error(ops, fresh_ctx):
    from mdproptools_b200._lib import MdpropError
    rng = np.random.default_rng(106)
    vel, mass, q, seg_off, type_off = _exact_system(rng, [[4] * 300], 4)
    fresh_ctx(4096)
    with pytest.raises(MdpropError, match="exceeds the context limit"):
        ops.charge_flux(_dev(vel), _dev(mass), _dev(q), _dev(seg_off, torch.int32), type_off, VS_EXACT, QS_EXACT)


# ------------------------------------------------------------------------------------------------
# charge flux on realistic inputs: against the exact sum, to a rounding bound
# ------------------------------------------------------------------------------------------------
def _flux_exact_and_bound(vel, mass, q, seg_off, type_off, vs, qs, oracle=False):
    """(exact J [3, G, F] as Fractions of the double inputs, bound [3, G, F]).  Per molecule of k atoms the kernel's
    j = fl(fl(fl(acc / ws) * vs) * fl(qsum * qs)) carries, first order, (k + (k - 1) + (k - 1) + 4) u of
    P = |vs qs| * sum|m v| / sum m * sum|q|  (acc, ws and qsum are sequential sums); the sum over the molecules of a
    type is a tree of depth <= ceil(nchunks / 32) + 14 (two warp shuffles, four warp partials, the chunk loop of
    k_flux_finish).  So |got - exact| <= (3 kmax + ceil(nchunks / 32) + ceil(log2 M) + 16) 2^-53 sum P, the log2 M
    term covering the higher-order ones.  With ``oracle`` the bound is the numpy oracle's, whose dot product over the
    molecules is any order: M in place of the tree depth."""
    Fv = [[[Fraction(x) for x in row] for row in fr] for fr in vel]
    Fm = [Fraction(x) for x in mass]
    Fq = [Fraction(x) for x in q]
    fvs, fqs = Fraction(vs), Fraction(qs)
    T, G = len(vel), len(type_off) - 1
    exact = np.empty((3, G, T), dtype=object)
    bound = np.empty((3, G, T), dtype=object)
    u = Fraction(1, 2 ** 53)
    for g in range(G):
        mols = range(type_off[g], type_off[g + 1])
        M = len(mols)
        kmax = int(max(seg_off[s + 1] - seg_off[s] for s in mols))
        nchunks = -(-M // FLUX_B)
        depth = M if oracle else math.ceil(nchunks / 32) + math.ceil(math.log2(max(M, 2)))
        coef = 3 * kmax + depth + 16
        W = [sum(Fm[seg_off[s]:seg_off[s + 1]]) for s in mols]
        Q = [sum(Fq[seg_off[s]:seg_off[s + 1]]) * fqs for s in mols]
        Qabs = [sum(abs(x) for x in Fq[seg_off[s]:seg_off[s + 1]]) * abs(fqs) for s in mols]
        for t in range(T):
            for c in range(3):
                row = Fv[t][c]
                e = p = Fraction(0)
                for i, s in enumerate(mols):
                    a, b = seg_off[s], seg_off[s + 1]
                    e += sum(Fm[k] * row[k] for k in range(a, b)) / W[i] * fvs * Q[i]
                    p += sum(Fm[k] * abs(row[k]) for k in range(a, b)) / W[i] * abs(fvs) * Qabs[i]
                exact[c, g, t] = e
                bound[c, g, t] = coef * u * p
    return exact, bound


def _assert_within(got, exact, bound, what):
    for idx in np.ndindex(exact.shape):
        err = abs(Fraction(float(got[idx])) - exact[idx])
        assert err <= bound[idx], (what, idx, float(err), float(bound[idx]))


def test_charge_flux_realistic_inputs_within_rounding_bound(ops):
    """Real masses and unit conversions, velocities ~1e-3, ragged molecule types (591 x 16, 66 x 15, 33 x 1 atoms):
    every J within the rounding bound of the exact value."""
    from mdproptools_b200.common import constants
    rng = np.random.default_rng(107)
    num_mols, num_atoms = [591, 66, 33], [16, 15, 1]
    sizes = np.repeat(num_atoms, num_mols)
    seg_off = np.concatenate(([0], np.cumsum(sizes))).astype(np.int64)
    type_off = np.concatenate(([0], np.cumsum(num_mols))).astype(np.int64)
    n, F = int(seg_off[-1]), 3
    mass = rng.choice(np.asarray(MASS), n)
    q = rng.normal(0.0, 0.4, n)
    vel = rng.normal(0.0, 1e-3, (F, 3, n))
    vs, qs = constants.VELOCITY_CONVERSION["real"], constants.CHARGE_CONVERSION["real"]
    got = ops.charge_flux(_dev(vel), _dev(mass), _dev(q), _dev(seg_off, torch.int32), type_off, vs, qs).cpu().numpy()
    exact, bound = _flux_exact_and_bound(vel, mass, q, seg_off, type_off, vs, qs)
    _assert_within(got, exact, bound, "kernel")


def test_charge_flux_fluctuating_charges_through_the_api(ops, tmp_path, monkeypatch):
    """A dump whose charges change every frame: Conductivity.get_charge_flux takes one call per frame (on one-frame
    views of the batch) and equals the exact flux to the rounding bound, and the oracle applied frame by frame to the
    sum of both bounds."""
    from mdproptools_b200.common import constants
    from mdproptools_b200.dynamical import conductivity as cmod
    rng = np.random.default_rng(108)
    num_mols, num_atoms = [20, 15, 6], [5, 3, 1]
    templates = [[1, 2, 3, 3, 3], [4, 5, 6], [9]]
    types = np.concatenate([np.tile(t, k) for t, k in zip(templates, num_mols)])
    n, F, L = len(types), 6, 30.0
    seg_off = np.concatenate(([0], np.cumsum(np.repeat(num_atoms, num_mols)))).astype(np.int64)
    type_off = np.concatenate(([0], np.cumsum(num_mols))).astype(np.int64)
    q = rng.normal(0.0, 0.5, (F, n))
    vel = rng.normal(0.0, 1e-3, (F, 3, n))
    for t in range(F):
        with open(tmp_path / f"dump.fq.{t * 10}.dump", "w") as f:
            f.write(f"ITEM: TIMESTEP\n{t * 10}\nITEM: NUMBER OF ATOMS\n{n}\nITEM: BOX BOUNDS pp pp pp\n")
            f.write(f"0.0 {L!r}\n0.0 {L!r}\n0.0 {L!r}\nITEM: ATOMS id type q vx vy vz\n")
            for i in rng.permutation(n):
                vals = (float(q[t, i]), float(vel[t, 0, i]), float(vel[t, 1, i]), float(vel[t, 2, i]))
                f.write(f"{i + 1} {int(types[i])} " + " ".join(repr(v) for v in vals) + "\n")
    frames_per_call = []
    real = cmod.ops.charge_flux

    def counting(vel_d, *a, **k):
        frames_per_call.append(vel_d.shape[0])
        return real(vel_d, *a, **k)

    monkeypatch.setattr(cmod.ops, "charge_flux", counting)
    c = cmod.Conductivity("dump.fq.*.dump", num_mols, num_atoms, volume=L ** 3, mass=MASS, working_dir=str(tmp_path))
    J = c.get_charge_flux()
    assert frames_per_call == [1] * F
    mass = np.asarray(MASS)[types - 1]
    vs, qs = constants.VELOCITY_CONVERSION["real"], constants.CHARGE_CONVERSION["real"]
    for t in range(F):
        exact, bound = _flux_exact_and_bound(vel[t:t + 1], mass, q[t], seg_off, type_off, vs, qs)
        _, bound_o = _flux_exact_and_bound(vel[t:t + 1], mass, q[t], seg_off, type_off, vs, qs, oracle=True)
        _assert_within(J[:, :, t:t + 1], exact, bound, ("api", t))
        want = O.charge_flux(vel[t:t + 1], mass, q[t], seg_off, type_off, vs, qs)
        _assert_within(want, exact, bound_o, ("oracle", t))
        for idx in np.ndindex(want.shape):
            assert abs(Fraction(float(J[idx[0], idx[1], t])) - Fraction(float(want[idx]))) <= bound[idx] + bound_o[idx]


# ------------------------------------------------------------------------------------------------
# scratch-limited batching: pair engine frame sub-batches, FFT channel groups
# ------------------------------------------------------------------------------------------------
LIMIT_MAX = 64 << 20


def _sweep(install, run, count, fine_step, fine_span):
    """Run ``run()`` on a fresh context for each scratch limit of a ladder: a bisection down to 256 B towards the
    smallest limit that works, a few limits just below, steps of ``fine_step`` over ``fine_span`` below and above (the
    bisection lands on *a* boundary; if success were not monotone, working limits below it would show up), then x1.5
    up to 64 MB.  Returns {limit: (result, count(ctx)) or the error message}."""
    from mdproptools_b200._lib import MdpropError
    seen = {}

    def attempt(limit):
        if limit not in seen:
            ctx = install(limit)
            try:
                seen[limit] = (run(), count(ctx))
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
    for k in range(1, 4):
        attempt(hi - 64 * k)
    for k in range(-(fine_span // fine_step), fine_span // fine_step + 1):
        if hi + k * fine_step > 0:
            attempt(hi + k * fine_step)
    lim = hi + fine_span
    while lim < LIMIT_MAX:
        attempt(lim)
        lim = int(lim * 1.5)
    return seen


def _check_sweep(seen, same):
    """Success is monotone in the limit, failures are the scratch refusal and nothing else, the unit count (sub-batches,
    channel groups) never grows with the limit, and every result equals ``same``.  Returns the unit counts seen."""
    ok = sorted(l for l, v in seen.items() if not isinstance(v, str))
    bad = sorted(l for l, v in seen.items() if isinstance(v, str))
    for l in bad:
        assert "exceeds the context limit" in seen[l], (l, seen[l])
    first = ok[0]
    above = [l for l in bad if l > first]

    def units_below(l):
        lower = [k for k in ok if k < l]
        return seen[lower[-1]][1] if lower else None

    assert not above, ("limits that fail above the smallest working limit %d B: " % first +
                       ", ".join("%d B (%d units just below)" % (l, units_below(l)) for l in above[:8]) +
                       " -- %d of %d such limits" % (len(above), len([l for l in seen if l > first])))
    units = [seen[l][1] for l in ok]
    assert all(a >= b for a, b in zip(units, units[1:])), list(zip(ok, units))
    for l in ok:
        assert same(seen[l][0]), l
    return set(units)


def _pair_inputs():
    rng = np.random.default_rng(111)
    F, n, nb_pts = 9, 2000, 700
    Ls = np.stack([rng.uniform(24.0, 28.0, F), rng.uniform(24.0, 28.0, F), rng.uniform(24.0, 28.0, F)], axis=1)
    cells = np.concatenate([Ls, rng.uniform(-4.0, 4.0, (F, 3))], axis=1)
    xa = rng.uniform(0, 1, (F, 3, n)) * Ls[:, :, None]
    xb = rng.uniform(0, 1, (F, 3, nb_pts)) * Ls[:, :, None]
    s = rng.uniform(0, 1, (F, 3, n))
    tri = np.stack([s[:, 0] * cells[:, 0:1] + s[:, 1] * cells[:, 3:4] + s[:, 2] * cells[:, 4:5],
                    s[:, 1] * cells[:, 1:2] + s[:, 2] * cells[:, 5:6], s[:, 2] * cells[:, 2:3]], axis=1)
    ca = rng.integers(0, 2, (F, n)).astype(np.int32)          # per-frame classes: the class rows move with the frames
    cb = rng.integers(0, 2, (F, nb_pts)).astype(np.int32)
    return Ls, cells, xa, xb, tri, ca, cb


PAIR_RC, PAIR_DDR, PAIR_NB = 6.0, 0.1, 60
REL = np.array([[1, 1], [1, 2], [2, 2]])


@pytest.mark.parametrize("variant", ["symmetric", "symmetric_f64", "rectangular", "rectangular_f64", "triclinic",
                                     "triclinic_f64", "shell_list"])
def test_pair_engine_frame_subbatches_under_scratch_limits(ops, fresh_ctx, monkeypatch, variant):
    """9 frames with their own boxes (and classes), swept over scratch limits on fresh contexts: every limit that works
    gives the unlimited result, which equals the oracle frame by frame; the sweep sees one frame per sub-batch and
    sub-batches that do not divide 9; sub-batches never grow and calls never fail again above the smallest working
    limit (the batch size accounts for everything the scratch request adds)."""
    from mdproptools_b200._lib import PAIR_F64, PAIR_TRICLINIC, bin_edges
    Ls, cells, xa, xb, tri, ca, cb = _pair_inputs()
    F = len(Ls)
    edges = bin_edges(PAIR_DDR, PAIR_NB)
    rc2 = O.rcut_sq(PAIR_RC)
    flags = PAIR_F64 if variant.endswith("_f64") else 0
    if variant.startswith("symmetric"):
        a, cl = _dev(xa), _dev(ca)

        def run():
            return ops.pair_hist(a, cl, 2, Ls, rc2, edges, PAIR_DDR, flags=flags)
    elif variant.startswith("rectangular"):
        a, b, cl, clb = _dev(xa), _dev(xb), _dev(ca), _dev(cb)

        def run():
            return ops.pair_hist(a, cl, 2, Ls, rc2, edges, PAIR_DDR, xyz_b=b, cls_b=clb, ncls_b=2, flags=flags)
    elif variant.startswith("triclinic"):
        a, cl = _dev(tri), _dev(ca)

        def run():
            return ops.pair_hist(a, cl, 2, cells, rc2, edges, PAIR_DDR, flags=flags | PAIR_TRICLINIC)
    else:
        monkeypatch.setenv("MDP_SHELL_GRID", "0")                 # the general engine's list mode
        a, b = _dev(xa[:, :, :150]), _dev(xa)
        r_in, r_out = 1.0, 4.0

        def run():
            lst, _ = ops.pair_list(a, b, Ls, r_in * r_in, r_out * r_out, 1)
            lst = lst.cpu().numpy().astype(np.int64)
            return torch.from_numpy(np.sort((lst[:, 0] * 150 + lst[:, 1]) * xa.shape[2] + lst[:, 2]))

    ref = run()                                                    # the default context: one sub-batch
    got = ref.cpu().numpy()
    for f in range(F):
        if variant.startswith("symmetric") or variant.startswith("triclinic"):
            pos = tri[f] if variant.startswith("triclinic") else xa[f]
            loop = O.rdf_loop_tri if variant.startswith("triclinic") else O.rdf_loop
            full, part = loop(ca[f] + 1.0, pos[0], pos[1], pos[2], REL, cells[f] if variant.startswith("triclinic") else Ls[f],
                              PAIR_RC, PAIR_DDR, PAIR_NB, nthreads=0)
            h = got[f]                                             # rows (0,0), (0,1), (1,1)
            assert np.array_equal(2 * h.sum(axis=0), full), f
            assert np.array_equal(np.stack([2 * h[0], h[1], 2 * h[2]]), part), f
        elif variant.startswith("rectangular"):
            rel = np.array([[1, 1], [1, 2], [2, 1], [2, 2]])       # row i * 2 + j
            part = O.rdf_rect(ca[f] + 1.0, xa[f, 0], xa[f, 1], xa[f, 2], cb[f] + 1.0, xb[f, 0], xb[f, 1], xb[f, 2], rel,
                              Ls[f], PAIR_RC, PAIR_DDR, PAIR_NB, nthreads=0)
            assert np.array_equal(got[f], part), f
        else:
            h = O.shell_mask(xa[f, 0, :150], xa[f, 1, :150], xa[f, 2, :150], xa[f, 0], xa[f, 1], xa[f, 2], Ls[f], r_in, r_out,
                             False)
            ia, ib = np.nonzero(h)
            want = np.sort((f * 150 + ia.astype(np.int64)) * xa.shape[2] + ib)
            mine = got[(got // (150 * xa.shape[2])) == f]
            assert len(want) > 0 and np.array_equal(mine, want), f
    assert got.sum() > 0

    seen = _sweep(fresh_ctx, run, lambda ctx: ctx.timing_read(0)[1], 16 << 10, 1 << 20)
    batches = _check_sweep(seen, lambda r: torch.equal(r, ref))
    # 9 sub-batches = one frame each; 5 = two frames each (the last sub-batch holds one); 1 = all frames
    assert {9, 5, 1} <= batches, sorted(batches)


def test_fft_correlation_channel_groups_under_scratch_limits(ops, fresh_ctx, monkeypatch):
    """7 channels of 4097 steps, 1500 lags, swept over scratch limits on fresh contexts: groups of 1, 2 and 3 channels
    occur; every grouping gives the same bits (a channel's arithmetic does not depend on its group), within 1e-10 of
    max|C| of the direct kernel; groups never shrink and calls never fail again above the smallest working limit."""
    rng = np.random.default_rng(112)
    C, T, nlags = 7, 4097, 1500
    a = np.cumsum(rng.normal(0, 1, (C, T)), axis=1) * 0.05 + rng.normal(0, 1, (C, T))
    b = a.copy()
    b[4:] = rng.normal(0, 2, (C - 4, T))
    a_d, b_d = _dev(a), _dev(b)
    monkeypatch.setenv("MDP_XCORR_FFT", "0")
    direct = ops.xcorr_unbiased(a_d, b_d, nlags).cpu().numpy()
    monkeypatch.setenv("MDP_XCORR_FFT", "1")
    ref = ops.xcorr_unbiased(a_d, b_d, nlags)
    for c in range(C):
        assert np.abs(ref[c].cpu().numpy() - direct[c]).max() <= 1e-10 * np.abs(direct[c]).max()

    # launches of one call: the twiddle table, then the same passes for every group
    ctx = fresh_ctx(LIMIT_MAX)
    ops.xcorr_unbiased(a_d, b_d, nlags)
    per_group = ctx.launch_count() - 1

    def groups(ctx):
        k = ctx.launch_count() - 1
        assert k % per_group == 0, k
        return k // per_group

    seen = _sweep(fresh_ctx, lambda: ops.xcorr_unbiased(a_d, b_d, nlags), groups, 4 << 10, 1 << 20)
    ngroups = _check_sweep(seen, lambda r: torch.equal(r, ref))
    assert {7, 4, 3, 1} <= ngroups, sorted(ngroups)            # groups of one, two, three and all seven channels
