"""Every sample rate the engine accepts (N = s * 1023 samples per ms, s in 1, 2, 3, 4, 5, 6, 8, 10, 12, 16) on every build of
the correlate kernel, through the C ABI, against the float64 oracle.

The planner picks a build from the launch shape; GB200_W2048, GB200_NP and GB200_RSPLIT (INTEGRATION.md) force the others.
They are read when an engine is created, so every engine here is created under its own settings.  Tolerances (DESIGN.md
section 6): peak and sum |gpu - ref| <= 1e-5 * max(ref); count exact; argmax exact except where the oracle's own float64 profile
ties to within that tolerance; strength within 1e-4.  Builds that share a kernel body compute the same per-lag values and merge
their per-warp peaks order-free, so they agree bit for bit in peak / argmax / count (the float64 sum to its summation order)."""
import functools
import math
import multiprocessing as mp
import os

import numpy as np
import pytest

from oracle import gypsum_oracle as o

pytestmark = pytest.mark.gpu
MAG_TOL = 1e-5
RATES = [1, 2, 3, 4, 5, 6, 8, 10, 12, 16]
LAG_CHIPS = [0, 31, 32, 511, 512, 1021, 1022]  # chip lags q at the lane / half / end boundaries of the kernels' lag layout
DOP = np.array([-7500.0, -5000.0, -2500.0, 0.0, 2500.0, 5000.0, 7500.0])  # a prime count: every PRN's last chunk is partly filled
N_BLOCKS = 8
SVS = list(range(1, 33))
KNOBS = ("GB200_W2048", "GB200_NP", "GB200_RSPLIT", "GB200_SPEC_BUDGET_MB")

# (build, settings, CTA slots a cell's polyphase branches are split over: warps of the one-warp kernel, pairs of the pair kernel)
SINGLE_MS = [("w2048<12>", {}, 12), ("w2048<10>", {"GB200_W2048": 10}, 10), ("pair np10", {"GB200_W2048": 0}, 10),
             ("pair np8", {"GB200_W2048": 0, "GB200_NP": 8}, 8)]
FOUR_MS = [("w2048<8>", {}, 8), ("pair np8", {"GB200_W2048": 0}, 8)]
COHERENT = [("pair np8", {}, 8)]  # coherent launches always run on the 8-pair build

ERR = {}  # s -> largest |gpu - ref| / max(ref) seen by this file


def rsplits(s, slots):
    """Every split GB200_RSPLIT can force on this build: the divisors of gcd(s, slots) (pick_rsplit ignores any other)."""
    g = math.gcd(s, slots)
    return [d for d in range(1, g + 1) if g % d == 0]


def variants(s, builds):
    """(build name, engine settings) of every build x every valid split."""
    return [(f"{name} rsplit {d}", dict(knobs, GB200_RSPLIT=d)) for name, knobs, slots in builds for d in rsplits(s, slots)]


@pytest.fixture(scope="module")
def engine(native_lib):
    from gypsum_b200 import _native

    cache = {}
    chips = np.stack([o.ca_code(sv) for sv in SVS]).astype(np.uint8)

    def get(s, **knobs):
        key = (s, tuple(sorted(knobs.items())))
        if key not in cache:
            saved = {k: os.environ.pop(k, None) for k in KNOBS}
            os.environ.update({k: str(v) for k, v in knobs.items()})
            try:
                e = _native.Engine(1023 * s * 1000, 1023 * s)
            finally:
                for k, v in saved.items():
                    os.environ.pop(k, None)
                    if v is not None:
                        os.environ[k] = v
            e.set_replicas(chips)
            cache[key] = e
        return cache[key]

    yield get
    for e in cache.values():
        e.close()
    print("\nlargest |gpu - ref| / max(ref) per s:", {s: float(f"{v:.2e}") for s, v in sorted(ERR.items())})


def note_err(s, got, ref):
    ERR[s] = max(ERR.get(s, 0.0), float(np.abs(got - ref).max() / np.abs(ref).max()))


def _pool_map(fn, jobs):
    with mp.get_context("fork").Pool(max(1, min(len(jobs), os.cpu_count() or 1))) as pool:
        return pool.map(fn, jobs)


@functools.lru_cache(maxsize=None)
def planted_input(s, n_ms):
    """N_BLOCKS independent blocks of n_ms ms.  In block b every PRN a is planted at its own code phase tau[b, a] and Doppler
    DOP[dbin[b, a]]; over the 256 (block, PRN) slots the code phases take every pair (q, r) of a boundary chip lag q in
    LAG_CHIPS and a residue r (tau = s q + r, so also 0 and N - 1), the other slots random ones."""
    n = 1023 * s
    rng = np.random.default_rng(s)
    tau = rng.integers(0, n, N_BLOCKS * 32)
    tau[rng.permutation(N_BLOCKS * 32)[:7 * s]] = [s * q + r for r in range(s) for q in LAG_CHIPS]
    tau = tau.reshape(N_BLOCKS, 32)
    dbin = rng.integers(0, len(DOP), (N_BLOCKS, 32))
    phase = rng.uniform(0, 2 * np.pi, (N_BLOCKS, 32))
    x = np.concatenate([o.synth_iq(100 * s + b, n, n_ms, 1000 * n,
                                   [(a + 1, DOP[dbin[b, a]], int(tau[b, a]), phase[b, a], 1.0) for a in range(32)], sigma=0.3)
                        for b in range(N_BLOCKS)])
    return x, tau, dbin


def _oracle_block(args):
    x, n, dop, kind = args
    return o.grid_cells(x, 1000 * n, n, SVS, list(dop), kind)


@functools.lru_cache(maxsize=None)
def oracle_records(s, n_ms):
    """o.grid_cells of every block of planted_input(s, n_ms): (peak, argmax, sum, count), each [N_BLOCKS, 32, len(DOP)]."""
    n = 1023 * s
    x = planted_input(s, n_ms)[0]
    parts = _pool_map(_oracle_block, [(x[b * n_ms * n:(b + 1) * n_ms * n], n, DOP, o.NON_COHERENT) for b in range(N_BLOCKS)])
    return tuple(np.stack(p) for p in zip(*parts))


def check_records(rec, ref, x, s, dop, kind, what):
    """rec: [blocks, PRN, Doppler] records of the blocks of x; ref: the oracle's (peak, argmax, sum, count) of the same cells."""
    n = 1023 * s
    m = len(x) // (rec.shape[0] * n)
    peak, arg, total, count = ref
    note_err(s, rec["peak"], peak)
    note_err(s, rec["sum"], total)
    assert np.abs(rec["peak"] - peak).max() <= MAG_TOL * peak.max(), what
    assert np.abs(rec["sum"] - total).max() <= MAG_TOL * total.max(), what
    assert np.array_equal(rec["count"], count), what
    for b, a, d in np.argwhere(rec["argmax"] != arg):  # only where the float64 profile itself ties to within the tolerance
        prof = np.abs(o.integrate(kind, x[b * m * n:(b + 1) * m * n], 1000 * n, n, dop[d], o.replica(a + 1, n)))
        assert prof.max() - prof[rec["argmax"][b, a, d]] <= MAG_TOL * prof.max(), (what, b, a, d)
    strength = rec["peak"] / ((rec["sum"] - rec["count"] * rec["peak"].astype(np.float64)) / (n - rec["count"]))
    ref_strength = peak / ((total - count * peak) / (n - count))
    assert np.abs(strength - ref_strength).max() <= 1e-4 * ref_strength.max(), what


def assert_same_cells(a, b, what):
    """Two builds of one kernel body: bit-identical peak / argmax / count / probe, the float64 sum to its summation order."""
    for k in ("peak", "argmax", "count", "probe_re", "probe_im"):
        assert np.array_equal(a[k], b[k]), (what, k)
    assert (np.abs(a["sum"] - b["sum"]) <= 1e-12 * np.abs(b["sum"])).all(), what


@pytest.mark.parametrize("s", RATES)
def test_profiles_at_every_rate(engine, s):
    """Full profiles (the 8-pair build with PROFILE=true, rsplit gcd(s, 8)), non-coherent and coherent, 1 and 3 ms, at a
    fractional Doppler carrying a signal and at one beyond the search range, every value against the oracle."""
    from gypsum_b200 import _native

    n, fs = 1023 * s, 1023000 * s
    tau = s * 700 + s - 1
    x = o.synth_iq(40 + s, n, 3, fs, [(7, -2750.4, tau, 0.7, 0.5)])
    e = engine(s)
    e.upload_iq(x)
    for f in (-2750.4, 23000.0):
        for m in (1, 3):
            what = (f, m)
            prn = o.replica(7, n)
            ref = o.integrate(o.NON_COHERENT, x[:m * n], fs, n, f, prn)
            refc = o.integrate(o.COHERENT, x[:m * n], fs, n, f, prn)
            nc = e.correlation_profile(6, f, m, _native.NON_COHERENT)
            co = e.correlation_profile(6, f, m, _native.COHERENT)
            note_err(s, nc, ref)
            note_err(s, co, refc)
            assert np.abs(nc - ref).max() <= MAG_TOL * ref.max(), what
            assert np.abs(co - refc).max() <= MAG_TOL * np.abs(refc).max(), what
            for got, want in ((nc, ref), (np.abs(co), np.abs(refc))):
                assert want.max() - want[int(got.argmax())] <= MAG_TOL * want.max(), what
            if f < 0:
                assert int(nc.argmax()) == int(ref.argmax()) == tau and int(np.abs(co).argmax()) == tau, what


@pytest.mark.parametrize("s", RATES)
def test_index_map_at_every_rate(engine, s):
    """8 blocks x 32 PRNs x 7 Doppler bins on the default build: every (block, PRN) reports its planted code phase, exactly, at
    its planted bin -- residues 0 .. s-1, the chip lags either side of each lane / half boundary, 0 and N - 1 -- and every record
    matches the oracle."""
    x, tau, dbin = planted_input(s, 1)
    ref = oracle_records(s, 1)
    e = engine(s)
    e.upload_iq(x)
    rec = e.acquire_grid(N_BLOCKS, 1, np.arange(32), DOP)
    b, a = np.indices(tau.shape)
    assert np.array_equal(ref[1][b, a, dbin], tau)  # the input: every planted peak is unambiguous in float64
    assert np.array_equal(rec["argmax"][b, a, dbin], tau)
    check_records(rec, ref, x, s, DOP, o.NON_COHERENT, "default build")


def run_builds(engine, s, n_ms, builds, kind=None):
    """Records of the 8-block planted grid under every (build, split); the 1-block grid of each is its block 0, to the bit."""
    x = planted_input(s, n_ms)[0]
    out = {}
    for name, knobs in variants(s, builds):
        e = engine(s, **knobs)
        e.upload_iq(x)
        rec = e.acquire_grid(N_BLOCKS, n_ms, np.arange(32), DOP)
        one = e.acquire_grid(1, n_ms, np.arange(32), DOP)
        assert np.array_equal(one.view(np.uint8), rec[:1].view(np.uint8)), name
        out[name] = rec
    return x, out


@pytest.mark.parametrize("s", RATES)
def test_single_ms_builds(engine, s):
    """Non-coherent, 1 ms: w2048<12> (default), w2048<10>, pair np10, pair np8, each at every split, against the oracle; the
    splits of a build, w2048<12> vs w2048<10>, and pair np10 vs pair np8 bit for bit."""
    x, recs = run_builds(engine, s, 1, SINGLE_MS)
    ref = oracle_records(s, 1)
    for name, rec in recs.items():
        check_records(rec, ref, x, s, DOP, o.NON_COHERENT, name)
    for group in (("w2048<12>", "w2048<10>"), ("pair np10", "pair np8")):
        same = [rec for name, rec in recs.items() if name.rsplit(" rsplit", 1)[0] in group]
        for rec in same[1:]:
            assert_same_cells(rec, same[0], group)


@pytest.mark.parametrize("s", RATES)
def test_four_ms_builds(engine, s):
    """Non-coherent, 4 ms: w2048<8, multi-ms> (default) and pair np8, each at every split, against the oracle; the splits of
    one build bit for bit."""
    x, recs = run_builds(engine, s, 4, FOUR_MS)
    ref = oracle_records(s, 4)
    for name, rec in recs.items():
        check_records(rec, ref, x, s, DOP, o.NON_COHERENT, name)
    for build, _, _ in FOUR_MS:
        same = [rec for name, rec in recs.items() if name.startswith(build + " ")]
        for rec in same[1:]:
            assert_same_cells(rec, same[0], build)


def _coherent_sv(args):
    x, n, sv, probes = args
    out = []
    for f, p in zip(DOP, probes):
        prof = o.integrate(o.COHERENT, x, 1000 * n, n, f, o.replica(sv, n))
        mag = np.abs(prof)
        out.append((mag.max(), int(mag.argmax()), mag.sum(), int(np.count_nonzero(mag == mag.max())), prof[p]))
    return out


@pytest.mark.parametrize("s", RATES)
def test_coherent_builds_with_probes(engine, s):
    """Coherent, 2 ms, list mode on the split kernels: pair np8 at every split.  Probes at every residue mod s, at lags 0 and
    N - 1 and at each planted peak == the oracle's complex profile there; the splits bit for bit, probes included."""
    from gypsum_b200 import _native

    n = 1023 * s
    x_all, tau, dbin = planted_input(s, 2)
    x = x_all[:2 * n]  # list mode reads the first 2 ms: block 0
    cycle = [0, n - 1] + [s * LAG_CHIPS[r % 7] + r for r in range(s)]
    probe = np.array([cycle[k % len(cycle)] for k in range(32 * len(DOP))]).reshape(32, len(DOP))
    probe[np.arange(32), dbin[0]] = tau[0]
    ref = _pool_map(_coherent_sv, [(x, n, sv, probe[sv - 1]) for sv in SVS])
    peak, arg, total, count, pval = (np.array([[c[k] for c in row] for row in ref]) for k in range(5))
    prn = np.repeat(np.arange(32), len(DOP))
    dop = np.tile(DOP, 32)
    first = None
    for name, knobs in variants(s, COHERENT):
        e = engine(s, **knobs)
        e.upload_iq(x)
        e.set_fused(False)
        try:
            rec = e.acquire_cells(prn, dop, 2, _native.COHERENT, probe_idx=probe.ravel()).reshape(1, 32, len(DOP))
        finally:
            e.set_fused(None)
        check_records(rec, (peak[None], arg[None], total[None], count[None]), x, s, DOP, o.COHERENT, name)
        got = rec["probe_re"][0] + 1j * rec["probe_im"][0].astype(np.float64)
        note_err(s, got, pval)
        assert (np.abs(got - pval) <= MAG_TOL * peak).all(), name
        assert np.array_equal(rec["argmax"][0, np.arange(32), dbin[0]], tau[0]), name
        if first is None:
            first = rec
        assert_same_cells(rec, first, name)


def all_builds(s):
    """(launch, build, settings) of every non-coherent and coherent build at every split."""
    return ([("nc", 1, name, k) for name, k in variants(s, SINGLE_MS)] + [("nc", 4, name, k) for name, k in variants(s, FOUR_MS)]
            + [("co", 2, name, k) for name, k in variants(s, COHERENT)])


@pytest.mark.parametrize("s", RATES)
def test_all_zero_input(engine, s):
    """Every profile value ties at 0: peak 0, argmax 0, sum 0 and count exactly N on every build.  N + s would mean the lag
    q = 1023, which does not exist, took part in the reduction."""
    from gypsum_b200 import _native

    n = 1023 * s
    for launch, m, name, knobs in all_builds(s):
        e = engine(s, **knobs)
        e.upload_iq(np.zeros(8 * n, np.complex64))
        if launch == "nc":
            rec = e.acquire_grid(2, m, [0, 31], DOP[:3]).ravel()
        else:
            e.set_fused(False)
            try:
                rec = e.acquire_cells([0, 31, 5], DOP[:3], m, _native.COHERENT, probe_idx=[0, n - 1, s - 1])
            finally:
                e.set_fused(None)
        what = (launch, name)
        assert (rec["peak"] == 0).all() and (rec["argmax"] == 0).all() and (rec["sum"] == 0).all(), what
        assert (rec["count"] == n).all(), what
        assert (rec["probe_re"] == 0).all() and (rec["probe_im"] == 0).all(), what


@pytest.mark.parametrize("s", RATES)
def test_duplicate_doppler_bins(engine, s):
    """An axis with the same Doppler twice computes two identical records, and acquire_grid_best reports the first of the two
    bins (acquisition.py:180-182 takes the first bin among equal maxima), on every non-coherent build."""
    n, fs = 1023 * s, 1023000 * s
    axis = np.array([-1000.0, 500.0, 500.0, 2000.0, -3000.0])
    planted = [(sv, 500.0, (331 * sv) % n, 0.1 * sv, 0.4) for sv in (1, 4, 9, 17, 30)] + [(12, 2000.0, n - 1, 0.0, 0.4)]
    x = o.synth_iq(60 + s, n, 4, fs, planted)
    for launch, m, name, knobs in all_builds(s):
        if launch != "nc":
            continue
        e = engine(s, **knobs)
        e.upload_iq(x)
        rec = e.acquire_grid(1, m, np.arange(32), axis)[0]
        best = e.acquire_grid_best(1, m, np.arange(32), axis)[0]
        assert rec[:, 1].tobytes() == rec[:, 2].tobytes(), name
        want = np.argmax(rec["peak"], axis=1)  # first bin of the row maximum
        assert np.array_equal(best["bin"], want) and not (best["bin"] == 2).any(), name
        assert np.array_equal(best["code_phase"], rec["argmax"][np.arange(32), want]), name
        for sv, f, t, _, _ in planted:
            assert (best["bin"][sv - 1], best["code_phase"][sv - 1]) == (1 if f == 500.0 else 3, t), (name, sv)


def _long_sv(args):
    x, n, sv, dop = args
    return o.grid_cells(x, 1000 * n, n, [sv], list(dop))


@pytest.mark.parametrize("s", [1, 16])
def test_long_integration(engine, s):
    """M = 20 non-coherent: the multi-ms one-warp build accumulates 20 ms in its registers (and the pair build for comparison)."""
    n, fs, m = 1023 * s, 1023000 * s, 20
    dop = DOP[1:6]
    planted = [(1, -2500.0, n - 1, 0.3, 0.12), (2, 0.0, 0, 1.0, 0.12), (5, 5000.0, s * 512 + s // 2, 2.0, 0.12)]
    x = o.synth_iq(70 + s, n, m, fs, planted)
    svs = list(range(1, 9))
    parts = _pool_map(_long_sv, [(x, n, sv, dop) for sv in svs])
    ref = tuple(np.concatenate(p)[None] for p in zip(*parts))
    for name, knobs in (("w2048<8>", {}), ("pair np8", {"GB200_W2048": 0})):
        e = engine(s, **knobs)
        e.upload_iq(x)
        rec = e.acquire_grid(1, m, np.array(svs) - 1, dop)
        check_records(rec, ref, x, s, dop, o.NON_COHERENT, name)
        for sv, f, t, _, _ in planted:
            assert rec["argmax"][0, sv - 1, list(dop).index(f)] == t, (name, sv)


@pytest.mark.parametrize("s", [7, 9, 11, 13, 17])
def test_unsupported_rates_are_refused(native_lib, s):
    from gypsum_b200 import _native

    with pytest.raises(ValueError):
        _native.Engine(1023 * s * 1000, 1023 * s)


def test_generic_replica_at_s5(engine):
    """correlation_profile_replica (the direct kernel for any complex replica) at 5.115 Msps, both kinds, 2 ms."""
    from gypsum_b200 import _native

    s = 5
    n, fs = 1023 * s, 1023000 * s
    x = o.synth_iq(80, n, 2, fs, [(9, 1250.0, 4000, 0.4, 0.4)])
    rng = np.random.default_rng(5)
    rep = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    e = engine(s)
    e.upload_iq(x)
    for kind, okind in ((_native.NON_COHERENT, o.NON_COHERENT), (_native.COHERENT, o.COHERENT)):
        got = e.correlation_profile_replica(rep, 1250.0, 2, kind)
        ref = o.integrate(okind, x, fs, n, 1250.0, rep.astype(complex))
        note_err(s, got, ref)
        assert np.abs(got - ref).max() <= MAG_TOL * np.abs(ref).max(), kind


def test_grid_host_eager_capture_replay_at_s6(engine):
    """acquire_grid_host at 6.138 Msps: the eager call, the captured one and the replay == acquire_grid == the oracle."""
    s = 6
    x, _, _ = planted_input(s, 1)
    e = engine(s)
    e.upload_iq(x)
    want = e.acquire_grid(N_BLOCKS, 1, np.arange(32), DOP)
    check_records(want, oracle_records(s, 1), x, s, DOP, o.NON_COHERENT, "acquire_grid")
    for call in ("eager", "capture", "replay"):
        got = e.acquire_grid_host(x, N_BLOCKS, 1, np.arange(32), DOP)
        assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), call


def test_scratch_batches_at_s10(engine):
    """10.23 Msps with a 3 MB spectra budget (two blocks per batch): every record lands where one batch puts it, to the bit."""
    s = 10
    x, _, _ = planted_input(s, 1)
    small, big = engine(s, GB200_SPEC_BUDGET_MB=3), engine(s)
    for e in (small, big):
        e.upload_iq(x)
    a = small.acquire_grid(N_BLOCKS, 1, np.arange(32), DOP)
    b = big.acquire_grid(N_BLOCKS, 1, np.arange(32), DOP)
    assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    check_records(a, oracle_records(s, 1), x, s, DOP, o.NON_COHERENT, "batched")
