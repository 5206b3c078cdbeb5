"""Every BASELINE.json configuration compared with the oracle CELL FOR CELL at its full size, through the C ABI.

Tolerances (DESIGN.md section 6): magnitudes / sums |gpu - ref| <= 1e-5 * max(ref); count exact; code phase exact unless the
ORACLE's own profile shows a near-tie at the two indices (proved per mismatch, never as a percentage).  The oracle grids
are spread over the host's cores (fork pool) so the file runs in well under a minute on the GPU box."""
import multiprocessing as mp
import os

import numpy as np
import pytest

from oracle import gypsum_oracle as o
from oracle import tracker_oracle as t

pytestmark = pytest.mark.gpu
MAG_TOL = 1e-5


def _cells_worker(args):
    x, fs, n, svs, dop = args
    return o.grid_cells(x, fs, n, svs, dop)


def oracle_grid(x, fs, n, svs, dop):
    """o.grid_cells over all SVs, one process per SV group."""
    procs = max(1, min(len(svs), os.cpu_count() or 1))
    parts = [svs[i::procs] for i in range(procs)]
    with mp.get_context("fork").Pool(procs) as pool:
        res = pool.map(_cells_worker, [(x, fs, n, p, list(dop)) for p in parts])
    shape = (len(svs), len(dop))
    peak, arg, total, count = (np.zeros(shape), np.zeros(shape, np.int64), np.zeros(shape), np.zeros(shape, np.int64))
    for i, (pk, ag, tt, ct) in enumerate(res):
        rows = list(range(i, len(svs), procs))
        peak[rows], arg[rows], total[rows], count[rows] = pk, ag, tt, ct
    return peak, arg, total, count


def check_grid(rec, x, fs, n, svs, dop, what):
    peak, arg, total, count = oracle_grid(x, fs, n, svs, dop)
    assert rec.shape == peak.shape
    assert np.abs(rec["peak"] - peak).max() <= MAG_TOL * peak.max(), what
    assert np.abs(rec["sum"] - total).max() <= MAG_TOL * total.max(), what
    assert np.array_equal(rec["count"], count), what
    bad = np.argwhere(rec["argmax"] != arg)
    for a, b in bad:  # a different index is only acceptable where the float64 profile itself ties to within the tolerance
        prof = o.integrate(o.NON_COHERENT, x, fs, n, dop[b], o.replica(svs[a], n))
        assert prof.max() - prof[rec["argmax"][a, b]] <= MAG_TOL * prof.max(), (what, a, b)
    strength = rec["peak"].astype(np.float64) / ((rec["sum"] - rec["count"] * rec["peak"].astype(np.float64)) / (n - rec["count"]))
    ref_strength = peak / ((total - count * peak) / (n - count))
    assert np.abs(strength - ref_strength).max() <= 1e-4 * ref_strength.max(), what
    return len(bad)


@pytest.fixture(scope="module")
def engine_for(native_lib):
    from gypsum_b200 import _native

    cache = {}

    def get(n):
        if n not in cache:
            e = _native.Engine(n * 1000, n)
            e.set_replicas(np.stack([o.ca_code(sv) for sv in range(1, 33)]).astype(np.uint8))
            cache[n] = e
        return cache[n]

    yield get
    for e in cache.values():
        e.close()


PLANTED = [(3, -3000.0, 5, 1.0, 0.3), (11, 4500.0, 1234, 2.0, 0.3), (25, 1500.0, 777, 0.3, 0.3), (32, -9500.0, 2045, 2.5, 0.3)]
SVS = list(range(1, 33))


def test_config2_all_1312_cells(engine_for):
    """32 PRN x 41 Doppler x 1 ms @ 2.046 Msps: every record of the grid, by every entry point that produces it."""
    n, fs = 2046, 2046000
    dop = np.arange(-10000.0, 10001.0, 500.0)
    x = o.synth_iq(2, n, 1, fs, PLANTED)
    eng = engine_for(n)
    eng.upload_iq(x)
    rec = eng.acquire_grid(1, 1, np.arange(32), dop)[0]
    check_grid(rec, x, fs, n, SVS, dop, "acquire_grid")
    rec_h = eng.acquire_grid_host(x, 1, 1, np.arange(32), dop)[0]  # eager call of the shape ...
    rec_g = eng.acquire_grid_host(x, 1, 1, np.arange(32), dop)[0]  # ... captured into a graph ...
    rec_r = eng.acquire_grid_host(x, 1, 1, np.arange(32), dop)[0]  # ... replayed
    for other in (rec_h, rec_g, rec_r):
        for k in ("peak", "argmax", "sum", "count"):
            assert np.array_equal(other[k], rec[k]), k
    # the replayed graph reads the grid's axes and the replica spectra from device buffers other calls reuse: a list-mode call
    # with other Dopplers, a different grid, and a re-loaded replica table in between must not leak into the next replay
    eng.acquire_cells([3, 4], [123.0, -456.0], 1)
    eng.acquire_grid(1, 1, [5], [777.0])
    again = eng.acquire_grid_host(x, 1, 1, np.arange(32), dop)[0]
    assert all(np.array_equal(again[k], rec[k]) for k in ("peak", "argmax", "sum", "count"))
    chips = np.stack([o.ca_code(sv) for sv in range(1, 33)]).astype(np.uint8)
    eng.set_replicas(chips[::-1].copy())  # row a now holds SV 32 - a
    flipped = eng.acquire_grid_host(x, 1, 1, np.arange(32), dop)[0]
    assert all(np.array_equal(flipped[k], rec[k][::-1]) for k in ("peak", "argmax", "sum", "count"))
    eng.set_replicas(chips)
    eng.upload_iq(x)
    best = eng.acquire_grid_best(1, 1, np.arange(32), dop)[0]
    for a in range(32):  # acquisition.py:179-189 per PRN row
        b = int(np.argmax(rec["peak"][a]))
        assert (best["bin"][a], best["doppler"][a], best["code_phase"][a], best["peak"][a]) == (b, dop[b], rec["argmax"][a, b], rec["peak"][a, b])
    for sv, f, tau, _, _ in PLANTED:
        assert (best["doppler"][sv - 1], best["code_phase"][sv - 1]) == (f, tau) and best["strength"][sv - 1] > 8


def test_config3_all_cells_10ms_4092(engine_for):
    """32 PRN x 41 Doppler x 10 ms non-coherent @ 4.092 Msps."""
    n, fs = 4092, 4092000
    dop = np.arange(-10000.0, 10001.0, 500.0)
    planted = [(3, -3000.0, 5, 1.0, 0.1), (11, 4500.0, 2500, 2.0, 0.1), (25, 1500.0, 4091, 0.3, 0.08), (32, -9500.0, 2045, 2.5, 0.1)]
    x = o.synth_iq(3, n, 10, fs, planted)
    eng = engine_for(n)
    eng.upload_iq(x)
    rec = eng.acquire_grid(1, 10, np.arange(32), dop)[0]
    check_grid(rec, x, fs, n, SVS, dop, "config 3")
    for sv, f, tau, _, _ in planted:
        b = int(np.argmax(rec["peak"][sv - 1]))
        assert dop[b] == f and rec["argmax"][sv - 1, b] == tau


def test_config5_all_cells_two_blocks_16368(engine_for):
    """32 PRN x 81 Doppler @ 16.368 Msps, two independent 1-ms blocks in one call (the shape the 8-GPU job shards)."""
    n, fs = 16368, 16368000
    dop = np.arange(-10000.0, 10001.0, 250.0)
    assert len(dop) == 81
    planted = [(3, -3000.0, 5, 1.0, 0.12), (11, 4500.0, 12345, 2.0, 0.12), (25, 1500.0, 16367, 0.3, 0.1)]
    x = np.concatenate([o.synth_iq(50 + b, n, 1, fs, planted) for b in range(2)])
    eng = engine_for(n)
    eng.upload_iq(x)
    rec = eng.acquire_grid(2, 1, np.arange(32), dop)
    for b in range(2):
        check_grid(rec[b], x[b * n:(b + 1) * n], fs, n, SVS, dop, f"config 5 block {b}")


def test_config4_four_channels_ten_seconds_with_bits(engine_for):
    """Config 4 on a stated subset the CPU can afford: 4 channels x 10 s of ONE shared stream through TrackerBank (one
    launch) + the device bit integrator, against TrackerOracle per channel + the host integrator restatement (itself
    pinned to events recorded from the live reference).  Symbols / code phase exact bar per-millisecond proofs."""
    from gypsum_b200.gps_ca_prn_codes import GpsSatelliteId, generate_replica_prn_signals
    from gypsum_b200.navigation_bit_integrator import NavigationBitIntegrator
    from gypsum_b200.satellite import GpsSatellite
    from gypsum_b200.tracker import BitValue, EmittedPseudosymbol, NavigationBitPseudosymbol, TrackerBank

    n, fs, n_ms = 2046, 2046000, 10000
    chans = [(25, 1500.3, 0.0, 777, 0.3, 0.004), (7, -2212.7, 0.2, 100, 1.0, 0.005), (31, 3000.2, -0.3, 2045, 2.0, 0.004),
             (12, 640.4, 0.0, 1501, 0.7, 0.006)]
    inits = [(1500.0, 0.0, 777), (-2210.0, 0.5, 100), (3000.0, 0.0, 2045), (640.0, 0.0, 1501)]
    # every channel tracks its own satellite inside the SAME stream (sum of the four signals + one noise realisation)
    x = t.synth_tracking_iq(77, n, n_ms, fs, chans)

    class Attrs:
        samples_per_second, samples_per_prn_transmission = fs, n

    codes = generate_replica_prn_signals()
    sats = {c[0]: GpsSatellite(GpsSatelliteId(c[0]), codes[GpsSatelliteId(c[0])], 2) for c in chans}
    bank = TrackerBank([(sats[c[0]], i[0], i[1], i[2]) for c, i in zip(chans, inits)], Attrs)
    tt = np.array([t.chunk_times(k, fs, n) for k in range(n_ms)])
    rec = bank.process(x, tt[:, 0])
    bits = bank.integrate_bits(tt[:, 0], tt[:, 1])

    # oracle: one process per channel, each on the same stream
    with mp.get_context("fork").Pool(4) as pool:
        want = pool.map(oracle_channel_entry, [(x, chans[ci], inits[ci], n_ms) for ci in range(4)])
    for ci in range(4):
        w, g = want[ci], rec[ci]
        assert not g["lost"].any()
        scale = np.abs(w[:, 5]).max()
        for k in np.flatnonzero(g["symbol"] != w[:, 0].astype(int)):  # only where the in-phase value is float32 noise around 0
            assert abs(w[k, 5]) <= 1e-4 * scale, (ci, k)
        for k in np.flatnonzero(g["code_phase"] != w[:, 1].astype(int)):  # only where the accumulator sits on an integer boundary
            frac = w[k, 2] - np.floor(w[k, 2])
            assert min(frac, 1 - frac) <= 5e-3 and abs(g["phase_acc"][k] - w[k, 2]) <= 5e-3, (ci, k)
        assert np.abs(g["doppler"] - w[:, 3]).max() <= 5e-3
        d = np.abs(g["carrier_phase"] - w[:, 4])
        assert np.minimum(d, 2 * np.pi - d).max() <= 2e-3
        # bits: the host integrator on the ORACLE's pseudosymbols vs the device integrator on the device's records
        integ = NavigationBitIntegrator(chans[ci][0])
        code = {BitValue.ONE: 1, BitValue.ZERO: 0, BitValue.UNKNOWN: -1}
        ref_bits = []
        for k in range(n_ms):
            ps = EmittedPseudosymbol(w[k, 6], w[k, 7], NavigationBitPseudosymbol.from_val(int(w[k, 0])), 0)
            ref_bits += [(k, e.receiver_timestamp, e.trailing_edge_receiver_timestamp, code[e.bit_value])
                         for e in integ.process_pseudosymbol(tt[k, 0], ps)]
        got_bits = [(int(e["ms_index"]), float(e["receiver_timestamp"]), float(e["trailing_edge_receiver_timestamp"]),
                     int(e["bit_value"])) for e in bits[ci]]
        if np.array_equal(g["symbol"], w[:, 0].astype(int)) and np.array_equal(g["code_phase"], w[:, 1].astype(int)):
            assert got_bits == ref_bits, ci  # same symbols and code phases in => same bits and edges out, event for event
        assert len(got_bits) >= 480  # 10 s at 50 bit/s minus the synchronisation backlog


def oracle_channel_entry(args):
    x, ch, init, n_ms = args
    n, fs = 2046, 2046000
    tr = t.TrackerOracle(ch[0], init[0], init[1], init[2], fs, n)
    rows = []
    for k in range(n_ms):
        a, b = t.chunk_times(k, fs, n)
        r = tr.step(x[k * n:(k + 1) * n], a, b)
        rows.append((r["symbol"], r["code_phase"], tr.phase, r["doppler"], r["carrier_phase"], r["peak"].real, r["start"], r["end"]))
    return np.array(rows)


_WINDOW_CHILD = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from gypsum_b200 import _native
from gypsum_b200.gps_ca_prn_codes import ca_code_chips
n, nb = int(sys.argv[2]), int(sys.argv[3])
x = np.load(sys.argv[4])
e = _native.Engine(n * 1000, n)
e.set_replicas(np.stack([ca_code_chips(sv) for sv in range(1, 33)]).astype(np.uint8))
e.upload_iq(x)
rec = e.acquire_grid(nb, 1, np.arange(32, dtype=np.int32), np.arange(-10000.0, 10001.0, 500.0))
np.save(sys.argv[5], rec.view(np.uint8))
e.close()
"""


@pytest.mark.parametrize("n, nb", [(2046, 20), (16368, 3), (12276, 3)])
def test_l2_windows_leave_every_record_unchanged(engine_for, tmp_path, n, nb):
    """The one-warp kernel walks batches larger than L2 in windows of units (group order window / PRN / chunk, extra groups going
    round the CTAs).  That only reorders independent cells: with windows forced onto a small batch (a child process, the knobs
    are read once per process) every record is byte-identical to the single-window launch's, also with a ragged last window."""
    import subprocess
    import sys

    rng = np.random.default_rng(n + nb)
    x = (rng.standard_normal(2 * n * nb).astype(np.float32)).view(np.complex64)
    x[:n] += o.synth_iq(0, n, 1, n * 1000, [(25, 1500.0, 777, 0.3, 0.3)], sigma=0.0)
    e = engine_for(n)
    e.upload_iq(x)
    ref = e.acquire_grid(nb, 1, np.arange(32, dtype=np.int32), np.arange(-10000.0, 10001.0, 500.0))
    assert int(ref["argmax"][0, 24, 23]) == 777
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    np.save(tmp_path / "x.npy", x)
    for mb in ("1", "3"):
        env = dict(os.environ, GB200_L2_WINDOW_MB=mb, GB200_L2_WINDOW_MIN_GROUPS="0")
        subprocess.run([sys.executable, "-c", _WINDOW_CHILD, root, str(n), str(nb), str(tmp_path / "x.npy"), str(tmp_path / f"r{mb}.npy")],
                       check=True, env=env, timeout=600)
        got = np.load(tmp_path / f"r{mb}.npy")
        assert np.array_equal(got, ref.view(np.uint8)), mb
