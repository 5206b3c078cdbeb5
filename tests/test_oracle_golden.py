"""The oracle (oracle/gypsum_oracle.py) against fixtures produced by the live reference (tools/make_golden.py)
and against the only known-answer table the reference holds (IS-GPS-200 first ten chips)."""
import hashlib
import os

import numpy as np
import pytest

from oracle import gypsum_oracle as o
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def test_ca_codes_match_reference_and_is_gps_200():
    g = np.load(os.path.join(GOLDEN, "ca_codes.npz"))["chips"]
    for sv in range(1, 33):
        c = o.ca_code(sv)
        assert np.array_equal(c, g[sv - 1])
        assert c.sum() == 512  # balanced Gold code
        assert int("".join(map(str, c[:10])), 2) == int(str(o.FIRST_10_CHIPS_OCTAL[sv - 1]), 8)


def test_product_code_generator_matches_golden():
    from gypsum_b200.gps_ca_prn_codes import GpsSatelliteId, generate_replica_prn_signals

    g = np.load(os.path.join(GOLDEN, "ca_codes.npz"))["chips"]
    codes = generate_replica_prn_signals()
    for sv in range(1, 33):
        assert np.array_equal(codes[GpsSatelliteId(sv)].inner, g[sv - 1])


def _cases():
    z = np.load(os.path.join(GOLDEN, "cell_profiles.npz"))
    names = sorted({k.split("__")[0] for k in z.files})
    for name in names:
        n = int(name.split("_")[0][1:])
        n_ms = int(name.split("_m")[1])
        k = 0
        while f"{name}__{k}__sv" in z.files:
            yield name, n, n_ms, k, z
            k += 1


@pytest.mark.parametrize("name,n,n_ms,k", [(a, b, c, d) for a, b, c, d, _ in _cases()])
def test_oracle_profiles_bit_exact_with_reference(name, n, n_ms, k):
    z = np.load(os.path.join(GOLDEN, "cell_profiles.npz"))
    planted = [(int(p[0]), p[1], int(p[2]), p[3], p[4]) for p in z[f"{name}__planted"]]
    fs = n * 1000
    x = o.synth_iq(1234, n, n_ms, fs, planted)
    sv, f = int(z[f"{name}__{k}__sv"]), float(z[f"{name}__{k}__doppler"])
    prn = o.replica(sv, n)
    nc = o.integrate(o.NON_COHERENT, x, fs, n, f, prn)
    co = o.integrate(o.COHERENT, x, fs, n, f, prn)
    # the recorded sample first (a failure shows the values), then the digest of every value
    idx = z[f"{name}__{k}__sample_idx"]
    assert np.array_equal(nc[idx], z[f"{name}__{k}__noncoherent_sample"])
    assert np.array_equal(co[idx], z[f"{name}__{k}__coherent_sample"])
    assert hashlib.sha256(nc.tobytes()).digest() == z[f"{name}__{k}__noncoherent_sha256"].tobytes()
    assert hashlib.sha256(co.tobytes()).digest() == z[f"{name}__{k}__coherent_sha256"].tobytes()
    assert o.peak_strength(nc) == float(z[f"{name}__{k}__strength"])


def test_oracle_detector_matches_reference_detector():
    z = np.load(os.path.join(GOLDEN, "detector_n2046.npz"))
    planted = [(int(p[0]), p[1], int(p[2]), p[3], p[4]) for p in z["planted"]]
    x = o.synth_iq(int(z["seed"]), 2046, 10, 2046000, planted)
    for row in z["results"][:2]:  # two satellites keep the CPU suite short; the GPU suite checks all five
        r = o.acquire_sv(int(row[0]), x, 2046000, 2046)
        assert (r.doppler, r.code_phase) == (int(row[1]), int(row[3]))
        assert r.carrier_phase == row[2] and r.strength == row[4]


def test_doppler_bins_semantics():
    assert o.doppler_bins(0.0, 7000.0) == list(range(-7000, 7000, 700))
    assert o.doppler_bins(-700, 13.671875) == list(range(-713, -686, 1))
    from gypsum_b200.acquisition import doppler_search_bins

    for c, s in [(0.0, 7000.0), (1400, 3500.0), (-3150, 54.6875), (-1, 13.671875)]:
        assert list(doppler_search_bins(c, s)) == o.doppler_bins(c, s)


def test_strength_from_record_equals_profile_formula():
    rng = np.random.default_rng(3)
    p = rng.random(2046)
    p[17] = p[400] = 5.0
    m = p.max()
    assert np.isclose(o.strength_from_record(m, p.sum(), 2, p.size), o.peak_strength(p), rtol=1e-12)
