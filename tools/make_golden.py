"""Generate tests/golden/*.npz by running the LIVE reference (the original gypsum project).

The reference has no golden vectors of its own (SURVEY.md F2), so parity is pinned on the reference's own
outputs: this script imports gypsum.* from a checkout of the reference (read-only, unmodified) and records what
its functions return on seeded synthetic input.  Run:  python tools/make_golden.py PATH_TO_REFERENCE_CHECKOUT
The tests read only the fixtures; they never need the reference itself.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
if len(sys.argv) != 2:
    sys.exit("usage: python tools/make_golden.py PATH_TO_REFERENCE_CHECKOUT")
sys.path.insert(0, os.path.abspath(sys.argv[1]))

from gypsum.acquisition import GpsSatelliteDetector  # noqa: E402
from gypsum.antenna_sample_provider import SampleProviderAttributes  # noqa: E402
from gypsum.gps_ca_prn_codes import GpsSatelliteId, generate_replica_prn_signals  # noqa: E402
from gypsum.satellite import GpsSatellite  # noqa: E402
from gypsum.utils import (  # noqa: E402
    IntegrationType,
    get_normalized_correlation_peak_strength,
    integrate_correlation_with_doppler_shifted_prn,
)

from oracle import gypsum_oracle as o  # noqa: E402  (only for synth_iq: identical input bytes everywhere)

OUT = os.path.join(ROOT, "tests", "golden")
PROFILE_SAMPLE = 64  # profile values stored per cell beside the digests; the peak index is always one of them


def sha256(a: np.ndarray) -> np.ndarray:
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


class _Bytes(np.ndarray):
    """acquisition.py:203 calls ndarray.tostring(), removed in numpy 2.x; supply it from the caller side so the
    reference file runs unmodified (SURVEY.md F10)."""

    def tostring(self):
        return self.tobytes()


class _Sat:
    def __init__(self, sat):
        self.satellite_id = sat.satellite_id
        self.prn_as_complex = sat.prn_as_complex.view(_Bytes)


def main():
    os.makedirs(OUT, exist_ok=True)
    codes = generate_replica_prn_signals()
    np.savez_compressed(
        os.path.join(OUT, "ca_codes.npz"),
        chips=np.stack([codes[GpsSatelliteId(i)].inner for i in range(1, 33)]).astype(np.uint8),
    )

    # ---- per-cell profiles (utils.py:77) at the three sample rates ----
    # Whole profiles would exceed 1 MB, so each is kept as the SHA-256 of its bytes (the oracle's float64 profile must
    # hash to it: bit-exact over every value) plus a seeded sample of values that shows the size of any difference.
    cases = {}
    for name, n, n_ms, planted, cells in [
        ("n2046_m1", 2046, 1, [(25, 1500.0, 777, 0.3, 0.5)], [(25, 1500), (25, -3500), (3, 0), (25, 1000.5)]),
        ("n2046_m10", 2046, 10, [(25, 1500.0, 777, 0.3, 0.12), (3, -3250.0, 5, 1.0, 0.1)],
         [(25, 1500), (25, 1250), (3, -3250), (11, 4875)]),
        ("n4092_m3", 4092, 3, [(11, 4875.5, 4000, 2.0, 0.2)], [(11, 4875), (11, 5000), (32, -10000)]),
        ("n16368_m1", 16368, 1, [(32, -250.0, 16367, 0.0, 0.1)], [(32, -250), (1, 10000)]),
    ]:
        fs = n * 1000
        attrs = SampleProviderAttributes(fs, n)
        x = o.synth_iq(1234, n, n_ms, fs, planted)
        for k, (sv, f) in enumerate(cells):
            sat = GpsSatellite(GpsSatelliteId(sv), codes[GpsSatelliteId(sv)], n // 1023)
            nc = integrate_correlation_with_doppler_shifted_prn(IntegrationType.NonCoherent, x, attrs, f,
                                                                sat.prn_as_complex)
            co = integrate_correlation_with_doppler_shifted_prn(IntegrationType.Coherent, x, attrs, f,
                                                                sat.prn_as_complex)
            cases[f"{name}__{k}__sv"] = np.int64(sv)
            cases[f"{name}__{k}__doppler"] = np.float64(f)
            idx = np.union1d(np.random.default_rng(k).choice(n, PROFILE_SAMPLE - 1, replace=False), [int(np.argmax(nc))])
            cases[f"{name}__{k}__sample_idx"] = idx.astype(np.int64)
            cases[f"{name}__{k}__noncoherent_sample"] = nc[idx]
            cases[f"{name}__{k}__coherent_sample"] = co[idx]
            cases[f"{name}__{k}__noncoherent_sha256"] = sha256(nc)
            cases[f"{name}__{k}__coherent_sha256"] = sha256(co)
            cases[f"{name}__{k}__strength"] = np.float64(get_normalized_correlation_peak_strength(nc))
        cases[f"{name}__planted"] = np.array(planted, dtype=np.float64)
    np.savez_compressed(os.path.join(OUT, "cell_profiles.npz"), **cases)

    # ---- the real detector (acquisition.py:52-152), 10 ms @ 2.046 Msps ----
    n, fs = 2046, 2046000
    planted = [(25, 1504.0, 777, 0.3, 0.12), (3, -3250.0, 5, 1.0, 0.1), (32, 4875.5, 2045, 2.5, 0.15)]
    x = o.synth_iq(7, n, 10, fs, planted)
    sats = {GpsSatelliteId(i): _Sat(GpsSatellite(GpsSatelliteId(i), codes[GpsSatelliteId(i)], 2)) for i in range(1, 33)}
    det = GpsSatelliteDetector(sats)
    svs = [1, 3, 11, 25, 32]
    rows = []
    for sv in svs:
        r = det._attempt_acquisition_for_satellite_id(GpsSatelliteId(sv), x, SampleProviderAttributes(fs, n))
        rows.append([sv, r.doppler_shift, r.carrier_wave_phase_shift, r.prn_phase_shift, r.correlation_strength])
    found = det.detect_satellites_in_antenna_data([GpsSatelliteId(s) for s in svs], x, SampleProviderAttributes(fs, n))
    np.savez_compressed(
        os.path.join(OUT, "detector_n2046.npz"),
        seed=np.int64(7), planted=np.array(planted), svs=np.array(svs), results=np.array(rows, dtype=np.float64),
        detected=np.array([r.satellite_id.id for r in found]),
    )
    print("golden written:", sorted(os.listdir(OUT)))


if __name__ == "__main__":
    main()
