"""The product's lane-level device functions (warp FFT-1024, polyphase split, padded-FFT correlation, replica
spectra) executed on the CPU by the lane emulator and compared with the oracle.  No GPU needed."""
import ctypes

import numpy as np
import pytest

from oracle import gypsum_oracle as o


@pytest.mark.parametrize("inverse", [0, 1])
def test_warp_fft1024(emu_lib, inverse):
    rng = np.random.default_rng(inverse)
    x = (rng.standard_normal(1024) + 1j * rng.standard_normal(1024)).astype(np.complex64)
    y = x.copy()
    emu_lib.emu_fft1024(y.ctypes.data_as(ctypes.c_void_p), inverse)
    ref = np.fft.ifft(x.astype(complex)) * 1024 if inverse else np.fft.fft(x.astype(complex))
    assert np.abs(y - ref).max() <= 5e-7 * np.abs(ref).max()


@pytest.mark.parametrize("n,n_ms,sv,f", [(2046, 1, 25, 1500.0), (2046, 3, 7, -3250.0), (4092, 2, 11, 4875.5),
                                         (16368, 1, 32, -250.0), (1023, 2, 1, 700.0), (3069, 1, 19, 10000.0),
                                         (5115, 1, 3, -2750.0), (6138, 3, 14, 1250.5), (8184, 1, 22, 6000.0),
                                         (10230, 3, 5, -9000.0), (12276, 1, 28, 333.0)])
def test_polyphase_correlation_matches_oracle(emu_lib, n, n_ms, sv, f):
    emu_lib.emu_cell_profile.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                         ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    rec = np.zeros(1, dtype=[("peak", "<f4"), ("argmax", "<i4"), ("sum", "<f8"), ("count", "<i4"), ("pr", "<f4"),
                             ("pi", "<f4"), ("pad", "<i4")])
    fs = n * 1000
    iq = o.synth_iq(1, n, n_ms, fs, [(sv, f + 3, n - 7, 0.3, 0.3)])
    chips = o.ca_code(sv).astype(np.uint8)
    prn = o.replica(sv, n)
    nc = np.zeros(n, np.float32)
    emu_lib.emu_cell_profile(iq.ctypes.data, n, n_ms, float(fs), float(f), chips.ctypes.data, 2, nc.ctypes.data, rec.ctypes.data)
    ref = o.integrate(o.NON_COHERENT, iq, fs, n, f, prn)
    assert np.abs(nc - ref).max() <= 1e-6 * ref.max()
    assert nc.argmax() == ref.argmax() == n - 7
    # the branch-free per-thread reduction + merges reproduce np.max / np.argmax / count / sum of the profile
    assert rec["peak"][0] == nc.max() and rec["argmax"][0] == int(nc.argmax())
    assert rec["count"][0] == int(np.count_nonzero(nc == nc.max()))
    assert abs(rec["sum"][0] - nc.astype(np.float64).sum()) <= 2e-6 * rec["sum"][0]
    co = np.zeros(n, np.complex64)
    emu_lib.emu_cell_profile(iq.ctypes.data, n, n_ms, float(fs), float(f), chips.ctypes.data, 1, co.ctypes.data, None)
    refc = o.integrate(o.COHERENT, iq, fs, n, f, prn)
    assert np.abs(co - refc).max() <= 1e-6 * np.abs(refc).max()


RATES = [1, 2, 3, 4, 5, 6, 8, 10, 12, 16]  # every s = N / 1023 the engine accepts
LAG_CHIPS = [0, 31, 32, 511, 512, 1021, 1022]  # chip lags q at the lane / half / end boundaries of the lag layout


@pytest.mark.parametrize("n_ms", [1, 4])
@pytest.mark.parametrize("s", RATES)
def test_one_warp_cell_record_matches_oracle(emu_lib, s, n_ms):
    """One cell of the one-warp kernel (k_correlate_w2048): lag q = lane + 32 k of branch r lands at profile index s q + r,
    and the two 16-lag halves reduce to the record of the whole profile.  Copies of the replica are planted at delays of every
    residue r = 0 .. s-1 and every boundary lag q, the strongest at tau = N - 1 (1 ms) or 0 (4 ms)."""
    emu_lib.emu_cell_record_w2048.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                              ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    rec = np.zeros(1, dtype=[("peak", "<f4"), ("argmax", "<i4"), ("sum", "<f8"), ("count", "<i4"), ("pr", "<f4"),
                             ("pi", "<f4"), ("pad", "<i4")])
    n = 1023 * s
    fs, sv, f = n * 1000, 13, -2750.0
    main = n - 1 if n_ms == 1 else 0
    taus = {s * LAG_CHIPS[r % 7] + r for r in range(s)} | {s * q + k % s for k, q in enumerate(LAG_CHIPS)}
    planted = [(sv, f, main, 0.2, 1.0)] + [(sv, f, t, 0.1 * k, 0.4) for k, t in enumerate(sorted(taus - {main}))]
    iq = o.synth_iq(2 + s, n, n_ms, fs, planted, sigma=0.5)
    chips = o.ca_code(sv).astype(np.uint8)
    nc = np.zeros(n, np.float32)
    emu_lib.emu_cell_record_w2048(iq.ctypes.data, n, n_ms, float(fs), f, chips.ctypes.data, nc.ctypes.data, rec.ctypes.data)
    ref = o.integrate(o.NON_COHERENT, iq, fs, n, f, o.replica(sv, n))
    assert np.abs(nc - ref).max() <= 1e-6 * ref.max()
    assert nc.argmax() == ref.argmax() == main
    assert rec["peak"][0] == nc.max() and rec["argmax"][0] == main
    assert rec["count"][0] == int(np.count_nonzero(nc == nc.max()))
    assert abs(rec["sum"][0] - nc.astype(np.float64).sum()) <= 2e-6 * rec["sum"][0]


def test_one_warp_pruned_ifft2048(emu_lib):
    """w2048_phase1/2: out[k] = sum_g Y[g] exp(+2 pi i g k / 2048) for k < 1024, Y[2f+h] = Y_h[f]."""
    rng = np.random.default_rng(5)
    ye = (rng.standard_normal(1024) + 1j * rng.standard_normal(1024)).astype(np.complex64)
    yo = (rng.standard_normal(1024) + 1j * rng.standard_normal(1024)).astype(np.complex64)
    out = np.zeros(1024, np.complex64)
    emu_lib.emu_ifft2048_pruned(ye.ctypes.data_as(ctypes.c_void_p), yo.ctypes.data_as(ctypes.c_void_p),
                                out.ctypes.data_as(ctypes.c_void_p))
    y = np.empty(2048, complex)
    y[0::2], y[1::2] = ye, yo
    ref = (np.fft.ifft(y) * 2048)[:1024]
    assert np.abs(out - ref).max() <= 5e-7 * np.abs(ref).max()
