// Host lane emulator: runs the product's lane-level device functions (gypsum_b200/csrc/warp_fft.cuh) with the
// 32 lanes of each warp as a plain loop, following the same dataflow as kernels.cu (doppler_spectra ->
// correlate_cells).  Lets the -m "not gpu" suite check the polyphase / padded-FFT algebra and every index map
// against the oracle without a GPU.  Test infrastructure; never loaded by the product.
#include <cmath>
#include <cstring>
#include <vector>

#include "../../gypsum_b200/csrc/warp_fft.cuh"

using namespace gb;

static std::vector<float2> g_tw1, g_tw2;
static void init_tables() {
    if (!g_tw1.empty()) return;
    g_tw1.resize(1024);
    g_tw2.resize(1024);
    for (int k1 = 0; k1 < 32; ++k1)
        for (int l = 0; l < 32; ++l) {
            double a = -2.0 * M_PI * ((l * k1) % 1024) / 1024.0;
            g_tw1[pidx(k1, l)] = make_float2((float)cos(a), (float)sin(a));
        }
    for (int n = 0; n < 1024; ++n) {
        double a = -2.0 * M_PI * n / 2048.0;
        g_tw2[zpos(n)] = make_float2((float)cos(a), (float)sin(a));
    }
}

struct WarpRegs {
    float2 x[32][32];  // [lane][j]
};

static void warp_fft1024(WarpRegs& w, bool inverse, float2* tile) {
    for (int lane = 0; lane < 32; ++lane) {
        if (inverse) wfft_phase1<true>(w.x[lane], lane, g_tw1.data(), tile);
        else wfft_phase1<false>(w.x[lane], lane, g_tw1.data(), tile);
    }
    for (int lane = 0; lane < 32; ++lane) {
        if (inverse) wfft_phase2<true>(w.x[lane], lane, tile);
        else wfft_phase2<false>(w.x[lane], lane, tile);
    }
}

extern "C" {

// plain warp FFT-1024 check: x[1024] complex64 in/out (natural order)
void emu_fft1024(float2* x, int inverse) {
    init_tables();
    std::vector<float2> tile(kTileF2);
    WarpRegs* w = new WarpRegs;
    for (int lane = 0; lane < 32; ++lane)
        for (int j = 0; j < 32; ++j) w->x[lane][j] = x[lane + 32 * j];
    warp_fft1024(*w, inverse != 0, tile.data());
    for (int lane = 0; lane < 32; ++lane)
        for (int j = 0; j < 32; ++j) x[lane + 32 * j] = w->x[lane][j];
    delete w;
}

// crep[2][1024] for one PRN
void emu_replica_spectrum(const uint8_t* chips, float2* crep) {
    std::vector<double2> cs(kPad);
    for (int t = 0; t < kPad; ++t) cs[t] = make_double2(cos(2.0 * M_PI * t / kPad), sin(2.0 * M_PI * t / kPad));
    for (int g = 0; g < kPad; ++g) {
        double re, im;
        replica_spectrum_bin(chips, g, cs.data(), re, im);
        crep[(g & 1) * 1024 + zpos(g >> 1)] = make_float2((float)re, (float)im);
    }
}

}  // extern "C"

// ---- doppler_spectra (mirrors k_doppler_spectra<S>: 256 "threads", carrier = coarse x fine table) ----
// spec[i][r][half][1024] for the n_ms milliseconds of one Doppler bin
static std::vector<float2> emu_spectra(const float2* iq, int N, int n_ms, double fs, double doppler) {
    const int s = N / kChips;
    std::vector<float2> tile(kTileF2);
    std::vector<float2> ypoly((size_t)s * kFft);
    std::vector<float2> spec((size_t)n_ms * s * 2 * kFft);
    WarpRegs* w = new WarpRegs;
    const double inv_fs = 1.0 / fs;
    for (int i = 0; i < n_ms; ++i) {
        float2 coarse[64], fine[256];
        for (int k = 0; k < (N + 255) / 256; ++k) coarse[k] = carrier_at(doppler, (double)(k * 256 + i * N), inv_fs);
        for (int t = 0; t < 256; ++t) fine[t] = carrier_at(doppler, (double)t, inv_fs);
        for (int n = 0; n < N; ++n) {
            const float2 y = cmul(iq[(size_t)i * N + n], cmul(coarse[n / 256], fine[n % 256]));
            ypoly[(size_t)(n % s) * kFft + zpos(n / s)] = y;
        }
        for (int t = 0; t < s; ++t) ypoly[(size_t)t * kFft + zpos(kFft - 1)] = ypoly[(size_t)t * kFft + zpos(0)];
        if (s > 1) {
            std::vector<float2> znew((size_t)s * kFft);
            for (int m = 0; m < kChips; ++m) {
                switch (s) {
#define EMU_CASE(S) case S: { float2 z[S]; boxcar_column<S>(ypoly.data(), m, z); for (int r = 0; r < S; ++r) znew[(size_t)r * kFft + zpos(m)] = z[r]; } break;
                    EMU_CASE(2) EMU_CASE(3) EMU_CASE(4) EMU_CASE(5) EMU_CASE(6) EMU_CASE(8) EMU_CASE(10) EMU_CASE(12) EMU_CASE(16)
#undef EMU_CASE
                }
            }
            for (int t = 0; t < s; ++t)
                for (int m = 0; m < kChips; ++m) ypoly[(size_t)t * kFft + zpos(m)] = znew[(size_t)t * kFft + zpos(m)];
        }
        for (int t = 0; t < s; ++t) ypoly[(size_t)t * kFft + zpos(kFft - 1)] = make_float2(0.f, 0.f);
        for (int r = 0; r < s; ++r)
            for (int half = 0; half < 2; ++half) {
                for (int lane = 0; lane < 32; ++lane) {
                    load_vec(w->x[lane], lane, ypoly.data() + (size_t)r * kFft);
                    if (half) mul_tw2(w->x[lane], lane, g_tw2.data());
                }
                warp_fft1024(*w, false, tile.data());
                float2* dst = &spec[(((size_t)i * s + r) * 2 + half) * kFft];
                for (int lane = 0; lane < 32; ++lane) store_vec(w->x[lane], lane, dst);
            }
    }
    delete w;
    return spec;
}

extern "C" {

// Full per-cell pipeline.  iq: complex64[n_ms*N]; out: float[N] (non-coherent) or float2[N] (coherent).
// kind: 1 coherent, 2 non-coherent (utils.py:23-25).
void emu_cell_profile(const float2* iq, int N, int n_ms, double fs, double doppler, const uint8_t* chips, int kind,
                      float* out, CellRecord* rec_out) {
    init_tables();
    const int s = N / kChips;
    std::vector<float2> crep(2048);
    emu_replica_spectrum(chips, crep.data());
    std::vector<float2> tile(kTileF2), tileO(kTileF2);
    const std::vector<float2> spec = emu_spectra(iq, N, n_ms, fs, doppler);
    WarpRegs* w = new WarpRegs;
    WarpRegs* wo = new WarpRegs;
    // ---- correlate_cells ----
    if (kind == 2) memset(out, 0, sizeof(float) * N);
    else memset(out, 0, sizeof(float) * 2 * N);
    const int n_iter = kind == 1 ? 1 : n_ms;
    Peak cell;
    peak_init(cell);
    std::vector<float> acc((size_t)2 * 32 * 16);  // [h][lane][jj]
    for (int r = 0; r < s; ++r) {
        std::fill(acc.begin(), acc.end(), 0.f);
        for (int it = 0; it < n_iter; ++it) {
            for (int half = 0; half < 2; ++half) {
                WarpRegs* ww = half ? wo : w;
                for (int lane = 0; lane < 32; ++lane) {
                    if (kind == 1) {
                        for (int j = 0; j < 32; ++j) ww->x[lane][j] = make_float2(0.f, 0.f);
                        for (int i = 0; i < n_ms; ++i) {
                            float2 t[32];
                            load_vec(t, lane, &spec[(((size_t)i * s + r) * 2 + half) * kFft]);
                            for (int j = 0; j < 32; ++j) ww->x[lane][j] = c_add(ww->x[lane][j], t[j]);
                        }
                        mul_vec(ww->x[lane], lane, crep.data() + half * 1024);
                    } else {
                        load_mul_vec(ww->x[lane], lane, &spec[(((size_t)it * s + r) * 2 + half) * kFft], crep.data() + half * 1024);
                    }
                }
                warp_fft1024(*ww, true, half ? tileO.data() : tile.data());
                // (all lanes have finished phase 2 before the tile is reused for the exchange)
                for (int lane = 0; lane < 32; ++lane)
                    exchange_store(ww->x[lane], lane, half, half ? tileO.data() : tile.data());
            }
            for (int half = 0; half < 2; ++half)
                for (int lane = 0; lane < 32; ++lane) {
                    float2 o16[16];
                    if (half == 0) combine_even(w->x[lane], lane, g_tw2.data(), tileO.data(), o16);
                    else combine_odd(wo->x[lane], lane, g_tw2.data(), tile.data(), o16);
                    for (int jj = 0; jj < 16; ++jj) {
                        const int q = lane + 32 * (16 * half + jj);
                        const int n = s * q + r;
                        float& a = acc[((size_t)half * 32 + lane) * 16 + jj];
                        if (kind == 2) a += gb_mag(o16[jj]);
                        else {
                            a = gb_mag(o16[jj]);
                            if (q < kChips) {
                                out[2 * n] = o16[jj].x;
                                out[2 * n + 1] = o16[jj].y;
                            }
                        }
                    }
                }
        }
        for (int half = 0; half < 2; ++half)
            for (int lane = 0; lane < 32; ++lane) {
                float v[16];
                for (int jj = 0; jj < 16; ++jj) {
                    v[jj] = acc[((size_t)half * 32 + lane) * 16 + jj];
                    const int q = lane + 32 * (16 * half + jj);
                    if (kind == 2 && q < kChips) out[s * q + r] = v[jj];
                }
                Peak t;
                float fsum;
                thread_peak16(v, lane, half, s, r, t, fsum);
                t.sum = (double)fsum;
                peak_merge(cell, t);
            }
    }
    if (rec_out) {
        rec_out->peak = cell.mx;
        rec_out->argmax = cell.idx;
        rec_out->sum = cell.sum;
        rec_out->count = cell.cnt;
        rec_out->probe_re = rec_out->probe_im = 0.f;
        rec_out->pad_ = 0;
    }
    delete w;
    delete wo;
}

// One cell of k_correlate_w2048 (non-coherent): per polyphase branch r, one warp loads both half-spectra times the replica
// spectrum, runs the pruned inverse FFT-2048 and accumulates |.| of its 32 lags q = lane + 32 k over the n_ms milliseconds;
// the lags k < 16 and k >= 16 are reduced as the halves h = 0 / 1 of thread_peak16, and every thread's peaks are merged
// into the cell record.  out: float[N], the accumulated profile at index s q + r.
void emu_cell_record_w2048(const float2* iq, int N, int n_ms, double fs, double doppler, const uint8_t* chips, float* out,
                           CellRecord* rec_out) {
    init_tables();
    const int s = N / kChips;
    std::vector<float2> crep(2048);
    emu_replica_spectrum(chips, crep.data());
    std::vector<float2> tile(kTile64F2);
    const std::vector<float2> spec = emu_spectra(iq, N, n_ms, fs, doppler);
    static float acc[32][32];  // [lane][k]
    Peak cell;
    peak_init(cell);
    for (int r = 0; r < s; ++r) {
        memset(acc, 0, sizeof(acc));
        for (int it = 0; it < n_ms; ++it) {
            const float2* p = &spec[((size_t)it * s + r) * 2 * kFft];
            for (int lane = 0; lane < 32; ++lane) {
                float2 hx[32];
                load_mul_vec(hx, lane, p, crep.data());  // even bins
                w2048_phase1<0>(hx, lane, g_tw1.data(), tile.data());
                load_mul_vec(hx, lane, p + kFft, crep.data() + kFft);  // odd bins
                w2048_phase1<1>(hx, lane, g_tw1.data(), tile.data());
            }
            for (int lane = 0; lane < 32; ++lane) {
                float2 x[64];
                w2048_phase2(x, lane, tile.data());
                for (int k = 0; k < 32; ++k) acc[lane][k] += gb_mag(x[k]);
            }
        }
        for (int lane = 0; lane < 32; ++lane) {
            for (int k = 0; k < 32; ++k) {
                const int q = lane + 32 * k;
                if (q < kChips) out[s * q + r] = acc[lane][k];
            }
            for (int hh = 0; hh < 2; ++hh) {
                float v[16];
                for (int jj = 0; jj < 16; ++jj) v[jj] = acc[lane][16 * hh + jj];
                Peak t;
                float fsum;
                thread_peak16(v, lane, hh, s, r, t, fsum);
                t.sum = (double)fsum;
                peak_merge(cell, t);
            }
        }
    }
    rec_out->peak = cell.mx;
    rec_out->argmax = cell.idx;
    rec_out->sum = cell.sum;
    rec_out->count = cell.cnt;
    rec_out->probe_re = rec_out->probe_im = 0.f;
    rec_out->pad_ = 0;
}
}

// ---- scalar tracking loop (tracker_core.cuh) on the host ----
#include "../../gypsum_b200/csrc/tracker_core.cuh"
extern "C" {
int emu_track_state_size() { return (int)sizeof(TrackState); }
void emu_track_init(TrackState* st, int prn, double doppler, double carrier_phase, int code_phase) {
    track_state_init(*st, prn, doppler, carrier_phase, code_phase);
}
void emu_track_update(TrackState* st, const float* elp /* E.re E.im L.re L.im P.re P.im */, float strength, int off,
                      double t0, double fs, TrackMsRecord* out) {
    const TrackConsts tc = track_consts(fs);
    track_update(*st, make_float2(elp[0], elp[1]), make_float2(elp[2], elp[3]), make_float2(elp[4], elp[5]), strength, off,
                 t0, tc, nullptr, *out);
}
}

extern "C" int emu_track_rot_ok(double mr, double mi, int fast) { return fast ? track_rot_ok_fast(mr, mi) : track_rot_ok(mr, mi); }

// ---- one-warp pruned inverse FFT-2048 (w2048_phase1/2) ----
extern "C" void emu_ifft2048_pruned(const float2* y_even, const float2* y_odd, float2* out /*[1024]*/) {
    init_tables();
    std::vector<float2> tile(kTile64F2);
    static float2 a[32][32], b[32][32];
    for (int lane = 0; lane < 32; ++lane)
        for (int j = 0; j < 32; ++j) {
            a[lane][j] = y_even[lane + 32 * j];
            b[lane][j] = y_odd[lane + 32 * j];
        }
    for (int lane = 0; lane < 32; ++lane) {
        w2048_phase1<0>(a[lane], lane, g_tw1.data(), tile.data());
        w2048_phase1<1>(b[lane], lane, g_tw1.data(), tile.data());
    }
    for (int lane = 0; lane < 32; ++lane) {
        float2 x[64];
        w2048_phase2(x, lane, tile.data());
        for (int k2 = 0; k2 < 32; ++k2) out[lane + 32 * k2] = x[k2];
    }
}

// ---- navigation bit integration (bits_core.cuh) on the host ----
#include "../../gypsum_b200/csrc/bits_core.cuh"
extern "C" {
int emu_bit_state_size() { return (int)sizeof(BitState); }
void emu_bit_init(BitState* st) {
    memset(st, 0, sizeof(BitState));
    bit_state_init(*st);
}
// n symbols of one channel; returns the number of events (may exceed max_events)
int emu_bit_run(BitState* st, int n, const int* symbols, const double* recv_ts, const double* start, const double* end,
                BitEvent* out, int max_events) {
    int n_out = 0;
    for (int k = 0; k < n; ++k) bit_step(st->h, *st, symbols[k], recv_ts[k], start[k], end[k], k, out, max_events, n_out);
    return n_out;
}
void emu_bit_summary(const BitState* st, long long* out /*[8]*/) {
    out[0] = st->h.emitted;
    out[1] = st->h.failed;
    out[2] = st->h.processed;
    out[3] = st->h.slide;
    out[4] = st->h.determined;
    out[5] = st->h.prev_decision;
    out[6] = st->h.cursor;
    out[7] = st->h.overflow;
}
}
