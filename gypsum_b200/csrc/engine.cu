// C ABI of the engine (include/gypsum_b200.h): owns device memory, builds launch plans, drives the kernels.
// Host side of the reference path it replaces: gypsum/acquisition.py:154-219 (the per-bin scan and its memo
// wrapper) and gypsum/utils.py:77-108.
#include <algorithm>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <numeric>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

#include "../../include/gypsum_b200.h"
#include "bits_core.cuh"
#include "kernels.cuh"

using namespace gb;

static_assert(sizeof(gb200_cell_record) == sizeof(CellRecord), "ABI record and device record must match");

namespace {

thread_local std::string g_create_error;

// A growable allocation that frees itself.  The engine's device must be current when it is destroyed or grown.
template <class T, cudaError_t (*Alloc)(void**, size_t), cudaError_t (*Free)(void*)>
class Buf {
public:
    T* p = nullptr;
    size_t cap = 0;
    Buf() = default;
    Buf(Buf&& o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    Buf(const Buf&) = delete;
    Buf& operator=(const Buf&) = delete;
    ~Buf() { release(); }
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        release();
        size_t want = std::max(n, static_cast<size_t>(16));
        cudaError_t e = Alloc(reinterpret_cast<void**>(&p), want * sizeof(T));
        if (e == cudaSuccess) cap = want;
        return e;
    }

private:
    void release() {
        if (p) Free(p);
        p = nullptr;
        cap = 0;
    }
};
template <class T>
using DevBuf = Buf<T, cudaMalloc, cudaFree>;
template <class T>
using PinnedBuf = Buf<T, cudaMallocHost, cudaFreeHost>;

int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

}  // namespace

struct gb200_engine {
    int device = 0, fs = 0, N = 0, s = 0, num_sms = 148;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    DevBuf<float2> tw1, tw2, crep, iq_own, spec, d_replica;
    DevBuf<uint8_t> chips;
    DevBuf<double> d_doppler;
    DevBuf<int> d_ints;
    DevBuf<CellRecord> d_records;
    DevBuf<float> d_profile;
    // on-device refinement (gb200_detect)
    DevBuf<RefineState> r_state;
    DevBuf<double> r_doppler;
    DevBuf<CellRecord> r_records;
    DevBuf<int> r_ints;
    DevBuf<RefineResult> r_results;
    DevBuf<int> r_cell_prn;
    PinnedBuf<int> rh_cell_prn;
    PinnedBuf<int> rh_ints;
    PinnedBuf<RefineResult> rh_results;
    PinnedBuf<float2> h_iq;
    PinnedBuf<CellRecord> h_records;
    PinnedBuf<int> h_ints;
    PinnedBuf<double> h_doubles;
    PinnedBuf<float> h_profile;
    std::vector<double> doppler_cache;  // what d_doppler[0..] currently holds (grid mode)
    std::vector<int> prn_cache;         // what d_ints[0..] currently holds (grid mode)
    bool grid_cache_valid = false;
    int n_prn = 0;
    const float2* iq = nullptr;
    int64_t iq_samples = 0;
    int64_t launches = 0;
    size_t spec_budget_bytes = 512u << 20;
    int np_override = 0, rsplit_override = 0;
    int w2048 = 12;  // one-warp-per-transform correlate kernel: warps per CTA for single-ms searches (0 = use the pair kernel)
    bool timing = false;
    int fused = -1;  // acquire_cells kernel choice: -1 automatic, 0 doppler_spectra + correlate_cells, 1 fused block-per-cell
    bool detect_fused = true;  // gb200_detect: fused block-per-cell kernel (every cell has its own Doppler)
    bool fused_configured = false;
    DevBuf<BestRecord> d_best;
    PinnedBuf<BestRecord> h_best;
    // gb200_acquire_grid_host: one CUDA graph (copy-in, doppler_spectra, correlate_cells, copy-out) per grid shape
    struct HostGraph {
        // What a captured graph bakes in: the grid's shape, every buffer its nodes dereference and the capture stream.
        struct Key {
            int n_blocks, M, P, D, kind;
            const void *iq_dev, *rec_dev, *iq_stage, *rec_stage, *spec, *d_dop, *d_prn, *crep;
            const void* rec_target;  // where the captured correlate kernel stores its records
            cudaStream_t stream;
            auto tie() const {
                return std::tie(n_blocks, M, P, D, kind, iq_dev, rec_dev, iq_stage, rec_stage, spec, d_dop, d_prn, crep, rec_target,
                                stream);
            }
            bool operator==(const Key& o) const { return tie() == o.tie(); }
        };
        cudaGraphExec_t exec = nullptr;
        int seen = 0;
        Key key{};
        std::vector<double> dop;  // the grid's axes, compared in place against the caller's
        std::vector<int> prn;
    } hg;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev[2];
    size_t ev_used[2] = {0, 0};
    std::string err;

    ~gb200_engine() {
        if (hg.exec) cudaGraphExecDestroy(hg.exec);
        for (auto& pool : ev)
            for (auto& pr : pool) {
                cudaEventDestroy(pr.first);
                cudaEventDestroy(pr.second);
            }
        if (own_stream) cudaStreamDestroy(own_stream);
    }
};

struct gb200_tracker {
    gb200_engine* e = nullptr;
    int n_channels = 0;
    std::vector<char> seeded;     // pool slots that hold a channel (gb200_tracker_create seeds all)
    std::vector<char> undo_ok;    // shadow[c] holds channel c's state before its last keep_undo launch
    std::vector<int> sel_cache;   // what d_sel currently holds
    DevBuf<TrackState> states, shadow;
    DevBuf<int> d_sel;
    PinnedBuf<int> h_sel;
    DevBuf<TrackMsRecord> d_out;
    DevBuf<double> d_times;
    DevBuf<float> d_prof;
    PinnedBuf<TrackMsRecord> h_out;
    PinnedBuf<double> h_times;
    PinnedBuf<float> h_prof;
    int last_n_ms = 0;  // records of the last gb200_tracker_process call still in d_out
    DevBuf<BitState> bit_states;
    DevBuf<BitEvent> d_events;
    DevBuf<int> d_counts;
    DevBuf<double> d_bit_times;
    PinnedBuf<BitEvent> h_events;
    PinnedBuf<int> h_counts;
    PinnedBuf<double> h_bit_times;
};
// A pipelined stream of grid batches: slot k's host->device copy, compute and device->host copy run on three streams.
struct gb200_grid_stream {
    gb200_engine* e = nullptr;
    int n_blocks = 0, M = 0, P = 0, D = 0, kind = 0, depth = 0;
    std::vector<int32_t> prn;
    std::vector<double> dop;
    struct Slot {
        DevBuf<float2> iq;
        DevBuf<CellRecord> rec;
        PinnedBuf<float2> h_iq;       // staging, only when the caller's IQ is pageable
        PinnedBuf<CellRecord> h_rec;  // staging, only when the caller's record buffer is pageable
        gb200_cell_record* out = nullptr;  // where this batch's records go
        bool staged_out = false;
        cudaEvent_t h2d = nullptr, done = nullptr, d2h = nullptr;
        ~Slot() {
            for (cudaEvent_t ev : {h2d, done, d2h})
                if (ev) cudaEventDestroy(ev);
        }
    };
    std::vector<Slot> slots;
    cudaStream_t s_in = nullptr, s_out = nullptr;
    long long head = 0, tail = 0;  // batches submitted / collected
    ~gb200_grid_stream() {
        if (s_in) cudaStreamDestroy(s_in);
        if (s_out) cudaStreamDestroy(s_out);
    }
};

// Device-resident rolling window of the newest milliseconds; every millisecond is stored at slot k and at slot
// k + capacity, so the newest n <= capacity milliseconds are contiguous whatever the write position.
struct gb200_ring {
    gb200_engine* e = nullptr;
    int capacity = 0;
    int64_t appended = 0;
    DevBuf<float2> buf;        // [2 * capacity][N]
    PinnedBuf<float2> h_stage;  // staging for pageable callers
};

static_assert(sizeof(gb200_track_record) == sizeof(TrackMsRecord), "ABI track record and device record must match");
static_assert(sizeof(gb200_best_record) == sizeof(BestRecord), "ABI best record and device record must match");
static_assert(sizeof(gb200_bit_event) == sizeof(BitEvent), "ABI bit event and device event must match");

#define GB_FAIL(e, code, ...)                        \
    do {                                             \
        char buf_[512];                              \
        snprintf(buf_, sizeof(buf_), __VA_ARGS__);   \
        (e)->err = buf_;                             \
        return code;                                 \
    } while (0)

#define GB_CUDA(e, expr)                                                                                   \
    do {                                                                                                   \
        cudaError_t ce_ = (expr);                                                                          \
        if (ce_ != cudaSuccess) {                                                                          \
            cudaGetLastError();                                                                            \
            GB_FAIL(e, GB200_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(ce_), __FILE__, __LINE__); \
        }                                                                                                  \
    } while (0)

// passes on the GB200_* code of a call that has already set the error message
#define GB_TRY(expr)            \
    do {                        \
        const int rc_ = (expr); \
        if (rc_) return rc_;    \
    } while (0)

namespace {

// optional event bracket around one kernel launch (measurement aid, off by default)
struct TimedLaunch {
    gb200_engine* e;
    int which;
    cudaEvent_t stop = nullptr;
    TimedLaunch(gb200_engine* e_, int which_) : e(e_), which(which_) {
        if (!e->timing) return;
        auto& pool = e->ev[which];
        if (e->ev_used[which] == pool.size()) {
            cudaEvent_t a, b;
            if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return;
            pool.emplace_back(a, b);
        }
        auto& pr = pool[e->ev_used[which]++];
        cudaEventRecord(pr.first, e->stream);
        stop = pr.second;
    }
    ~TimedLaunch() {
        if (stop) cudaEventRecord(stop, e->stream);
    }
};

// How many warp pairs share one cell.  With plenty of cells per pair each pair keeps a whole cell (no cross-pair
// merge, no CTA-wide barrier); small launches split a cell's polyphase branches over pairs to fill the machine.
int pick_rsplit(const gb200_engine* e, int np, long long n_cells) {
    if (e->rsplit_override > 0 && e->s % e->rsplit_override == 0 && np % e->rsplit_override == 0) return e->rsplit_override;
    if (n_cells >= 8LL * e->num_sms * np) return 1;
    return std::gcd(e->s, np);
}

// Non-coherent, record-only launches use the one-warp-per-transform kernel: 12 warps per CTA (168 registers) for
// single-millisecond searches, 8 warps (the 32 accumulators live across the milliseconds: 226 registers) for longer
// integrations.  With the packed-FP32 codelets it beats the warp-pair kernel everywhere (config 3: 0.219 -> 0.181 ms,
// profiles/ablation_r2.md), so the pair kernel keeps only the coherent and full-profile launches.
// Returns the warps per CTA, or 0 for the pair kernel.  GB200_W2048=0 disables it, =10 runs single-ms searches with 10 warps.
int pick_w2048(const gb200_engine* e, int M, int kind, bool profile) {
    if (e->w2048 <= 0 || kind != GB200_NON_COHERENT || profile) return 0;
    if (M == 1) return e->w2048 == 10 ? 10 : 12;
    return 8;
}

// Warp pairs per CTA: 10 (20 warps / SM) for single-millisecond non-coherent searches, 8 otherwise (the
// multi-millisecond accumulators need the larger register budget).  GB200_NP=8 forces the 8-pair build.
int pick_np(const gb200_engine* e, int M, int kind, bool profile) {
    if (e->np_override == 8) return 8;
    return (M == 1 && kind == GB200_NON_COHERENT && !profile) ? 10 : 8;
}

// The correlate kernel of one launch shape: nw warps per CTA of the one-warp kernel, or (nw = 0) the pair kernel with np pairs;
// rsplit slots share a cell, so a group holds cpg cells.
struct CorrPlan {
    int nw, np, rsplit, cpg;
};

CorrPlan plan_correlate(const gb200_engine* e, int M, int kind, bool profile, long long n_cells) {
    const int nw = pick_w2048(e, M, kind, profile);
    const int np = nw ? nw : pick_np(e, M, kind, profile);  // CTA "slots": warps (one-warp kernel) or warp pairs
    const int rsplit = pick_rsplit(e, np, n_cells);
    return {nw, np, rsplit, np / rsplit};
}

size_t unit_floats2(const gb200_engine* e, int M) { return static_cast<size_t>(M) * e->s * 2 * kFft; }

// need_replicas = false: the caller brings its own replica (gb200_correlation_profile_replica)
int check_common(gb200_engine* e, int n_ms, int kind, bool need_replicas = true) {
    if (!e) return GB200_EINVAL;
    if (kind != GB200_COHERENT && kind != GB200_NON_COHERENT) GB_FAIL(e, GB200_EINVAL, "Unexpected integration type");
    if (need_replicas && e->n_prn == 0) GB_FAIL(e, GB200_ESTATE, "no PRN replicas loaded (gb200_set_replicas)");
    if (!e->iq) GB_FAIL(e, GB200_ESTATE, "no IQ loaded (gb200_upload_iq / gb200_bind_iq_device)");
    if (n_ms < 1) GB_FAIL(e, GB200_EINVAL, "need at least one whole millisecond of samples");
    return GB200_OK;
}

int check_prns(gb200_engine* e, const int32_t* prn_idx, int n) {
    for (int i = 0; i < n; ++i)
        if (prn_idx[i] < 0 || prn_idx[i] >= e->n_prn) GB_FAIL(e, GB200_EINVAL, "prn index %d out of range", prn_idx[i]);
    return GB200_OK;
}

// n_ms milliseconds from the start of the bound IQ
int check_samples(gb200_engine* e, int n_ms) {
    const long long need = static_cast<long long>(n_ms) * e->N;
    if (need > e->iq_samples)
        GB_FAIL(e, GB200_EINVAL, "need %lld samples, %lld loaded", need, static_cast<long long>(e->iq_samples));
    return GB200_OK;
}

int check_channel(gb200_tracker* t, int channel) {
    if (channel < 0 || channel >= t->n_channels) GB_FAIL(t->e, GB200_EINVAL, "channel %d out of range", channel);
    return GB200_OK;
}

// A device buffer and its pinned host staging, both grown to at least n elements.
template <class T>
cudaError_t ensure_staging(DevBuf<T>& dev, PinnedBuf<T>& host, size_t n) {
    const cudaError_t ce = dev.ensure(n);
    return ce == cudaSuccess ? host.ensure(n) : ce;
}

// The staging pair (device buffer, pinned host buffer) receives n elements of src and queues their upload.  The caller makes
// sure the host buffer is no longer in flight.
template <class T>
int stage_upload(gb200_engine* e, DevBuf<T>& dev, PinnedBuf<T>& host, const T* src, size_t n) {
    GB_CUDA(e, ensure_staging(dev, host, n));
    memcpy(host.p, src, sizeof(T) * n);
    GB_CUDA(e, cudaMemcpyAsync(dev.p, host.p, sizeof(T) * n, cudaMemcpyHostToDevice, e->stream));
    return GB200_OK;
}

// n elements from the device to the caller through pinned staging (already large enough): one copy, one synchronise.
template <class T>
int download(gb200_engine* e, void* out_host, PinnedBuf<T>& stage, const T* src_dev, size_t n) {
    GB_CUDA(e, cudaMemcpyAsync(stage.p, src_dev, n * sizeof(T), cudaMemcpyDeviceToHost, e->stream));
    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    memcpy(out_host, stage.p, n * sizeof(T));
    return GB200_OK;
}

// The device address of page-locked host memory, or null when p is pageable.
void* pinned_alias(const void* p) {
    cudaPointerAttributes attr{};
    const bool pinned = cudaPointerGetAttributes(&attr, p) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    return pinned ? attr.devicePointer : nullptr;
}

// Where a copy of n samples from the caller's buffer starts: the buffer itself when it is pinned, else the pinned staging
// buffer, refilled once the stream has stopped reading it.
int pinned_source(gb200_engine* e, PinnedBuf<float2>& stage, const float* host, size_t n, const float2** src) {
    *src = reinterpret_cast<const float2*>(host);
    if (pinned_alias(host)) return GB200_OK;
    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    GB_CUDA(e, stage.ensure(std::max<size_t>(n, 1)));
    memcpy(stage.p, host, n * sizeof(float2));
    *src = stage.p;
    return GB200_OK;
}

cudaError_t ensure_fused_configured(gb200_engine* e) {
    if (e->fused_configured) return cudaSuccess;
    const cudaError_t ce = configure_fused_kernel();
    e->fused_configured = ce == cudaSuccess;
    return ce;
}

// The three acquisition kernels, each with its optional timing events and counted in e->launches.
int enqueue_spectra(gb200_engine* e, const float2* iq, long long block_stride, const double* dop, int M, int n_doppler,
                    int n_units) {
    SpectraArgs sa{};
    sa.iq = iq;
    sa.doppler = dop;
    sa.spec = e->spec.p;
    sa.tw1 = e->tw1.p;
    sa.tw2 = e->tw2.p;
    sa.block_stride = block_stride;
    sa.inv_fs = 1.0 / static_cast<double>(e->fs);
    sa.N = e->N;
    sa.s = e->s;
    sa.M = M;
    sa.n_doppler = n_doppler;
    sa.n_units = n_units;
    TimedLaunch tl(e, 0);
    GB_CUDA(e, launch_doppler_spectra(sa, e->stream));
    e->launches++;
    return GB200_OK;
}

// The engine's part of a correlate launch; the caller adds the grid-mode or list-mode cell layout.
CorrelateArgs correlate_args(const gb200_engine* e, int M, int kind, CellRecord* records) {
    CorrelateArgs ca{};
    ca.spec = e->spec.p;
    ca.crep = e->crep.p;
    ca.tw1 = e->tw1.p;
    ca.tw2 = e->tw2.p;
    ca.records = records;
    ca.N = e->N;
    ca.s = e->s;
    ca.M = M;
    ca.kind = kind;
    return ca;
}

int enqueue_correlate(gb200_engine* e, const CorrPlan& plan, CorrelateArgs ca, int grid) {
    ca.rsplit = plan.rsplit;
    TimedLaunch tl(e, 1);
    if (plan.nw) GB_CUDA(e, launch_correlate_w2048(ca, plan.nw, grid, e->stream));
    else GB_CUDA(e, launch_correlate_cells(ca, plan.np, grid, e->stream));
    e->launches++;
    return GB200_OK;
}

// one CTA per cell, whole pipeline in one kernel
int enqueue_fused(gb200_engine* e, int M, int kind, const double* dop, const int* prn, const int* probe, CellRecord* records,
                  int n_cells) {
    FusedArgs fa{};
    fa.iq = e->iq;
    fa.doppler = dop;
    fa.prn = prn;
    fa.probe = probe;
    fa.records = records;
    fa.crep = e->crep.p;
    fa.tw1 = e->tw1.p;
    fa.tw2 = e->tw2.p;
    fa.inv_fs = 1.0 / static_cast<double>(e->fs);
    fa.N = e->N;
    fa.M = M;
    fa.n_cells = n_cells;
    TimedLaunch tl(e, 1);
    GB_CUDA(e, launch_acquire_fused(fa, e->s, kind, e->stream));
    e->launches++;
    return GB200_OK;
}

// L2 windows of the one-warp kernel (see the kernel): a batch whose spectra exceed L2 is walked in equal runs of units of
// about GB200_L2_WINDOW_MB (default 40; 0 = off), as long as a window still gives every CTA at least two groups (config 5's
// heavy cells: 2.8 groups per CTA and window; the kernel's round-robin of the extra groups keeps the CTAs together).
// Returns the chunks per window, 0 for one window over the whole batch.
int l2_window_chunks(size_t batch_bytes, int chunks, int P, int grid) {
    static const size_t win_bytes = static_cast<size_t>(std::max(0, env_int("GB200_L2_WINDOW_MB", 40))) << 20;
    if (!win_bytes || batch_bytes <= win_bytes + win_bytes / 2) return 0;
    const long long n_win = static_cast<long long>((batch_bytes + win_bytes - 1) / win_bytes);
    long long wc = (chunks + n_win - 1) / n_win;
    // a window whose P * wc groups divide evenly among the CTAs, when one exists within a quarter of the target size
    const long long q = grid / std::gcd(P, grid);
    const long long even = ((wc + q / 2) / q) * q;
    if (even > 0 && even * 4 >= wc * 3 && even * 4 <= wc * 5) wc = even;
    static const int min_groups = env_int("GB200_L2_WINDOW_MIN_GROUPS", 2);
    return (wc * P >= static_cast<long long>(min_groups) * grid && wc < chunks) ? static_cast<int>(wc) : 0;
}

// The grid's axes (PRN rows in d_ints, Doppler bins in d_doppler) are uploaded only when they changed -- or when a list-mode
// call (gb200_acquire_cells / gb200_detect) has reused those device buffers since.
int upload_grid_axes(gb200_engine* e, const int32_t* prn_idx, int P, const double* dop, int D) {
    const bool same = e->grid_cache_valid && static_cast<int>(e->doppler_cache.size()) == D &&
                      static_cast<int>(e->prn_cache.size()) == P &&
                      memcmp(e->doppler_cache.data(), dop, sizeof(double) * D) == 0 &&
                      memcmp(e->prn_cache.data(), prn_idx, sizeof(int) * P) == 0;
    if (same) return GB200_OK;
    GB_CUDA(e, cudaStreamSynchronize(e->stream));  // staging buffers may still be in flight
    e->grid_cache_valid = false;                   // until both axes are queued
    GB_TRY(stage_upload(e, e->d_doppler, e->h_doubles, dop, D));
    GB_TRY(stage_upload(e, e->d_ints, e->h_ints, prn_idx, P));
    e->doppler_cache.assign(dop, dop + D);
    e->prn_cache.assign(prn_idx, prn_idx + P);
    e->grid_cache_valid = true;
    return GB200_OK;
}

// grid mode: all cells of n_blocks x prn list x doppler list; records written to rec_dev (device)
int run_grid(gb200_engine* e, int n_blocks, int M, const int32_t* prn_idx, int P, const double* dop, int D, int kind,
             CellRecord* rec_dev) {
    GB_TRY(check_common(e, M, kind));
    if (n_blocks < 1 || P < 1 || D < 1 || !prn_idx || !dop) GB_FAIL(e, GB200_EINVAL, "empty grid");
    if (static_cast<int64_t>(n_blocks) * M * e->N > e->iq_samples)
        GB_FAIL(e, GB200_EINVAL, "grid needs %lld samples, %lld loaded", static_cast<long long>(n_blocks) * M * e->N,
                static_cast<long long>(e->iq_samples));
    GB_TRY(check_prns(e, prn_idx, P));

    GB_TRY(upload_grid_axes(e, prn_idx, P, dop, D));

    const size_t unit = unit_floats2(e, M);
    const size_t per_block = unit * D;
    int nb = static_cast<int>(std::max<size_t>(1, e->spec_budget_bytes / (per_block * sizeof(float2))));
    nb = std::min(nb, n_blocks);
    GB_CUDA(e, e->spec.ensure(per_block * nb));

    const CorrPlan plan = plan_correlate(e, M, kind, false, static_cast<long long>(nb) * P * D);
    for (int b0 = 0; b0 < n_blocks; b0 += nb) {
        const int nbb = std::min(nb, n_blocks - b0);
        const int chunks = (nbb * D + plan.cpg - 1) / plan.cpg;  // groups per PRN: its nbb*D cells in chunks of cpg
        const long long stride = static_cast<long long>(M) * e->N;
        GB_TRY(enqueue_spectra(e, e->iq + static_cast<size_t>(b0) * stride, stride, e->d_doppler.p, M, D, nbb * D));

        CorrelateArgs ca = correlate_args(e, M, kind, rec_dev + static_cast<size_t>(b0) * P * D);
        ca.n_groups = P * chunks;
        ca.grid_mode = 1;
        ca.P = P;
        ca.D = D;
        ca.n_blocks = nbb;
        ca.chunks = chunks;
        ca.prn_idx = e->d_ints.p;
        const int grid = std::min(ca.n_groups, e->num_sms);
        if (plan.nw) ca.win_chunks = l2_window_chunks(static_cast<size_t>(nbb) * per_block * sizeof(float2), chunks, P, grid);
        GB_TRY(enqueue_correlate(e, plan, ca, grid));
    }
    return GB200_OK;
}

// list mode.  Cells are sorted by PRN and cut into chunks whose spectra fit the scratch budget.
int run_cells(gb200_engine* e, int n_cells, const int32_t* prn_idx, const double* dop, const int32_t* probe, int M,
              int kind, CellRecord* rec_dev, float* profile_dev) {
    GB_TRY(check_common(e, M, kind));
    if (n_cells < 1 || !prn_idx || !dop) GB_FAIL(e, GB200_EINVAL, "empty cell list");
    GB_TRY(check_samples(e, M));
    GB_TRY(check_prns(e, prn_idx, n_cells));
    e->grid_cache_valid = false;  // d_ints / d_doppler are about to be overwritten

    bool use_fused = e->fused == 1;
    if (e->fused < 0 && fused_supports(e->s) && !profile_dev) {
        // Automatic choice.  The split kernels pay off when many cells share a Doppler bin (the PRN-independent half is
        // computed once per bin); lists with mostly distinct Dopplers (the refinement passes of acquisition.py:81-101)
        // and small lists are faster through the fused block-per-cell kernel (profiles/configs_r1l.jsonl).
        std::vector<double> u(dop, dop + n_cells);
        std::sort(u.begin(), u.end());
        const long long n_unique = std::unique(u.begin(), u.end()) - u.begin();
        use_fused = n_unique * 4 > n_cells || static_cast<long long>(n_cells) * M <= 8192;
    }
    if (use_fused && fused_supports(e->s) && !profile_dev) {
        GB_CUDA(e, ensure_fused_configured(e));
        GB_CUDA(e, cudaStreamSynchronize(e->stream));
        GB_CUDA(e, ensure_staging(e->d_ints, e->h_ints, static_cast<size_t>(n_cells) * 2));
        GB_CUDA(e, ensure_staging(e->d_doppler, e->h_doubles, n_cells));
        for (int i = 0; i < n_cells; ++i) {
            e->h_ints.p[i] = prn_idx[i];
            e->h_ints.p[n_cells + i] = probe ? probe[i] : -1;
            e->h_doubles.p[i] = dop[i];
        }
        GB_CUDA(e, cudaMemcpyAsync(e->d_ints.p, e->h_ints.p, sizeof(int) * 2 * n_cells, cudaMemcpyHostToDevice, e->stream));
        GB_CUDA(e, cudaMemcpyAsync(e->d_doppler.p, e->h_doubles.p, sizeof(double) * n_cells, cudaMemcpyHostToDevice, e->stream));
        return enqueue_fused(e, M, kind, e->d_doppler.p, e->d_ints.p, e->d_ints.p + n_cells, rec_dev, n_cells);
    }

    const CorrPlan plan = plan_correlate(e, M, kind, profile_dev != nullptr, n_cells);
    const int cpg = plan.cpg;
    std::vector<int> order(n_cells);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return prn_idx[a] < prn_idx[b]; });

    const size_t unit = unit_floats2(e, M);
    const int max_cells = static_cast<int>(std::max<size_t>(cpg, e->spec_budget_bytes / (unit * sizeof(float2)) / cpg * cpg));

    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    // probe indices live at the front of the int buffer for the whole call
    const size_t ints_needed = static_cast<size_t>(n_cells) * 3 + 3 * (static_cast<size_t>(n_cells) + 1);
    GB_CUDA(e, ensure_staging(e->d_ints, e->h_ints, ints_needed));
    GB_CUDA(e, ensure_staging(e->d_doppler, e->h_doubles, n_cells));
    for (int i = 0; i < n_cells; ++i) e->h_ints.p[i] = probe ? probe[i] : -1;
    GB_CUDA(e, cudaMemcpyAsync(e->d_ints.p, e->h_ints.p, sizeof(int) * n_cells, cudaMemcpyHostToDevice, e->stream));
    GB_CUDA(e, e->spec.ensure(unit * std::min(max_cells, n_cells)));

    int c0 = 0;
    while (c0 < n_cells) {
        // take up to max_cells sorted cells, ending on a PRN-group boundary where possible
        int c1 = std::min(n_cells, c0 + max_cells);
        // plan arrays for this chunk (indices into the chunk)
        std::map<double, int> uniq;
        std::vector<double> udop;
        std::vector<int> cell_u, cell_out, g_first, g_count, g_prn;
        for (int c = c0; c < c1; ++c) {
            const int orig = order[c];
            auto it = uniq.find(dop[orig]);
            int u;
            if (it == uniq.end()) {
                u = static_cast<int>(udop.size());
                uniq.emplace(dop[orig], u);
                udop.push_back(dop[orig]);
            } else {
                u = it->second;
            }
            cell_u.push_back(u);
            cell_out.push_back(orig);
            if (g_prn.empty() || g_prn.back() != prn_idx[orig] || g_count.back() == cpg) {
                g_first.push_back(c - c0);
                g_count.push_back(1);
                g_prn.push_back(prn_idx[orig]);
            } else {
                g_count.back()++;
            }
        }
        const int nc = c1 - c0, ng = static_cast<int>(g_prn.size()), nu = static_cast<int>(udop.size());
        // the staging buffers are reused per chunk: wait for the previous chunk's copies
        if (c0 > 0) GB_CUDA(e, cudaStreamSynchronize(e->stream));
        int* hi = e->h_ints.p + n_cells;
        int* di = e->d_ints.p + n_cells;
        memcpy(hi, cell_u.data(), sizeof(int) * nc);
        memcpy(hi + nc, cell_out.data(), sizeof(int) * nc);
        memcpy(hi + 2 * nc, g_first.data(), sizeof(int) * ng);
        memcpy(hi + 2 * nc + ng, g_count.data(), sizeof(int) * ng);
        memcpy(hi + 2 * nc + 2 * ng, g_prn.data(), sizeof(int) * ng);
        memcpy(e->h_doubles.p, udop.data(), sizeof(double) * nu);
        GB_CUDA(e, cudaMemcpyAsync(di, hi, sizeof(int) * (2 * nc + 3 * ng), cudaMemcpyHostToDevice, e->stream));
        GB_CUDA(e, cudaMemcpyAsync(e->d_doppler.p, e->h_doubles.p, sizeof(double) * nu, cudaMemcpyHostToDevice, e->stream));

        GB_TRY(enqueue_spectra(e, e->iq, 0, e->d_doppler.p, M, nu, nu));

        CorrelateArgs ca = correlate_args(e, M, kind, rec_dev);
        ca.profile = profile_dev;
        ca.n_groups = ng;
        ca.cell_u = di;
        ca.cell_out = di + nc;
        ca.grp_first = di + 2 * nc;
        ca.grp_count = di + 2 * nc + ng;
        ca.grp_prn = di + 2 * nc + 2 * ng;
        ca.cell_probe = e->d_ints.p;
        GB_TRY(enqueue_correlate(e, plan, ca, std::min(ng, e->num_sms)));
        c0 = c1;
    }
    return GB200_OK;
}

// Records to the caller: straight DMA when the caller's buffer is pinned, else through the engine's pinned staging.
int fetch_records(gb200_engine* e, size_t n, gb200_cell_record* out_host) {
    if (pinned_alias(out_host)) {
        GB_CUDA(e, cudaMemcpyAsync(out_host, e->d_records.p, n * sizeof(CellRecord), cudaMemcpyDeviceToHost, e->stream));
        GB_CUDA(e, cudaStreamSynchronize(e->stream));
        return GB200_OK;
    }
    GB_CUDA(e, e->h_records.ensure(n));
    return download(e, out_host, e->h_records, e->d_records.p, n);
}

}  // namespace

extern "C" {

int gb200_abi_version(void) { return GB200_ABI_VERSION; }

const char* gb200_last_error(const gb200_engine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

int gb200_create(int device, int fs, int n, gb200_engine** out) {
    if (!out) return GB200_EINVAL;
    *out = nullptr;
    if (n <= 0 || n % kChips != 0 || fs <= 0) {
        g_create_error = "samples_per_ms must be a positive multiple of 1023 and samples_per_second positive";
        return GB200_EINVAL;
    }
    int count = 0;
    cudaError_t ce = cudaGetDeviceCount(&count);
    if (ce != cudaSuccess || device < 0 || device >= count) {
        cudaGetLastError();
        g_create_error = std::string("no usable CUDA device (there is no CPU fallback): ") +
                         (ce != cudaSuccess ? cudaGetErrorString(ce) : "ordinal out of range");
        return GB200_ECUDA;
    }
    gb200_engine* e = new gb200_engine;
    e->device = device;
    e->fs = fs;
    e->N = n;
    e->s = n / kChips;
    // Spectra scratch per launch pair.  It does not have to stay in L2: a launch writes and re-reads 21 MB per 16.368 Msps block
    // in ~0.15 ms (< 0.3 TB/s), and launches that carry more cells run the correlate kernel without cross-warp merges and with a
    // shorter tail (config 5: 99.7 -> 121.6 Msamples/s going from 80 MB to 512 MB; config 2 x 512 blocks +3 %).
    e->spec_budget_bytes = static_cast<size_t>(env_int("GB200_SPEC_BUDGET_MB", 512)) << 20;
    e->np_override = env_int("GB200_NP", 0);
    e->w2048 = env_int("GB200_W2048", 12);
    e->rsplit_override = env_int("GB200_RSPLIT", 0);
    e->detect_fused = env_int("GB200_DETECT_FUSED", 1) != 0;
    auto fail = [&](cudaError_t c, const char* what) {
        g_create_error = std::string(what) + ": " + cudaGetErrorString(c);
        cudaGetLastError();
        delete e;
        return GB200_ECUDA;
    };
    if ((ce = cudaSetDevice(device)) != cudaSuccess) return fail(ce, "cudaSetDevice");
    cudaDeviceProp prop;
    if ((ce = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return fail(ce, "cudaGetDeviceProperties");
    if (prop.major != 10) {
        g_create_error = "this build targets sm_100a (B200) only";
        delete e;
        return GB200_ECUDA;
    }
    e->num_sms = prop.multiProcessorCount;
    if (!spectra_supports(e->s)) {
        g_create_error = "samples_per_ms / 1023 must be one of 1,2,3,4,5,6,8,10,12,16";
        delete e;
        return GB200_EINVAL;
    }
    if ((ce = cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking)) != cudaSuccess) return fail(ce, "cudaStreamCreate");
    e->stream = e->own_stream;
    if ((ce = configure_kernels()) != cudaSuccess) return fail(ce, "cudaFuncSetAttribute");
    if ((ce = e->tw1.ensure(kFft)) != cudaSuccess) return fail(ce, "cudaMalloc");
    if ((ce = e->tw2.ensure(kFft)) != cudaSuccess) return fail(ce, "cudaMalloc");
    if ((ce = launch_init_tables(e->tw1.p, e->tw2.p, e->stream)) != cudaSuccess) return fail(ce, "init_tables");
    e->launches++;
    if ((ce = cudaStreamSynchronize(e->stream)) != cudaSuccess) return fail(ce, "init_tables sync");
    *out = e;
    return GB200_OK;
}

int gb200_destroy(gb200_engine* e) {
    if (!e) return GB200_OK;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    delete e;  // ~gb200_engine releases every device / pinned allocation, the events and the stream
    return GB200_OK;
}

int gb200_set_stream(gb200_engine* e, void* st) {
    if (!e) return GB200_EINVAL;
    GB_CUDA(e, cudaSetDevice(e->device));
    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    e->stream = st ? static_cast<cudaStream_t>(st) : e->own_stream;
    return GB200_OK;
}

int gb200_set_replicas(gb200_engine* e, const uint8_t* chips, int n_prn) {
    if (!e) return GB200_EINVAL;
    if (!chips || n_prn < 1) GB_FAIL(e, GB200_EINVAL, "need at least one PRN code");
    for (int i = 0; i < n_prn * kChips; ++i)
        if (chips[i] > 1) GB_FAIL(e, GB200_EINVAL, "chips must be 0 or 1");
    GB_CUDA(e, cudaSetDevice(e->device));
    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    GB_CUDA(e, e->chips.ensure(static_cast<size_t>(n_prn) * kChips));
    GB_CUDA(e, e->crep.ensure(static_cast<size_t>(n_prn) * 2 * kFft));
    GB_CUDA(e, cudaMemcpyAsync(e->chips.p, chips, static_cast<size_t>(n_prn) * kChips, cudaMemcpyHostToDevice, e->stream));
    GB_CUDA(e, launch_replica_spectra(e->chips.p, n_prn, e->crep.p, e->stream));
    e->launches++;
    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    e->n_prn = n_prn;
    return GB200_OK;
}

int gb200_upload_iq(gb200_engine* e, const float* iq_host, int64_t n_samples) {
    if (!e) return GB200_EINVAL;
    if (!iq_host || n_samples < 0) GB_FAIL(e, GB200_EINVAL, "bad IQ buffer");
    GB_CUDA(e, cudaSetDevice(e->device));
    GB_CUDA(e, e->iq_own.ensure(static_cast<size_t>(std::max<int64_t>(n_samples, 1))));
    const float2* src = nullptr;
    GB_TRY(pinned_source(e, e->h_iq, iq_host, static_cast<size_t>(n_samples), &src));
    GB_CUDA(e, cudaMemcpyAsync(e->iq_own.p, src, static_cast<size_t>(n_samples) * sizeof(float2), cudaMemcpyHostToDevice,
                               e->stream));
    e->iq = e->iq_own.p;
    e->iq_samples = n_samples;
    return GB200_OK;
}

int gb200_bind_iq_device(gb200_engine* e, const void* iq_device, int64_t n_samples) {
    if (!e) return GB200_EINVAL;
    if (!iq_device || n_samples < 0) GB_FAIL(e, GB200_EINVAL, "bad IQ buffer");
    // the fused acquisition kernel stages the IQ with cp.async.bulk and the tracking kernel with 16-byte cp.async
    if (reinterpret_cast<uintptr_t>(iq_device) % 16 != 0) GB_FAIL(e, GB200_EINVAL, "IQ buffer must be 16-byte aligned");
    e->iq = static_cast<const float2*>(iq_device);
    e->iq_samples = n_samples;
    return GB200_OK;
}

int gb200_acquire_grid_device(gb200_engine* e, int n_blocks, int M, const int32_t* prn_idx, int P, const double* dop, int D,
                              int kind, void* out_device) {
    if (!e) return GB200_EINVAL;
    if (!out_device) GB_FAIL(e, GB200_EINVAL, "null output");
    GB_CUDA(e, cudaSetDevice(e->device));
    return run_grid(e, n_blocks, M, prn_idx, P, dop, D, kind, static_cast<CellRecord*>(out_device));
}

int gb200_acquire_grid(gb200_engine* e, int n_blocks, int M, const int32_t* prn_idx, int P, const double* dop, int D,
                       int kind, gb200_cell_record* out_host) {
    if (!e) return GB200_EINVAL;
    if (!out_host) GB_FAIL(e, GB200_EINVAL, "null output");
    GB_CUDA(e, cudaSetDevice(e->device));
    if (n_blocks < 1 || P < 1 || D < 1) GB_FAIL(e, GB200_EINVAL, "empty grid");
    const size_t n = static_cast<size_t>(n_blocks) * P * D;
    GB_CUDA(e, e->d_records.ensure(n));
    GB_TRY(run_grid(e, n_blocks, M, prn_idx, P, dop, D, kind, e->d_records.p));
    return fetch_records(e, n, out_host);
}

// acquisition.py:179-189 per (block, prn) row on the device: the grid, then one reduction kernel over its records.
int gb200_acquire_grid_best_device(gb200_engine* e, int n_blocks, int M, const int32_t* prn_idx, int P, const double* dop, int D,
                                   int kind, void* out_device) {
    if (!e) return GB200_EINVAL;
    if (!out_device) GB_FAIL(e, GB200_EINVAL, "null output");
    GB_CUDA(e, cudaSetDevice(e->device));
    if (n_blocks < 1 || P < 1 || D < 1) GB_FAIL(e, GB200_EINVAL, "empty grid");
    const size_t n = static_cast<size_t>(n_blocks) * P * D;
    GB_CUDA(e, e->d_records.ensure(n));
    GB_TRY(run_grid(e, n_blocks, M, prn_idx, P, dop, D, kind, e->d_records.p));
    GB_CUDA(e, launch_best_bins(n_blocks * P, D, e->N, e->d_records.p, e->d_doppler.p, static_cast<BestRecord*>(out_device),
                                e->stream));
    e->launches++;
    return GB200_OK;
}

int gb200_acquire_grid_best(gb200_engine* e, int n_blocks, int M, const int32_t* prn_idx, int P, const double* dop, int D,
                            int kind, gb200_best_record* out_host) {
    if (!e) return GB200_EINVAL;
    if (!out_host) GB_FAIL(e, GB200_EINVAL, "null output");
    GB_CUDA(e, cudaSetDevice(e->device));
    if (n_blocks < 1 || P < 1 || D < 1) GB_FAIL(e, GB200_EINVAL, "empty grid");
    const size_t n = static_cast<size_t>(n_blocks) * P;
    GB_CUDA(e, cudaStreamSynchronize(e->stream));  // h_best may still be in flight
    GB_CUDA(e, ensure_staging(e->d_best, e->h_best, n));
    GB_TRY(gb200_acquire_grid_best_device(e, n_blocks, M, prn_idx, P, dop, D, kind, e->d_best.p));
    return download(e, out_host, e->h_best, e->d_best.p, n);
}

// Host to host in one call.  The first call of a shape runs eagerly (it may have to upload the axes and grow buffers,
// which synchronise); the second captures {copy-in, doppler_spectra, correlate_cells, copy-out} into a CUDA graph; from
// then on a call is: 16 KB memcpy into pinned staging, one cudaGraphLaunch, one stream synchronise, memcpy out.
int gb200_acquire_grid_host(gb200_engine* e, const float* iq_host, int n_blocks, int M, const int32_t* prn_idx, int P,
                            const double* dop, int D, int kind, gb200_cell_record* out_host) {
    if (!e) return GB200_EINVAL;
    if (!iq_host || !out_host) GB_FAIL(e, GB200_EINVAL, "null buffer");
    if (n_blocks < 1 || M < 1 || P < 1 || D < 1 || !prn_idx || !dop) GB_FAIL(e, GB200_EINVAL, "empty grid");
    GB_CUDA(e, cudaSetDevice(e->device));
    const size_t n_iq = static_cast<size_t>(n_blocks) * M * e->N, n_rec = static_cast<size_t>(n_blocks) * P * D;
    const size_t spec_bytes = unit_floats2(e, M) * D * sizeof(float2) * n_blocks;
    static const bool graphs = env_int("GB200_GRAPH", 1) != 0;
    if (!graphs || e->timing || spec_bytes > e->spec_budget_bytes) {  // several scratch batches / per-kernel events: plain path
        GB_TRY(gb200_upload_iq(e, iq_host, static_cast<int64_t>(n_iq)));
        return gb200_acquire_grid(e, n_blocks, M, prn_idx, P, dop, D, kind, out_host);
    }
    GB_CUDA(e, cudaStreamSynchronize(e->stream));  // the pinned staging buffers may still be in flight
    GB_CUDA(e, ensure_staging(e->iq_own, e->h_iq, n_iq));
    GB_CUDA(e, ensure_staging(e->d_records, e->h_records, n_rec));
    // Large pinned inputs (a 10-ms window is 327 KB) are copied by the DMA engine straight from the caller's buffer: staging them
    // would cost a 15-20 us host memcpy.  The copy node of the graph has its source baked in, so those calls launch eagerly
    // (1.7 us more than a replay on this host, profiles/launch_latency_r2.log).  Small inputs are staged and replayed.
    const bool eager_src = n_iq * sizeof(float2) > (64u << 10) && pinned_alias(iq_host);
    const float2* h2d_src = eager_src ? reinterpret_cast<const float2*>(iq_host) : e->h_iq.p;
    if (!eager_src) memcpy(e->h_iq.p, iq_host, n_iq * sizeof(float2));
    e->iq = e->iq_own.p;
    e->iq_samples = static_cast<int64_t>(n_iq);

    // The captured kernels read the axes from d_doppler / d_ints and the replica spectra from crep: make sure those hold THIS
    // grid's axes now (a list-mode call may have reused them since the last replay; cheap when nothing changed), and treat a
    // moved buffer (gb200_set_replicas with a larger table, a larger list-mode call) as a new shape.
    {
        if (e->n_prn == 0) GB_FAIL(e, GB200_ESTATE, "no PRN replicas loaded (gb200_set_replicas)");
        GB_TRY(check_prns(e, prn_idx, P));
        GB_TRY(upload_grid_axes(e, prn_idx, P, dop, D));
    }
    // Small grids: the correlate kernel stores its 32-byte records straight into pinned (device-mapped under UVA) memory --
    // posted PCIe writes at the kernel's tail instead of a separate copy node behind it -- and into the CALLER's buffer when that
    // is itself pinned, which also saves the host copy out of the staging buffer.
    const bool direct = n_rec * sizeof(CellRecord) <= (256u << 10);
    CellRecord* caller_alias = direct ? static_cast<CellRecord*>(pinned_alias(out_host)) : nullptr;
    CellRecord* rec_target = caller_alias ? caller_alias : direct ? e->h_records.p : e->d_records.p;
    auto& g = e->hg;
    // what a graph captured now would bake in (a first eager call may still grow the spectra scratch)
    auto key_now = [&] {
        return gb200_engine::HostGraph::Key{n_blocks, M, P, D, kind, e->iq_own.p, e->d_records.p, e->h_iq.p, e->h_records.p,
                                            e->spec.p, e->d_doppler.p, e->d_ints.p, e->crep.p, rec_target, e->stream};
    };
    const bool same = g.seen && g.key == key_now() && memcmp(g.dop.data(), dop, sizeof(double) * D) == 0 &&
                      memcmp(g.prn.data(), prn_idx, sizeof(int) * P) == 0;
    auto enqueue = [&]() -> int {
        GB_CUDA(e, cudaMemcpyAsync(e->iq_own.p, h2d_src, n_iq * sizeof(float2), cudaMemcpyHostToDevice, e->stream));
        GB_TRY(run_grid(e, n_blocks, M, prn_idx, P, dop, D, kind, rec_target));
        if (!direct)
            GB_CUDA(e, cudaMemcpyAsync(e->h_records.p, e->d_records.p, n_rec * sizeof(CellRecord), cudaMemcpyDeviceToHost, e->stream));
        return GB200_OK;
    };
    if (eager_src) {
        GB_TRY(enqueue());
    } else if (same && g.exec) {
        GB_CUDA(e, cudaGraphLaunch(g.exec, e->stream));
        e->launches += 2;
    } else if (same && !g.exec && g.seen == 1) {
        // second call of this shape: the axes are on the device and every buffer has its size, so nothing below synchronises
        g.seen = 2;  // capture is attempted once per shape
        GB_CUDA(e, cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
        int rc = enqueue();
        cudaGraph_t graph = nullptr;
        cudaError_t ce = cudaStreamEndCapture(e->stream, &graph);
        if (rc == GB200_OK && ce == cudaSuccess && graph) ce = cudaGraphInstantiate(&g.exec, graph, 0);
        if (graph) cudaGraphDestroy(graph);
        if (rc != GB200_OK || ce != cudaSuccess || !g.exec) {
            cudaGetLastError();
            g.exec = nullptr;
            rc = enqueue();  // capture unavailable: stay on the eager path for this shape
            if (rc) return rc;
        } else {
            GB_CUDA(e, cudaGraphLaunch(g.exec, e->stream));
        }
    } else {
        if (!same) {
            if (g.exec) cudaGraphExecDestroy(g.exec);
            g.exec = nullptr;
        }
        GB_TRY(enqueue());
        if (!same) {
            g.key = key_now();
            g.dop.assign(dop, dop + D);
            g.prn.assign(prn_idx, prn_idx + P);
            g.seen = 1;
        }
    }
    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    if (!caller_alias) memcpy(out_host, e->h_records.p, n_rec * sizeof(CellRecord));
    return GB200_OK;
}

// ---------------------------------------------------------------------------------------------------------
// device-resident rolling sample window (receiver.py:68,100,219)
// ---------------------------------------------------------------------------------------------------------
int gb200_ring_create(gb200_engine* e, int capacity_ms, gb200_ring** out) {
    if (!e) return GB200_EINVAL;
    if (!out) GB_FAIL(e, GB200_EINVAL, "null output");
    *out = nullptr;
    if (capacity_ms < 1) GB_FAIL(e, GB200_EINVAL, "ring capacity must be at least one millisecond");
    GB_CUDA(e, cudaSetDevice(e->device));
    gb200_ring* r = new gb200_ring;
    r->e = e;
    r->capacity = capacity_ms;
    cudaError_t ce = r->buf.ensure(static_cast<size_t>(2) * capacity_ms * e->N);
    if (ce != cudaSuccess) {
        delete r;
        cudaGetLastError();
        GB_FAIL(e, GB200_ECUDA, "ring allocation failed: %s", cudaGetErrorString(ce));
    }
    *out = r;
    return GB200_OK;
}

int gb200_ring_destroy(gb200_ring* r) {
    if (!r) return GB200_OK;
    gb200_engine* e = r->e;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    if (e->iq >= r->buf.p && e->iq < r->buf.p + r->buf.cap) {  // the engine was reading the ring: unbind
        e->iq = nullptr;
        e->iq_samples = 0;
    }
    delete r;
    return GB200_OK;
}

int gb200_ring_append(gb200_ring* r, const float* iq_host, int n_ms) {
    if (!r) return GB200_EINVAL;
    gb200_engine* e = r->e;
    if (!iq_host || n_ms < 1) GB_FAIL(e, GB200_EINVAL, "need at least one whole millisecond of samples");
    if (n_ms > r->capacity) GB_FAIL(e, GB200_EINVAL, "%d ms do not fit a ring of %d ms", n_ms, r->capacity);
    GB_CUDA(e, cudaSetDevice(e->device));
    const size_t N = static_cast<size_t>(e->N);
    const float2* src = nullptr;
    GB_TRY(pinned_source(e, r->h_stage, iq_host, N * n_ms, &src));
    int done = 0;
    while (done < n_ms) {
        const int slot = static_cast<int>((r->appended + done) % r->capacity);
        const int run = std::min(n_ms - done, r->capacity - slot);
        float2* lo = r->buf.p + static_cast<size_t>(slot) * N;
        float2* hi = lo + static_cast<size_t>(r->capacity) * N;
        GB_CUDA(e, cudaMemcpyAsync(lo, src + static_cast<size_t>(done) * N, run * N * sizeof(float2), cudaMemcpyHostToDevice,
                                   e->stream));
        GB_CUDA(e, cudaMemcpyAsync(hi, lo, run * N * sizeof(float2), cudaMemcpyDeviceToDevice, e->stream));
        done += run;
    }
    r->appended += n_ms;
    return GB200_OK;
}

int gb200_ring_bind_newest(gb200_ring* r, int n_ms) {
    if (!r) return GB200_EINVAL;
    gb200_engine* e = r->e;
    if (n_ms < 1 || n_ms > r->capacity || n_ms > r->appended)
        GB_FAIL(e, GB200_EINVAL, "the ring holds %lld of at most %d ms; %d asked for",
                static_cast<long long>(std::min<int64_t>(r->appended, r->capacity)), r->capacity, n_ms);
    const int first = static_cast<int>((r->appended - n_ms) % r->capacity);
    e->iq = r->buf.p + static_cast<size_t>(first) * e->N;
    e->iq_samples = static_cast<int64_t>(n_ms) * e->N;
    return GB200_OK;
}

int gb200_ring_appended(const gb200_ring* r, int64_t* total_ms) {
    if (!r || !total_ms) return GB200_EINVAL;
    *total_ms = r->appended;
    return GB200_OK;
}

int gb200_acquire_cells(gb200_engine* e, int n_cells, const int32_t* prn_idx, const double* dop, const int32_t* probe,
                        int n_ms, int kind, gb200_cell_record* out_host) {
    if (!e) return GB200_EINVAL;
    if (!out_host) GB_FAIL(e, GB200_EINVAL, "null output");
    GB_CUDA(e, cudaSetDevice(e->device));
    if (n_cells < 1) GB_FAIL(e, GB200_EINVAL, "empty cell list");
    GB_CUDA(e, e->d_records.ensure(n_cells));
    GB_TRY(run_cells(e, n_cells, prn_idx, dop, probe, n_ms, kind, e->d_records.p, nullptr));
    return fetch_records(e, n_cells, out_host);
}

int gb200_correlation_profile(gb200_engine* e, int prn, double dop, int n_ms, int kind, float* out_host) {
    if (!e) return GB200_EINVAL;
    if (!out_host) GB_FAIL(e, GB200_EINVAL, "null output");
    GB_CUDA(e, cudaSetDevice(e->device));
    const size_t nf = static_cast<size_t>(e->N) * (kind == GB200_COHERENT ? 2 : 1);
    GB_CUDA(e, ensure_staging(e->d_profile, e->h_profile, nf));
    GB_CUDA(e, e->d_records.ensure(1));
    const int32_t p = prn;
    GB_TRY(run_cells(e, 1, &p, &dop, nullptr, n_ms, kind, e->d_records.p, e->d_profile.p));
    return download(e, out_host, e->h_profile, e->d_profile.p, nf);
}

int gb200_correlation_profile_replica(gb200_engine* e, const float* replica_host, double dop, int n_ms, int kind,
                                      float* out_host) {
    if (!e) return GB200_EINVAL;
    if (!replica_host || !out_host) GB_FAIL(e, GB200_EINVAL, "null buffer");
    GB_TRY(check_common(e, n_ms, kind, false));
    GB_TRY(check_samples(e, n_ms));
    GB_CUDA(e, cudaSetDevice(e->device));
    const size_t nf = static_cast<size_t>(e->N) * (kind == GB200_COHERENT ? 2 : 1);
    GB_CUDA(e, cudaStreamSynchronize(e->stream));  // staging buffers may still be in flight
    GB_CUDA(e, e->d_profile.ensure(nf));
    GB_CUDA(e, e->h_profile.ensure(std::max(nf, static_cast<size_t>(2) * e->N)));
    GB_CUDA(e, e->d_replica.ensure(e->N));
    memcpy(e->h_profile.p, replica_host, sizeof(float2) * e->N);  // the pinned profile buffer doubles as replica staging
    GB_CUDA(e, cudaMemcpyAsync(e->d_replica.p, e->h_profile.p, sizeof(float2) * e->N, cudaMemcpyHostToDevice, e->stream));
    GB_CUDA(e, launch_correlate_generic(e->iq, e->d_replica.p, e->N, n_ms, dop, 1.0 / static_cast<double>(e->fs), kind,
                                        e->d_profile.p, e->stream));
    e->launches++;
    return download(e, out_host, e->h_profile, e->d_profile.p, nf);
}

int gb200_enable_kernel_timing(gb200_engine* e, int on) {
    if (!e) return GB200_EINVAL;
    GB_CUDA(e, cudaSetDevice(e->device));
    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    e->timing = on != 0;
    e->ev_used[0] = e->ev_used[1] = 0;
    return GB200_OK;
}

int gb200_kernel_timing(gb200_engine* e, int which, double* total_ms, int64_t* launches) {
    if (!e || which < 0 || which > 1 || !total_ms || !launches) return GB200_EINVAL;
    GB_CUDA(e, cudaSetDevice(e->device));
    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    double t = 0.0;
    for (size_t i = 0; i < e->ev_used[which]; ++i) {
        float ms = 0.f;
        GB_CUDA(e, cudaEventElapsedTime(&ms, e->ev[which][i].first, e->ev[which][i].second));
        t += ms;
    }
    *total_ms = t;
    *launches = static_cast<int64_t>(e->ev_used[which]);
    return GB200_OK;
}

// ---------------------------------------------------------------------------------------------------------
// on-device acquisition search (acquisition.py:70-152)
// ---------------------------------------------------------------------------------------------------------
static_assert(sizeof(gb200_acquisition_result) == sizeof(RefineResult), "ABI acquisition result must match");

int gb200_detect(gb200_engine* e, int n_sv, const int32_t* prn_idx, int n_ms, gb200_acquisition_result* out_host) {
    if (!e) return GB200_EINVAL;
    if (!out_host) GB_FAIL(e, GB200_EINVAL, "null output");
    GB_CUDA(e, cudaSetDevice(e->device));
    GB_TRY(check_common(e, n_ms, GB200_NON_COHERENT));
    if (n_sv < 1 || !prn_idx) GB_FAIL(e, GB200_EINVAL, "no satellites to search for");
    GB_TRY(check_samples(e, n_ms));
    GB_TRY(check_prns(e, prn_idx, n_sv));

    const int MAXB = kRefineMaxBins;
    const int n_cells = n_sv * MAXB;
    const CorrPlan plan = plan_correlate(e, n_ms, GB200_NON_COHERENT, false, n_cells);
    const int cpg = plan.cpg;
    const int gps = (MAXB + cpg - 1) / cpg;  // groups per satellite
    const size_t unit = unit_floats2(e, n_ms);
    int sv_per_chunk = static_cast<int>(std::max<size_t>(1, e->spec_budget_bytes / (unit * sizeof(float2) * MAXB)));
    sv_per_chunk = std::min(sv_per_chunk, n_sv);

    // ---- static plan: cell c = sv*MAXB + b ----
    // ints: [cell_u n_cells][cell_out n_cells][grp_first][grp_count][grp_prn] (n_sv*gps each)
    //       then the coherent pass: [ccell_u n_sv][ccell_out n_sv][cgrp_first][cgrp_count][cgrp_prn] (n_sv each), [probe n_sv]
    const int ng = n_sv * gps;
    const size_t n_ints = static_cast<size_t>(2) * n_cells + 3 * ng + 6 * n_sv;
    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    GB_CUDA(e, ensure_staging(e->r_ints, e->rh_ints, n_ints));
    int* cell_u = e->rh_ints.p;
    int* cell_out = cell_u + n_cells;
    int* g_first = cell_out + n_cells;
    int* g_count = g_first + ng;
    int* g_prn = g_count + ng;
    int* cc_u = g_prn + ng;
    int* cc_out = cc_u + n_sv;
    int* cg_first = cc_out + n_sv;
    int* cg_count = cg_first + n_sv;
    int* cg_prn = cg_count + n_sv;
    for (int sv = 0; sv < n_sv; ++sv) {
        for (int b = 0; b < MAXB; ++b) {
            cell_u[sv * MAXB + b] = (sv % sv_per_chunk) * MAXB + b;
            cell_out[sv * MAXB + b] = sv * MAXB + b;
        }
        for (int g = 0; g < gps; ++g) {
            g_first[sv * gps + g] = sv * MAXB + g * cpg;
            g_count[sv * gps + g] = std::min(cpg, MAXB - g * cpg);
            g_prn[sv * gps + g] = prn_idx[sv];
        }
        cc_u[sv] = sv;
        cc_out[sv] = sv;
        cg_first[sv] = sv;
        cg_count[sv] = 1;
        cg_prn[sv] = prn_idx[sv];
    }
    int* di = e->r_ints.p;
    GB_CUDA(e, cudaMemcpyAsync(di, cell_u, sizeof(int) * (n_ints - n_sv), cudaMemcpyHostToDevice, e->stream));
    int* d_probe = di + (n_ints - n_sv);

    GB_CUDA(e, e->r_state.ensure(n_sv));
    GB_CUDA(e, e->r_doppler.ensure(static_cast<size_t>(n_cells) + n_sv));
    GB_CUDA(e, e->r_records.ensure(static_cast<size_t>(n_cells) + n_sv));
    GB_CUDA(e, ensure_staging(e->r_results, e->rh_results, n_sv));
    GB_CUDA(e, e->spec.ensure(unit * std::max(sv_per_chunk * MAXB, n_sv)));
    double* d_coh_doppler = e->r_doppler.p + n_cells;
    CellRecord* d_coh_records = e->r_records.p + n_cells;

    // Every (satellite, bin) cell of a refinement pass has its own Doppler, so nothing is shared between PRNs: the
    // fused block-per-cell kernel does the same arithmetic without the spectra round trip through HBM.
    const bool use_fused = fused_supports(e->s) && e->detect_fused;
    if (use_fused) {
        GB_CUDA(e, ensure_fused_configured(e));
        // [n_cells] replica row of every (satellite, bin) slot, then [n_sv] one per satellite for the coherent pass
        GB_CUDA(e, ensure_staging(e->r_cell_prn, e->rh_cell_prn, static_cast<size_t>(n_cells) + n_sv));
        for (int c = 0; c < n_cells; ++c) e->rh_cell_prn.p[c] = prn_idx[c / MAXB];
        for (int sv = 0; sv < n_sv; ++sv) e->rh_cell_prn.p[n_cells + sv] = prn_idx[sv];
        GB_CUDA(e, cudaMemcpyAsync(e->r_cell_prn.p, e->rh_cell_prn.p, sizeof(int) * (n_cells + n_sv), cudaMemcpyHostToDevice,
                                   e->stream));
    }

    GB_CUDA(e, launch_refine_init(n_sv, e->r_state.p, e->stream));
    e->launches++;
    for (double spread = 7000.0; spread >= 10.0; spread /= 2.0) {  // acquisition.py:78-89
        GB_CUDA(e, launch_refine_plan(n_sv, spread, e->r_state.p, e->r_doppler.p, e->stream));
        e->launches++;
        if (use_fused) {
            // one launch per pass: a CTA per (satellite, bin) slot, no spectra scratch
            GB_TRY(enqueue_fused(e, n_ms, GB200_NON_COHERENT, e->r_doppler.p, e->r_cell_prn.p, nullptr, e->r_records.p, n_cells));
        }
        for (int sv0 = 0; !use_fused && sv0 < n_sv; sv0 += sv_per_chunk) {
            const int nsv = std::min(sv_per_chunk, n_sv - sv0);
            GB_TRY(enqueue_spectra(e, e->iq, 0, e->r_doppler.p + static_cast<size_t>(sv0) * MAXB, n_ms, nsv * MAXB, nsv * MAXB));
            CorrelateArgs ca = correlate_args(e, n_ms, GB200_NON_COHERENT, e->r_records.p);
            ca.n_groups = nsv * gps;
            ca.cell_u = di;
            ca.cell_out = di + n_cells;
            ca.grp_first = di + 2 * n_cells + sv0 * gps;
            ca.grp_count = di + 2 * n_cells + ng + sv0 * gps;
            ca.grp_prn = di + 2 * n_cells + 2 * ng + sv0 * gps;
            ca.cell_gate = e->r_doppler.p;
            GB_TRY(enqueue_correlate(e, plan, ca, std::min(ca.n_groups, e->num_sms)));
        }
        GB_CUDA(e, launch_refine_select(n_sv, e->N, e->r_records.p, e->r_doppler.p, e->r_state.p, e->stream));
        e->launches++;
    }
    // coherent integration at the kept Doppler (acquisition.py:120-136)
    GB_CUDA(e, launch_refine_coherent_plan(n_sv, e->r_state.p, d_coh_doppler, d_probe, e->stream));
    e->launches++;
    if (use_fused) {
        GB_TRY(enqueue_fused(e, n_ms, GB200_COHERENT, d_coh_doppler, e->r_cell_prn.p + n_cells, d_probe, d_coh_records, n_sv));
    } else {
        GB_TRY(enqueue_spectra(e, e->iq, 0, d_coh_doppler, n_ms, n_sv, n_sv));
        const int* cbase = di + 2 * n_cells + 3 * ng;
        CorrelateArgs ca = correlate_args(e, n_ms, GB200_COHERENT, d_coh_records);
        ca.n_groups = n_sv;
        ca.cell_u = cbase;
        ca.cell_out = cbase + n_sv;
        ca.grp_first = cbase + 2 * n_sv;
        ca.grp_count = cbase + 3 * n_sv;
        ca.grp_prn = cbase + 4 * n_sv;
        ca.cell_probe = d_probe;
        const int rsplit = pick_rsplit(e, 8, n_sv);  // the coherent pass always runs on the 8-pair build
        GB_TRY(enqueue_correlate(e, CorrPlan{0, 8, rsplit, 8 / rsplit}, ca, std::min(n_sv, e->num_sms)));
    }
    GB_CUDA(e, launch_refine_finalize(n_sv, e->r_state.p, d_coh_records, e->r_results.p, e->stream));
    e->launches++;
    return download(e, out_host, e->rh_results, e->r_results.p, n_sv);
}

// ---------------------------------------------------------------------------------------------------------
// tracking
// ---------------------------------------------------------------------------------------------------------
// Both tracker constructors: n channel slots whose device states are uploaded from init with every slot seeded
// (gb200_tracker_create, whose PRN rows prn_idx are checked first) or, with init null, zeroed and unseeded (a pool).
static int new_tracker(gb200_engine* e, int n, const int32_t* prn_idx, const TrackState* init, gb200_tracker** out) {
    if (e->s != 2 && e->s != 4) GB_FAIL(e, GB200_EINVAL, "tracking needs 2046 or 4092 samples per ms (reference tracker.py:301 hard-wires 2046)");
    if (init) {
        if (e->n_prn == 0) GB_FAIL(e, GB200_ESTATE, "no PRN replicas loaded (gb200_set_replicas)");
        GB_TRY(check_prns(e, prn_idx, n));
    }
    GB_CUDA(e, cudaSetDevice(e->device));
    GB_CUDA(e, configure_track_kernel());
    gb200_tracker* t = new gb200_tracker;
    t->e = e;
    t->n_channels = n;
    t->seeded.assign(n, init ? 1 : 0);
    t->undo_ok.assign(n, 0);
    const size_t bytes = sizeof(TrackState) * n;
    cudaError_t ce = t->states.ensure(n);
    if (ce == cudaSuccess)
        ce = init ? cudaMemcpy(t->states.p, init, bytes, cudaMemcpyHostToDevice) : cudaMemset(t->states.p, 0, bytes);
    if (ce != cudaSuccess) {
        delete t;
        cudaGetLastError();
        GB_FAIL(e, GB200_ECUDA, "tracker state allocation failed: %s", cudaGetErrorString(ce));
    }
    *out = t;
    return GB200_OK;
}

int gb200_tracker_create(gb200_engine* e, int n_channels, const int32_t* prn_idx, const double* doppler_hz,
                         const double* carrier_phase, const int32_t* code_phase, gb200_tracker** out) {
    if (!e) return GB200_EINVAL;
    if (!out) GB_FAIL(e, GB200_EINVAL, "null output");
    *out = nullptr;
    if (n_channels < 1 || !prn_idx || !doppler_hz || !carrier_phase || !code_phase) GB_FAIL(e, GB200_EINVAL, "no channels");
    std::vector<TrackState> init(n_channels);
    for (int c = 0; c < n_channels; ++c) {
        memset(&init[c], 0, sizeof(TrackState));
        track_state_init(init[c], prn_idx[c], doppler_hz[c], carrier_phase[c], code_phase[c]);
    }
    return new_tracker(e, n_channels, prn_idx, init.data(), out);
}

int gb200_tracker_destroy(gb200_tracker* t) {
    if (!t) return GB200_OK;
    cudaSetDevice(t->e->device);
    cudaStreamSynchronize(t->e->stream);
    delete t;
    return GB200_OK;
}

// One launch of k_track_channels.  sel (host, may be null = every channel in order): the n_sel channels to advance; CTA i
// writes records out_dev[i * n_ms ...].  keep_undo: the kernel also stores every launched channel's previous state.
static int tracker_launch(gb200_tracker* t, int n_sel, const int32_t* sel, int n_ms, const double* start_times,
                          TrackMsRecord* out_dev, float* prof_dev, bool keep_undo) {
    gb200_engine* e = t->e;
    if (n_ms < 1 || !start_times) GB_FAIL(e, GB200_EINVAL, "need at least one whole millisecond of samples");
    if (!e->iq) GB_FAIL(e, GB200_ESTATE, "no IQ loaded (gb200_upload_iq / gb200_bind_iq_device)");
    GB_TRY(check_samples(e, n_ms));
    if (reinterpret_cast<uintptr_t>(e->iq) % 16 != 0) GB_FAIL(e, GB200_EINVAL, "IQ buffer must be 16-byte aligned for tracking");
    if (sel) {
        for (int i = 0; i < n_sel; ++i) {
            GB_TRY(check_channel(t, sel[i]));
            if (!t->seeded[sel[i]]) GB_FAIL(e, GB200_ESTATE, "channel %d was never seeded (gb200_tracker_reset_channel)", sel[i]);
            for (int j = 0; j < i; ++j)
                if (sel[j] == sel[i]) GB_FAIL(e, GB200_EINVAL, "channel %d listed twice", sel[i]);
        }
    } else {
        for (int c = 0; c < t->n_channels; ++c)
            if (!t->seeded[c]) GB_FAIL(e, GB200_ESTATE, "channel %d was never seeded (gb200_tracker_reset_channel)", c);
    }
    TrackArgs a{};
    if (n_ms == 1) {
        a.start_times = nullptr;  // a single millisecond's start time travels in the kernel arguments
        a.t0_single = start_times[0];
    } else {
        GB_CUDA(e, cudaStreamSynchronize(e->stream));  // h_times may still be in flight
        GB_TRY(stage_upload(e, t->d_times, t->h_times, start_times, n_ms));
        a.start_times = t->d_times.p;
    }
    if (sel) {
        const bool cached = static_cast<int>(t->sel_cache.size()) == n_sel && memcmp(t->sel_cache.data(), sel, sizeof(int) * n_sel) == 0;
        if (!cached) {  // the subset rarely changes between calls: upload it only when it did
            GB_CUDA(e, cudaStreamSynchronize(e->stream));
            GB_TRY(stage_upload(e, t->d_sel, t->h_sel, sel, n_sel));
            t->sel_cache.assign(sel, sel + n_sel);
        }
        a.channel_idx = t->d_sel.p;
    }
    if (keep_undo) {
        GB_CUDA(e, t->shadow.ensure(t->n_channels));
        a.shadow = t->shadow.p;
    }
    a.iq = e->iq;
    a.states = t->states.p;
    a.out = out_dev;
    a.profiles = prof_dev;
    a.crep = e->crep.p;
    a.tw1 = e->tw1.p;
    a.tw2 = e->tw2.p;
    a.fs = static_cast<double>(e->fs);
    a.inv_fs = 1.0 / static_cast<double>(e->fs);
    a.N = e->N;
    a.s = e->s;
    a.n_ms = n_ms;
    a.n_channels = sel ? n_sel : t->n_channels;
    GB_CUDA(e, launch_track_channels(a, e->stream));
    e->launches++;
    for (int i = 0; i < a.n_channels; ++i) t->undo_ok[sel ? sel[i] : i] = keep_undo ? 1 : 0;
    return GB200_OK;
}

int gb200_tracker_process_device(gb200_tracker* t, int n_ms, const double* start_times, void* out_device) {
    if (!t) return GB200_EINVAL;
    gb200_engine* e = t->e;
    if (!out_device) GB_FAIL(e, GB200_EINVAL, "null output");
    GB_CUDA(e, cudaSetDevice(e->device));
    return tracker_launch(t, t->n_channels, nullptr, n_ms, start_times, static_cast<TrackMsRecord*>(out_device), nullptr, false);
}

static int tracker_process_host(gb200_tracker* t, int n_sel, const int32_t* sel, int n_ms, const double* start_times,
                                bool keep_undo, gb200_track_record* out_host, float* profiles_host) {
    gb200_engine* e = t->e;
    if (!out_host) GB_FAIL(e, GB200_EINVAL, "null output");
    GB_CUDA(e, cudaSetDevice(e->device));
    if (n_ms < 1) GB_FAIL(e, GB200_EINVAL, "need at least one whole millisecond of samples");
    if (n_sel < 1) GB_FAIL(e, GB200_EINVAL, "no channels");
    const size_t n = static_cast<size_t>(n_sel) * n_ms;
    GB_CUDA(e, ensure_staging(t->d_out, t->h_out, n));
    const size_t np = profiles_host ? n * e->N : 0;
    if (np) GB_CUDA(e, ensure_staging(t->d_prof, t->h_prof, np));
    t->last_n_ms = 0;
    GB_TRY(tracker_launch(t, n_sel, sel, n_ms, start_times, t->d_out.p, np ? t->d_prof.p : nullptr, keep_undo));
    if (!sel) t->last_n_ms = n_ms;  // gb200_tracker_integrate_bits reads [channel][n_ms] of the whole bank
    GB_CUDA(e, cudaMemcpyAsync(t->h_out.p, t->d_out.p, n * sizeof(TrackMsRecord), cudaMemcpyDeviceToHost, e->stream));
    if (np) GB_CUDA(e, cudaMemcpyAsync(t->h_prof.p, t->d_prof.p, np * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    memcpy(out_host, t->h_out.p, n * sizeof(TrackMsRecord));
    if (np) memcpy(profiles_host, t->h_prof.p, np * sizeof(float));
    return GB200_OK;
}

int gb200_tracker_process(gb200_tracker* t, int n_ms, const double* start_times, gb200_track_record* out_host,
                          float* profiles_host) {
    if (!t) return GB200_EINVAL;
    return tracker_process_host(t, t->n_channels, nullptr, n_ms, start_times, false, out_host, profiles_host);
}

int gb200_tracker_process_channels(gb200_tracker* t, int n_sel, const int32_t* channels, int n_ms, const double* start_times,
                                   int keep_undo, gb200_track_record* out_host, float* profiles_host) {
    if (!t) return GB200_EINVAL;
    if (!channels) GB_FAIL(t->e, GB200_EINVAL, "null channel list");
    return tracker_process_host(t, n_sel, channels, n_ms, start_times, keep_undo != 0, out_host, profiles_host);
}

int gb200_tracker_undo_channel(gb200_tracker* t, int channel) {
    if (!t) return GB200_EINVAL;
    gb200_engine* e = t->e;
    GB_TRY(check_channel(t, channel));
    if (!t->undo_ok[channel]) GB_FAIL(e, GB200_ESTATE, "channel %d has no kept state to go back to", channel);
    GB_CUDA(e, cudaSetDevice(e->device));
    GB_CUDA(e, cudaMemcpyAsync(t->states.p + channel, t->shadow.p + channel, sizeof(TrackState), cudaMemcpyDeviceToDevice, e->stream));
    t->undo_ok[channel] = 0;
    return GB200_OK;
}

int gb200_tracker_create_pool(gb200_engine* e, int capacity, gb200_tracker** out) {
    if (!e) return GB200_EINVAL;
    if (!out) GB_FAIL(e, GB200_EINVAL, "null output");
    *out = nullptr;
    if (capacity < 1) GB_FAIL(e, GB200_EINVAL, "no channels");
    return new_tracker(e, capacity, nullptr, nullptr, out);
}

int gb200_tracker_reset_channel(gb200_tracker* t, int channel, int32_t prn_idx, double doppler_hz, double carrier_phase,
                                int32_t code_phase) {
    if (!t) return GB200_EINVAL;
    gb200_engine* e = t->e;
    GB_TRY(check_channel(t, channel));
    GB_TRY(check_prns(e, &prn_idx, 1));
    GB_CUDA(e, cudaSetDevice(e->device));
    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    std::vector<TrackState> init(1);
    memset(init.data(), 0, sizeof(TrackState));
    track_state_init(init[0], prn_idx, doppler_hz, carrier_phase, code_phase);
    GB_CUDA(e, cudaMemcpy(t->states.p + channel, init.data(), sizeof(TrackState), cudaMemcpyHostToDevice));
    t->seeded[channel] = 1;
    t->undo_ok[channel] = 0;
    return GB200_OK;
}

int gb200_tracker_get_state(gb200_tracker* t, int channel, double* doppler_hz, double* carrier_phase, double* phase_acc,
                            int32_t* code_phase, int32_t* lost) {
    if (!t) return GB200_EINVAL;
    gb200_engine* e = t->e;
    GB_TRY(check_channel(t, channel));
    GB_CUDA(e, cudaSetDevice(e->device));
    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    TrackState st;
    GB_CUDA(e, cudaMemcpy(&st, t->states.p + channel, offsetof(TrackState, err_ring), cudaMemcpyDeviceToHost));
    if (doppler_hz) *doppler_hz = st.doppler;
    if (carrier_phase) *carrier_phase = st.carrier_phase;
    if (phase_acc) *phase_acc = st.phase_acc;
    if (code_phase) *code_phase = st.code_phase;
    if (lost) *lost = st.lost;
    return GB200_OK;
}

int gb200_tracker_set_state(gb200_tracker* t, int channel, double doppler_hz, double carrier_phase, double phase_acc,
                            int32_t code_phase) {
    if (!t) return GB200_EINVAL;
    gb200_engine* e = t->e;
    GB_TRY(check_channel(t, channel));
    GB_CUDA(e, cudaSetDevice(e->device));
    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    TrackState st;
    const size_t head = offsetof(TrackState, err_ring);
    GB_CUDA(e, cudaMemcpy(&st, t->states.p + channel, head, cudaMemcpyDeviceToHost));
    st.doppler = doppler_hz;
    st.carrier_phase = carrier_phase;
    st.phase_acc = phase_acc;
    st.code_phase = code_phase;
    st.lost = 0;  // the reference tracker object keeps processing after it raised LostSatelliteLockError
    GB_CUDA(e, cudaMemcpy(t->states.p + channel, &st, head, cudaMemcpyHostToDevice));
    t->undo_ok[channel] = 0;
    return GB200_OK;
}

int gb200_tracker_integrate_bits(gb200_tracker* t, int n_ms, const double* start_times, const double* end_times,
                                 const void* records_device, gb200_bit_event* events_host, int32_t max_events,
                                 int32_t* counts_host) {
    if (!t) return GB200_EINVAL;
    gb200_engine* e = t->e;
    if (n_ms < 1 || !start_times || !end_times) GB_FAIL(e, GB200_EINVAL, "need at least one millisecond and its timestamps");
    if (!events_host || !counts_host || max_events < 1) GB_FAIL(e, GB200_EINVAL, "null / empty event buffer");
    if (!records_device && t->last_n_ms != n_ms)
        GB_FAIL(e, GB200_ESTATE, "no records of %d ms on the device (last gb200_tracker_process call held %d)", n_ms, t->last_n_ms);
    GB_CUDA(e, cudaSetDevice(e->device));
    GB_CUDA(e, cudaStreamSynchronize(e->stream));  // pinned staging may still be in flight
    const int nc = t->n_channels;
    if (!t->bit_states.p) {
        std::vector<BitState> init(nc);
        for (int c = 0; c < nc; ++c) {
            memset(&init[c], 0, sizeof(BitState));
            bit_state_init(init[c]);
        }
        GB_CUDA(e, t->bit_states.ensure(nc));
        GB_CUDA(e, cudaMemcpy(t->bit_states.p, init.data(), sizeof(BitState) * nc, cudaMemcpyHostToDevice));
    }
    const size_t ne = static_cast<size_t>(nc) * max_events;
    GB_CUDA(e, ensure_staging(t->d_events, t->h_events, ne));
    GB_CUDA(e, ensure_staging(t->d_counts, t->h_counts, nc));
    GB_CUDA(e, ensure_staging(t->d_bit_times, t->h_bit_times, 2 * static_cast<size_t>(n_ms)));
    memcpy(t->h_bit_times.p, start_times, sizeof(double) * n_ms);
    memcpy(t->h_bit_times.p + n_ms, end_times, sizeof(double) * n_ms);
    GB_CUDA(e, cudaMemcpyAsync(t->d_bit_times.p, t->h_bit_times.p, 2 * sizeof(double) * n_ms, cudaMemcpyHostToDevice, e->stream));
    BitArgs a{};
    a.records = records_device ? static_cast<const TrackMsRecord*>(records_device) : t->d_out.p;
    a.start_times = t->d_bit_times.p;
    a.end_times = t->d_bit_times.p + n_ms;
    a.states = t->bit_states.p;
    a.events = t->d_events.p;
    a.counts = t->d_counts.p;
    a.n_ms = n_ms;
    a.n_channels = nc;
    a.max_events = max_events;
    GB_CUDA(e, launch_integrate_bits(a, e->stream));
    e->launches++;
    GB_CUDA(e, cudaMemcpyAsync(t->h_events.p, t->d_events.p, ne * sizeof(BitEvent), cudaMemcpyDeviceToHost, e->stream));
    GB_CUDA(e, cudaMemcpyAsync(t->h_counts.p, t->d_counts.p, nc * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    GB_CUDA(e, cudaStreamSynchronize(e->stream));
    memcpy(events_host, t->h_events.p, ne * sizeof(BitEvent));
    memcpy(counts_host, t->h_counts.p, nc * sizeof(int));
    return GB200_OK;
}

int gb200_tracker_bit_state(gb200_tracker* t, int channel, int64_t out[8]) {
    if (!t) return GB200_EINVAL;
    gb200_engine* e = t->e;
    if (channel < 0 || channel >= t->n_channels || !out) GB_FAIL(e, GB200_EINVAL, "channel %d out of range", channel);
    BitState st;
    memset(&st, 0, sizeof(st));
    bit_state_init(st);
    if (t->bit_states.p) {
        GB_CUDA(e, cudaSetDevice(e->device));
        GB_CUDA(e, cudaStreamSynchronize(e->stream));
        GB_CUDA(e, cudaMemcpy(&st, t->bit_states.p + channel, sizeof(BitHead), cudaMemcpyDeviceToHost));
    }
    out[0] = st.h.emitted;
    out[1] = st.h.failed;
    out[2] = st.h.processed;
    out[3] = st.h.slide;
    out[4] = st.h.determined;
    out[5] = st.h.prev_decision;
    out[6] = st.h.cursor;
    out[7] = st.h.stopped;
    return GB200_OK;
}

// ---------------------------------------------------------------------------------------------------------
// pipelined grid batches
// ---------------------------------------------------------------------------------------------------------
int gb200_grid_stream_destroy(gb200_grid_stream* g) {
    if (!g) return GB200_OK;
    cudaSetDevice(g->e->device);
    cudaStreamSynchronize(g->e->stream);
    if (g->s_in) cudaStreamSynchronize(g->s_in);
    if (g->s_out) cudaStreamSynchronize(g->s_out);
    delete g;
    return GB200_OK;
}

int gb200_grid_stream_create(gb200_engine* e, int n_blocks, int M, const int32_t* prn_idx, int P, const double* dop, int D,
                             int kind, int depth, gb200_grid_stream** out) {
    if (!e) return GB200_EINVAL;
    if (!out) GB_FAIL(e, GB200_EINVAL, "null output");
    *out = nullptr;
    if (n_blocks < 1 || P < 1 || D < 1 || !prn_idx || !dop) GB_FAIL(e, GB200_EINVAL, "empty grid");
    if (depth < 1 || depth > 8) GB_FAIL(e, GB200_EINVAL, "depth must be 1..8");
    GB_TRY(check_common(e, M, kind));
    GB_TRY(check_prns(e, prn_idx, P));
    GB_CUDA(e, cudaSetDevice(e->device));
    gb200_grid_stream* g = new gb200_grid_stream;
    g->e = e;
    g->n_blocks = n_blocks;
    g->M = M;
    g->P = P;
    g->D = D;
    g->kind = kind;
    g->depth = depth;
    g->prn.assign(prn_idx, prn_idx + P);
    g->dop.assign(dop, dop + D);
    g->slots = std::vector<gb200_grid_stream::Slot>(depth);
    const size_t n_iq = static_cast<size_t>(n_blocks) * M * e->N, n_rec = static_cast<size_t>(n_blocks) * P * D;
    cudaError_t ce = cudaStreamCreateWithFlags(&g->s_in, cudaStreamNonBlocking);
    if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&g->s_out, cudaStreamNonBlocking);
    for (auto& sl : g->slots) {
        if (ce == cudaSuccess) ce = sl.iq.ensure(n_iq);
        if (ce == cudaSuccess) ce = sl.rec.ensure(n_rec);
        for (cudaEvent_t* ev : {&sl.h2d, &sl.done, &sl.d2h})
            if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(ev, cudaEventDisableTiming);
    }
    if (ce != cudaSuccess) {
        gb200_grid_stream_destroy(g);
        cudaGetLastError();
        GB_FAIL(e, GB200_ECUDA, "grid stream allocation failed: %s", cudaGetErrorString(ce));
    }
    *out = g;
    return GB200_OK;
}

int gb200_grid_stream_submit(gb200_grid_stream* g, const float* iq_host, gb200_cell_record* out_host) {
    if (!g) return GB200_EINVAL;
    gb200_engine* e = g->e;
    if (!iq_host || !out_host) GB_FAIL(e, GB200_EINVAL, "null buffer");
    if (g->head - g->tail >= g->depth) GB_FAIL(e, GB200_ESTATE, "%d batches in flight: collect one first", g->depth);
    GB_CUDA(e, cudaSetDevice(e->device));
    auto& sl = g->slots[g->head % g->depth];
    const size_t n_iq = static_cast<size_t>(g->n_blocks) * g->M * e->N, n_rec = static_cast<size_t>(g->n_blocks) * g->P * g->D;
    // the slot's previous batch was collected, so its device buffers and staging are free
    const void* src = iq_host;
    if (!pinned_alias(iq_host)) {
        GB_CUDA(e, sl.h_iq.ensure(n_iq));
        memcpy(sl.h_iq.p, iq_host, n_iq * sizeof(float2));
        src = sl.h_iq.p;
    }
    sl.out = out_host;
    sl.staged_out = !pinned_alias(out_host);
    if (sl.staged_out) GB_CUDA(e, sl.h_rec.ensure(n_rec));
    GB_CUDA(e, cudaMemcpyAsync(sl.iq.p, src, n_iq * sizeof(float2), cudaMemcpyHostToDevice, g->s_in));
    GB_CUDA(e, cudaEventRecord(sl.h2d, g->s_in));
    GB_CUDA(e, cudaStreamWaitEvent(e->stream, sl.h2d, 0));
    e->iq = sl.iq.p;
    e->iq_samples = static_cast<int64_t>(n_iq);
    GB_TRY(run_grid(e, g->n_blocks, g->M, g->prn.data(), g->P, g->dop.data(), g->D, g->kind, sl.rec.p));
    GB_CUDA(e, cudaEventRecord(sl.done, e->stream));
    GB_CUDA(e, cudaStreamWaitEvent(g->s_out, sl.done, 0));
    GB_CUDA(e, cudaMemcpyAsync(sl.staged_out ? reinterpret_cast<gb200_cell_record*>(sl.h_rec.p) : out_host, sl.rec.p,
                               n_rec * sizeof(CellRecord), cudaMemcpyDeviceToHost, g->s_out));
    GB_CUDA(e, cudaEventRecord(sl.d2h, g->s_out));
    g->head++;
    return GB200_OK;
}

int gb200_grid_stream_collect(gb200_grid_stream* g) {
    if (!g) return GB200_EINVAL;
    gb200_engine* e = g->e;
    if (g->head == g->tail) GB_FAIL(e, GB200_ESTATE, "no batch in flight");
    GB_CUDA(e, cudaSetDevice(e->device));
    auto& sl = g->slots[g->tail % g->depth];
    GB_CUDA(e, cudaEventSynchronize(sl.d2h));
    if (sl.staged_out)
        memcpy(sl.out, sl.h_rec.p, static_cast<size_t>(g->n_blocks) * g->P * g->D * sizeof(CellRecord));
    g->tail++;
    return GB200_OK;
}

int gb200_set_fused(gb200_engine* e, int mode) {
    if (!e) return GB200_EINVAL;
    if (mode < -1 || mode > 1) GB_FAIL(e, GB200_EINVAL, "mode must be -1 (automatic), 0 or 1");
    if (mode == 1 && !fused_supports(e->s)) GB_FAIL(e, GB200_EINVAL, "the fused kernel needs 2046 or 4092 samples per ms");
    e->fused = mode;
    return GB200_OK;
}

int gb200_launch_count(const gb200_engine* e, int64_t* out) {
    if (!e || !out) return GB200_EINVAL;
    *out = e->launches;
    return GB200_OK;
}

}  // extern "C"
