// C-ABI entry points and host-side orchestration (see include/acoss_b200.h).
//
// Pipeline per acoss_score_pairs* call (all asynchronous on the context stream):
//   K1 oti_kernel over all pairs -> pairs are processed in fixed-pitch chunks ("slots"):
//   K2 (fast sweep path, exact fallback) -> bit-packed CRP per slot -> K3 DP -> scores[k].
// Nothing here computes on the CPU: without a usable device every call fails with ACOSS_E_CUDA.
#include <nvtx3/nvToolsExt.h>   // header-only NVTX 3: ranges around stages / K2 kernels (visible to nsys / ncu --nvtx)
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <vector>

#include "common.cuh"
#include "k2_fast.cuh"

static thread_local char g_err[512] = "";

void acoss_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

struct Buf {
    void *p = nullptr;
    size_t cap = 0;
};

struct acoss_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    // resident track set
    float *d_frames = nullptr;
    bool own_frames = false;
    int64_t *d_offsets = nullptr;
    float *d_gchroma = nullptr;
    int32_t n_tracks = 0;
    int32_t max_frames = 0, min_frames = 0;
    int64_t total_frames = 0;
    int32_t fx_exp = -1000, nonneg = 0, q_exp = -1;
    int64_t ws_limit = (int64_t)24 << 30;
    // grow-only scratch
    Buf pairs, scores, oti, status, crp, rows, cols, thr_q, thr_r, rrot, aa, bb, D, halo, misc, fast, fbmap, dbg, glive;
    uint32_t *h_flag = nullptr;   // pinned
    uint32_t *h_dbg = nullptr;    // pinned, 32 diagnostic counters
    int64_t stats[8] = {0};
    // deferred exact fallback of the last asynchronous call (pairs the fast CRP path flagged): the first
    // FB_ROUNDS * fb_slots of them are re-scored inside the call's own stream work; if more were flagged, acoss_sync()
    // scores the rest
    struct PendingFb {
        int active = 0;
        const int32_t *pairs_dev = nullptr;
        float *scores_dev = nullptr, *scores2_dev = nullptr;
        acoss_params p;
        SlotGeom g;
        int64_t ldd = 0, halo_pitch = 0, K = 0;
        int fb_slots = 0, done = 0;
    } fb;
    Buf fbtmp;
    int pending_status_check = 0;
    int stats_reason_pending = 0;
    int64_t pending_pairs = 0;
    // optional per-stage timing (CUDA events on the context stream)
    int profiling = 0;
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
    struct Span { int stage; cudaEvent_t a, b; };
    std::vector<Span> spans;
    double stage_ms[32] = {0};   // [0..3] Serra09 pipeline, [4..8] EarlyFusion pipeline, [9..12] SNF, [16 + K2K_*] K2 kernels
    // EarlyFusion block features (acoss_ef_set_tracks): float64, row pitch ef_dp[k], kinds mfccs / ssms / chromas
    Buf ef_feat[3], ef_sq[2], ef_cmed, ef_off;
    std::vector<int64_t> ef_hoff;
    int32_t ef_d[3] = {0, 0, 0}, ef_dp[3] = {0, 0, 0};
    int32_t ef_tracks = 0;
    Buf ef_csm, ef_stat, ef_shapes, ef_nn, ef_csmoff, ef_oti, ef_pairs, ef_scores, ef_bits, ef_bitoff, ef_stage;
    // SiMPle pair scoring (acoss_simple_*): per-slot workspace, pair list / scores / OTI of the host entry points
    Buf sp_ws, sp_pairs, sp_scores, sp_oti;
    int64_t ef_stats[4] = {0, 0, 0, 0};
};

static cudaEvent_t get_event(acoss_ctx *c) {
    if (c->ev_used == c->ev_pool.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        c->ev_pool.push_back(e);
    }
    return c->ev_pool[c->ev_used++];
}
static const char *const STAGE_NAMES[13] = {"acoss/K1 oti", "acoss/K2 crp", "acoss/K3 dp", "acoss/K2 emit", "acoss/EF csm", "acoss/EF knn",
                                            "acoss/EF sw", "acoss/EF radii", "acoss/EF fuse", "acoss/SNF h2d", "acoss/SNF affinity",
                                            "acoss/SNF diffusion", "acoss/SNF average"};
struct StageTimer {     // NVTX range around a pipeline stage (host side: the enqueue); CUDA events [a, b] when profiling is on
    acoss_ctx *c; int stage; cudaEvent_t a = nullptr; bool open = true;
    StageTimer(acoss_ctx *c_, int s) : c(c_), stage(s) {
        nvtxRangePushA(STAGE_NAMES[s < 13 ? s : 1]);
        if (c->profiling) { a = get_event(c); cudaEventRecord(a, c->stream); }
    }
    void stop() {
        if (c->profiling && a) { cudaEvent_t b = get_event(c); cudaEventRecord(b, c->stream); c->spans.push_back({stage, a, b}); a = nullptr; }
        if (open) { nvtxRangePop(); open = false; }
    }
    ~StageTimer() { if (open) nvtxRangePop(); }
};
struct CtxKernelTimer : KernelTimer {     // K2 per-kernel spans -> stage_ms[16 + id]; the emit kernel also feeds stage 3
    acoss_ctx *c; cudaEvent_t a[K2K_COUNT];
    explicit CtxKernelTimer(acoss_ctx *c_) : c(c_) {}
    void begin(int id) override { a[id] = get_event(c); cudaEventRecord(a[id], c->stream); }
    void end(int id) override {
        cudaEvent_t b = get_event(c);
        cudaEventRecord(b, c->stream);
        c->spans.push_back({16 + id, a[id], b});
        if (id == K2K_EMIT) c->spans.push_back({3, a[id], b});
    }
};
static void fold_spans(acoss_ctx *c) {
    for (auto &s : c->spans) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) c->stage_ms[s.stage] += ms;
    }
    c->spans.clear();
    c->ev_used = 0;
}

static int ensure(Buf &b, size_t bytes) {
    if (bytes <= b.cap) return ACOSS_OK;
    if (b.p) CUDA_TRY(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    size_t want = bytes + (bytes >> 3) + 256;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        acoss_set_error("cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
        return ACOSS_E_NOMEM;
    }
    b.cap = want;
    return ACOSS_OK;
}
#define TRY(x)                         \
    do {                               \
        int _rc = (x);                 \
        if (_rc != ACOSS_OK) return _rc; \
    } while (0)

extern "C" {

static int finish_tracks(acoss_ctx *c, const int64_t *offsets, int32_t n_tracks, int64_t mx, int64_t mn);

void acoss_default_params(acoss_params *p) {
    if (!p) return;
    p->m = 9; p->tau = 1; p->kappa = 0.095f; p->oti = 1; p->noti = 12;
    p->gamma_o = 0.5f; p->gamma_e = 0.5f; p->align = ACOSS_ALIGN_QMAX; p->integer_guard = 0;
    p->crp_path = ACOSS_CRP_AUTO;
    p->f2_strict = 0; p->f3_float_acc = 0; p->f4_keep_last = 0; p->f5_asymmetric = 0;
}

// stacked frames of a track with n frames: n - win_incr (F4: essentia drops one window)
static int win_incr(const acoss_params *p) { return p->f4_keep_last ? (p->m - 1) * p->tau : p->m * p->tau; }

const char *acoss_last_error(void) { return g_err; }
const char *acoss_version(void) { return "acoss_b200 0.1 (sm_100a)"; }
int acoss_compiled_sm(void) { return 100; }

int acoss_create(acoss_ctx **out, int device) {
    if (!out) { acoss_set_error("ctx is NULL"); return ACOSS_E_INVALID; }
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        acoss_set_error("no CUDA device available (%s); acoss_b200 has no CPU fallback",
                        e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return ACOSS_E_CUDA;
    }
    if (device < 0 || device >= ndev) { acoss_set_error("device %d out of range (%d devices)", device, ndev); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    // sm_100a code is architecture-specific: it does not run on any other compute capability, newer ones included
    if (prop.major != 10 || prop.minor != 0) {
        acoss_set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
        return ACOSS_E_CUDA;
    }
    acoss_ctx *c = new acoss_ctx();
    c->device = device;
    CUDA_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaMallocHost((void **)&c->h_flag, 64));
    CUDA_TRY(cudaMallocHost((void **)&c->h_dbg, 128));
    memset(c->h_dbg, 0, 128);
    *out = c;
    return ACOSS_OK;
}

static void free_buf(Buf &b) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; }

int acoss_destroy(acoss_ctx *c) {
    if (!c) return ACOSS_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    Buf *bufs[] = {&c->pairs, &c->scores, &c->oti, &c->status, &c->crp, &c->rows, &c->cols, &c->thr_q, &c->thr_r,
                   &c->rrot, &c->aa, &c->bb, &c->D, &c->halo, &c->misc, &c->fast, &c->fbmap, &c->dbg, &c->glive, &c->fbtmp,
                   &c->ef_feat[0], &c->ef_feat[1], &c->ef_feat[2], &c->ef_sq[0], &c->ef_sq[1], &c->ef_cmed, &c->ef_off,
                   &c->ef_csm, &c->ef_stat, &c->ef_shapes, &c->ef_nn, &c->ef_csmoff, &c->ef_oti, &c->ef_pairs,
                   &c->ef_scores, &c->ef_bits, &c->ef_bitoff, &c->ef_stage, &c->sp_ws, &c->sp_pairs, &c->sp_scores,
                   &c->sp_oti};
    for (Buf *b : bufs) free_buf(*b);
    if (c->own_frames && c->d_frames) cudaFree(c->d_frames);
    if (c->d_offsets) cudaFree(c->d_offsets);
    if (c->d_gchroma) cudaFree(c->d_gchroma);
    if (c->h_flag) cudaFreeHost(c->h_flag);
    if (c->h_dbg) cudaFreeHost(c->h_dbg);
    for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
    cudaStreamDestroy(c->stream);
    delete c;
    return ACOSS_OK;
}

int acoss_set_workspace_limit(acoss_ctx *c, int64_t bytes) {
    if (!c || bytes < ((int64_t)64 << 20)) { acoss_set_error("workspace limit must be >= 64 MiB"); return ACOSS_E_INVALID; }
    c->ws_limit = bytes;
    return ACOSS_OK;
}

void *acoss_stream(acoss_ctx *c) { return c ? (void *)c->stream : nullptr; }

int acoss_set_tracks(acoss_ctx *c, const float *frames, const int64_t *offsets, int32_t n_tracks, int on_device) {
    if (!c || !frames || !offsets || n_tracks <= 0) { acoss_set_error("set_tracks: bad arguments"); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    int64_t mx = 0, mn = INT64_MAX;
    for (int t = 0; t < n_tracks; ++t) {
        const int64_t n = offsets[t + 1] - offsets[t];
        if (n < 0 || offsets[0] != 0) { acoss_set_error("set_tracks: offsets must start at 0 and be non-decreasing"); return ACOSS_E_INVALID; }
        mx = std::max(mx, n);
        mn = std::min(mn, n);
    }
    if (mx > (1 << 20)) { acoss_set_error("set_tracks: track longer than 2^20 frames"); return ACOSS_E_INVALID; }
    const int64_t total = offsets[n_tracks];
    if (c->own_frames && c->d_frames) CUDA_TRY(cudaFree(c->d_frames));
    c->d_frames = nullptr;
    if (c->d_offsets) CUDA_TRY(cudaFree(c->d_offsets));
    if (c->d_gchroma) CUDA_TRY(cudaFree(c->d_gchroma));
    c->d_offsets = nullptr; c->d_gchroma = nullptr;
    if (on_device) {
        c->d_frames = const_cast<float *>(frames);
        c->own_frames = false;
    } else {
        // +16 floats of zero padding so vector loads past the last frame stay in bounds
        CUDA_TRY(cudaMalloc((void **)&c->d_frames, (size_t)(total * NBINS + 64) * sizeof(float)));
        c->own_frames = true;
        CUDA_TRY(cudaMemsetAsync(c->d_frames + total * NBINS, 0, 64 * sizeof(float), c->stream));
        CUDA_TRY(cudaMemcpyAsync(c->d_frames, frames, (size_t)total * NBINS * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    }
    return finish_tracks(c, offsets, n_tracks, mx, mn);
}

// common tail of acoss_set_tracks / acoss_set_tracks_raw: c->d_frames holds the frames (device), offsets on the host
static int finish_tracks(acoss_ctx *c, const int64_t *offsets, int32_t n_tracks, int64_t mx, int64_t mn) {
    const int64_t total = offsets[n_tracks];
    CUDA_TRY(cudaMalloc((void **)&c->d_offsets, (size_t)(n_tracks + 1) * sizeof(int64_t)));
    CUDA_TRY(cudaMalloc((void **)&c->d_gchroma, (size_t)n_tracks * NBINS * sizeof(float)));
    CUDA_TRY(cudaMemcpyAsync(c->d_offsets, offsets, (size_t)(n_tracks + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    c->n_tracks = n_tracks;
    c->max_frames = (int32_t)mx;
    c->min_frames = (int32_t)mn;
    c->total_frames = total;
    TRY(launch_global_chroma(c->d_frames, c->d_offsets, n_tracks, c->d_gchroma, c->stream));
    // feature range for the fast path's fixed point
    TRY(ensure(c->misc, 256));
    TRY(launch_frame_stats(c->d_frames, total, (float *)c->misc.p, c->stream));
    float st2[3] = {0.f, 0.f, 0.f};
    CUDA_TRY(cudaMemcpyAsync(st2, c->misc.p, 12, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->nonneg = (st2[1] >= 0.f) ? 1 : 0;
    c->fx_exp = -1000;
    if (st2[0] > 1e-30f && st2[0] < 1e30f) {
        int e = 0;
        frexp(2.0 * (double)st2[0] * 1.001, &e);     // 2*gmax2*1.001 = f * 2^e, f in [0.5, 1)  =>  < 2^e
        c->fx_exp = e;
    }
    if (((uintptr_t)c->d_frames & 15) != 0) c->fx_exp = -1000;   // vector loads need 16 B alignment
    // tensor sweeps: 24-bit quantisation x_q = rint(x * 2^q_exp) < 2^24 of the non-negative features.  The limb products the
    // sweeps keep weigh 2^e0, 2^(e0 - 8), 2^(e0 - 16) fixed-point units; their error against the exact item grows with e0
    // (quantisation 1.4 * 2^(e0/2) units, dropped limb products 0.84 * 2^e0: DESIGN.md 4.2), so e0 <= 6 keeps it inside EPS
    // (HPCP: frames normalised to max 1, largest squared frame norm in [4, 16)  =>  e0 = 5 or 6).
    c->q_exp = -1;
    if (c->fx_exp > -100 && c->nonneg && st2[2] > 0.f) {
        int e = 0;
        frexp((double)st2[2] * 1.000001, &e);        // max feature < 2^e / 1.000001  =>  rint(x * 2^(24 - e)) <= 2^24 - 2
        const int qe = 24 - e, e0 = 56 - 2 * qe - c->fx_exp;
        if (e0 >= 0 && e0 <= 6) c->q_exp = qe;
    }
    return ACOSS_OK;
}

// common tail of acoss_set_tracks_raw / acoss_set_tracks_pooled: uploads the raw frames, runs `reduce` (raw, raw
// offsets, output offsets, output frames: device) into the new resident set and finishes it; off = output offsets
using RawReduce = std::function<int(const float *, const int64_t *, const int64_t *, int64_t, float *)>;
static int reduce_raw_tracks(acoss_ctx *c, const float *raw_frames, const int64_t *raw_offsets, int32_t n_tracks,
                             const std::vector<int64_t> &off, int64_t mx, int64_t mn, int64_t *offsets_out,
                             const RawReduce &reduce) {
    const int64_t total_raw = raw_offsets[n_tracks], total = off[n_tracks];
    if (c->own_frames && c->d_frames) CUDA_TRY(cudaFree(c->d_frames));
    c->d_frames = nullptr;
    if (c->d_offsets) CUDA_TRY(cudaFree(c->d_offsets));
    if (c->d_gchroma) CUDA_TRY(cudaFree(c->d_gchroma));
    c->d_offsets = nullptr; c->d_gchroma = nullptr;
    float *d_raw = nullptr;
    int64_t *d_roff = nullptr, *d_ooff = nullptr;
    auto cleanup = [&]() { if (d_raw) cudaFree(d_raw); if (d_roff) cudaFree(d_roff); if (d_ooff) cudaFree(d_ooff); };
#define CUDA_TRYC(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) { acoss_set_error("%s -> %s", #x, cudaGetErrorString(_e)); cleanup(); return _e == cudaErrorMemoryAllocation ? ACOSS_E_NOMEM : ACOSS_E_CUDA; } } while (0)
    CUDA_TRYC(cudaMalloc((void **)&d_raw, (size_t)std::max<int64_t>(total_raw, 1) * NBINS * sizeof(float)));
    CUDA_TRYC(cudaMalloc((void **)&d_roff, (size_t)(n_tracks + 1) * sizeof(int64_t)));
    CUDA_TRYC(cudaMalloc((void **)&d_ooff, (size_t)(n_tracks + 1) * sizeof(int64_t)));
    CUDA_TRYC(cudaMalloc((void **)&c->d_frames, (size_t)(total * NBINS + 64) * sizeof(float)));
    c->own_frames = true;
    CUDA_TRYC(cudaMemsetAsync(c->d_frames + total * NBINS, 0, 64 * sizeof(float), c->stream));
    CUDA_TRYC(cudaMemcpyAsync(d_raw, raw_frames, (size_t)total_raw * NBINS * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRYC(cudaMemcpyAsync(d_roff, raw_offsets, (size_t)(n_tracks + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRYC(cudaMemcpyAsync(d_ooff, off.data(), (size_t)(n_tracks + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    int rc = reduce(d_raw, d_roff, d_ooff, total, c->d_frames);
    if (rc == ACOSS_OK) { cudaError_t e = cudaStreamSynchronize(c->stream); if (e != cudaSuccess) { acoss_set_error("on-ramp: %s", cudaGetErrorString(e)); rc = ACOSS_E_CUDA; } }
    cleanup();
#undef CUDA_TRYC
    if (rc != ACOSS_OK) return rc;
    if (offsets_out) memcpy(offsets_out, off.data(), (size_t)(n_tracks + 1) * sizeof(int64_t));
    return finish_tracks(c, off.data(), n_tracks, mx, mn);
}

int acoss_set_tracks_raw(acoss_ctx *c, const float *raw_frames, const int64_t *raw_offsets, int32_t n_tracks,
                         int32_t downsample_fac, int64_t *offsets_out) {
    if (!c || !raw_frames || !raw_offsets || n_tracks <= 0) { acoss_set_error("set_tracks_raw: bad arguments"); return ACOSS_E_INVALID; }
    if (downsample_fac < 1 || downsample_fac > onramp_max_fac()) {
        acoss_set_error("set_tracks_raw: downsample factor must be in 1..%d", onramp_max_fac());
        return ACOSS_E_INVALID;
    }
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (raw_offsets[0] != 0) { acoss_set_error("set_tracks_raw: offsets must start at 0"); return ACOSS_E_INVALID; }
    std::vector<int64_t> off(n_tracks + 1, 0);
    int64_t mx = 0, mn = INT64_MAX;
    for (int t = 0; t < n_tracks; ++t) {
        const int64_t n = raw_offsets[t + 1] - raw_offsets[t];
        if (n < 0) { acoss_set_error("set_tracks_raw: offsets must be non-decreasing"); return ACOSS_E_INVALID; }
        const int64_t no = (n + downsample_fac - 1) / downsample_fac;      // ceil(n / fac) blocks, last one short
        off[t + 1] = off[t] + no;
        mx = std::max(mx, no);
        mn = std::min(mn, no);
    }
    if (mx > (1 << 20)) { acoss_set_error("set_tracks_raw: track longer than 2^20 frames"); return ACOSS_E_INVALID; }
    return reduce_raw_tracks(c, raw_frames, raw_offsets, n_tracks, off, mx, mn, offsets_out,
                             [&](const float *raw, const int64_t *roff, const int64_t *ooff, int64_t total, float *out) {
                                 return launch_median_sync(raw, roff, ooff, n_tracks, downsample_fac, total, out, c->stream);
                             });
}

int acoss_set_tracks_pooled(acoss_ctx *c, const float *raw_frames, const int64_t *raw_offsets, int32_t n_tracks,
                            int32_t win, int32_t skip, int32_t keep_partial, int64_t *offsets_out) {
    if (!c || !raw_frames || !raw_offsets || n_tracks <= 0) { acoss_set_error("set_tracks_pooled: bad arguments"); return ACOSS_E_INVALID; }
    if (win < 1 || win > 65536 || skip < 1 || skip > 65536) { acoss_set_error("set_tracks_pooled: win and skip must be in 1..65536"); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (raw_offsets[0] != 0) { acoss_set_error("set_tracks_pooled: offsets must start at 0"); return ACOSS_E_INVALID; }
    std::vector<int64_t> off(n_tracks + 1, 0);
    int64_t mx = 0, mn = INT64_MAX;
    for (int t = 0; t < n_tracks; ++t) {
        const int64_t n = raw_offsets[t + 1] - raw_offsets[t];
        if (n < 0) { acoss_set_error("set_tracks_pooled: offsets must be non-decreasing"); return ACOSS_E_INVALID; }
        int64_t no;
        if (!keep_partial) {                                     // S5 default: full windows only
            if (n < win) { acoss_set_error("set_tracks_pooled: track %d has %lld raw frames, fewer than win = %d", t, (long long)n, win); return ACOSS_E_TOO_SHORT; }
            no = (n - win) / skip + 1;
        } else {                                                 // S5 = 1: a shorter last window covers the tail
            no = n <= win ? (n > 0 ? 1 : 0) : (n - win + skip - 1) / skip + 1;
        }
        off[t + 1] = off[t] + no;
        mx = std::max(mx, no);
        mn = std::min(mn, no);
    }
    if (mx > (1 << 20)) { acoss_set_error("set_tracks_pooled: track longer than 2^20 pooled frames"); return ACOSS_E_INVALID; }
    return reduce_raw_tracks(c, raw_frames, raw_offsets, n_tracks, off, mx, mn, offsets_out,
                             [&](const float *raw, const int64_t *roff, const int64_t *ooff, int64_t total, float *out) {
                                 return launch_mean_pool(raw, roff, ooff, n_tracks, win, skip, total, out, c->stream);
                             });
}

int acoss_get_tracks(acoss_ctx *c, float *frames_out, int64_t total_frames) {
    if (!c || !frames_out || !c->d_frames) { acoss_set_error("get_tracks: no tracks resident or NULL buffer"); return ACOSS_E_INVALID; }
    if (total_frames != c->total_frames) { acoss_set_error("get_tracks: buffer holds %lld frames, resident set has %lld", (long long)total_frames, (long long)c->total_frames); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaMemcpyAsync(frames_out, c->d_frames, (size_t)total_frames * NBINS * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return ACOSS_OK;
}

static TrackSet track_set(const acoss_ctx *c) {
    TrackSet ts;
    ts.frames = c->d_frames; ts.offsets = c->d_offsets; ts.gchroma = c->d_gchroma;
    ts.n_tracks = c->n_tracks; ts.max_frames = c->max_frames;
    ts.fx_exp = c->fx_exp; ts.nonneg = c->nonneg; ts.q_exp = c->q_exp;
    return ts;
}

static int check_params(const acoss_ctx *c, const acoss_params *p) {
    if (!c || !p) { acoss_set_error("NULL context or params"); return ACOSS_E_INVALID; }
    if (!c->d_frames) { acoss_set_error("no tracks resident: call acoss_set_tracks first"); return ACOSS_E_INVALID; }
    if (p->m < 1 || p->m > 64 || p->tau < 1 || p->tau > 64) { acoss_set_error("m and tau must be in 1..64"); return ACOSS_E_INVALID; }
    if (!(p->kappa >= 0.f && p->kappa <= 1.f)) { acoss_set_error("kappa must be in [0,1]"); return ACOSS_E_INVALID; }
    if (p->noti < 0 || p->noti > 64) { acoss_set_error("noti out of range"); return ACOSS_E_INVALID; }
    if (p->align != ACOSS_ALIGN_QMAX && p->align != ACOSS_ALIGN_DMAX && p->align != ACOSS_ALIGN_DMAX_PLAIN &&
        p->align != ACOSS_ALIGN_SW) {
        acoss_set_error("align mode %d not implemented for the pair pipeline", p->align);
        return ACOSS_E_INVALID;
    }
    const int incr = win_incr(p);
    if (c->min_frames < incr + 2) {
        acoss_set_error("a track has %d frames; essentia needs at least m*tau+2 = %d (F9)", c->min_frames, incr + 2);
        return ACOSS_E_TOO_SHORT;
    }
    return ACOSS_OK;
}

__global__ void or_reduce_kernel(const uint32_t *__restrict__ status, int64_t n, uint32_t *__restrict__ out) {
    uint32_t v = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) v |= status[i];
    v = __reduce_or_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0 && v) atomicOr(out, v);
}
__global__ void count_bits_kernel(const uint32_t *__restrict__ status, int64_t n, uint32_t bit, unsigned long long *out) {
    unsigned c = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) c += (status[i] & bit) ? 1u : 0u;
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, (unsigned long long)c);
}

struct DumpOut {
    int32_t *oti = nullptr;
    uint32_t *crp = nullptr;
    float *thr_q = nullptr, *thr_r = nullptr;
};

constexpr int FB_ROUNDS = 4;      // deferred exact-fallback rounds issued without knowing how many pairs were flagged

// One round of the deferred exact fallback: the pairs map[0 .. nslots) (absolute pair indices, negative = unused)
// are re-scored by the exact CRP path in scratch slots 0 .. nslots-1 and their scores overwrite scores_dev[map[.]].
static int fallback_round(acoss_ctx *c, const TrackSet &ts, const int32_t *pairs_dev, const acoss_params *p, const SlotGeom &g,
                          int64_t ldd, int64_t halo_pitch, const int32_t *map_dev, int nslots, float *scores_dev,
                          float *scores2_dev, int64_t *launches) {
    cudaStream_t st = c->stream;
    ExactScratch sc;
    sc.rrot = (float *)c->rrot.p; sc.aa = (float *)c->aa.p; sc.bb = (float *)c->bb.p; sc.D = (float *)c->D.p;
    sc.ldd = ldd; sc.slots = nslots;
    uint32_t *status = (uint32_t *)c->status.p;
    const int incr = win_incr(p);
    TRY(launch_k2_exact(ts, pairs_dev, (const int32_t *)c->oti.p, 0, nslots, *p, g, sc, (uint32_t *)c->crp.p, (float *)c->thr_q.p,
                        (float *)c->thr_r.p, status, map_dev, st, launches, true));
    TRY(launch_pair_geometry_map(ts, pairs_dev, map_dev, nslots, incr, (int32_t *)c->rows.p, (int32_t *)c->cols.p, st));
    float *tmp = (float *)c->fbtmp.p;
    if (!scores2_dev && p->align == ACOSS_ALIGN_SW)
        TRY(launch_sw_trim((uint32_t *)c->crp.p, g.crp_words, g.words, (int32_t *)c->rows.p, (int32_t *)c->cols.p, nslots, st));
    TRY(launch_dp_bits((const uint32_t *)c->crp.p, g.crp_words, g.words, (const int32_t *)c->rows.p, (const int32_t *)c->cols.p,
                       nslots, g.max_cols, scores2_dev ? ACOSS_ALIGN_QMAX : p->align, p->gamma_o, p->gamma_e, tmp,
                       (uint32_t *)c->halo.p, halo_pitch, st, launches));
    if (p->f5_asymmetric) TRY(launch_score_asymmetric(tmp, (const int32_t *)c->cols.p, nslots, st));
    TRY(launch_scatter_scores(tmp, map_dev, nslots, scores_dev, st));
    if (scores2_dev) {
        TRY(launch_dp_bits((const uint32_t *)c->crp.p, g.crp_words, g.words, (const int32_t *)c->rows.p, (const int32_t *)c->cols.p,
                           nslots, g.max_cols, ACOSS_ALIGN_DMAX, p->gamma_o, p->gamma_e, tmp, (uint32_t *)c->halo.p, halo_pitch, st,
                           launches));
        if (p->f5_asymmetric) TRY(launch_score_asymmetric(tmp, (const int32_t *)c->cols.p, nslots, st));
        TRY(launch_scatter_scores(tmp, map_dev, nslots, scores2_dev, st));
    }
    if (launches) *launches += 3;
    return ACOSS_OK;
}

// Core pipeline.  pairs_dev / scores_dev are device pointers.
// scores2_dev (optional): Dmax scores of the same CRPs (ChenFusion), scores_dev then holds Qmax.
static int run_pairs(acoss_ctx *c, const int32_t *pairs_dev, int64_t K, const acoss_params *p, float *scores_dev,
                     DumpOut *dump, float *scores2_dev = nullptr) {
    TRY(check_params(c, p));
    if (K <= 0) return ACOSS_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const TrackSet ts = track_set(c);
    const int incr = win_incr(p);
    SlotGeom g;
    g.max_rows = c->max_frames - incr;
    g.max_cols = c->max_frames - incr;
    g.words = (g.max_cols + 31) / 32 + 1;
    g.crp_words = (int64_t)g.max_rows * g.words;
    const int64_t ldd = ((int64_t)g.max_cols + 31) / 32 * 32;
    const int64_t halo_pitch = g.max_rows;
    memset(c->stats, 0, sizeof(c->stats));
    int64_t launches = 0;

    TRY(ensure(c->oti, (size_t)K * 4));
    TRY(ensure(c->status, (size_t)K * 4 + 64));
    TRY(ensure(c->misc, 256));
    CUDA_TRY(cudaMemsetAsync(c->status.p, 0, (size_t)K * 4 + 64, st));
    CUDA_TRY(cudaMemsetAsync(c->misc.p, 0, 256, st));
    TRY(ensure(c->dbg, 128));
    CUDA_TRY(cudaMemsetAsync(c->dbg.p, 0, 128, st));
    {
        StageTimer t1(c, 0);
        TRY(launch_oti(ts, pairs_dev, K, p->noti, p->oti, (int32_t *)c->oti.p, st));
        t1.stop();
    }
    ++launches;

    const bool fast = (p->crp_path == ACOSS_CRP_AUTO) && !p->f2_strict && !p->f3_float_acc && !p->f4_keep_last &&
                      k2_fast_supported(*p, g, ts);
    // bytes per slot
    const size_t exact_slot = (size_t)g.max_rows * ldd * 4 + (size_t)c->max_frames * NBINS * 4 + (size_t)(g.max_rows + g.max_cols) * 4;
    const size_t common_slot = (size_t)g.crp_words * 4 + (size_t)(g.max_rows + g.max_cols) * 4 + 8 + (size_t)2 * halo_pitch * 16;
    const size_t fast_slot = fast ? k2_fast_slot_bytes(g, c->max_frames) : 0;
    const size_t per_slot = common_slot + (fast ? fast_slot : exact_slot);
    int64_t slots = std::max<int64_t>(1, (int64_t)(c->ws_limit / (int64_t)per_slot));
    slots = std::min<int64_t>(slots, std::min<int64_t>(K, 16384));
    // exact-fallback slots available to the fast path (flagged pairs are re-run in small groups)
    const int fb_slots = fast ? (int)std::max<int64_t>(1, std::min<int64_t>(16, ((int64_t)2 << 30) / (int64_t)exact_slot)) : 0;
    const int64_t ex_slots = fast ? fb_slots : slots;

    const int64_t oslots = std::max<int64_t>(slots, fb_slots);   // the deferred fallback rounds reuse these buffers
    TRY(ensure(c->crp, (size_t)oslots * g.crp_words * 4));
    TRY(ensure(c->rows, (size_t)oslots * 4));
    TRY(ensure(c->cols, (size_t)oslots * 4));
    TRY(ensure(c->thr_q, (size_t)oslots * g.max_rows * 4));
    TRY(ensure(c->thr_r, (size_t)oslots * g.max_cols * 4));
    TRY(ensure(c->halo, (size_t)oslots * 2 * halo_pitch * 16));
    TRY(ensure(c->fbtmp, (size_t)std::max(fb_slots, 1) * 4 + 64));
    const bool defer = fast && (dump == nullptr);               // single-pair dumps resolve their fallback at once
    c->fb.active = 0;
    TRY(ensure(c->rrot, (size_t)ex_slots * c->max_frames * NBINS * 4));
    TRY(ensure(c->aa, (size_t)ex_slots * g.max_rows * 4));
    TRY(ensure(c->bb, (size_t)ex_slots * g.max_cols * 4));
    TRY(ensure(c->D, (size_t)ex_slots * g.max_rows * ldd * 4));
    if (fast) TRY(ensure(c->fast, (size_t)slots * fast_slot + 4096));
    const uint32_t gcap = k2_fast_sparse_cap(slots);
    if (fast) TRY(ensure(c->glive, ((size_t)gcap + 16) * 4));
    ExactScratch sc;
    sc.rrot = (float *)c->rrot.p; sc.aa = (float *)c->aa.p; sc.bb = (float *)c->bb.p; sc.D = (float *)c->D.p;
    sc.ldd = ldd; sc.slots = (int32_t)ex_slots;

    uint32_t *status = (uint32_t *)c->status.p;
    for (int64_t first = 0; first < K; first += slots) {
        const int n = (int)std::min<int64_t>(slots, K - first);
        ++c->stats[6];
        TRY(launch_pair_geometry(ts, pairs_dev, first, n, incr, (int32_t *)c->rows.p, (int32_t *)c->cols.p, st));
        ++launches;
        StageTimer t2(c, 1);
        if (fast) {
            CtxKernelTimer kt(c);
            TRY(launch_k2_fast(ts, pairs_dev, (const int32_t *)c->oti.p, first, n, *p, g, c->fast.p, fast_slot,
                               (uint32_t *)c->crp.p, (float *)c->thr_q.p, (float *)c->thr_r.p, status, (uint32_t *)c->dbg.p, st, &launches,
                               c->profiling ? &kt : nullptr, (uint32_t *)c->glive.p, gcap));
            // exact fallback for pairs the fast path flagged.  Batched calls defer it to the end of the call (no host
            // synchronisation between chunks); a debug dump compacts the flagged slots and re-runs them at once
            int nfb = 0;
            if (!defer) {
                TRY(ensure(c->fbmap, (size_t)slots * 4 + 64));
                TRY(k2_fast_collect_fallback(status, first, n, (int32_t *)c->fbmap.p, (int32_t *)((char *)c->misc.p + 128), &nfb, st));
            }
            if (nfb > 0) {
                c->stats[1] += nfb;
                for (int b0 = 0; b0 < nfb; b0 += fb_slots) {
                    const int nb = std::min(fb_slots, nfb - b0);
                    TRY(launch_k2_exact(ts, pairs_dev, (const int32_t *)c->oti.p, first, nb, *p, g, sc, (uint32_t *)c->crp.p,
                                        (float *)c->thr_q.p, (float *)c->thr_r.p, status, (const int32_t *)c->fbmap.p + b0, st,
                                        &launches));
                }
            }
        } else {
            TRY(launch_k2_exact(ts, pairs_dev, (const int32_t *)c->oti.p, first, n, *p, g, sc, (uint32_t *)c->crp.p,
                                (float *)c->thr_q.p, (float *)c->thr_r.p, status, nullptr, st, &launches));
        }
        t2.stop();
        if (dump && first == 0) {
            // single-pair debug dump (K == 1); before the DP stage: the SW trim below edits rows / cols / CRP
            const int q = 0;
            (void)q;
            if (dump->oti) CUDA_TRY(cudaMemcpyAsync(dump->oti, c->oti.p, 4, cudaMemcpyDeviceToHost, st));
            int32_t rc[2];
            CUDA_TRY(cudaMemcpyAsync(&rc[0], c->rows.p, 4, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaMemcpyAsync(&rc[1], c->cols.p, 4, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            const int wout = (rc[1] + 31) / 32;
            if (dump->crp)
                CUDA_TRY(cudaMemcpy2DAsync(dump->crp, (size_t)wout * 4, c->crp.p, (size_t)g.words * 4, (size_t)wout * 4,
                                           rc[0], cudaMemcpyDeviceToHost, st));
            if (dump->thr_q) CUDA_TRY(cudaMemcpyAsync(dump->thr_q, c->thr_q.p, (size_t)rc[0] * 4, cudaMemcpyDeviceToHost, st));
            if (dump->thr_r) CUDA_TRY(cudaMemcpyAsync(dump->thr_r, c->thr_r.p, (size_t)rc[1] * 4, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
        }
        StageTimer t3(c, 2);
        if (!scores2_dev && p->align == ACOSS_ALIGN_SW) {        // SW drops the last row / column of the CRP
            TRY(launch_sw_trim((uint32_t *)c->crp.p, g.crp_words, g.words, (int32_t *)c->rows.p, (int32_t *)c->cols.p, n, st));
            ++launches;
        }
        TRY(launch_dp_bits((const uint32_t *)c->crp.p, g.crp_words, g.words, (const int32_t *)c->rows.p,
                           (const int32_t *)c->cols.p, n, g.max_cols, scores2_dev ? ACOSS_ALIGN_QMAX : p->align,
                           p->gamma_o, p->gamma_e, scores_dev + first, (uint32_t *)c->halo.p, halo_pitch, st, &launches));
        if (scores2_dev)
            TRY(launch_dp_bits((const uint32_t *)c->crp.p, g.crp_words, g.words, (const int32_t *)c->rows.p,
                               (const int32_t *)c->cols.p, n, g.max_cols, ACOSS_ALIGN_DMAX, p->gamma_o, p->gamma_e,
                               scores2_dev + first, (uint32_t *)c->halo.p, halo_pitch, st, &launches));
        if (p->f5_asymmetric) {                                  // F5: sqrt(N') / max(Q) (essentia 'asymmetric')
            TRY(launch_score_asymmetric(scores_dev + first, (const int32_t *)c->cols.p, n, st));
            if (scores2_dev) TRY(launch_score_asymmetric(scores2_dev + first, (const int32_t *)c->cols.p, n, st));
            ++launches;
        }
        t3.stop();
    }
    if (defer) {
        // Deferred exact fallback: compact the flagged pairs of the whole call on the device, re-score the first
        // FB_ROUNDS * fb_slots of them right here (kernels skip unused map entries, so no count is needed on the
        // host); the count travels to the host with the status word and acoss_sync() finishes any remainder.
        TRY(ensure(c->fbmap, (size_t)(K + FB_ROUNDS * fb_slots) * 4 + 64));
        int32_t *map = (int32_t *)c->fbmap.p;
        CUDA_TRY(cudaMemsetAsync(map, 0xff, (size_t)(K + FB_ROUNDS * fb_slots) * 4, st));
        TRY(k2_fast_collect_fallback(status, 0, (int)K, map, (int32_t *)((char *)c->misc.p + 128), nullptr, st));
        ++launches;
        StageTimer t4(c, 1);
        for (int r = 0; r < FB_ROUNDS; ++r)
            TRY(fallback_round(c, ts, pairs_dev, p, g, ldd, halo_pitch, map + r * fb_slots, fb_slots, scores_dev, scores2_dev,
                               &launches));
        t4.stop();
        CUDA_TRY(cudaMemcpyAsync(c->h_flag + 2, (char *)c->misc.p + 128, 4, cudaMemcpyDeviceToHost, st));
        c->fb.active = 1; c->fb.pairs_dev = pairs_dev; c->fb.scores_dev = scores_dev; c->fb.scores2_dev = scores2_dev;
        c->fb.p = *p; c->fb.g = g; c->fb.ldd = ldd; c->fb.halo_pitch = halo_pitch; c->fb.K = K; c->fb.fb_slots = fb_slots;
        c->fb.done = FB_ROUNDS * fb_slots;
    }
    // fold per-pair status into one word; read back at sync time
    or_reduce_kernel<<<148, 256, 0, st>>>(status, K, (uint32_t *)c->misc.p);
    CUDA_TRY(cudaGetLastError());
    ++launches;
    CUDA_TRY(cudaMemcpyAsync(c->h_flag, c->misc.p, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(c->h_dbg, c->dbg.p, 128, cudaMemcpyDeviceToHost, st));
    c->pending_status_check = 1;
    c->pending_pairs = K;
    c->stats[0] = K;
    c->stats[2] = launches;
    c->stats_reason_pending = 1;
    return ACOSS_OK;
}

// waits for the stream and completes the deferred exact fallback of the last asynchronous call
static int finish_pending(acoss_ctx *c) {
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (c->fb.active) {
        // the asynchronous call re-scored the first fb.done flagged pairs itself; the (rare) remainder is scored here
        c->fb.active = 0;
        const int nfb = (int)c->h_flag[2];
        c->stats[1] = nfb;
        if (nfb > c->fb.done) {
            const TrackSet ts = track_set(c);
            int64_t launches = 0;
            const int32_t *map = (const int32_t *)c->fbmap.p;
            for (int b0 = c->fb.done; b0 < nfb; b0 += c->fb.fb_slots)
                TRY(fallback_round(c, ts, c->fb.pairs_dev, &c->fb.p, c->fb.g, c->fb.ldd, c->fb.halo_pitch, map + b0,
                                   c->fb.fb_slots, c->fb.scores_dev, c->fb.scores2_dev, &launches));
            // the remainder may have raised the NaN status of its pairs: fold the status words again
            CUDA_TRY(cudaMemsetAsync(c->misc.p, 0, 4, c->stream));
            or_reduce_kernel<<<148, 256, 0, c->stream>>>((const uint32_t *)c->status.p, c->fb.K, (uint32_t *)c->misc.p);
            CUDA_TRY(cudaMemcpyAsync(c->h_flag, c->misc.p, 4, cudaMemcpyDeviceToHost, c->stream));
            CUDA_TRY(cudaStreamSynchronize(c->stream));
            c->stats[2] += launches;
        }
    }
    return ACOSS_OK;
}

int acoss_sync(acoss_ctx *c) {
    if (!c) { acoss_set_error("NULL context"); return ACOSS_E_INVALID; }
    TRY(finish_pending(c));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    fold_spans(c);
    if (c->pending_status_check) {
        c->pending_status_check = 0;
        c->stats[5] = c->h_flag[0];
        if (c->h_flag[0] & PAIR_ST_NAN) {
            acoss_set_error("a squared distance was negative -> NaN distance (essentia would raise: non-binary CRP, F7)");
            return ACOSS_E_NAN;
        }
    }
    return ACOSS_OK;
}

int acoss_score_pairs_device(acoss_ctx *c, const int32_t *pairs_dev, int64_t K, const acoss_params *p, float *scores_dev) {
    if (!c || (K > 0 && (!pairs_dev || !scores_dev))) { acoss_set_error("score_pairs_device: NULL argument"); return ACOSS_E_INVALID; }
    return run_pairs(c, pairs_dev, K, p, scores_dev, nullptr);
}

int acoss_score_pairs(acoss_ctx *c, const int32_t *pairs, int64_t K, const acoss_params *p, float *scores) {
    if (!c || (K > 0 && (!pairs || !scores))) { acoss_set_error("score_pairs: NULL argument"); return ACOSS_E_INVALID; }
    if (K <= 0) return check_params(c, p);
    for (int64_t k = 0; k < 2 * K; ++k)
        if (pairs[k] < 0 || pairs[k] >= c->n_tracks) { acoss_set_error("pair index %d out of range", pairs[k]); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    TRY(ensure(c->pairs, (size_t)K * 8));
    TRY(ensure(c->scores, (size_t)K * 4));
    CUDA_TRY(cudaMemcpyAsync(c->pairs.p, pairs, (size_t)K * 8, cudaMemcpyHostToDevice, c->stream));
    TRY(run_pairs(c, (const int32_t *)c->pairs.p, K, p, (float *)c->scores.p, nullptr));
    TRY(finish_pending(c));                                    // every flagged pair is re-scored before the read-back
    CUDA_TRY(cudaMemcpyAsync(scores, c->scores.p, (size_t)K * 4, cudaMemcpyDeviceToHost, c->stream));
    return acoss_sync(c);
}

int acoss_score_pairs_chen(acoss_ctx *c, const int32_t *pairs, int64_t K, const acoss_params *p, float *qmax_scores,
                           float *dmax_scores) {
    if (!c || (K > 0 && (!pairs || !p || !qmax_scores || !dmax_scores))) { acoss_set_error("score_pairs_chen: NULL argument"); return ACOSS_E_INVALID; }
    if (K <= 0) return check_params(c, p);
    for (int64_t k = 0; k < 2 * K; ++k)
        if (pairs[k] < 0 || pairs[k] >= c->n_tracks) { acoss_set_error("pair index %d out of range", pairs[k]); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    TRY(ensure(c->pairs, (size_t)K * 8));
    TRY(ensure(c->scores, (size_t)K * 8));
    CUDA_TRY(cudaMemcpyAsync(c->pairs.p, pairs, (size_t)K * 8, cudaMemcpyHostToDevice, c->stream));
    acoss_params pp = *p;
    pp.align = ACOSS_ALIGN_QMAX;
    TRY(run_pairs(c, (const int32_t *)c->pairs.p, K, &pp, (float *)c->scores.p, nullptr, (float *)c->scores.p + K));
    TRY(finish_pending(c));
    CUDA_TRY(cudaMemcpyAsync(qmax_scores, c->scores.p, (size_t)K * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(dmax_scores, (float *)c->scores.p + K, (size_t)K * 4, cudaMemcpyDeviceToHost, c->stream));
    return acoss_sync(c);
}

int acoss_score_pairs_chen_device(acoss_ctx *c, const int32_t *pairs_dev, int64_t K, const acoss_params *p, float *qmax_dev,
                                  float *dmax_dev) {
    if (!c || (K > 0 && (!pairs_dev || !qmax_dev || !dmax_dev))) { acoss_set_error("score_pairs_chen_device: NULL argument"); return ACOSS_E_INVALID; }
    TRY(check_params(c, p));
    if (K <= 0) return ACOSS_OK;
    acoss_params pp = *p;                                    // run_pairs keeps its own copy for the deferred fallback
    pp.align = ACOSS_ALIGN_QMAX;
    return run_pairs(c, pairs_dev, K, &pp, qmax_dev, nullptr, dmax_dev);
}

int acoss_oti_pairs(acoss_ctx *c, const int32_t *pairs, int64_t K, int32_t noti, int32_t *oti) {
    if (!c || !pairs || !oti || K < 0 || !c->d_frames) { acoss_set_error("oti_pairs: bad arguments"); return ACOSS_E_INVALID; }
    if (K == 0) return ACOSS_OK;
    for (int64_t k = 0; k < 2 * K; ++k)
        if (pairs[k] < 0 || pairs[k] >= c->n_tracks) { acoss_set_error("pair index %d out of range", pairs[k]); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    TRY(ensure(c->pairs, (size_t)K * 8));
    TRY(ensure(c->oti, (size_t)K * 4));
    CUDA_TRY(cudaMemcpyAsync(c->pairs.p, pairs, (size_t)K * 8, cudaMemcpyHostToDevice, c->stream));
    TRY(launch_oti(track_set(c), (const int32_t *)c->pairs.p, K, noti, 1, (int32_t *)c->oti.p, c->stream));
    CUDA_TRY(cudaMemcpyAsync(oti, c->oti.p, (size_t)K * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return ACOSS_OK;
}

int acoss_dump_pair(acoss_ctx *c, int32_t q, int32_t r, const acoss_params *p, int32_t *oti, uint32_t *crp_bits,
                    float *thr_q, float *thr_r, float *score) {
    TRY(check_params(c, p));
    if (q < 0 || r < 0 || q >= c->n_tracks || r >= c->n_tracks) { acoss_set_error("dump_pair: track index out of range"); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    TRY(ensure(c->pairs, 8));
    TRY(ensure(c->scores, 4));
    const int32_t pr[2] = {q, r};
    CUDA_TRY(cudaMemcpyAsync(c->pairs.p, pr, 8, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    DumpOut d;
    d.oti = oti; d.crp = crp_bits; d.thr_q = thr_q; d.thr_r = thr_r;
    TRY(run_pairs(c, (const int32_t *)c->pairs.p, 1, p, (float *)c->scores.p, &d));
    if (score) CUDA_TRY(cudaMemcpyAsync(score, c->scores.p, 4, cudaMemcpyDeviceToHost, c->stream));
    return acoss_sync(c);
}

int acoss_dp_bytes(acoss_ctx *c, const uint8_t *mats, const int64_t *offsets, const int32_t *shapes, int64_t n,
                   int32_t mode, float gamma_o, float gamma_e, float *scores) {
    if (!c || (n > 0 && (!mats || !offsets || !shapes || !scores))) { acoss_set_error("dp_bytes: NULL argument"); return ACOSS_E_INVALID; }
    if (mode != ACOSS_ALIGN_QMAX && mode != ACOSS_ALIGN_SW && mode != ACOSS_ALIGN_DMAX && mode != ACOSS_ALIGN_DMAX_PLAIN) {
        acoss_set_error("dp_bytes: mode %d not implemented", mode);
        return ACOSS_E_INVALID;
    }
    if (n == 0) return ACOSS_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    int max_r = 1, max_c = 1;
    int64_t total = 0;
    for (int64_t k = 0; k < n; ++k) {
        if (shapes[2 * k] < 0 || shapes[2 * k + 1] < 0 || shapes[2 * k] > (1 << 20) || shapes[2 * k + 1] > (1 << 20)) { acoss_set_error("dp_bytes: bad shape"); return ACOSS_E_INVALID; }
        max_r = std::max(max_r, shapes[2 * k]);
        max_c = std::max(max_c, shapes[2 * k + 1]);
        total = std::max<int64_t>(total, offsets[k] + (int64_t)shapes[2 * k] * shapes[2 * k + 1]);
    }
    const int words = (max_c + 31) / 32 + 1;
    const int64_t slot_words = (int64_t)max_r * words;
    const size_t per_slot = (size_t)slot_words * 4 + (size_t)2 * max_r * 16 + 16;
    int64_t slots = std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(n, 16384), c->ws_limit / (int64_t)per_slot));
    Buf dm, doff, dsh;
    int rc = ACOSS_OK;
    auto cleanup = [&]() { free_buf(dm); free_buf(doff); free_buf(dsh); };
#define TRYC(x) do { rc = (x); if (rc != ACOSS_OK) { cleanup(); return rc; } } while (0)
#define CUDA_TRYC(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) { acoss_set_error("%s -> %s", #x, cudaGetErrorString(_e)); cleanup(); return ACOSS_E_CUDA; } } while (0)
    TRYC(ensure(dm, (size_t)total + 16));
    TRYC(ensure(doff, (size_t)n * 8));
    TRYC(ensure(dsh, (size_t)n * 8));
    TRYC(ensure(c->crp, (size_t)slots * slot_words * 4));
    TRYC(ensure(c->rows, (size_t)slots * 4));
    TRYC(ensure(c->cols, (size_t)slots * 4));
    TRYC(ensure(c->halo, (size_t)slots * 2 * max_r * 16));
    TRYC(ensure(c->scores, (size_t)n * 4));
    TRYC(ensure(c->misc, 256));
    CUDA_TRYC(cudaMemsetAsync(c->misc.p, 0, 256, st));
    CUDA_TRYC(cudaMemcpyAsync(dm.p, mats, (size_t)total, cudaMemcpyHostToDevice, st));
    CUDA_TRYC(cudaMemcpyAsync(doff.p, offsets, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRYC(cudaMemcpyAsync(dsh.p, shapes, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    int64_t launches = 0;
    for (int64_t first = 0; first < n; first += slots) {
        const int nn = (int)std::min<int64_t>(slots, n - first);
        TRYC(launch_pack_bytes((const uint8_t *)dm.p, (const int64_t *)doff.p + first, (const int32_t *)dsh.p + 2 * first, nn,
                               mode, (uint32_t *)c->crp.p, slot_words, words, (int32_t *)c->rows.p, (int32_t *)c->cols.p,
                               (uint32_t *)c->misc.p, st));
        TRYC(launch_dp_bits((const uint32_t *)c->crp.p, slot_words, words, (const int32_t *)c->rows.p, (const int32_t *)c->cols.p,
                            nn, max_c, mode, gamma_o, gamma_e, (float *)c->scores.p + first, (uint32_t *)c->halo.p, max_r, st,
                            &launches));
    }
    CUDA_TRYC(cudaMemcpyAsync(scores, c->scores.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRYC(cudaMemcpyAsync(c->h_flag, c->misc.p, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRYC(cudaStreamSynchronize(st));
    cleanup();
#undef TRYC
#undef CUDA_TRYC
    if (c->h_flag[0]) { acoss_set_error("Non-binary elements found in input"); return ACOSS_E_NONBINARY; }
    return ACOSS_OK;
}

int acoss_knn_sw(acoss_ctx *c, const double *csms, const int64_t *offsets, const int32_t *shapes, const int32_t *nn,
                 int64_t n, float *scores, uint32_t *bits_out) {
    if (!c || (n > 0 && (!csms || !offsets || !shapes || !nn || !scores))) { acoss_set_error("knn_sw: NULL argument"); return ACOSS_E_INVALID; }
    if (n == 0) return ACOSS_OK;
    if (n > 60000) { acoss_set_error("knn_sw: at most 60000 matrices per call"); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    int max_r = 1, max_c = 1;
    int64_t total = 0, out_total = 0;
    std::vector<int64_t> out_off(n);
    for (int64_t k = 0; k < n; ++k) {
        const int M = shapes[2 * k], N = shapes[2 * k + 1];
        if (M <= 0 || N <= 0 || M > 65535 || N > (1 << 20)) { acoss_set_error("knn_sw: bad shape"); return ACOSS_E_INVALID; }
        // np.argpartition(D, NNeighbs, 1) needs kth < N (cross_recurrence.py:156): a count equal to the column count raises
        if (nn[k] >= N) { acoss_set_error("knn_sw: nn >= columns (np.argpartition raises: kth out of bounds)"); return ACOSS_E_INVALID; }
        max_r = std::max(max_r, M); max_c = std::max(max_c, N);
        total = std::max<int64_t>(total, offsets[k] + (int64_t)M * N);
        out_off[k] = out_total;
        out_total += (int64_t)M * ((N + 31) / 32);
    }
    const int words = (max_c + 31) / 32 + 1;
    const int64_t slot_words = (int64_t)max_r * words;
    Buf dcsm, doff, dsh, dnn, dout, dooff;
    int rc = ACOSS_OK;
    auto cleanup = [&]() { free_buf(dcsm); free_buf(doff); free_buf(dsh); free_buf(dnn); free_buf(dout); free_buf(dooff); };
#define TRYC(x) do { rc = (x); if (rc != ACOSS_OK) { cleanup(); return rc; } } while (0)
#define CUDA_TRYC(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) { acoss_set_error("%s -> %s", #x, cudaGetErrorString(_e)); cleanup(); return ACOSS_E_CUDA; } } while (0)
    TRYC(ensure(dcsm, (size_t)total * 8));
    TRYC(ensure(doff, (size_t)n * 8)); TRYC(ensure(dsh, (size_t)n * 8)); TRYC(ensure(dnn, (size_t)n * 4));
    TRYC(ensure(dooff, (size_t)n * 8));
    if (bits_out) TRYC(ensure(dout, (size_t)out_total * 4));
    TRYC(ensure(c->crp, (size_t)n * slot_words * 4));
    TRYC(ensure(c->rows, (size_t)n * 4)); TRYC(ensure(c->cols, (size_t)n * 4));
    TRYC(ensure(c->halo, (size_t)n * 2 * max_r * 16));
    TRYC(ensure(c->scores, (size_t)n * 4));
    CUDA_TRYC(cudaMemcpyAsync(dcsm.p, csms, (size_t)total * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRYC(cudaMemcpyAsync(doff.p, offsets, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRYC(cudaMemcpyAsync(dsh.p, shapes, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRYC(cudaMemcpyAsync(dnn.p, nn, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRYC(cudaMemcpyAsync(dooff.p, out_off.data(), (size_t)n * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRYC(cudaMemsetAsync(c->crp.p, 0, (size_t)n * slot_words * 4, st));
    TRYC(launch_knn_rows((const double *)dcsm.p, (const int64_t *)doff.p, (const int32_t *)dsh.p, (const int32_t *)dnn.p, (int)n,
                         max_r, max_c, (uint32_t *)c->crp.p, slot_words, words, bits_out ? (uint32_t *)dout.p : nullptr,
                         (const int64_t *)dooff.p, (int32_t *)c->rows.p, (int32_t *)c->cols.p, st));
    int64_t launches = 0;
    TRYC(launch_dp_bits((const uint32_t *)c->crp.p, slot_words, words, (const int32_t *)c->rows.p, (const int32_t *)c->cols.p,
                        (int)n, max_c, ACOSS_ALIGN_SW, 0.5f, 0.5f, (float *)c->scores.p, (uint32_t *)c->halo.p, max_r, st, &launches));
    CUDA_TRYC(cudaMemcpyAsync(scores, c->scores.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    if (bits_out) CUDA_TRYC(cudaMemcpyAsync(bits_out, dout.p, (size_t)out_total * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRYC(cudaStreamSynchronize(st));
    cleanup();
#undef TRYC
#undef CUDA_TRYC
    return ACOSS_OK;
}

int acoss_debug_counters(acoss_ctx *c, int64_t out[32]) {
    if (!c || !out) { acoss_set_error("debug_counters: NULL argument"); return ACOSS_E_INVALID; }
    for (int i = 0; i < 32; ++i) out[i] = c->h_dbg ? (int64_t)c->h_dbg[i] : 0;
    return ACOSS_OK;
}

int acoss_set_profiling(acoss_ctx *c, int on) {
    if (!c) { acoss_set_error("NULL context"); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    fold_spans(c);
    c->profiling = on ? 1 : 0;
    for (double &m : c->stage_ms) m = 0.0;
    return ACOSS_OK;
}

int acoss_stage_ms(acoss_ctx *c, double ms[4]) {
    if (!c || !ms) { acoss_set_error("stage_ms: NULL argument"); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    fold_spans(c);
    for (int i = 0; i < 4; ++i) ms[i] = c->stage_ms[i];
    return ACOSS_OK;
}

int acoss_kernel_ms(acoss_ctx *c, double ms[16]) {
    if (!c || !ms) { acoss_set_error("kernel_ms: NULL argument"); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    fold_spans(c);
    for (int i = 0; i < 16; ++i) ms[i] = c->stage_ms[16 + i];
    return ACOSS_OK;
}

int acoss_last_stats(acoss_ctx *c, int64_t stats[8]) {
    if (!c || !stats) { acoss_set_error("last_stats: NULL argument"); return ACOSS_E_INVALID; }
    memcpy(stats, c->stats, sizeof(c->stats));
    return ACOSS_OK;
}

// ---------------------------------------------------------------------------------------------
// EarlyFusion pair scoring (k5_earlyfusion.cu + k4_knn.cu + k3_dp.cu)
// ---------------------------------------------------------------------------------------------
int acoss_ef_set_tracks(acoss_ctx *c, const void *mfccs, int32_t d_mfccs, const void *ssms, int32_t d_ssms,
                        const void *chromas, int32_t d_chromas, const double *chroma_med, const int64_t *offsets,
                        int32_t n_tracks, int32_t elem_size) {
    if (!c || !mfccs || !ssms || !chromas || !chroma_med || !offsets || n_tracks <= 0) { acoss_set_error("ef_set_tracks: bad arguments"); return ACOSS_E_INVALID; }
    if (elem_size != 4 && elem_size != 8) { acoss_set_error("ef_set_tracks: elem_size must be 4 (float32) or 8 (float64)"); return ACOSS_E_INVALID; }
    if (d_mfccs <= 0 || d_ssms <= 0 || d_chromas <= 0 || d_chromas % NBINS) { acoss_set_error("ef_set_tracks: feature dimensions must be positive, chroma blocks a multiple of 12"); return ACOSS_E_INVALID; }
    if (offsets[0] != 0) { acoss_set_error("ef_set_tracks: offsets must start at 0"); return ACOSS_E_INVALID; }
    for (int t = 0; t < n_tracks; ++t) {
        const int64_t n = offsets[t + 1] - offsets[t];
        if (n <= 0 || n > 65535) { acoss_set_error("ef_set_tracks: track %d has %lld blocks (1..65535 supported)", t, (long long)n); return ACOSS_E_INVALID; }
    }
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    CUDA_TRY(cudaStreamSynchronize(st));
    c->ef_tracks = 0;
    const int64_t rows = offsets[n_tracks];
    const void *src[3] = {mfccs, ssms, chromas};
    const int32_t d[3] = {d_mfccs, d_ssms, d_chromas};
    Buf &stage = c->ef_stage;                                  // upload staging, released below (also by acoss_destroy)
    for (int k = 0; k < 3; ++k) {
        const int dp = (d[k] + 15) / 16 * 16;
        TRY(ensure(c->ef_feat[k], (size_t)rows * dp * 8));
        TRY(ensure(stage, (size_t)rows * d[k] * elem_size));
        if (k < 2) TRY(ensure(c->ef_sq[k], (size_t)rows * 8));
        CUDA_TRY(cudaMemcpyAsync(stage.p, src[k], (size_t)rows * d[k] * elem_size, cudaMemcpyHostToDevice, st));
        TRY(launch_ef_widen(stage.p, elem_size, rows, d[k], dp, (double *)c->ef_feat[k].p, st));
        TRY(launch_ef_rownorm((double *)c->ef_feat[k].p, rows, dp, k == 2 ? 1 : 0, k < 2 ? (double *)c->ef_sq[k].p : nullptr, st));
        CUDA_TRY(cudaStreamSynchronize(st));                  // the staging buffer is reused by the next kind
        c->ef_d[k] = d[k];
        c->ef_dp[k] = dp;
    }
    free_buf(stage);
    TRY(ensure(c->ef_cmed, (size_t)n_tracks * NBINS * 8));
    TRY(ensure(c->ef_off, (size_t)(n_tracks + 1) * 8));
    CUDA_TRY(cudaMemcpyAsync(c->ef_cmed.p, chroma_med, (size_t)n_tracks * NBINS * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(c->ef_off.p, offsets, (size_t)(n_tracks + 1) * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    c->ef_hoff.assign(offsets, offsets + n_tracks + 1);
    c->ef_tracks = n_tracks;
    return ACOSS_OK;
}

// One chunk of n pairs (device pair list d_pairs) -> four device score arrays sc[kind][0..n).
// bits_dev / bit_off (optional): bit-packed binary matrices of every kind, kind-major; csm stays in c->ef_csm.
static int ef_run_chunk(acoss_ctx *c, const int32_t *d_pairs, int n, int max_r, int max_c, double kappa, int K,
                        float *const sc[4], uint32_t *bits_dev, const int64_t *bit_off_dev, int64_t bits_per_kind,
                        int32_t *oti_dev) {
    cudaStream_t st = c->stream;
    const int64_t slot_elems = (int64_t)max_r * max_c;
    const int64_t kind_stride = slot_elems * n;
    const int words = (max_c + 31) / 32 + 1;
    const int64_t slot_words = (int64_t)max_r * words;
    const int stat_pitch = max_r + max_c;
    TRY(ensure(c->ef_csm, (size_t)kind_stride * 4 * 8));
    TRY(ensure(c->ef_stat, (size_t)stat_pitch * n * 3 * 8));
    TRY(ensure(c->ef_shapes, (size_t)n * 8)); TRY(ensure(c->ef_nn, (size_t)n * 4)); TRY(ensure(c->ef_csmoff, (size_t)n * 8));
    TRY(ensure(c->ef_oti, (size_t)n * 4));
    TRY(ensure(c->crp, (size_t)n * slot_words * 4));
    TRY(ensure(c->rows, (size_t)n * 4)); TRY(ensure(c->cols, (size_t)n * 4));
    TRY(ensure(c->halo, (size_t)n * 2 * max_r * 16));
    double *csm = (double *)c->ef_csm.p;
    const int64_t *off = (const int64_t *)c->ef_off.p;
    int32_t *oti = oti_dev ? oti_dev : (int32_t *)c->ef_oti.p;
    TRY(launch_ef_geom(off, d_pairs, n, kappa, slot_elems, (int32_t *)c->ef_shapes.p, (int32_t *)c->ef_nn.p,
                       (int64_t *)c->ef_csmoff.p, st));
    TRY(launch_ef_oti((const double *)c->ef_cmed.p, d_pairs, n, oti, st));
    c->ef_stats[2] += 2;
    {
        StageTimer t(c, 4);
        for (int k = 0; k < 3; ++k) {
            TRY(launch_ef_csm(k == 2 ? 1 : 0, (const double *)c->ef_feat[k].p, c->ef_dp[k], c->ef_d[k],
                              k < 2 ? (const double *)c->ef_sq[k].p : nullptr, off, d_pairs, oti, n, max_r, max_c,
                              csm + k * kind_stride, slot_elems, st));
            ++c->ef_stats[2];
        }
        t.stop();
    }
    {
        StageTimer t(c, 7);
        TRY(launch_ef_linestat(csm, kind_stride, slot_elems, off, d_pairs, n, max_r, max_c, K, (double *)c->ef_stat.p,
                               (int64_t)stat_pitch * n, stat_pitch, st));
        t.stop();
    }
    {
        StageTimer t(c, 8);
        TRY(launch_ef_fuse(csm, kind_stride, slot_elems, off, d_pairs, n, max_r, max_c, (const double *)c->ef_stat.p,
                           (int64_t)stat_pitch * n, stat_pitch, csm + 3 * kind_stride, st));
        t.stop();
    }
    c->ef_stats[2] += 2;
    for (int k = 0; k < 4; ++k) {
        {
            StageTimer t(c, 5);
            CUDA_TRY(cudaMemsetAsync(c->crp.p, 0, (size_t)n * slot_words * 4, st));
            TRY(launch_knn_rows(csm + k * kind_stride, (const int64_t *)c->ef_csmoff.p, (const int32_t *)c->ef_shapes.p,
                                (const int32_t *)c->ef_nn.p, n, max_r, max_c, (uint32_t *)c->crp.p, slot_words, words,
                                bits_dev ? bits_dev + k * bits_per_kind : nullptr, bit_off_dev, (int32_t *)c->rows.p,
                                (int32_t *)c->cols.p, st));
            t.stop();
        }
        {
            StageTimer t(c, 6);
            int64_t launches = 0;
            TRY(launch_dp_bits((const uint32_t *)c->crp.p, slot_words, words, (const int32_t *)c->rows.p,
                               (const int32_t *)c->cols.p, n, max_c, ACOSS_ALIGN_SW, 0.5f, 0.5f, sc[k],
                               (uint32_t *)c->halo.p, max_r, st, &launches));
            t.stop();
        }
        c->ef_stats[2] += 2;
    }
    return ACOSS_OK;
}

static int ef_check_pairs(acoss_ctx *c, const int32_t *pairs, int64_t n, double kappa, int K, int *max_r, int *max_c,
                          int64_t *cells) {
    if (c->ef_tracks <= 0) { acoss_set_error("EarlyFusion features are not loaded: call acoss_ef_set_tracks first"); return ACOSS_E_INVALID; }
    if (!(kappa >= 0.0)) { acoss_set_error("kappa must be >= 0"); return ACOSS_E_INVALID; }
    if (K < 1 || K > ef_linestat_max_k()) { acoss_set_error("K must be in 1..%d", ef_linestat_max_k()); return ACOSS_E_INVALID; }
    int mr = 1, mc = 1;
    int64_t cl = 0;
    for (int64_t k = 0; k < n; ++k) {
        const int q = pairs[2 * k], r = pairs[2 * k + 1];
        if (q < 0 || r < 0 || q >= c->ef_tracks || r >= c->ef_tracks) { acoss_set_error("pair %lld: track index out of range", (long long)k); return ACOSS_E_INVALID; }
        const int M = (int)(c->ef_hoff[q + 1] - c->ef_hoff[q]), N = (int)(c->ef_hoff[r + 1] - c->ef_hoff[r]);
        // np.partition(CSM, K, axis) raises ValueError when K is not a valid index (similarity_fusion.py:48-51)
        if (K >= M || K >= N) { acoss_set_error("pair %lld: K = %d needs more than K blocks per track (%d x %d); the reference raises ValueError", (long long)k, K, M, N); return ACOSS_E_INVALID; }
        // csm_to_binary (cross_recurrence.py:151-156): NNeighbs = kappa (a count) or int(round(kappa * N)); argpartition
        // needs kth < N, so a neighbour count equal to the column count raises in the reference
        {
            const int nnk = (kappa >= 1.0) ? (int)kappa : (int)nearbyint(kappa * (double)N);
            if (kappa > 0.0 && nnk >= N) { acoss_set_error("pair %lld: %d neighbours >= %d columns (np.argpartition raises: kth out of bounds)", (long long)k, nnk, N); return ACOSS_E_INVALID; }
        }
        mr = std::max(mr, M); mc = std::max(mc, N);
        cl += (int64_t)M * N;
    }
    if (mc > 200 * 1024 / 8) { acoss_set_error("tracks longer than %d blocks are not supported by the k-NN kernel", 200 * 1024 / 8); return ACOSS_E_INVALID; }
    *max_r = mr; *max_c = mc; *cells = cl;
    return ACOSS_OK;
}

int acoss_ef_score_pairs(acoss_ctx *c, const int32_t *pairs, int64_t n_pairs, double kappa, int32_t K, float *scores) {
    if (!c || (n_pairs > 0 && (!pairs || !scores)) || n_pairs < 0) { acoss_set_error("ef_score_pairs: bad arguments"); return ACOSS_E_INVALID; }
    if (n_pairs == 0) return ACOSS_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    int max_r, max_c;
    int64_t cells;
    TRY(ef_check_pairs(c, pairs, n_pairs, kappa, K, &max_r, &max_c, &cells));
    cudaStream_t st = c->stream;
    TRY(ensure(c->ef_pairs, (size_t)n_pairs * 8));
    TRY(ensure(c->ef_scores, (size_t)n_pairs * 4 * 4));
    CUDA_TRY(cudaMemcpyAsync(c->ef_pairs.p, pairs, (size_t)n_pairs * 8, cudaMemcpyHostToDevice, st));
    // slots per chunk from the workspace limit: 4 float64 matrices + the bit-packed copy + line statistics per slot
    const int words = (max_c + 31) / 32 + 1;
    const int64_t per_slot = (int64_t)max_r * max_c * 8 * 4 + (int64_t)max_r * words * 4 + (int64_t)(max_r + max_c) * 24 + 2 * (int64_t)max_r * 16 + 64;
    int64_t slots = std::max<int64_t>(1, std::min<int64_t>(c->ws_limit / per_slot, 32768));
    slots = std::min<int64_t>(slots, n_pairs);
    c->ef_stats[0] = n_pairs; c->ef_stats[1] = cells; c->ef_stats[2] = 0; c->ef_stats[3] = 0;
    float *dsc = (float *)c->ef_scores.p;
    for (int64_t first = 0; first < n_pairs; first += slots) {
        const int n = (int)std::min<int64_t>(slots, n_pairs - first);
        float *const sc[4] = {dsc + first, dsc + n_pairs + first, dsc + 2 * n_pairs + first, dsc + 3 * n_pairs + first};
        TRY(ef_run_chunk(c, (const int32_t *)c->ef_pairs.p + 2 * first, n, max_r, max_c, kappa, K, sc, nullptr, nullptr, 0, nullptr));
        ++c->ef_stats[3];
    }
    CUDA_TRY(cudaMemcpyAsync(scores, dsc, (size_t)n_pairs * 4 * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return ACOSS_OK;
}

int acoss_ef_dump_pair(acoss_ctx *c, int32_t q, int32_t r, double kappa, int32_t K, int32_t *oti, double *csms,
                       uint32_t *bits, float *scores) {
    if (!c) { acoss_set_error("NULL context"); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    const int32_t pr[2] = {q, r};
    int max_r, max_c;
    int64_t cells;
    TRY(ef_check_pairs(c, pr, 1, kappa, K, &max_r, &max_c, &cells));
    cudaStream_t st = c->stream;
    const int64_t wpm = (int64_t)max_r * ((max_c + 31) / 32);
    TRY(ensure(c->ef_pairs, 8)); TRY(ensure(c->ef_scores, 16)); TRY(ensure(c->ef_bits, (size_t)wpm * 4 * 4)); TRY(ensure(c->ef_bitoff, 8));
    TRY(ensure(c->ef_oti, 4));
    CUDA_TRY(cudaMemcpyAsync(c->ef_pairs.p, pr, 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(c->ef_bitoff.p, 0, 8, st));
    float *dsc = (float *)c->ef_scores.p;
    float *const sc[4] = {dsc, dsc + 1, dsc + 2, dsc + 3};
    TRY(ef_run_chunk(c, (const int32_t *)c->ef_pairs.p, 1, max_r, max_c, kappa, K, sc, (uint32_t *)c->ef_bits.p,
                     (const int64_t *)c->ef_bitoff.p, wpm, nullptr));
    if (oti) CUDA_TRY(cudaMemcpyAsync(oti, c->ef_oti.p, 4, cudaMemcpyDeviceToHost, st));
    if (csms) CUDA_TRY(cudaMemcpyAsync(csms, c->ef_csm.p, (size_t)cells * 4 * 8, cudaMemcpyDeviceToHost, st));
    if (bits) CUDA_TRY(cudaMemcpyAsync(bits, c->ef_bits.p, (size_t)wpm * 4 * 4, cudaMemcpyDeviceToHost, st));
    if (scores) CUDA_TRY(cudaMemcpyAsync(scores, dsc, 16, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return ACOSS_OK;
}

int acoss_ef_stage_ms(acoss_ctx *c, double ms[5]) {
    if (!c || !ms) { acoss_set_error("ef_stage_ms: NULL argument"); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    fold_spans(c);
    for (int i = 0; i < 5; ++i) ms[i] = c->stage_ms[4 + i];
    return ACOSS_OK;
}

int acoss_ef_last_stats(acoss_ctx *c, int64_t stats[4]) {
    if (!c || !stats) { acoss_set_error("ef_last_stats: NULL argument"); return ACOSS_E_INVALID; }
    memcpy(stats, c->ef_stats, sizeof(c->ef_stats));
    return ACOSS_OK;
}

// ---- Simple (SiMPle) pair scoring -------------------------------------------------------------------------------

void acoss_simple_default_params(acoss_simple_params *p) {
    if (!p) return;
    p->m = 10; p->oti = 1; p->s2_squared = 0; p->s3_positive = 0; p->s4_roll_first = 0;
}

static int simple_check(const acoss_ctx *c, const acoss_simple_params *p) {
    if (!c || !p) { acoss_set_error("NULL context or params"); return ACOSS_E_INVALID; }
    if (!c->d_frames) { acoss_set_error("no tracks resident: call acoss_set_tracks_pooled first"); return ACOSS_E_INVALID; }
    if (p->m < 1 || p->m > 128) { acoss_set_error("subsequence length m = %d outside 1..128", p->m); return ACOSS_E_INVALID; }
    if (c->min_frames < p->m) {
        acoss_set_error("a track has %d pooled frames, fewer than the subsequence length m = %d", c->min_frames, p->m);
        return ACOSS_E_TOO_SHORT;
    }
    return ACOSS_OK;
}

// Enqueues the scoring of K pairs (device list) in workspace-limited chunks; oti_dev (may be NULL) receives the OTIs,
// prof0 / idx0 (may be NULL) the profile and index arrays of workspace slot 0 (the first pair of the last chunk).
static int simple_run(acoss_ctx *c, const int32_t *pairs_dev, int64_t K, const acoss_simple_params *p, float *scores_dev,
                      int32_t *oti_dev, const double **prof0 = nullptr, const int32_t **idx0 = nullptr) {
    TRY(simple_check(c, p));
    if (K <= 0) return ACOSS_OK;
    CUDA_TRY(cudaSetDevice(c->device));
    const size_t per_slot = simple_slot_bytes(c->max_frames, p->m);
    const int64_t slots = std::max<int64_t>(1, std::min<int64_t>({K, (int64_t)8192, c->ws_limit / (int64_t)per_slot}));
    TRY(ensure(c->sp_ws, (size_t)slots * per_slot));
    const int64_t rows = std::max(1, c->max_frames - p->m + 1);
    SimpleArgs a;
    a.frames = c->d_frames; a.offsets = c->d_offsets; a.pairs = pairs_dev;
    a.m = p->m; a.oti = p->oti ? 1 : 0; a.s2_squared = p->s2_squared ? 1 : 0; a.s3_positive = p->s3_positive ? 1 : 0;
    a.s4_roll_first = p->s4_roll_first ? 1 : 0;
    a.max_frames = c->max_frames;
    a.stage_pitch = (int64_t)2 * c->max_frames * NBINS;
    a.row_pitch = rows;
    char *w = (char *)c->sp_ws.p;                                 // [stage][thr][cnt][prof][idx][cand], each slots x pitch
    a.stage = (float *)w; w += (size_t)slots * a.stage_pitch * 4;
    a.prof = (double *)w; w += (size_t)slots * rows * 8;
    a.thr = (uint32_t *)w; w += (size_t)slots * rows * 4;
    a.cnt = (int32_t *)w; w += (size_t)slots * rows * 4;
    a.idx = (int32_t *)w; w += (size_t)slots * rows * 4;
    a.cand = (int32_t *)w;
    a.scores = scores_dev; a.oti_out = oti_dev;
    if (prof0) *prof0 = a.prof;
    if (idx0) *idx0 = a.idx;
    for (int64_t first = 0; first < K; first += slots) {
        a.first = first;
        TRY(launch_simple_pairs(a, (int)std::min<int64_t>(slots, K - first), c->stream));
    }
    return ACOSS_OK;
}

static int simple_pairs_in_range(const acoss_ctx *c, const int32_t *pairs, int64_t K) {
    for (int64_t k = 0; k < 2 * K; ++k)
        if (pairs[k] < 0 || pairs[k] >= c->n_tracks) { acoss_set_error("pair index %d out of range", pairs[k]); return ACOSS_E_INVALID; }
    return ACOSS_OK;
}

int acoss_simple_score_pairs(acoss_ctx *c, const int32_t *pairs, int64_t K, const acoss_simple_params *p, float *scores) {
    if (!c || (K > 0 && (!pairs || !scores))) { acoss_set_error("simple_score_pairs: NULL argument"); return ACOSS_E_INVALID; }
    TRY(simple_check(c, p));
    if (K <= 0) return ACOSS_OK;
    TRY(simple_pairs_in_range(c, pairs, K));
    CUDA_TRY(cudaSetDevice(c->device));
    TRY(ensure(c->sp_pairs, (size_t)K * 8));
    TRY(ensure(c->sp_scores, (size_t)K * 4));
    CUDA_TRY(cudaMemcpyAsync(c->sp_pairs.p, pairs, (size_t)K * 8, cudaMemcpyHostToDevice, c->stream));
    TRY(simple_run(c, (const int32_t *)c->sp_pairs.p, K, p, (float *)c->sp_scores.p, nullptr));
    CUDA_TRY(cudaMemcpyAsync(scores, c->sp_scores.p, (size_t)K * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return ACOSS_OK;
}

int acoss_simple_score_pairs_device(acoss_ctx *c, const int32_t *pairs_dev, int64_t K, const acoss_simple_params *p,
                                    float *scores_dev) {
    if (!c || (K > 0 && (!pairs_dev || !scores_dev))) { acoss_set_error("simple_score_pairs_device: NULL argument"); return ACOSS_E_INVALID; }
    return simple_run(c, pairs_dev, K, p, scores_dev, nullptr);
}

int acoss_simple_dump_pair(acoss_ctx *c, int32_t q, int32_t r, const acoss_simple_params *p, int32_t *oti,
                           double *profile, int32_t *index, float *score) {
    TRY(simple_check(c, p));
    const int32_t pr[2] = {q, r};
    TRY(simple_pairs_in_range(c, pr, 1));
    CUDA_TRY(cudaSetDevice(c->device));
    TRY(ensure(c->sp_pairs, 8));
    TRY(ensure(c->sp_scores, 4));
    TRY(ensure(c->sp_oti, 4));
    CUDA_TRY(cudaMemcpyAsync(c->sp_pairs.p, pr, 8, cudaMemcpyHostToDevice, c->stream));
    const double *prof = nullptr;
    const int32_t *idx = nullptr;
    TRY(simple_run(c, (const int32_t *)c->sp_pairs.p, 1, p, (float *)c->sp_scores.p, (int32_t *)c->sp_oti.p, &prof, &idx));
    int64_t hoff[2];
    CUDA_TRY(cudaMemcpyAsync(hoff, c->d_offsets + q, 16, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    const int64_t rows = hoff[1] - hoff[0] - p->m + 1;          // profile length of the query
    if (profile) CUDA_TRY(cudaMemcpyAsync(profile, prof, (size_t)rows * 8, cudaMemcpyDeviceToHost, c->stream));
    if (index) CUDA_TRY(cudaMemcpyAsync(index, idx, (size_t)rows * 4, cudaMemcpyDeviceToHost, c->stream));
    if (oti) CUDA_TRY(cudaMemcpyAsync(oti, c->sp_oti.p, 4, cudaMemcpyDeviceToHost, c->stream));
    if (score) CUDA_TRY(cudaMemcpyAsync(score, c->sp_scores.p, 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return ACOSS_OK;
}


// ---- Similarity-network fusion (k7_snf.cu) -----------------------------------------------------------------------

int acoss_snf(acoss_ctx *c, const float *const *D, int32_t n_mats, int32_t n, int32_t K, int32_t niters, double reg_diag,
              double reg_neighbs, int32_t jacobi, double *fused, float *W, float *P, int32_t *S_idx, float *S_val) {
    if (!c || !D || !fused) { acoss_set_error("snf: NULL argument"); return ACOSS_E_INVALID; }
    if (n_mats < 2 || n_mats > ACOSS_SNF_MAX_MATS) {
        acoss_set_error("snf: %d score matrices; 2..%d supported (the reference divides by n_mats - 1)", n_mats, ACOSS_SNF_MAX_MATS);
        return ACOSS_E_INVALID;
    }
    for (int m = 0; m < n_mats; ++m)
        if (!D[m]) { acoss_set_error("snf: score matrix %d is NULL", m); return ACOSS_E_INVALID; }
    if (K < 1 || K > ACOSS_SNF_MAX_K) { acoss_set_error("snf: K = %d outside 1..%d", K, ACOSS_SNF_MAX_K); return ACOSS_E_INVALID; }
    if (n < 2 || n > 65535 || K + 1 >= n) {
        acoss_set_error("snf: n = %d with K = %d; K + 1 < n <= 65535 required (np.partition raises for kth >= n)", n, K);
        return ACOSS_E_INVALID;
    }
    if (niters < 0) { acoss_set_error("snf: niters = %d < 0", niters); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int64_t N2 = (int64_t)n * n;
    const int sets = niters == 0 ? 0 : (jacobi ? 2 : 1);     // float64 Pts sets: Jacobi keeps the previous iteration
    const std::vector<int32_t> leaves = snf_leaf_offsets(n);
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t b_p = up((size_t)n_mats * N2 * 4), b_s = up((size_t)n_mats * n * K * 4), b_pts = up((size_t)sets * n_mats * N2 * 8),
                 b_x = up((size_t)N2 * 8), b_t = niters ? up((size_t)N2 * 8) : 0, b_md = up((size_t)n * 4), b_leaf = up(leaves.size() * 4);
    const size_t total = b_p + 2 * b_s + b_pts + b_x + b_t + b_md + b_leaf;
    if ((int64_t)total > c->ws_limit) {
        acoss_set_error("snf: %zu bytes of device workspace needed, limit %lld (acoss_set_workspace_limit)", total, (long long)c->ws_limit);
        return ACOSS_E_NOMEM;
    }
    struct Scratch { void *p = nullptr; ~Scratch() { if (p) cudaFree(p); } } ws;   // released when the call returns
    if (cudaMalloc(&ws.p, total) != cudaSuccess) {
        cudaGetLastError();
        ws.p = nullptr;
        acoss_set_error("snf: cudaMalloc(%zu bytes) failed", total);
        return ACOSS_E_NOMEM;
    }
    char *p = (char *)ws.p;
    float *dP = (float *)p; p += b_p;                          // P of every matrix (the first iteration's Pts)
    int32_t *dSi = (int32_t *)p; p += b_s;
    float *dSv = (float *)p; p += b_s;
    double *dPts = (double *)p; p += b_pts;                    // [set][matrix] float64 Pts
    double *dX = (double *)p; p += b_x;                        // X^T; the score staging + DSym / W before; fused after
    double *dT = (double *)p; p += b_t;                        // A^T
    float *dmd = (float *)p; p += b_md;
    int32_t *dleaf = (int32_t *)p;
    float *dstage = (float *)dX, *dw = (float *)dX + N2;
    CUDA_TRY(cudaMemcpyAsync(dleaf, leaves.data(), leaves.size() * 4, cudaMemcpyHostToDevice, st));
    for (int m = 0; m < n_mats; ++m) {
        StageTimer h2d(c, 9);
        CUDA_TRY(cudaMemcpyAsync(dstage, D[m], (size_t)N2 * 4, cudaMemcpyHostToDevice, st));
        h2d.stop();
        StageTimer aff(c, 10);
        TRY(launch_snf_affinity(dstage, n, K, dw, dmd, dleaf, (int)leaves.size() - 1, dP + m * N2, dSi + (int64_t)m * n * K,
                                dSv + (int64_t)m * n * K, st));
        aff.stop();
        if (W) CUDA_TRY(cudaMemcpyAsync(W + m * N2, dw, (size_t)N2 * 4, cudaMemcpyDeviceToHost, st));
    }
    if (P) CUDA_TRY(cudaMemcpyAsync(P, dP, (size_t)n_mats * N2 * 4, cudaMemcpyDeviceToHost, st));
    if (S_idx) CUDA_TRY(cudaMemcpyAsync(S_idx, dSi, (size_t)n_mats * n * K * 4, cudaMemcpyDeviceToHost, st));
    if (S_val) CUDA_TRY(cudaMemcpyAsync(S_val, dSv, (size_t)n_mats * n * K * 4, cudaMemcpyDeviceToHost, st));
    // Iteration 0 reads the float32 P; later ones read set (it - 1) % sets and write set it % sets, so with one set
    // (jacobi = 0) Pts[k < i] already hold this iteration's values
    auto pts = [&](int set, int m) { return dPts + ((int64_t)set * n_mats + m) * N2; };
    StageTimer dif(c, 11);
    for (int it = 0; it < niters; ++it) {
        for (int i = 0; i < n_mats; ++i) {
            const void *src[ACOSS_SNF_MAX_MATS];
            int ns = 0;
            for (int k = 0; k < n_mats; ++k)
                if (k != i) src[ns++] = it == 0 ? (const void *)(dP + k * N2) : (const void *)pts((it - 1) % sets, k);
            TRY(launch_snf_mix(src, ns, it == 0, it == 0 ? nullptr : pts((it - 1) % sets, i), n, (double)(n_mats - 1), dX, st));
            TRY(launch_snf_spmm(dX, dSi + (int64_t)i * n * K, dSv + (int64_t)i * n * K, n, K, true, 0.0, 0.0, dT, st));
            TRY(launch_snf_spmm(dT, dSi + (int64_t)i * n * K, dSv + (int64_t)i * n * K, n, K, false, reg_diag, reg_neighbs,
                                pts(it % sets, i), st));
        }
    }
    dif.stop();
    StageTimer fin(c, 12);
    const void *src[ACOSS_SNF_MAX_MATS];
    for (int m = 0; m < n_mats; ++m) src[m] = niters == 0 ? (const void *)(dP + m * N2) : (const void *)pts((niters - 1) % sets, m);
    TRY(launch_snf_average(src, n_mats, niters == 0, N2, dX, st));
    CUDA_TRY(cudaMemcpyAsync(fused, dX, (size_t)N2 * 8, cudaMemcpyDeviceToHost, st));
    fin.stop();
    CUDA_TRY(cudaStreamSynchronize(st));
    return ACOSS_OK;
}

int acoss_snf_stage_ms(acoss_ctx *c, double ms[4]) {
    if (!c || !ms) { acoss_set_error("snf_stage_ms: NULL argument"); return ACOSS_E_INVALID; }
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    fold_spans(c);
    for (int i = 0; i < 4; ++i) ms[i] = c->stage_ms[9 + i];
    return ACOSS_OK;
}

}  // extern "C"
