// K0 — feature on-ramp: median downsampling (Serra09) and mean pooling (SiMPle) of raw HPCP frames on the GPU.
//
// Replaces the aggregation inside Serra09.load_features / ChenFusion.load_features
//   /root/reference/acoss/algorithms/rqa_serra09.py:47-53
//       chroma = sync(chroma.T, np.arange(0, chroma.shape[0], self.downsample_fac), aggregate=np.median)
// (librosa.util.sync, SURVEY.md App. A7): output frame k of a track = per-bin np.median of the raw frames
// [fac*k, min(fac*k + fac, n)); float32 in, float32 out; an even block takes
// float32(float32(a + b) / 2) of its two middle values, which is what np.median computes on float32 data.
//
// One warp per output frame.  The block's fac x 12 raw floats are contiguous in HBM (48 B per frame): the warp
// copies them to shared memory with coalesced loads, every lane then ranks a share of the block's values
// inside their own bin by counting (ties broken by frame index, so exactly one value has each rank) and the
// values of rank (L-1)/2 and L/2 are published per bin.  NaN features are not supported (np.median would
// return NaN and warn).
#include "common.cuh"

namespace {

constexpr int ONRAMP_MAX_FAC = 128;   // raw frames per output frame this kernel stages in shared memory
constexpr int ONRAMP_WPC = 4;         // warps (output frames) per CTA

__global__ void __launch_bounds__(32 * ONRAMP_WPC) median_sync_kernel(const float *__restrict__ raw,
                                                                    const int64_t *__restrict__ raw_off,
                                                                    const int64_t *__restrict__ out_off,
                                                                    int n_tracks, int fac,
                                                                    float *__restrict__ out) {
    __shared__ float s_x[ONRAMP_WPC][ONRAMP_MAX_FAC * NBINS];
    __shared__ float s_sel[ONRAMP_WPC][2][NBINS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t f = (int64_t)blockIdx.x * ONRAMP_WPC + warp;      // global output frame
    if (f >= out_off[n_tracks]) return;
    // track of this output frame: last t with out_off[t] <= f
    int lo = 0, hi = n_tracks - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (out_off[mid] <= f) lo = mid; else hi = mid - 1;
    }
    const int t = lo;
    const int64_t k = f - out_off[t];
    const int64_t n_raw = raw_off[t + 1] - raw_off[t];
    const int L = (int)min((int64_t)fac, n_raw - k * fac);            // frames of this block (>= 1)
    const float *src = raw + (raw_off[t] + k * fac) * NBINS;
    float *x = s_x[warp];
    for (int i = lane; i < L * NBINS; i += 32) x[i] = __ldg(src + i);
    __syncwarp();
    const int r_lo = (L - 1) >> 1, r_hi = L >> 1;
    for (int i = lane; i < L * NBINS; i += 32) {
        const int r = i / NBINS, b = i - r * NBINS;
        const float v = x[i];
        int rank = 0;
        for (int r2 = 0; r2 < L; ++r2) {
            const float v2 = x[r2 * NBINS + b];
            rank += (v2 < v) || (v2 == v && r2 < r);
        }
        if (rank == r_lo) s_sel[warp][0][b] = v;
        if (rank == r_hi) s_sel[warp][1][b] = v;
    }
    __syncwarp();
    if (lane < NBINS) {
        const float a = s_sel[warp][0][lane], c = s_sel[warp][1][lane];
        out[f * NBINS + lane] = (r_lo == r_hi) ? a : __fmul_rn(__fadd_rn(a, c), 0.5f);
    }
}

// Mean pooling (the SiMPle on-ramp, simple_silva.py:38-41): output frame k of a track is the per-bin mean of raw
// frames [k*skip, min(k*skip + win, n)) as np.mean(X[a:b], axis=0) computes it on C-contiguous float32 data: a
// sequential float32 sum in frame order, then one float32 division by the frame count.  One warp per output frame,
// lanes 0..11 own the bins (one 48 B frame per step: coalesced).
__global__ void __launch_bounds__(32 * ONRAMP_WPC) mean_pool_kernel(const float *__restrict__ raw,
                                                                  const int64_t *__restrict__ raw_off,
                                                                  const int64_t *__restrict__ out_off,
                                                                  int n_tracks, int win, int skip,
                                                                  float *__restrict__ out) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t f = (int64_t)blockIdx.x * ONRAMP_WPC + warp;
    if (f >= out_off[n_tracks] || lane >= NBINS) return;
    int lo = 0, hi = n_tracks - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (out_off[mid] <= f) lo = mid; else hi = mid - 1;
    }
    const int64_t k = f - out_off[lo];
    const int64_t n_raw = raw_off[lo + 1] - raw_off[lo];
    const int64_t L = min((int64_t)win, n_raw - k * skip);
    const float *src = raw + (raw_off[lo] + k * skip) * NBINS + lane;
    float acc = 0.f;
    for (int64_t r = 0; r < L; ++r) acc = __fadd_rn(acc, __ldg(src + r * NBINS));
    out[f * NBINS + lane] = __fdiv_rn(acc, (float)L);
}

}  // namespace

int launch_mean_pool(const float *raw, const int64_t *raw_off, const int64_t *out_off, int n_tracks, int win, int skip,
                     int64_t total_out, float *out, cudaStream_t st) {
    if (total_out <= 0) return ACOSS_OK;
    const int64_t blocks = (total_out + ONRAMP_WPC - 1) / ONRAMP_WPC;
    mean_pool_kernel<<<(unsigned)blocks, 32 * ONRAMP_WPC, 0, st>>>(raw, raw_off, out_off, n_tracks, win, skip, out);
    CUDA_TRY(cudaGetLastError());
    return ACOSS_OK;
}

int onramp_max_fac() { return ONRAMP_MAX_FAC; }

// raw, raw_off, out_off, out: device pointers; out_off[n_tracks] output frames in total
int launch_median_sync(const float *raw, const int64_t *raw_off, const int64_t *out_off, int n_tracks, int fac,
                       int64_t total_out, float *out, cudaStream_t st) {
    if (total_out <= 0) return ACOSS_OK;
    if (fac < 1 || fac > ONRAMP_MAX_FAC) { acoss_set_error("downsample factor must be in 1..%d", ONRAMP_MAX_FAC); return ACOSS_E_INVALID; }
    const int64_t blocks = (total_out + ONRAMP_WPC - 1) / ONRAMP_WPC;
    median_sync_kernel<<<(unsigned)blocks, 32 * ONRAMP_WPC, 0, st>>>(raw, raw_off, out_off, n_tracks, fac, out);
    CUDA_TRY(cudaGetLastError());
    return ACOSS_OK;
}
