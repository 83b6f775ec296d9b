// Shared declarations for the acoss_b200 CUDA library (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <vector>

#include "../../include/acoss_b200.h"

#define NBINS ACOSS_NBINS

// ---------------------------------------------------------------------------------------------
// error plumbing (thread-local message, no exceptions across the ABI)
// ---------------------------------------------------------------------------------------------
void acoss_set_error(const char *fmt, ...);

#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) {                                                                \
            acoss_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return (_e == cudaErrorMemoryAllocation) ? ACOSS_E_NOMEM : ACOSS_E_CUDA;            \
        }                                                                                       \
    } while (0)

// ---------------------------------------------------------------------------------------------
// Device-side description of the resident track set (HBM layout, see DESIGN.md §3)
// ---------------------------------------------------------------------------------------------
struct TrackSet {
    const float *frames;      // [total_frames][12] float32, 48 B per frame (16 B aligned)
    const int64_t *offsets;   // [n_tracks + 1] first frame of each track
    const float *gchroma;     // [n_tracks][12] global chroma: sequential f32 frame sum / max (App. A1)
    int32_t n_tracks;
    int32_t max_frames;
    int32_t fx_exp;           // fast path fixed point: 2 * <frame, frame> < 2^fx_exp for every frame pair
    int32_t nonneg;           // 1 when every feature value is >= 0 (HPCP); the fast path requires it
    int32_t q_exp;            // tensor sweeps: features are quantised as rint(x * 2^q_exp) < 2^24 (three byte limbs); < 0: unavailable
};

// Per-pair status bits written by the kernels
#define PAIR_ST_NAN 1u        // a NaN distance was produced (F7)
#define PAIR_ST_FALLBACK 2u   // the fast CRP path failed a consistency check; exact path re-ran it

// One work slot of the pair pipeline (fixed pitch so no device-side scan is needed)
struct SlotGeom {
    int32_t max_rows;     // max M' over the call
    int32_t max_cols;     // max N' over the call
    int32_t words;        // CRP row pitch in 32-bit words (ceil(max_cols/32) + 1 pad word)
    int64_t crp_words;    // words per slot = max_rows * words
};

// ---------------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int rot_src(int b, int s) {   // rotR(x, s)[b] = x[(b - s) mod 12]
    int k = b - s;
    return k < 0 ? k + NBINS : k;
}

// essentia dotProduct arithmetic (App. A3, F3): float32 product (one rounding), sequential
// float64 accumulate.  __fmul_rn / __dadd_rn block FMA contraction.
__device__ __forceinline__ double acc_f32prod(double acc, float a, float b) {
    return __dadd_rn(acc, (double)__fmul_rn(a, b));
}

// Optional per-kernel timing hook of the K2 fast path (api.cu records CUDA events on the context stream)
#define K2K_PREP 0
#define K2K_SAMPLE 1
#define K2K_SELECT 2
#define K2K_HIST_COL 3
#define K2K_HIST_ROW 4
#define K2K_HIST_COL2 5
#define K2K_HIST_ROW2 6
#define K2K_SPARSE 7
#define K2K_EMIT 8
#define K2K_SCATTER 9
#define K2K_THR 10
#define K2K_BITS 11
#define K2K_EXACT 12
#define K2K_FINAL 13
#define K2K_COUNT 14
struct KernelTimer {
    virtual void begin(int id) = 0;
    virtual void end(int id) = 0;
};

// F3 switch: the same with a float32 accumulator (std::inner_product(..., 0.f)); the accumulator variable stays a
// double that always holds a float32 value
__device__ __forceinline__ double acc_f32prod_f32(double acc, float a, float b) {
    return (double)__fadd_rn((float)acc, __fmul_rn(a, b));
}

// host launchers (one per translation unit) -----------------------------------------------------
struct Params;   // fwd

int onramp_max_fac();
int launch_median_sync(const float *raw, const int64_t *raw_off, const int64_t *out_off, int n_tracks, int fac,
                       int64_t total_out, float *out, cudaStream_t st);
int launch_global_chroma(const float *frames, const int64_t *offsets, int n_tracks, float *gchroma,
                         cudaStream_t st);
int launch_frame_stats(const float *frames, int64_t total_frames, float *stats2, cudaStream_t st);
int launch_oti(const TrackSet &ts, const int32_t *pairs, int64_t n_pairs, int noti, int apply,
               int32_t *oti_out, cudaStream_t st);

// K2 exact path: CRP bits + thresholds for `n` pairs (pairs[first..first+n)) into slots 0..n-1
struct ExactScratch {
    float *rrot;     // [slots][max_frames][12] rotated reference frames
    float *aa;       // [slots][max_rows]
    float *bb;       // [slots][max_cols]
    float *D;        // [slots][max_rows][ldd] float32 distances
    int64_t ldd;
    int32_t slots;
};
int launch_k2_exact(const TrackSet &ts, const int32_t *pairs, const int32_t *oti, int64_t first, int n,
                    const acoss_params &p, const SlotGeom &g, const ExactScratch &sc,
                    uint32_t *crp, float *thr_q, float *thr_r, uint32_t *status,
                    const int32_t *slot_pair_map, cudaStream_t st, int64_t *launches, bool out_by_slot = false);

// K3: alignment DP over bit-packed matrices.  rows[k], cols[k] give the DP matrix of slot k.
int launch_dp_bits(const uint32_t *bits, int64_t slot_words, int words_per_row, const int32_t *rows,
                   const int32_t *cols, int n, int max_cols, int mode, float gamma_o, float gamma_e,
                   float *scores, uint32_t *halo_scratch, int64_t halo_pitch, cudaStream_t st,
                   int64_t *launches);
// pair geometry (rows = n_q - m*tau, cols = n_r - m*tau) for pairs[first..first+n)
int launch_pair_geometry(const TrackSet &ts, const int32_t *pairs, int64_t first, int n, int incr,
                         int32_t *rows, int32_t *cols, cudaStream_t st);
// F5 switch: scores[k] = sqrtf(cols[k]) / scores[k] (essentia distanceType 'asymmetric', App. A6)
int launch_score_asymmetric(float *scores, const int32_t *cols, int n, cudaStream_t st);
// the same for mapped pairs: slot k scores pair map[k]; map[k] < 0 -> rows = cols = 0 (the DP returns at once)
int launch_pair_geometry_map(const TrackSet &ts, const int32_t *pairs, const int32_t *map, int n, int incr,
                             int32_t *rows, int32_t *cols, cudaStream_t st);
// dst[map[k]] = src[k] for map[k] >= 0
int launch_scatter_scores(const float *src, const int32_t *map, int n, float *dst, cudaStream_t st);
int launch_sw_trim(uint32_t *bits, int64_t slot_words, int words_per_row, int32_t *rows, int32_t *cols, int n,
                   cudaStream_t st);
int launch_pack_bytes(const uint8_t *mats, const int64_t *offsets, const int32_t *shapes, int n,
                      int mode, uint32_t *bits, int64_t slot_words, int words_per_row,
                      int32_t *rows, int32_t *cols, uint32_t *nonbinary_flag, cudaStream_t st);
int launch_knn_rows(const double *csms, const int64_t *offsets, const int32_t *shapes, const int32_t *nn, int n,
                    int max_rows, int max_cols, uint32_t *bits_dp, int64_t slot_words, int wpr, uint32_t *bits_out,
                    const int64_t *out_offsets, int32_t *rows, int32_t *cols, cudaStream_t st);

// K0: mean pooling of raw frames (the SiMPle on-ramp): out frame k of a track = mean of raw frames
// [k*skip, min(k*skip + win, n)), sequential float32 sum, one float32 division
int launch_mean_pool(const float *raw, const int64_t *raw_off, const int64_t *out_off, int n_tracks, int win, int skip,
                     int64_t total_out, float *out, cudaStream_t st);

// K6: SiMPle pair scoring (k6_simple.cu), one CTA per pair of pairs[first .. first + n) in workspace slots 0 .. n-1
#define SIMPLE_CAND 32        // listed candidate cells per profile row; a row with more is evaluated over all j
struct SimpleArgs {
    const float *frames;      // resident track set
    const int64_t *offsets;
    const int32_t *pairs;     // device, absolute pair indices
    int64_t first;
    int32_t m, oti, s2_squared, s3_positive, s4_roll_first;
    int32_t max_frames;
    float *stage;             // [slot][2][max_frames][12] both tracks of the pair, rolled
    int64_t stage_pitch;      // floats per slot
    uint32_t *thr;            // [slot][row_pitch] row minima, then candidate thresholds (fixed point)
    int32_t *cnt;             // [slot][row_pitch] candidates per row
    int32_t *cand;            // [slot][row_pitch][SIMPLE_CAND] candidate columns
    double *prof;             // [slot][row_pitch] matrix profile
    int32_t *idx;             // [slot][row_pitch] profile index
    int64_t row_pitch;
    float *scores;            // [pair]
    int32_t *oti_out;         // [pair] or NULL
};
size_t simple_slot_bytes(int max_frames, int m);
int launch_simple_pairs(const SimpleArgs &args, int n, cudaStream_t st);

// EarlyFusion stages (k5_earlyfusion.cu)
int launch_ef_widen(const void *src, int elem_size, int64_t rows, int d, int dp, double *dst, cudaStream_t st);
int launch_ef_rownorm(double *feat, int64_t rows, int dp, int mode, double *sq, cudaStream_t st);
int launch_ef_oti(const double *cmed, const int32_t *pairs, int n, int32_t *oti, cudaStream_t st);
int launch_ef_geom(const int64_t *offsets, const int32_t *pairs, int n, double kappa, int64_t slot_elems,
                   int32_t *shapes, int32_t *nn, int64_t *csm_off, cudaStream_t st);
int launch_ef_csm(int mode, const double *feat, int dp, int d, const double *sq, const int64_t *offsets,
                  const int32_t *pairs, const int32_t *oti, int n, int max_rows, int max_cols, double *csm,
                  int64_t slot_elems, cudaStream_t st);
int ef_linestat_max_k();
int launch_ef_linestat(const double *csm, int64_t kind_stride, int64_t slot_elems, const int64_t *offsets,
                       const int32_t *pairs, int n, int max_rows, int max_cols, int K, double *stat,
                       int64_t stat_kind_stride, int stat_pitch, cudaStream_t st);
int launch_ef_fuse(const double *csm, int64_t kind_stride, int64_t slot_elems, const int64_t *offsets,
                   const int32_t *pairs, int n, int max_rows, int max_cols, const double *stat,
                   int64_t stat_kind_stride, int stat_pitch, double *out, cudaStream_t st);

// K7: similarity-network fusion (k7_snf.cu).  Leaf boundaries of numpy's pairwise sum over n elements (n_leaves + 1
// entries); the affinity stages of one matrix (d: the scores, dw: DSym, then W, in place; md: MeanDist); one diffusion
// input written transposed; S . Y (transposed output, or the regularised row-major one); the final average.
std::vector<int32_t> snf_leaf_offsets(int n);
int launch_snf_affinity(const float *d, int n, int K, float *dw, float *md, const int32_t *leaf_off, int n_leaves,
                        float *P, int32_t *s_idx, float *s_val, cudaStream_t st);
int launch_snf_mix(const void *const *src, int nsrc, bool f32, const double *prev, int n, double den, double *xt,
                   cudaStream_t st);
int launch_snf_spmm(const double *Y, const int32_t *s_idx, const float *s_val, int n, int K, bool transposed,
                    double reg_diag, double reg_neighbs, double *out, cudaStream_t st);
int launch_snf_average(const void *const *src, int nsrc, bool f32, int64_t cells, double *out, cudaStream_t st);
