/* acoss_b200 — C ABI of the B200-native all-pairs cover-song scoring hot path.
 *
 * Drop-in boundary.  The reference (furkanyesiler/acoss) has no FFI of its own: its hot path is
 * the body of a Python plugin method that calls two essentia C++ algorithms per pair,
 *     acoss/algorithms/rqa_serra09.py:55-69        Serra09.similarity(idxs)
 *     acoss/algorithms/rqa_serra09.py:60-67        ChromaCrossSimilarity(...)(query, reference)
 *                                                  CoverSongSimilarity('serra09','symmetric')(csm)
 * and, for the EarlyFusion flavour, the in-tree numba kernels
 *     acoss/algorithms/utils/alignment_tools.py:26-46     smith_waterman_constrained(B)
 *     acoss/algorithms/utils/cross_recurrence.py:76-103   get_oti(C1, C2)
 *     acoss/algorithms/utils/cross_recurrence.py:137-161  csm_to_binary(D, kappa)
 * Each entry point below names the reference interface it replaces.  A maintainer binds them
 * with ctypes (see INTEGRATION.md); acoss_b200/_lib.py is that binding.
 *
 * Conventions: extern "C"; plain pointers and sizes; every function returns 0 on success or a
 * negative ACOSS_E_* code, with a human-readable message available from acoss_last_error()
 * (thread-local).  No exceptions cross the ABI.  One context per device; a context is not
 * thread-safe.  There is NO CPU fallback: every entry point fails with ACOSS_E_CUDA when no
 * sm_100-class device is usable.
 */
#ifndef ACOSS_B200_H
#define ACOSS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACOSS_OK 0
#define ACOSS_E_INVALID (-1)    /* bad argument                                                    */
#define ACOSS_E_CUDA (-2)       /* CUDA runtime error / no device                                  */
#define ACOSS_E_TOO_SHORT (-3)  /* a track has fewer than m*tau+2 frames (essentia throws; F9)     */
#define ACOSS_E_NAN (-4)        /* a squared distance was negative -> NaN (essentia: non-binary)   */
#define ACOSS_E_NONBINARY (-5)  /* DP input holds values other than 0/1 (reference: IOError)       */
#define ACOSS_E_NOMEM (-6)      /* device memory exhausted                                         */

#define ACOSS_NBINS 12          /* chroma bins per HPCP frame (rqa_serra09.py: 12-bin HPCP)        */

/* alignment recurrences (acoss_params.align / acoss_dp_* mode) */
#define ACOSS_ALIGN_QMAX 0      /* essentia CoverSongSimilarity alignmentType='serra09'            */
#define ACOSS_ALIGN_SW 1        /* alignment_tools.py:26-46 smith_waterman_constrained             */
#define ACOSS_ALIGN_DMAX 2      /* essentia alignmentType='chen17' (latefusion_chen.py:69-71)      */
#define ACOSS_ALIGN_DMAX_PLAIN 3 /* F10 switch: Dmax without Chen's bridging terms                 */

/* CRP construction path (acoss_params.crp_path) */
#define ACOSS_CRP_AUTO 0        /* fast sweep kernels, exact per-pair fallback when a check fails  */
#define ACOSS_CRP_EXACT 1       /* exact reference-order kernels only (slow; debugging / fallback) */

typedef struct acoss_ctx acoss_ctx;

/* Parameters of Serra09.__init__ (rqa_serra09.py:31-32) + essentia defaults (SURVEY App. A). */
typedef struct acoss_params {
    int32_t m;              /* frameStackSize, 9                                                   */
    int32_t tau;            /* frameStackStride, 1                                                 */
    float kappa;            /* binarizePercentile, 0.095                                           */
    int32_t oti;            /* 1: transpose the reference by the optimal transposition index       */
    int32_t noti;           /* 12                                                                  */
    float gamma_o;          /* disOnset, 0.5                                                       */
    float gamma_e;          /* disExtension, 0.5                                                   */
    int32_t align;          /* ACOSS_ALIGN_QMAX (Serra09), ACOSS_ALIGN_DMAX (ChenFusion) or        */
                            /* ACOSS_ALIGN_SW: smith_waterman_constrained over the same CRP        */
    int32_t integer_guard;  /* F1 switch: 0 = essentia behaviour (integer rank -> threshold 0)     */
    int32_t crp_path;       /* ACOSS_CRP_AUTO / ACOSS_CRP_EXACT                                    */
    /* Switches for the points where the restatement of essentia is uncertain (SURVEY.md App. A F2-F5;    */
    /* the oracle carries the same switches).  All 0 = the App. A defaults.  Pairs scored with F2-F4 set   */
    /* take the exact CRP path (the fast path's bounds are derived for the defaults).                      */
    int32_t f2_strict;      /* F2: 1 = heaviside(x) = 1 iff x > 0 (d == threshold is NOT similar)          */
    int32_t f3_float_acc;   /* F3: 1 = dotProduct accumulates in float32 (init 0.f) instead of float64      */
    int32_t f4_keep_last;   /* F4: 1 = n - (m-1)*tau stacked frames (the natural count) instead of n - m*tau */
    int32_t f5_asymmetric;  /* F5: 1 = distanceType 'asymmetric': score = sqrt(N') / max(Q)                  */
} acoss_params;

/* Fills *p with the reference defaults (m=9, tau=1, kappa=0.095, oti=1, noti=12, 0.5, 0.5, Qmax). */
void acoss_default_params(acoss_params *p);

const char *acoss_last_error(void);
/* Library version string, and the sm target the kernels were compiled for (100). */
const char *acoss_version(void);
int acoss_compiled_sm(void);

/* Context on CUDA device `device` (its primary context; torch tensors of the same device can be
 * passed as raw pointers). */
int acoss_create(acoss_ctx **ctx, int device);
int acoss_destroy(acoss_ctx *ctx);
/* Upper bound, in bytes, of per-call scratch the context may allocate (default 24 GiB). */
int acoss_set_workspace_limit(acoss_ctx *ctx, int64_t bytes);

/* Replaces the per-process feature cache Serra09.all_feats / load_features (rqa_serra09.py:44-53):
 * uploads (or adopts, when frames_on_device != 0 — the pointer must stay valid) all tracks'
 * post-downsampling HPCP frames, concatenated: frames[(offsets[t] + f) * 12 + bin], float32;
 * offsets has n_tracks + 1 entries (host memory).  Precomputes the per-track global chroma. */
int acoss_set_tracks(acoss_ctx *ctx, const float *frames, const int64_t *offsets, int32_t n_tracks,
                     int frames_on_device);

/* The same from RAW (not yet downsampled) chroma features: replaces the median aggregation of
 * Serra09.load_features (rqa_serra09.py:47-53, librosa.util.sync with aggregate=np.median): output frame k
 * of a track is the per-bin median of raw frames [fac*k, min(fac*k+fac, n)), float32, computed on the GPU,
 * and the downsampled tracks become the resident set.  raw_frames / raw_offsets: host memory, layout as
 * above.  offsets_out (may be NULL, n_tracks + 1 entries) receives the downsampled offsets.  fac in 1..128. */
int acoss_set_tracks_raw(acoss_ctx *ctx, const float *raw_frames, const int64_t *raw_offsets, int32_t n_tracks,
                         int32_t downsample_fac, int64_t *offsets_out);
/* Copies the resident (post-downsampling) frames back to the host: total_frames * 12 floats. */
int acoss_get_tracks(acoss_ctx *ctx, float *frames_out, int64_t total_frames);

/* Replaces Serra09.similarity(idxs) (rqa_serra09.py:55-69) for a whole batch: pairs[2k] = query
 * track, pairs[2k+1] = reference track; scores[k] = the float the reference stores in
 * Ds[key][i][j].  Host buffers; H2D of the pair list and D2H of the scores happen inside. */
int acoss_score_pairs(acoss_ctx *ctx, const int32_t *pairs, int64_t n_pairs, const acoss_params *p,
                      float *scores);
/* Same with DEVICE buffers (pairs and scores in HBM), asynchronous on the context's stream: the call enqueues all
 * its work and returns without a host synchronisation; acoss_sync() waits for it.  Pairs the fast CRP path flags
 * (a consistency check failed) are re-scored by the exact path inside the same enqueued work, up to 4 x 16 of them
 * per call; if a call flags more, acoss_sync() scores the remainder before it returns, so scores_dev is complete
 * after acoss_sync() in every case.  Used for device-resident timing and for NCCL hand-off. */
int acoss_score_pairs_device(acoss_ctx *ctx, const int32_t *pairs_dev, int64_t n_pairs,
                             const acoss_params *p, float *scores_dev);
int acoss_sync(acoss_ctx *ctx);
/* Returns the context's CUDA stream (a cudaStream_t) so callers can record events on it. */
void *acoss_stream(acoss_ctx *ctx);

/* Replaces ChenFusion.similarity(idxs) (latefusion_chen.py:58-73) for a whole batch: the same CRP per
 * pair feeds both alignments; qmax_scores[k] / dmax_scores[k] are the floats the reference stores in
 * Ds["qmax"][i][j] / Ds["dmax"][i][j].  p->align is ignored.  Host buffers. */
int acoss_score_pairs_chen(acoss_ctx *ctx, const int32_t *pairs, int64_t n_pairs, const acoss_params *p,
                           float *qmax_scores, float *dmax_scores);
/* Same with DEVICE buffers (pairs, qmax_dev and dmax_dev in HBM), asynchronous on the context's stream like
 * acoss_score_pairs_device: the call enqueues all its work and returns without a host synchronisation; acoss_sync()
 * waits for it.  Flagged pairs are re-scored by the exact path for both alignments, inside the enqueued work up to
 * 4 x 16 of them and the remainder inside acoss_sync(), so both outputs are complete after acoss_sync().  p->align is
 * ignored.  Used for device-resident timing and for NCCL hand-off. */
int acoss_score_pairs_chen_device(acoss_ctx *ctx, const int32_t *pairs_dev, int64_t n_pairs, const acoss_params *p,
                                  float *qmax_dev, float *dmax_dev);

/* K1 only — essentia optimalTranspositionIndex (inside ChromaCrossSimilarity, App. A1). */
int acoss_oti_pairs(acoss_ctx *ctx, const int32_t *pairs, int64_t n_pairs, int32_t noti, int32_t *oti);

/* Debug dump of one pair (query track q, reference track r): OTI, bit-packed CRP
 * (rows = n_q - m*tau, words_per_row = ceil((n_r - m*tau)/32), bit b of word w = column 32w+b),
 * thresholds and the alignment score.  Any output pointer may be NULL.  Host buffers. */
int acoss_dump_pair(acoss_ctx *ctx, int32_t q, int32_t r, const acoss_params *p, int32_t *oti,
                    uint32_t *crp_bits, float *thr_q, float *thr_r, float *score);

/* K3 only — batched alignment DP over caller-supplied binary matrices (uint8, row-major, back to
 * back: matrix k starts at mats[offsets[k]], shape (shapes[2k], shapes[2k+1])).  Host buffers.
 *   ACOSS_ALIGN_SW   replaces smith_waterman_constrained(B) (alignment_tools.py:26-46)
 *   ACOSS_ALIGN_QMAX replaces CoverSongSimilarity('serra09','symmetric')(csm)[1]
 *   ACOSS_ALIGN_DMAX replaces CoverSongSimilarity('chen17','symmetric')(csm)[1]
 * Non-binary input -> ACOSS_E_NONBINARY (reference raises IOError / EssentiaException). */
int acoss_dp_bytes(acoss_ctx *ctx, const uint8_t *mats, const int64_t *offsets, const int32_t *shapes,
                   int64_t n_mats, int32_t mode, float gamma_o, float gamma_e, float *scores);

/* Row-only k-NN binarisation + SW of caller-supplied float64 CSMs — replaces
 * smith_waterman_constrained(csm_to_binary(D, kappa)) (earlyfusion_traile.py:168,171,175,183).
 * nn[k] = neighbours per row for matrix k (cross_recurrence.py:151-155 rule, computed by the
 * host).  bits_out (may be NULL) receives the bit-packed binary matrices back to back
 * (rows * ceil(cols/32) words each).  Ties at the nn-th value: lowest column index first. */
int acoss_knn_sw(acoss_ctx *ctx, const double *csms, const int64_t *offsets, const int32_t *shapes,
                 const int32_t *nn, int64_t n_mats, float *scores, uint32_t *bits_out);

/* ---- EarlyFusion pair scoring (earlyfusion_traile.py:157-198) ------------------------------------------
 * Replaces the per-process block-feature cache EarlyFusion.all_block_feats / load_features
 * (earlyfusion_traile.py:66-155): uploads every track's beat-synchronous block features, concatenated over
 * tracks: mfccs[(offsets[t] + b) * d_mfccs + k] etc., offsets in BLOCKS (n_tracks + 1 entries, all three kinds
 * have the same number of blocks per track), chroma_med[t * 12 + bin] = the song-level chroma median
 * (float64).  elem_size: 4 = float32 features (what the reference stores), 8 = float64.  Host memory.  The
 * device keeps float64 copies (chroma blocks pre-normalised for the cosine CSM) and the squared norms. */
int acoss_ef_set_tracks(acoss_ctx *ctx, const void *mfccs, int32_t d_mfccs, const void *ssms, int32_t d_ssms,
                        const void *chromas, int32_t d_chromas, const double *chroma_med, const int64_t *offsets,
                        int32_t n_tracks, int32_t elem_size);

/* Replaces EarlyFusion.similarity(idxs) (earlyfusion_traile.py:157-198) for a whole batch: per pair
 * (pairs[2k] = first song i, pairs[2k+1] = second song j) the Euclidean CSMs of the mfcc and ssm blocks
 * (get_csm, cross_recurrence.py:31-48), the blocked-OTI cosine CSM of the chroma blocks
 * (get_csm_blocked_oti / get_csm_cosine, :54-134), exp(-sum of getWCSM(CSM, K, K)) (similarity_fusion.py:38-54),
 * and smith_waterman_constrained(csm_to_binary(., kappa)) of all four.  scores is [4][n_pairs] float32, kind-major:
 * mfccs, ssms, chromas, early — the values the reference stores in Ds[kind][i][j].  kappa as in
 * csm_to_binary (0: all ones, < 1: fraction of the columns, else a count); K in 1..64 and smaller than the
 * block count of every track involved (np.partition raises otherwise: ACOSS_E_INVALID).  Host buffers. */
int acoss_ef_score_pairs(acoss_ctx *ctx, const int32_t *pairs, int64_t n_pairs, double kappa, int32_t K,
                         float *scores);

/* Debug dump of one pair (M = blocks of q, N = blocks of r): OTI, the four float64 matrices [4][M * N]
 * (mfccs, ssms, chromas CSMs and the fused matrix), their binarisations [4][M * ceil(N / 32)] bit-packed, and
 * the four scores.  Any output pointer may be NULL.  Host buffers. */
int acoss_ef_dump_pair(acoss_ctx *ctx, int32_t q, int32_t r, double kappa, int32_t K, int32_t *oti, double *csms,
                       uint32_t *bits, float *scores);

/* ---- Simple (SiMPle) pair scoring (simple_silva.py:17-126) ----------------------------------------------------
 * Parity is unpinned against the reference and pinned against the restatement of DESIGN.md §2 (switches S1-S5),
 * which oracle/simple_np.py implements. */

/* Replaces the mean pooling of Simple.load_features (simple_silva.py:38-41): pooled frame k of a track is the
 * per-bin mean of raw frames [k*skip, k*skip + win) (a sequential float32 sum, one float32 division: np.mean on
 * float32), computed on the GPU; the pooled tracks become the resident set and acoss_get_tracks reads them back.
 * keep_partial = 0 (S5 default): only full windows, (n - win)/skip + 1 frames, and a track with n < win is
 * ACOSS_E_TOO_SHORT.  keep_partial = 1: one more, shorter window [k*skip, n) covers a tail the full windows miss (a
 * track with 1 <= n <= win gives one frame).  raw_frames / raw_offsets: host memory, layout of acoss_set_tracks.
 * offsets_out (may be NULL, n_tracks + 1 entries) receives the pooled offsets.  win, skip in 1..65536. */
int acoss_set_tracks_pooled(acoss_ctx *ctx, const float *raw_frames, const int64_t *raw_offsets, int32_t n_tracks,
                            int32_t win, int32_t skip, int32_t keep_partial, int64_t *offsets_out);

typedef struct acoss_simple_params {
    int32_t m;              /* S1: subsequence length in pooled frames, 10 (unconfirmed against the reference); 1..128 */
    int32_t oti;            /* 1: transpose by the optimal transposition index (simple_silva.py:45-54)                  */
    int32_t s2_squared;     /* S2: 1 = the profile keeps squared distances (default 0: d = sqrt(d2))                   */
    int32_t s3_positive;    /* S3: 1 = score = +median (default 0: -median, so that higher means more similar)         */
    int32_t s4_roll_first;  /* S4: 1 = the query is rolled, oti = argmax <roll(g_q, s), g_r> (get_oti); default 0 rolls */
                            /*     the reference, oti = argmax <g_q, roll(g_r, s)> (essentia)                             */
} acoss_simple_params;

/* Fills *p with the defaults: m = 10, oti = 1, S2 = S3 = S4 = 0. */
void acoss_simple_default_params(acoss_simple_params *p);

/* Replaces Simple.similarity(idxs) for a whole batch: scores[k] = the float stored in Ds["main"][q][r] for
 * pairs[2k] = q (query), pairs[2k+1] = r.  Host buffers.  ACOSS_E_TOO_SHORT when a resident track has fewer than m
 * frames, ACOSS_E_INVALID for m outside 1..128. */
int acoss_simple_score_pairs(acoss_ctx *ctx, const int32_t *pairs, int64_t n_pairs, const acoss_simple_params *p,
                             float *scores);
/* Same with DEVICE buffers, asynchronous on the context's stream (no host synchronisation); acoss_sync() waits. */
int acoss_simple_score_pairs_device(acoss_ctx *ctx, const int32_t *pairs_dev, int64_t n_pairs,
                                    const acoss_simple_params *p, float *scores_dev);
/* Debug dump of one pair: OTI, the float64 matrix profile and its index (n_q - m + 1 entries each) and the score.
 * Any output pointer may be NULL.  Host buffers. */
int acoss_simple_dump_pair(acoss_ctx *ctx, int32_t q, int32_t r, const acoss_simple_params *p, int32_t *oti,
                           double *profile, int32_t *index, float *score);

/* ---- Similarity-network fusion (similarity_fusion.py, doSimilarityFusion) ------------------------------------------
 * The late fusion of ChenFusion.do_late_fusion (latefusion_chen.py:87-91: Ds["Late"]) and EarlyFusion.do_late_fusion
 * (earlyfusion_traile.py:200-206: Ds["late"], Ds["early+late"]) over the finished N x N score matrices. */
#define ACOSS_SNF_MAX_K 63      /* neighbours K of getS / getW (the plugins use 20)                                  */
#define ACOSS_SNF_MAX_MATS 16   /* score matrices per fusion                                                         */

/* Replaces doSimilarityFusion(D, K, niters, reg_diag, reg_neighbs) (similarity_fusion.py: getW, getP, getS,
 * doSimilarityFusionWs).  D[m] (m < n_mats) are row-major n x n float32 host matrices; fused (n x n float64, host)
 * receives the fused matrix.  getW: DSym = 0.5 (D + D^T) with a zero diagonal, MeanDist = mean of the K+1 smallest
 * DSym of the row * (K+1) / K, W = exp(-DSym^2 / (2 (0.5 Eps)^2)), Eps = (MeanDist_r + MeanDist_c + DSym) / 3, in
 * float32 and numpy's operation order (the K+1 smallest are added in ascending order).  getP: W / numpy's pairwise
 * float32 row sum.  getS: the K largest W of each row (ties: lowest column; NaN after +inf as in np.argpartition),
 * normalised by their sum and stored in ascending column order.  Diffusion: niters iterations of, for i in order,
 * Pts[i] = S_i ((nextPts[i] * 0 + sum_{k != i} Pts[k]) / (n_mats - 1)) S_i^T + reg_diag I (if reg_diag > 0)
 * + reg_neighbs on |r - c| == 1 (if reg_neighbs > 0), float64, each sparse product in stored-slot order with separate
 * roundings (scipy csr_matvecs).  jacobi = 0 (switch L1 default) is the reference's `Pts = nextPts` aliasing: the
 * first iteration reads the float32 P of every matrix, later ones read the Pts[k] already updated in the same
 * iteration for k < i; jacobi = 1 reads the previous iteration's Pts for every k.  fused = (sum of Pts) / n_mats.
 * W (n_mats x n x n float32), P (same), S_idx (n_mats x n x K int32) and S_val (same, float32) may be NULL; they
 * receive the affinities, the transition matrices and the neighbour lists.  ACOSS_E_INVALID for n_mats outside
 * 2..ACOSS_SNF_MAX_MATS (the reference divides by n_mats - 1 and returns NaN for one matrix), K outside
 * 1..ACOSS_SNF_MAX_K, K + 1 >= n (np.partition raises), n > 65535 or niters < 0; ACOSS_E_NOMEM when the device
 * workspace, n_mats n^2 (4 + 8 * (1 + jacobi)) + 16 n^2 bytes, exceeds the workspace limit.  Host buffers. */
int acoss_snf(acoss_ctx *ctx, const float *const *D, int32_t n_mats, int32_t n, int32_t K, int32_t niters,
              double reg_diag, double reg_neighbs, int32_t jacobi, double *fused, float *W, float *P, int32_t *S_idx,
              float *S_val);
/* Device milliseconds of the fusion stages since acoss_set_profiling(ctx, 1): [0] H2D of the score matrices,
 * [1] affinity (DSym, W, P, S), [2] diffusion, [3] the final average and the D2H of the fused matrix. */
int acoss_snf_stage_ms(acoss_ctx *ctx, double ms[4]);

/* Device milliseconds of the EarlyFusion stages since acoss_set_profiling(ctx, 1): [0] CSM contractions,
 * [1] k-NN binarisation, [2] Smith-Waterman DP, [3] getWCSM row/column radii, [4] fusion (exp) pass. */
int acoss_ef_stage_ms(acoss_ctx *ctx, double ms[5]);
/* Counters of the last acoss_ef_score_pairs call: [0] pairs, [1] cells (sum of M * N), [2] kernel launches,
 * [3] slot chunks. */
int acoss_ef_last_stats(acoss_ctx *ctx, int64_t stats[4]);

/* Counters of the last acoss_score_pairs* call: [0] pairs, [1] pairs that took the exact
 * fallback, [2] kernel launches, [3] cells (sum of M'*N'), [4] exact re-evaluated candidate cells, [5] OR of the
 * per-pair status words, [6] slot chunks the call was processed in (= launches of each K2 / K3 kernel). */
int acoss_last_stats(acoss_ctx *ctx, int64_t stats[8]);

/* Diagnostic counters of the last acoss_score_pairs* call (valid after acoss_sync).  Dense histogram
 * level, columns out[0..3] and rows out[4..7]: strips that swept, live lines on entry, lines whose wanted
 * ranks fell outside the sampled bracket, lines handed to the sparse refinement.  Sparse refinement
 * out[8..10]: warps, sweeps, lines still crowded at the end.  out[12..15] / out[16..19]: the same four
 * counters for the second (gated) dense level, columns / rows.  out[24] uncertain cells the emit sweep
 * listed, out[25] candidate cells evaluated exactly, out[26] listed cells whose coarse item the scatter kernel recomputed
 * (tensor-core sweeps: cells within dz below a line's bracket). */
int acoss_debug_counters(acoss_ctx *ctx, int64_t out[32]);

/* Per-stage device timing of the pair pipeline, measured with CUDA events on the context stream:
 * acoss_set_profiling(ctx, 1) resets and enables it; acoss_stage_ms returns the accumulated
 * milliseconds of [0] K1 OTI, [1] K2 CRP construction, [2] K3 alignment DP, [3] the emit sweep alone
 * (fast_emit_kernel, the dominant kernel of K2; part of [1]). */
int acoss_set_profiling(acoss_ctx *ctx, int on);
int acoss_stage_ms(acoss_ctx *ctx, double ms[4]);
/* Device milliseconds of every kernel of the fast K2 path since acoss_set_profiling(ctx, 1) (CUDA events around each
 * launch): [0] prep, [1] diagonal sampler, [2] sample selection, [3] / [4] dense histogram sweep columns / rows,
 * [5] / [6] the gated second level, [7] sparse refinement, [8] emit sweep, [9] candidate scatter, [10] candidate
 * ranking (z order statistics, window cells), [11] candidate bits, [12] exact evaluation of the window cells,
 * [13] thresholds; [14..15] reserved (0). */
int acoss_kernel_ms(acoss_ctx *ctx, double ms[16]);

#ifdef __cplusplus
}
#endif
#endif /* ACOSS_B200_H */
