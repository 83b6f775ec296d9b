// K6 — SiMPle pair scoring: OTI, matrix-profile join, median of the profile.
//
// Replaces Simple.similarity (acoss/algorithms/simple_silva.py:17-126): per pair the SiMPle join
// (simple_sim, :68-118, FFT sliding dot products on the CPU) of the query's length-m subsequences against the
// reference's, and the median of the resulting matrix profile.  Restated from Silva, Yeh, Batista, Keogh (ISMIR 2016);
// parity is unpinned against the reference and pinned against that restatement (oracle/simple_np.py, DESIGN.md §2
// switches S1-S5):
//   oti    = first argmax_s sum_b g_A[b] * g_B[(b - s) mod 12] (S4 = 0: the reference is rolled by oti) or
//            first argmax_s sum_b g_A[(b - s) mod 12] * g_B[b]  (S4 = 1: the query is rolled by oti), g = the float64
//            sequential frame sum of a track, products and sums rounded one by one
//   d2(i,j)= sum_{t<m} sum_b (A[i+t][b] - B[j+t][b])^2 in float64, sequential over t then b, no contraction
//   P[i]   = min_j d(i,j), d = sqrt(d2) (S2 = 1: d2);  I[i] = lowest j attaining it
//   score  = float32(-median(P)) (S3 = 1: +median), median = (a + b) / 2 of the two middle values when even
//
// One CTA per pair, four phases separated by __syncthreads:
//   0  stage: both tracks (the rolled one rolled) are copied to the pair's workspace slot; per-pair fixed-point scale.
//   1  filter sweep: each lane walks one diagonal j - i = d; the frame item e = sum_b (a_b - b_b)^2 (float32) is
//      quantised to u = rint(e * 2^k) and the m-tap box sum along the diagonal is an exact uint32 (a sliding sum
//      over a shared-memory ring of the last m items).  All lanes of a warp sit in the same row i at every step, so
//      the row minimum is a warp min plus one atomicMin per warp and row.
//   2  the same sweep again lists every cell whose box sum is within the error bound of its row minimum (up to
//      SIMPLE_CAND per row; a row with more is re-evaluated over all of its j).
//   3  exact float64 evaluation of the listed cells (or of whole rows), lexicographic min (d, j) per row.
//   4  median: rank of each profile value by counting (ties by index), the two middle ranks.
//
// Why the filter is exact.  Let Y be the box sum in fixed-point units, X the float64 d2 and E = sum of the real frame
// items.  |e32 - e| <= 14 u32 e + (underflow) per item, quantisation adds <= 1/2 unit per item, and the float64 sum
// is within (12 m + 2) u64 X of E.  Hence |X - Y| <= R (Y + c) + c with R = 2^-19, c = m units.  Any j attaining the
// minimum of X (or of sqrt(X), which merges values within 2 ulps) then has Y(j) <= ((Ymin + 2c)(1 + R'))/(1 - R') with
// R' = 2^-17 > R + 2^-51, which is the candidate threshold.  DESIGN.md §4.6 has the derivation.
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace {

constexpr int SIMPLE_THREADS = 256;
constexpr int SIMPLE_WARPS = SIMPLE_THREADS / 32;

__device__ __forceinline__ float frame_item(const float4 *a, const float4 *b) {
    const float4 a0 = a[0], a1 = a[1], a2 = a[2], b0 = b[0], b1 = b[1], b2 = b[2];
    const float x[12] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w, a2.x, a2.y, a2.z, a2.w};
    const float y[12] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w, b2.x, b2.y, b2.z, b2.w};
    float e = 0.f;
#pragma unroll
    for (int k = 0; k < NBINS; ++k) {
        const float d = __fsub_rn(x[k], y[k]);
        e = __fmaf_rn(d, d, e);
    }
    return e;
}

// float64 d2 of cell (i, j) in the order of the definition
__device__ __forceinline__ double exact_d2(const float *A, const float *B, int i, int j, int m) {
    double acc = 0.0;
    const float *a = A + (int64_t)i * NBINS, *b = B + (int64_t)j * NBINS;
    for (int t = 0; t < m * NBINS; ++t) {
        const double d = __dsub_rn((double)a[t], (double)b[t]);
        acc = __dadd_rn(acc, __dmul_rn(d, d));
    }
    return acc;
}

// One filter sweep over the pair.  pass 0: row minima into thr[]; pass 1: list the cells with box sum <= thr[i].
template <int PASS>
__device__ void sweep(const float4 *A4, const float4 *B4, int na, int nb, int m, float scale, uint32_t *ring,
                      uint32_t *thr, int32_t *cnt, int32_t *cand) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int La = na - m + 1, Lb = nb - m + 1;
    const int ndiag = La + Lb - 1;
    uint32_t *my_ring = ring + threadIdx.x;
    for (int g = warp; g * 32 < ndiag; g += SIMPLE_WARPS) {
        const int d0 = g * 32 - (La - 1);                 // first diagonal of the group
        const int d = d0 + lane;
        const bool dvalid = d <= Lb - 1;
        const int f_lo = max(0, -min(d0 + 31, Lb - 1));   // first A frame any lane of the group touches
        const int f_hi = min(na, nb - d0);                // one past the last
        const int my_lo = max(0, -d);
        const int my_hi = dvalid ? min(na, nb - d) : 0;
        for (int s = 0; s < m; ++s) my_ring[s * SIMPLE_THREADS] = 0u;
        uint32_t sum = 0u;
        int pos = 0;
        for (int f = f_lo; f < f_hi; ++f) {
            const bool fv = f >= my_lo && f < my_hi;
            uint32_t u = 0u;
            if (fv) u = __float2uint_rn(frame_item(A4 + 3 * f, B4 + 3 * (f + d)) * scale);
            const uint32_t old = my_ring[pos * SIMPLE_THREADS];
            my_ring[pos * SIMPLE_THREADS] = u;
            sum += u - old;
            pos = (pos + 1 == m) ? 0 : pos + 1;
            const int i = f - m + 1;                      // the row every lane of the warp is in
            if (i < 0) continue;
            const bool cell = fv && i >= my_lo;
            if (PASS == 0) {
                const uint32_t mn = __reduce_min_sync(0xffffffffu, cell ? sum : 0xffffffffu);
                // no cell of this warp in row i gives 0xffffffff: real box sums stay below 2^32 - 1 (choice of scale)
                if (lane == 0 && mn != 0xffffffffu) atomicMin(thr + i, mn);
            } else {
                const bool hit = cell && sum <= thr[i];
                const unsigned bal = __ballot_sync(0xffffffffu, hit);
                if (bal) {
                    int base = 0;
                    if (lane == 0) base = atomicAdd(cnt + i, __popc(bal));
                    base = __shfl_sync(0xffffffffu, base, 0);
                    const int slot = base + __popc(bal & ((1u << lane) - 1u));
                    if (hit && slot < SIMPLE_CAND) cand[(int64_t)i * SIMPLE_CAND + slot] = i + d;
                }
            }
        }
    }
}

__global__ void __launch_bounds__(SIMPLE_THREADS) simple_pair_kernel(SimpleArgs a) {
    extern __shared__ uint32_t s_ring[];                  // [m][SIMPLE_THREADS]
    __shared__ double s_g[2][NBINS];
    __shared__ double s_nrm[2][SIMPLE_WARPS];
    __shared__ double s_mid[2];
    __shared__ int s_oti;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t p = a.first + blockIdx.x;
    const int slot = blockIdx.x;
    const int q = a.pairs[2 * p], r = a.pairs[2 * p + 1];
    const int64_t oq = a.offsets[q], orr = a.offsets[r];
    const int na = (int)(a.offsets[q + 1] - oq), nb = (int)(a.offsets[r + 1] - orr);
    const int m = a.m, La = na - m + 1, Lb = nb - m + 1;
    const float *Aq = a.frames + oq * NBINS, *Br = a.frames + orr * NBINS;

    // ---- phase 0: OTI, staging, scale
    if (tid < 2 * NBINS) {                                // per-track float64 sequential frame sums
        const int side = tid / NBINS, b = tid % NBINS;
        const float *src = side ? Br : Aq;
        const int n = side ? nb : na;
        double g = 0.0;
        if (a.oti)
            for (int f = 0; f < n; ++f) g = __dadd_rn(g, (double)src[(int64_t)f * NBINS + b]);
        s_g[side][b] = g;
    }
    __syncthreads();
    if (tid == 0) {
        int best_s = 0;
        double best = -INFINITY;
        if (a.oti) {
            for (int s = 0; s < NBINS; ++s) {
                double acc = 0.0;
                for (int b = 0; b < NBINS; ++b) {
                    const int k = rot_src(b, s);
                    acc = __dadd_rn(acc, a.s4_roll_first ? __dmul_rn(s_g[0][k], s_g[1][b]) : __dmul_rn(s_g[0][b], s_g[1][k]));
                }
                if (acc > best) { best = acc; best_s = s; }
            }
        }
        s_oti = best_s;
        if (a.oti_out) a.oti_out[p] = best_s;
    }
    __syncthreads();
    const int oti = s_oti;
    float *A = a.stage + (int64_t)slot * a.stage_pitch;   // query frames, rolled by oti under S4 = 1
    float *B = A + (int64_t)a.max_frames * NBINS;         // reference frames, rolled by oti under S4 = 0
    const int rot_a = a.s4_roll_first ? oti : 0, rot_b = a.s4_roll_first ? 0 : oti;
    double nmax[2] = {0.0, 0.0};
    for (int side = 0; side < 2; ++side) {
        const float *src = side ? Br : Aq;
        float *dst = side ? B : A;
        const int n = side ? nb : na, rot = side ? rot_b : rot_a;
        for (int f = tid; f < n; f += SIMPLE_THREADS) {
            double n2 = 0.0;
#pragma unroll
            for (int b = 0; b < NBINS; ++b) {
                const float v = src[(int64_t)f * NBINS + rot_src(b, rot)];
                dst[(int64_t)f * NBINS + b] = v;
                n2 = fma((double)v, (double)v, n2);
            }
            nmax[side] = fmax(nmax[side], n2);
        }
    }
    for (int o = 16; o >= 1; o >>= 1) {
        nmax[0] = fmax(nmax[0], __shfl_xor_sync(0xffffffffu, nmax[0], o));
        nmax[1] = fmax(nmax[1], __shfl_xor_sync(0xffffffffu, nmax[1], o));
    }
    if (lane == 0) { s_nrm[0][warp] = nmax[0]; s_nrm[1][warp] = nmax[1]; }
    uint32_t *thr = a.thr + (int64_t)slot * a.row_pitch;
    int32_t *cnt = a.cnt + (int64_t)slot * a.row_pitch;
    int32_t *cand = a.cand + (int64_t)slot * a.row_pitch * SIMPLE_CAND;
    double *prof = a.prof + (int64_t)slot * a.row_pitch;
    int32_t *idx = a.idx + (int64_t)slot * a.row_pitch;
    for (int i = tid; i < La; i += SIMPLE_THREADS) { thr[i] = 0xffffffffu; cnt[i] = 0; }
    __syncthreads();
    double na2 = 0.0, nb2 = 0.0;
    for (int w = 0; w < SIMPLE_WARPS; ++w) { na2 = fmax(na2, s_nrm[0][w]); nb2 = fmax(nb2, s_nrm[1][w]); }
    // every frame item e <= (|a| + |b|)^2; the margin covers the float32 rounding of e and of the norms
    const double emax = (sqrt(na2) + sqrt(nb2)) * (sqrt(na2) + sqrt(nb2)) * (1.0 + 1.0 / 1024);
    // Too large for float32 items (or not finite): every row is evaluated exactly
    const bool all_exact = !(emax < 0x1p100);
    int k = 64;
    if (emax > 0.0 && !all_exact) k = min(64, (int)floor(log2((4294967295.0 / m - 2.0) / emax)));
    const float scale = ldexpf(1.f, k);

    // ---- phases 1 and 2: filter sweeps
    const float4 *A4 = reinterpret_cast<const float4 *>(A), *B4 = reinterpret_cast<const float4 *>(B);
    if (!all_exact) {
        sweep<0>(A4, B4, na, nb, m, scale, s_ring, thr, cnt, cand);
        __syncthreads();
        const double R = 0x1p-17, c = (double)m;
        for (int i = tid; i < La; i += SIMPLE_THREADS) {
            const double t = floor(((double)thr[i] + 2.0 * c) * (1.0 + R) / (1.0 - R)) + 1.0;
            thr[i] = t >= 4294967295.0 ? 0xffffffffu : (uint32_t)t;
        }
        __syncthreads();
        sweep<1>(A4, B4, na, nb, m, scale, s_ring, thr, cnt, cand);
    } else {
        for (int i = tid; i < La; i += SIMPLE_THREADS) cnt[i] = SIMPLE_CAND + 1;
    }
    __syncthreads();

    // ---- phase 3: exact evaluation, one warp per row
    for (int i = warp; i < La; i += SIMPLE_WARPS) {
        const int c = cnt[i];
        double best = INFINITY;
        int bj = 0x7fffffff;
        if (c <= SIMPLE_CAND) {
            if (lane < c) {
                bj = cand[(int64_t)i * SIMPLE_CAND + lane];
                best = exact_d2(A, B, i, bj, m);
            }
        } else {
            for (int j = lane; j < Lb; j += 32) {
                const double v = exact_d2(A, B, i, j, m);
                if (v < best) { best = v; bj = j; }          // j ascending per lane: strict < keeps the lowest
            }
        }
        if (!a.s2_squared && bj != 0x7fffffff) best = __dsqrt_rn(best);
        for (int o = 16; o >= 1; o >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
            if (ob < best || (ob == best && oj < bj)) { best = ob; bj = oj; }
        }
        if (lane == 0) { prof[i] = best; idx[i] = bj; }
    }
    __syncthreads();

    // ---- phase 4: median of prof[0 .. La)
    const int r_lo = (La - 1) >> 1, r_hi = La >> 1;
    for (int i = tid; i < La; i += SIMPLE_THREADS) {
        const double v = prof[i];
        int rank = 0;
        for (int l = 0; l < La; ++l) {
            const double w = prof[l];
            rank += (w < v) || (w == v && l < i);
        }
        if (rank == r_lo) s_mid[0] = v;
        if (rank == r_hi) s_mid[1] = v;
    }
    __syncthreads();
    if (tid == 0) {
        const double med = (r_lo == r_hi) ? s_mid[0] : __ddiv_rn(__dadd_rn(s_mid[0], s_mid[1]), 2.0);
        a.scores[p] = (float)(a.s3_positive ? med : -med);
    }
}

}  // namespace

size_t simple_slot_bytes(int max_frames, int m) {
    const int64_t rows = std::max(1, max_frames - m + 1);
    return (size_t)2 * max_frames * NBINS * 4 + (size_t)rows * (4 + 4 + 8 + 4 + 4 * SIMPLE_CAND);
}

int launch_simple_pairs(const SimpleArgs &args, int n, cudaStream_t st) {
    if (n <= 0) return ACOSS_OK;
    const size_t smem = (size_t)args.m * SIMPLE_THREADS * 4;
    CUDA_TRY(cudaFuncSetAttribute(simple_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    simple_pair_kernel<<<n, SIMPLE_THREADS, smem, st>>>(args);
    CUDA_TRY(cudaGetLastError());
    return ACOSS_OK;
}
