// EarlyFusion pair scoring on the device: cross-similarity matrices of the block features and the
// "early" similarity-network fusion of one pair.
//
// Replaces, per pair, the body of EarlyFusion.similarity
// (/root/reference/acoss/algorithms/earlyfusion_traile.py:157-198):
//   get_csm(X, Y)                          utils/cross_recurrence.py:31-48     (mfccs, ssms)
//   get_csm_blocked_oti(.., get_csm_cosine) utils/cross_recurrence.py:54-134   (chromas)
//   getWCSM(CSM, K, K)                     utils/similarity_fusion.py:38-54
//   exp(-sum of the three WCSMs)           earlyfusion_traile.py:178-182
// The binarisation (k4_knn.cu) and the Smith-Waterman DP (k3_dp.cu) consume the float64 matrices
// straight from HBM; nothing goes back to the host between the stages.
//
// Arithmetic: float64 throughout (the reference's numba/numpy code computes in the dtype of its
// inputs; its float32 features make BLAS-order-dependent float32 CSMs — the float64 value is the
// one every BLAS approximates, and it is what the pinned oracle computes).  These are genuine
// GEMMs (K = 480 / 1000 / 1225) but float64 ones, so tcgen05 (no float64 kind) does not apply; the
// float64 tensor path of sm_100a is the warp-level DMMA (ef_csm3_kernel: m8n8k4, 2x2 warps of 32x32,
// cp.async, 30.4 TFLOP/s).  It adds the k terms of a cell as an ascending-k FMA chain.  The two DFMA
// generations it replaced are described, with their measurements, in DESIGN.md §4.5.
#include <algorithm>

#include "common.cuh"

// ---------------------------------------------------------------------------------------------
// feature upload: [rows][d] (float32 or float64) -> [rows][dp] float64, zero padded to dp = 16 * ceil(d / 16)
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void ef_widen_kernel(const T *__restrict__ src, int64_t rows, int d, int dp, double *__restrict__ dst) {
    const int64_t total = rows * dp;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / dp;
        const int k = (int)(e - r * dp);
        dst[e] = k < d ? (double)src[r * d + k] : 0.0;
    }
}

// One warp per block row.  mode 0: sq[row] = sum x^2 (np.sum(X**2, 1), cross_recurrence.py:45).
// mode 1: row /= sqrt(sum x^2), zero norms replaced by 1 (cross_recurrence.py:67-71; the norm of a row is
// the same for every roll of its chroma groups, so normalising before the roll gives the same quotients).
__global__ void __launch_bounds__(256) ef_rownorm_kernel(double *__restrict__ feat, int64_t rows, int dp, int mode,
                                                         double *__restrict__ sq) {
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    double *x = feat + row * dp;
    double s = 0.0;
    for (int k = lane; k < dp; k += 32) s = fma(x[k], x[k], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (mode == 0) {
        if (lane == 0) sq[row] = s;
    } else {
        double nrm = sqrt(s);
        if (nrm == 0.0) nrm = 1.0;
        for (int k = lane; k < dp; k += 32) x[k] = x[k] / nrm;
    }
}

int launch_ef_widen(const void *src, int elem_size, int64_t rows, int d, int dp, double *dst, cudaStream_t st) {
    if (rows <= 0) return ACOSS_OK;
    const int64_t total = rows * dp;
    const int blocks = (int)std::min<int64_t>((total + 255) / 256, 148 * 16);
    if (elem_size == 4) ef_widen_kernel<float><<<blocks, 256, 0, st>>>((const float *)src, rows, d, dp, dst);
    else ef_widen_kernel<double><<<blocks, 256, 0, st>>>((const double *)src, rows, d, dp, dst);
    CUDA_TRY(cudaGetLastError());
    return ACOSS_OK;
}

int launch_ef_rownorm(double *feat, int64_t rows, int dp, int mode, double *sq, cudaStream_t st) {
    if (rows <= 0) return ACOSS_OK;
    ef_rownorm_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(feat, rows, dp, mode, sq);
    CUDA_TRY(cudaGetLastError());
    return ACOSS_OK;
}

// ---------------------------------------------------------------------------------------------
// OTI of the song-level chroma medians: argmax_i sum(roll(C1, i) * C2), first maximum
// (cross_recurrence.py:94-103).  The 12 products are added in the order numpy's pairwise sum uses
// for a contiguous 12-element array (8 running sums folded as a tree, then the 4 leftovers).
// ---------------------------------------------------------------------------------------------
__global__ void ef_oti_kernel(const double *__restrict__ cmed, const int32_t *__restrict__ pairs, int n,
                              int32_t *__restrict__ oti) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const double *c1 = cmed + (int64_t)pairs[2 * k] * NBINS;
    const double *c2 = cmed + (int64_t)pairs[2 * k + 1] * NBINS;
    double a[NBINS], b[NBINS];
#pragma unroll
    for (int t = 0; t < NBINS; ++t) { a[t] = c1[t]; b[t] = c2[t]; }
    int best = 0;
    double bestv = 0.0;
    for (int s = 0; s < NBINS; ++s) {
        double p[NBINS];
#pragma unroll
        for (int t = 0; t < NBINS; ++t) {
            int src = t - s;
            if (src < 0) src += NBINS;                       // np.roll(C1, s)[t] = C1[(t - s) mod 12]
            double av = a[0];
#pragma unroll
            for (int u = 1; u < NBINS; ++u) av = (u == src) ? a[u] : av;
            p[t] = __dmul_rn(av, b[t]);
        }
        double r = __dadd_rn(__dadd_rn(__dadd_rn(p[0], p[1]), __dadd_rn(p[2], p[3])),
                             __dadd_rn(__dadd_rn(p[4], p[5]), __dadd_rn(p[6], p[7])));
        r = __dadd_rn(r, p[8]); r = __dadd_rn(r, p[9]); r = __dadd_rn(r, p[10]); r = __dadd_rn(r, p[11]);
        if (s == 0 || r > bestv) { bestv = r; best = s; }
    }
    oti[k] = best;
}

int launch_ef_oti(const double *cmed, const int32_t *pairs, int n, int32_t *oti, cudaStream_t st) {
    if (n <= 0) return ACOSS_OK;
    ef_oti_kernel<<<(n + 127) / 128, 128, 0, st>>>(cmed, pairs, n, oti);
    CUDA_TRY(cudaGetLastError());
    return ACOSS_OK;
}

// ---------------------------------------------------------------------------------------------
// CSM: one 64x64 tile of one pair per CTA, on the float64 tensor path (DMMA, mma.sync.m8n8k4.f64 — tcgen05
// has no float64 kind; on sm_100a the legacy warp-level MMA is the only float64 tensor instruction).  One
// DMMA replaces 8 DFMA per lane and needs one A and one B double per lane: 2 x 2 warps of 32 x 32 (4 x 4
// MMA tiles, 32 accumulator doubles per lane), 8 LDS.64 per 16 DMMA.  Shared tiles are row-major [row][k]
// with a pitch of 20 doubles, so the 4 rows x 4 k a half-warp reads fall in 32 distinct banks.  Global ->
// shared goes through cp.async (16 B chunks, two-stage ring, no staging registers).
// ---------------------------------------------------------------------------------------------
#define EF_BM 64
#define EF_BN 64
#define EF_BK 16
#define EF3_LD 20
#define EF2_MAXDP 2048   // widest (padded) chroma block the rolled-column map covers
__device__ __forceinline__ void ef_cp_async16(void *smem, const void *g) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(g) : "memory");
}
__device__ __forceinline__ void ef_cp_async8(void *smem, const void *g) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(sa), "l"(g) : "memory");
}

__device__ __forceinline__ void ef_dmma(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// 16 k of one 32 x 32 warp quadrant, IMAX x JMAX of its 4 x 4 MMA tiles (compile-time bounds: the skipped
// tiles are not even issued — a predicated-off DMMA still takes its tensor-pipe slot)
template <int IMAX, int JMAX>
__device__ __forceinline__ void ef_quad_mma(const double *Ap, const double *Bp, double (&acc)[4][4][2]) {
#pragma unroll
    for (int k4 = 0; k4 < EF_BK; k4 += 4) {
        double a[IMAX], b[JMAX];
#pragma unroll
        for (int i = 0; i < IMAX; ++i) a[i] = Ap[i * 8 * EF3_LD + k4];
#pragma unroll
        for (int j = 0; j < JMAX; ++j) b[j] = Bp[j * 8 * EF3_LD + k4];
#pragma unroll
        for (int i = 0; i < IMAX; ++i)
#pragma unroll
            for (int j = 0; j < JMAX; ++j) ef_dmma(acc[i][j][0], acc[i][j][1], a[i], b[j]);
    }
}
template <int IMAX>
__device__ __forceinline__ void ef_quad_dispatch_j(int jmax, const double *Ap, const double *Bp, double (&acc)[4][4][2]) {
    switch (jmax) {
        case 4: ef_quad_mma<IMAX, 4>(Ap, Bp, acc); break;
        case 3: ef_quad_mma<IMAX, 3>(Ap, Bp, acc); break;
        case 2: ef_quad_mma<IMAX, 2>(Ap, Bp, acc); break;
        default: ef_quad_mma<IMAX, 1>(Ap, Bp, acc); break;
    }
}
__device__ __forceinline__ void ef_quad_dispatch(int imax, int jmax, const double *Ap, const double *Bp,
                                                 double (&acc)[4][4][2]) {
    switch (imax) {
        case 4: ef_quad_dispatch_j<4>(jmax, Ap, Bp, acc); break;
        case 3: ef_quad_dispatch_j<3>(jmax, Ap, Bp, acc); break;
        case 2: ef_quad_dispatch_j<2>(jmax, Ap, Bp, acc); break;
        default: ef_quad_dispatch_j<1>(jmax, Ap, Bp, acc); break;
    }
}

// MODE 0: sqrt(max(0, (|x|^2 + |y|^2) - 2 x.y)); MODE 1: 1 - xhat.yhat with the 12-bin groups of x rolled by oti.
// WIDE (MODE 1, dp > EF2_MAXDP): the gather computes each rolled source column instead of reading the column map.
template <int MODE, bool WIDE>
__global__ void __launch_bounds__(128) ef_csm3_kernel(const double *__restrict__ feat, int dp, int d,
                                                      const double *__restrict__ sq,
                                                      const int64_t *__restrict__ offsets,
                                                      const int32_t *__restrict__ pairs,
                                                      const int32_t *__restrict__ oti_a,
                                                      double *__restrict__ csm, int64_t slot_elems, int tiles_n) {
    __shared__ __align__(16) double As[2][EF_BM][EF3_LD];
    __shared__ __align__(16) double Bs[2][EF_BN][EF3_LD];
    __shared__ short kmap[MODE == 1 && !WIDE ? EF2_MAXDP : 1];
    const int slot = blockIdx.y;
    const int q = pairs[2 * slot], r = pairs[2 * slot + 1];
    const int64_t oq = offsets[q], orr = offsets[r];
    const int M = (int)(offsets[q + 1] - oq), N = (int)(offsets[r + 1] - orr);
    const int m0 = (blockIdx.x / tiles_n) * EF_BM, n0 = (blockIdx.x % tiles_n) * EF_BN;
    if (m0 >= M || n0 >= N) return;
    const int tid = threadIdx.x;
    const double *Abase = feat + oq * (int64_t)dp, *Bbase = feat + orr * (int64_t)dp;
    const int rot = MODE == 1 ? oti_a[slot] : 0;
    // np.roll(X1, oti, axis=2): out[b] = in[(b - oti) mod 12]
    auto rolled = [&](int k) {
        int src = k;
        if (k < d) {
            const int t = k / NBINS, b = k - t * NBINS;
            src = t * NBINS + rot_src(b, rot);
        }
        return src;
    };
    if (MODE == 1 && !WIDE) {
        for (int k = tid; k < dp; k += 128) kmap[k] = (short)rolled(k);
        __syncthreads();
    }
    auto issue = [&](int k0, int buf) {
        const int ch = tid & 7;
        if (MODE == 1) {
#pragma unroll 1
            for (int e = 0; e < 8; ++e) {                     // rolled chroma groups: element-wise gather
                const int id = tid + 128 * e, row = id >> 4, kk = id & 15;
                const int src = WIDE ? rolled(k0 + kk) : (int)kmap[k0 + kk];
                ef_cp_async8(&As[buf][row][kk], Abase + min(m0 + row, M - 1) * dp + src);
            }
        }
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
            const int row = (tid >> 3) + 16 * c;
            if (MODE == 0) ef_cp_async16(&As[buf][row][2 * ch], Abase + min(m0 + row, M - 1) * dp + k0 + 2 * ch);
            ef_cp_async16(&Bs[buf][row][2 * ch], Bbase + min(n0 + row, N - 1) * dp + k0 + 2 * ch);
        }
    };
    // warp (wr, wc) owns rows 32 wr .. +31 and columns 32 wc .. +31; MMA tile (rt, ct) of it: lane holds
    // C[8 rt + g][8 ct + 2 tg + {0,1}], reads A[8 rt + g][k + tg] and B[k + tg][8 ct + g]  (g = lane / 4, tg = lane % 4)
    const int lane = tid & 31, wr = (tid >> 5) >> 1, wc = (tid >> 5) & 1, g = lane >> 2, tg = lane & 3;
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    const bool warp_live = m0 + 32 * wr < M && n0 + 32 * wc < N;      // ragged edge tiles: idle quadrants only load
    const int imax = min(4, (M - m0 - 32 * wr + 7) >> 3), jmax = min(4, (N - n0 - 32 * wc + 7) >> 3);
    const int nt = dp / EF_BK;
    issue(0, 0);
    asm volatile("cp.async.commit_group;\n" ::: "memory");
    for (int t = 0; t < nt; ++t) {
        if (t + 1 < nt) issue((t + 1) * EF_BK, (t + 1) & 1);
        asm volatile("cp.async.commit_group;\n" ::: "memory");
        asm volatile("cp.async.wait_group 1;\n" ::: "memory");
        __syncthreads();
        if (warp_live) {
            const double *Ap = &As[t & 1][32 * wr + g][tg];
            const double *Bp = &Bs[t & 1][32 * wc + g][tg];
            ef_quad_dispatch(imax, jmax, Ap, Bp, acc);            // ragged edges: only the MMA tiles inside M x N
        }
        __syncthreads();
    }
    if (!warp_live) return;
    double *out = csm + (int64_t)slot * slot_elems;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int row = m0 + 32 * wr + 8 * i + g;
        if (row >= M) continue;
        const double sx = (MODE == 0) ? sq[oq + row] : 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int col = n0 + 32 * wc + 8 * j + 2 * tg + h;
                if (col >= N) continue;
                double v;
                if (MODE == 0) {
                    double c2 = __dsub_rn(__dadd_rn(sx, sq[orr + col]), __dmul_rn(2.0, acc[i][j][h]));
                    c2 = c2 < 0.0 ? 0.0 : c2;
                    v = sqrt(c2);
                } else {
                    v = __dsub_rn(1.0, acc[i][j][h]);
                }
                out[(int64_t)row * N + col] = v;
            }
    }
}

int launch_ef_csm(int mode, const double *feat, int dp, int d, const double *sq, const int64_t *offsets,
                  const int32_t *pairs, const int32_t *oti, int n, int max_rows, int max_cols, double *csm,
                  int64_t slot_elems, cudaStream_t st) {
    if (n <= 0) return ACOSS_OK;
    const int tiles_m = (max_rows + EF_BM - 1) / EF_BM, tiles_n = (max_cols + EF_BN - 1) / EF_BN;
    dim3 grid((unsigned)(tiles_m * tiles_n), (unsigned)n);
    static bool carve[16] = {false};                          // 40 KB static tiles per CTA: ask for the full carve-out
    int dev = 0;                                              // so that 5 CTAs fit an SM
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 16 && !carve[dev]) {
        cudaFuncSetAttribute(ef_csm3_kernel<0, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        cudaFuncSetAttribute(ef_csm3_kernel<1, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        cudaFuncSetAttribute(ef_csm3_kernel<1, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        carve[dev] = true;
    }
    if (mode == 0) ef_csm3_kernel<0, false><<<grid, 128, 0, st>>>(feat, dp, d, sq, offsets, pairs, oti, csm, slot_elems, tiles_n);
    else if (dp <= EF2_MAXDP) ef_csm3_kernel<1, false><<<grid, 128, 0, st>>>(feat, dp, d, sq, offsets, pairs, oti, csm, slot_elems, tiles_n);
    else ef_csm3_kernel<1, true><<<grid, 128, 0, st>>>(feat, dp, d, sq, offsets, pairs, oti, csm, slot_elems, tiles_n);
    CUDA_TRY(cudaGetLastError());
    return ACOSS_OK;
}

// ---------------------------------------------------------------------------------------------
// getWCSM neighbourhood radii: mean of the K smallest entries of every row and of every column
// (similarity_fusion.py:48-52).  One thread per line keeps the KMAX smallest values seen so far in a
// sorted register array (max/min insertion chain, no data-dependent indexing); which of several equal
// values is kept does not change the sum.  Line l < M is row l, line M + j is column j.
// ---------------------------------------------------------------------------------------------
template <int KMAX>
__global__ void __launch_bounds__(128) ef_linestat_kernel(const double *__restrict__ csm, int64_t kind_stride,
                                                          int64_t slot_elems, const int64_t *__restrict__ offsets,
                                                          const int32_t *__restrict__ pairs, int K,
                                                          double *__restrict__ stat, int64_t stat_kind_stride,
                                                          int stat_pitch) {
    const int slot = blockIdx.y, kind = blockIdx.z;
    const int q = pairs[2 * slot], r = pairs[2 * slot + 1];
    const int M = (int)(offsets[q + 1] - offsets[q]), N = (int)(offsets[r + 1] - offsets[r]);
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= M + N) return;
    const double *base = csm + kind * kind_stride + (int64_t)slot * slot_elems;
    const double *p;
    int len, stride;
    if (l < M) { p = base + (int64_t)l * N; len = N; stride = 1; }
    else { p = base + (l - M); len = M; stride = N; }
    double a[KMAX];
#pragma unroll
    for (int t = 0; t < KMAX; ++t) a[t] = __longlong_as_double(0x7ff0000000000000ll);
    // eight loads in flight per thread (the insertion branch would otherwise serialise the memory latency)
    for (int e0 = 0; e0 < len; e0 += 8) {
        double v8[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
            v8[u] = (e0 + u < len) ? p[(int64_t)(e0 + u) * stride] : __longlong_as_double(0x7ff0000000000000ll);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const double v = v8[u];
            if (v < a[KMAX - 1]) {
#pragma unroll
                for (int t = KMAX - 1; t > 0; --t) a[t] = fmax(a[t - 1], fmin(a[t], v));
                a[0] = fmin(a[0], v);
            }
        }
    }
    double s = 0.0;
#pragma unroll
    for (int t = 0; t < KMAX; ++t)
        if (t < K) s = __dadd_rn(s, a[t]);
    stat[kind * stat_kind_stride + (int64_t)slot * stat_pitch + l] = s / (double)K;
}

int ef_linestat_max_k() { return 64; }

int launch_ef_linestat(const double *csm, int64_t kind_stride, int64_t slot_elems, const int64_t *offsets,
                       const int32_t *pairs, int n, int max_rows, int max_cols, int K, double *stat,
                       int64_t stat_kind_stride, int stat_pitch, cudaStream_t st) {
    if (n <= 0) return ACOSS_OK;
    dim3 grid((unsigned)((max_rows + max_cols + 127) / 128), (unsigned)n, 3);
    if (K <= 16)
        ef_linestat_kernel<16><<<grid, 128, 0, st>>>(csm, kind_stride, slot_elems, offsets, pairs, K, stat,
                                                     stat_kind_stride, stat_pitch);
    else
        ef_linestat_kernel<64><<<grid, 128, 0, st>>>(csm, kind_stride, slot_elems, offsets, pairs, K, stat,
                                                     stat_kind_stride, stat_pitch);
    CUDA_TRY(cudaGetLastError());
    return ACOSS_OK;
}

// ---------------------------------------------------------------------------------------------
// early fusion: out = exp(-(W_mfccs + W_ssms + W_chromas)), W = exp(-d^2 / (2 (Mu Eps)^2)),
// Eps = ((rowmean + colmean) + d) / 3, Mu = 0.5   (similarity_fusion.py:52-54, earlyfusion_traile.py:178-182;
// same operation order, no contraction across the reference's separate numpy operations)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ef_fuse_kernel(const double *__restrict__ csm, int64_t kind_stride,
                                                      int64_t slot_elems, const int64_t *__restrict__ offsets,
                                                      const int32_t *__restrict__ pairs,
                                                      const double *__restrict__ stat, int64_t stat_kind_stride,
                                                      int stat_pitch, double mu, double *__restrict__ out) {
    const int slot = blockIdx.y;
    const int q = pairs[2 * slot], r = pairs[2 * slot + 1];
    const int M = (int)(offsets[q + 1] - offsets[q]), N = (int)(offsets[r + 1] - offsets[r]);
    const int64_t cells = (int64_t)M * N;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < cells; e += (int64_t)gridDim.x * blockDim.x) {
        const int i = (int)(e / N), j = (int)(e - (int64_t)i * N);
        double total = 0.0;
#pragma unroll
        for (int kind = 0; kind < 3; ++kind) {
            const double dd = csm[kind * kind_stride + (int64_t)slot * slot_elems + e];
            const double *st = stat + kind * stat_kind_stride + (int64_t)slot * stat_pitch;
            const double eps = __ddiv_rn(__dadd_rn(__dadd_rn(st[i], st[M + j]), dd), 3.0);
            const double me = __dmul_rn(mu, eps);
            const double den = __dmul_rn(2.0, __dmul_rn(me, me));
            const double w = exp(__ddiv_rn(-__dmul_rn(dd, dd), den));
            total = __dadd_rn(total, w);
        }
        out[(int64_t)slot * slot_elems + e] = exp(-total);
    }
}

int launch_ef_fuse(const double *csm, int64_t kind_stride, int64_t slot_elems, const int64_t *offsets,
                   const int32_t *pairs, int n, int max_rows, int max_cols, const double *stat,
                   int64_t stat_kind_stride, int stat_pitch, double *out, cudaStream_t st) {
    if (n <= 0) return ACOSS_OK;
    const int64_t cells = (int64_t)max_rows * max_cols;
    dim3 grid((unsigned)std::min<int64_t>((cells + 1023) / 1024, 4096), (unsigned)n);
    ef_fuse_kernel<<<grid, 256, 0, st>>>(csm, kind_stride, slot_elems, offsets, pairs, stat, stat_kind_stride,
                                         stat_pitch, 0.5, out);
    CUDA_TRY(cudaGetLastError());
    return ACOSS_OK;
}

// per-slot shapes, neighbour counts and CSM offsets for the k-NN kernel (cross_recurrence.py:151-155 rule:
// kappa == 0 -> all ones (-1), kappa < 1 -> int(np.round(kappa * columns)), else kappa)
__global__ void ef_geom_kernel(const int64_t *__restrict__ offsets, const int32_t *__restrict__ pairs, int n,
                               double kappa, int64_t slot_elems, int32_t *__restrict__ shapes,
                               int32_t *__restrict__ nn, int64_t *__restrict__ csm_off) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int q = pairs[2 * k], r = pairs[2 * k + 1];
    const int M = (int)(offsets[q + 1] - offsets[q]), N = (int)(offsets[r + 1] - offsets[r]);
    shapes[2 * k] = M;
    shapes[2 * k + 1] = N;
    int v;
    if (kappa == 0.0) v = -1;
    else if (kappa < 1.0) v = (int)rint(__dmul_rn(kappa, (double)N));      // np.round: half to even
    else v = (int)kappa;
    nn[k] = v;
    csm_off[k] = (int64_t)k * slot_elems;
}

int launch_ef_geom(const int64_t *offsets, const int32_t *pairs, int n, double kappa, int64_t slot_elems,
                   int32_t *shapes, int32_t *nn, int64_t *csm_off, cudaStream_t st) {
    if (n <= 0) return ACOSS_OK;
    ef_geom_kernel<<<(n + 127) / 128, 128, 0, st>>>(offsets, pairs, n, kappa, slot_elems, shapes, nn, csm_off);
    CUDA_TRY(cudaGetLastError());
    return ACOSS_OK;
}
