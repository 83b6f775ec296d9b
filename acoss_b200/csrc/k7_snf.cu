// K7: similarity-network fusion of finished N x N score matrices (acoss/algorithms/utils/similarity_fusion.py:
// getW, getP, getS, doSimilarityFusionWs), the late fusion of ChenFusion (latefusion_chen.py:87-91) and EarlyFusion
// (earlyfusion_traile.py:200-206).  The affinity stages repeat the reference's float32 numpy operations in their
// order; the diffusion repeats scipy's csr_matvecs in float64 (y += a * x per stored slot, multiply and add rounded
// separately).  DESIGN.md §4.7.
#include <algorithm>
#include <vector>

#include "common.cuh"

namespace {

constexpr int SNF_WARPS = 8;     // rows per CTA of the row kernels: one warp per row
constexpr int SP_BR = 32;        // SpMM output tile: 32 rows x 128 columns, 256 threads
constexpr int SP_BC = 128;
constexpr int SP_KMAX = 64;

template <typename T>
struct SnfSrc {                  // matrices summed element-wise, in this order
    const T *p[ACOSS_SNF_MAX_MATS];
    int n;
};

// numpy's sort order of float32 (NaN after +inf, -0 == +0) as an unsigned key
__device__ __forceinline__ uint32_t sort_key(float x) {
    if (x != x) return 0xffffffffu;
    const uint32_t b = (x == 0.0f) ? 0u : __float_as_uint(x);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// numpy's pairwise float32 sum (loops_utils.h.src, pairwise_sum) of a[0..n), n <= 128: below 8 elements a running
// sum from -0; otherwise 8 strided accumulators folded as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the rest in order
__device__ float np_sum_leaf(const float *a, int n) {
    if (n < 8) {
        float s = -0.0f;
        for (int i = 0; i < n; ++i) s = __fadd_rn(s, a[i]);
        return s;
    }
    float r[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) r[u] = a[u];
    int i = 8;
    for (; i < n - (n % 8); i += 8)
#pragma unroll
        for (int u = 0; u < 8; ++u) r[u] = __fadd_rn(r[u], a[i + u]);
    float s = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                        __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
    for (; i < n; ++i) s = __fadd_rn(s, a[i]);
    return s;
}

// The tree of numpy's pairwise sum above 128 elements, pw(n) = pw(n2) + pw(n - n2) with n2 = n/2 rounded down to a
// multiple of 8, over leaf sums given left to right (snf_leaf_offsets builds the same split on the host)
__device__ float np_sum_tree(int n, const float *leaf) {
    struct Frame { int n, n2; float left; bool right; };
    Frame st[32];
    int sp = 0, li = 0;
    for (;;) {
        while (n > 128) {
            int n2 = n / 2;
            n2 -= n2 % 8;
            st[sp++] = {n, n2, 0.0f, false};
            n = n2;
        }
        float v = leaf[li++];
        while (sp > 0 && st[sp - 1].right) v = __fadd_rn(st[--sp].left, v);
        if (sp == 0) return v;
        st[sp - 1].left = v;
        st[sp - 1].right = true;
        n = st[sp - 1].n - st[sp - 1].n2;
    }
}

// The ksel smallest (sort_key(v), column) pairs of a row, v = row[c] (largest = false) or -row[c] (largest = true), in
// ascending order into out[0..ksel): NaN last either way, equal values by lowest column (the keys are unique).  Each
// lane keeps the ksel smallest keys of its columns c = lane + 32i in a sorted register array with the insertion chain
// of ef_linestat_kernel (k5_earlyfusion.cu), here on 64-bit keys; the KMAX - ksel front slots hold 0 so that
// a[KMAX - 1] is the lane's ksel-th key.  ksel rounds of a warp minimum then merge the 32 lists.
template <int KMAX>
__device__ void warp_select(const float *__restrict__ row, int n, bool largest, int ksel, uint64_t *out) {
    const int lane = threadIdx.x & 31;
    uint64_t a[KMAX];
#pragma unroll
    for (int t = 0; t < KMAX; ++t) a[t] = t < KMAX - ksel ? 0ull : ~0ull;
    for (int c0 = lane; c0 < n; c0 += 256) {
        float v8[8];                                   // eight loads in flight before the insertion branches
#pragma unroll
        for (int u = 0; u < 8; ++u) v8[u] = c0 + 32 * u < n ? row[c0 + 32 * u] : 0.0f;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int c = c0 + 32 * u;
            const uint64_t k = ((uint64_t)sort_key(largest ? -v8[u] : v8[u]) << 32) | (uint32_t)c;
            if (c < n && k < a[KMAX - 1]) {
#pragma unroll
                for (int t = KMAX - 1; t > 0; --t) a[t] = max(a[t - 1], min(a[t], k));
                a[0] = min(a[0], k);
            }
        }
    }
#pragma unroll
    for (int t = 0; t < KMAX; ++t) a[t] = a[t] == 0ull ? ~0ull : a[t];
    for (int s = 0; s < ksel; ++s) {
        uint64_t m = a[0];
#pragma unroll
        for (int t = 1; t < KMAX; ++t) m = min(m, a[t]);
#pragma unroll
        for (int o = 16; o; o >>= 1) m = min(m, (uint64_t)__shfl_xor_sync(0xffffffffu, (unsigned long long)m, o));
#pragma unroll
        for (int t = 0; t < KMAX; ++t) a[t] = a[t] == m ? ~0ull : a[t];
        if (lane == 0) out[s] = m;
    }
    __syncwarp();
}

// getW, DSym = 0.5 * (D + D.T) with a zero diagonal (fill_diagonal), through a transposed 32 x 32 tile
__global__ void __launch_bounds__(256) snf_dsym_kernel(const float *__restrict__ D, int n, float *__restrict__ out) {
    __shared__ float tile[32][33];
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
    for (int j = threadIdx.y; j < 32; j += 8) {       // tile[j][x] = D[c0 + j][r0 + x]
        const int rr = c0 + j, cc = r0 + threadIdx.x;
        if (rr < n && cc < n) tile[j][threadIdx.x] = D[(int64_t)rr * n + cc];
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int r = r0 + j, c = c0 + threadIdx.x;
        if (r < n && c < n)
            out[(int64_t)r * n + c] = r == c ? 0.0f : __fmul_rn(0.5f, __fadd_rn(D[(int64_t)r * n + c], tile[threadIdx.x][j]));
    }
}

// getW, MeanDist = mean(partition(DSym, K+1, 1)[:, :K+1], 1) * float(K+1) / float(K).  The K+1 smallest values are
// added in ascending order (the reference adds them in introselect's order, which cannot be reproduced).
template <int KMAX>
__global__ void __launch_bounds__(SNF_WARPS * 32) snf_meandist_kernel(const float *__restrict__ dsym, int n, int K,
                                                                       float *__restrict__ md) {
    __shared__ uint64_t key[SNF_WARPS][KMAX];
    __shared__ float val[SNF_WARPS][KMAX];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * SNF_WARPS + w;
    if (r >= n) return;
    const float *row = dsym + (int64_t)r * n;
    warp_select<KMAX>(row, n, false, K + 1, key[w]);
    for (int s = lane; s <= K; s += 32) val[w][s] = row[(uint32_t)key[w][s]];
    __syncwarp();
    if (lane == 0) {
        const float mean = __fdiv_rn(__fadd_rn(0.0f, np_sum_leaf(val[w], K + 1)), (float)(K + 1));
        md[r] = __fdiv_rn(__fmul_rn(mean, (float)(K + 1)), (float)K);
    }
}

// getW, in place over DSym: Eps = (MeanDist[r] + MeanDist[c] + DSym) / 3, Denom = 2 * (0.5 * Eps)**2 (0 -> 1),
// W = exp(-DSym**2 / Denom), every step a separate float32 operation as numpy performs it
__global__ void __launch_bounds__(256) snf_w_kernel(float *__restrict__ dw, const float *__restrict__ md, int n) {
    const int r = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    const int64_t e = (int64_t)r * n + c;
    const float d = dw[e];
    const float eps = __fdiv_rn(__fadd_rn(__fadd_rn(md[r], md[c]), d), 3.0f);
    const float me = __fmul_rn(0.5f, eps);
    float den = __fmul_rn(2.0f, __fmul_rn(me, me));
    if (den == 0.0f) den = 1.0f;
    dw[e] = expf(__fdiv_rn(-__fmul_rn(d, d), den));
}

// getP and getS of one row per warp.  getS: the K largest W of the row (argpartition(-W, K)), stored in ascending
// column order (the CSR row coo_matrix.tocsr() builds) with values W / (0 + their pairwise sum in that order), a zero
// sum replaced by 1.  getP: W / (0 + numpy's pairwise row sum), a zero sum replaced by 1; the lanes sum the leaves.
template <int KMAX>
__global__ void __launch_bounds__(SNF_WARPS * 32) snf_rows_kernel(const float *__restrict__ W, int n, int K,
                                                                   const int32_t *__restrict__ leaf_off, int n_leaves,
                                                                   float *__restrict__ P, int32_t *__restrict__ s_idx,
                                                                   float *__restrict__ s_val) {
    extern __shared__ float leafsum[];               // [SNF_WARPS][n_leaves]
    __shared__ uint64_t key[SNF_WARPS][KMAX];
    __shared__ int32_t col[SNF_WARPS][KMAX];
    __shared__ float val[SNF_WARPS][KMAX];
    __shared__ float dv[SNF_WARPS][2];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * SNF_WARPS + w;
    if (r >= n) return;
    const float *row = W + (int64_t)r * n;
    warp_select<KMAX>(row, n, true, K, key[w]);
    for (int s = lane; s < K; s += 32) {
        const int cs = (int)(uint32_t)key[w][s];
        int rank = 0;
        for (int u = 0; u < K; ++u) rank += (int)(uint32_t)key[w][u] < cs;
        col[w][rank] = cs;
        val[w][rank] = row[cs];
    }
    float *ls = leafsum + w * n_leaves;
    for (int l = lane; l < n_leaves; l += 32) ls[l] = np_sum_leaf(row + leaf_off[l], leaf_off[l + 1] - leaf_off[l]);
    __syncwarp();
    if (lane == 0) {
        const float vs = __fadd_rn(0.0f, np_sum_leaf(val[w], K));
        const float rs = __fadd_rn(0.0f, np_sum_tree(n, ls));
        dv[w][0] = vs == 0.0f ? 1.0f : vs;
        dv[w][1] = rs == 0.0f ? 1.0f : rs;
    }
    __syncwarp();
    for (int s = lane; s < K; s += 32) {
        s_idx[(int64_t)r * K + s] = col[w][s];
        s_val[(int64_t)r * K + s] = __fdiv_rn(val[w][s], dv[w][0]);
    }
    const float rs = dv[w][1];
    for (int c = lane; c < n; c += 32) P[(int64_t)r * n + c] = __fdiv_rn(row[c], rs);
}

// One diffusion input, written transposed: X = (prev * 0 + src[0] + src[1] + ...) / den, out[c][r] = X[r][c].  prev is
// nextPts[i] before `nextPts[i] *= 0` (NULL: the zeros of the first iteration), so a NaN or inf there stays NaN.
template <typename T>
__global__ void __launch_bounds__(256) snf_mix_kernel(SnfSrc<T> src, const double *__restrict__ prev, int n, double den,
                                                      double *__restrict__ xt) {
    __shared__ double tile[32][33];
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int r = r0 + j, c = c0 + threadIdx.x;
        if (r < n && c < n) {
            const int64_t e = (int64_t)r * n + c;
            double acc = prev ? __dmul_rn(prev[e], 0.0) : 0.0;
            for (int k = 0; k < src.n; ++k) acc = __dadd_rn(acc, (double)src.p[k][e]);
            tile[j][threadIdx.x] = __ddiv_rn(acc, den);
        }
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int c = c0 + j, r = r0 + threadIdx.x;
        if (r < n && c < n) xt[(int64_t)c * n + r] = tile[threadIdx.x][j];
    }
}

// out = S . Y for the K-slot row-sparse S (s_idx ascending per row, float32 values) and dense row-major Y:
// out[r][c] = 0 + v_0 * Y[j_0][c] + v_1 * Y[j_1][c] + ... in slot order, each product and sum rounded on its own
// (scipy csr_matvecs).  blockIdx.x walks the row tiles of one 128-column panel of Y before the next panel, so the
// panel (N x 1 KB) is gathered from L2.  TRANSPOSED: write out[c][r] (T = A^T of A = S . X^T); otherwise add the
// reg_diag / reg_neighbs terms of doSimilarityFusionWs and write out[r][c].
template <bool TRANSPOSED>
__global__ void __launch_bounds__(256) snf_spmm_kernel(const double *__restrict__ Y, const int32_t *__restrict__ s_idx,
                                                       const float *__restrict__ s_val, int n, int K,
                                                       double reg_diag, double reg_neighbs, double *__restrict__ out) {
    __shared__ union {
        struct { int32_t j[SP_BR][SP_KMAX]; float v[SP_BR][SP_KMAX]; } s;
        double tile[SP_BC][SP_BR + 1];
    } sm;
    const int r0 = blockIdx.x * SP_BR, c0 = blockIdx.y * SP_BC;
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int e = threadIdx.x; e < SP_BR * K; e += blockDim.x) {
        const int rr = e / K, t = e - rr * K;
        const bool ok = r0 + rr < n;
        sm.s.j[rr][t] = ok ? s_idx[(int64_t)(r0 + rr) * K + t] : 0;
        sm.s.v[rr][t] = ok ? s_val[(int64_t)(r0 + rr) * K + t] : 0.0f;
    }
    __syncthreads();
    double acc[4][4];
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int u = 0; u < 4; ++u) acc[q][u] = 0.0;
    for (int t = 0; t < K; ++t) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const double v = (double)sm.s.v[w + 8 * q][t];
            const double *y = Y + (int64_t)sm.s.j[w + 8 * q][t] * n + c0 + lane;
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (c0 + lane + 32 * u < n) acc[q][u] = __dadd_rn(acc[q][u], __dmul_rn(v, __ldg(y + 32 * u)));
        }
    }
    if constexpr (TRANSPOSED) {
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int u = 0; u < 4; ++u) sm.tile[lane + 32 * u][w + 8 * q] = acc[q][u];
        __syncthreads();
        for (int cc = w; cc < SP_BC; cc += 8) {
            const int c = c0 + cc, r = r0 + lane;
            if (c < n && r < n) out[(int64_t)c * n + r] = sm.tile[cc][lane];
        }
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int r = r0 + w + 8 * q;
            if (r >= n) continue;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int c = c0 + lane + 32 * u;
                if (c >= n) continue;
                double x = acc[q][u];
                if (reg_diag > 0.0) x = __dadd_rn(x, r == c ? reg_diag : 0.0);          // += reg_diag * eye(N)
                if (reg_neighbs > 0.0 && (r - c == 1 || c - r == 1)) x = __dadd_rn(x, reg_neighbs);
                out[(int64_t)r * n + c] = x;
            }
        }
    }
}

// FusedScores = (0 + Pts[0] + Pts[1] + ...) / n_mats
template <typename T>
__global__ void __launch_bounds__(256) snf_average_kernel(SnfSrc<T> src, int64_t cells, double nm,
                                                          double *__restrict__ out) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < cells; e += (int64_t)gridDim.x * blockDim.x) {
        double acc = 0.0;
        for (int k = 0; k < src.n; ++k) acc = __dadd_rn(acc, (double)src.p[k][e]);
        out[e] = __ddiv_rn(acc, nm);
    }
}

template <typename T>
SnfSrc<T> make_src(const void *const *src, int nsrc) {
    SnfSrc<T> s{};
    for (int k = 0; k < nsrc; ++k) s.p[k] = (const T *)src[k];
    s.n = nsrc;
    return s;
}

void leaf_offsets(int64_t off, int64_t n, std::vector<int32_t> &out) {
    if (n <= 128) { out.push_back((int32_t)off); return; }
    int64_t n2 = n / 2;
    n2 -= n2 % 8;
    leaf_offsets(off, n2, out);
    leaf_offsets(off + n2, n - n2, out);
}

}  // namespace

std::vector<int32_t> snf_leaf_offsets(int n) {
    std::vector<int32_t> v;
    leaf_offsets(0, n, v);
    v.push_back(n);
    return v;
}

int launch_snf_affinity(const float *d, int n, int K, float *dw, float *md, const int32_t *leaf_off, int n_leaves,
                        float *P, int32_t *s_idx, float *s_val, cudaStream_t st) {
    const dim3 tiles((unsigned)((n + 31) / 32), (unsigned)((n + 31) / 32));
    snf_dsym_kernel<<<tiles, dim3(32, 8), 0, st>>>(d, n, dw);
    const unsigned row_ctas = (unsigned)((n + SNF_WARPS - 1) / SNF_WARPS);
    if (K + 1 <= 32) snf_meandist_kernel<32><<<row_ctas, SNF_WARPS * 32, 0, st>>>(dw, n, K, md);
    else snf_meandist_kernel<64><<<row_ctas, SNF_WARPS * 32, 0, st>>>(dw, n, K, md);
    snf_w_kernel<<<dim3((unsigned)((n + 255) / 256), (unsigned)n), 256, 0, st>>>(dw, md, n);
    const size_t dyn = (size_t)SNF_WARPS * n_leaves * sizeof(float);
    if (K <= 32) snf_rows_kernel<32><<<row_ctas, SNF_WARPS * 32, dyn, st>>>(dw, n, K, leaf_off, n_leaves, P, s_idx, s_val);
    else snf_rows_kernel<64><<<row_ctas, SNF_WARPS * 32, dyn, st>>>(dw, n, K, leaf_off, n_leaves, P, s_idx, s_val);
    CUDA_TRY(cudaGetLastError());
    return ACOSS_OK;
}

int launch_snf_mix(const void *const *src, int nsrc, bool f32, const double *prev, int n, double den, double *xt,
                   cudaStream_t st) {
    const dim3 tiles((unsigned)((n + 31) / 32), (unsigned)((n + 31) / 32));
    if (f32) snf_mix_kernel<float><<<tiles, dim3(32, 8), 0, st>>>(make_src<float>(src, nsrc), prev, n, den, xt);
    else snf_mix_kernel<double><<<tiles, dim3(32, 8), 0, st>>>(make_src<double>(src, nsrc), prev, n, den, xt);
    CUDA_TRY(cudaGetLastError());
    return ACOSS_OK;
}

int launch_snf_spmm(const double *Y, const int32_t *s_idx, const float *s_val, int n, int K, bool transposed,
                    double reg_diag, double reg_neighbs, double *out, cudaStream_t st) {
    const dim3 grid((unsigned)((n + SP_BR - 1) / SP_BR), (unsigned)((n + SP_BC - 1) / SP_BC));
    if (transposed) snf_spmm_kernel<true><<<grid, 256, 0, st>>>(Y, s_idx, s_val, n, K, 0.0, 0.0, out);
    else snf_spmm_kernel<false><<<grid, 256, 0, st>>>(Y, s_idx, s_val, n, K, reg_diag, reg_neighbs, out);
    CUDA_TRY(cudaGetLastError());
    return ACOSS_OK;
}

int launch_snf_average(const void *const *src, int nsrc, bool f32, int64_t cells, double *out, cudaStream_t st) {
    const unsigned grid = (unsigned)std::min<int64_t>((cells + 255) / 256, 148 * 16);
    if (f32) snf_average_kernel<float><<<grid, 256, 0, st>>>(make_src<float>(src, nsrc), cells, (double)nsrc, out);
    else snf_average_kernel<double><<<grid, 256, 0, st>>>(make_src<double>(src, nsrc), cells, (double)nsrc, out);
    CUDA_TRY(cudaGetLastError());
    return ACOSS_OK;
}
