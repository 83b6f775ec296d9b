// K2 (fast path) — cross-similarity, per-row / per-column k-th-nearest selection and bit-packed CRP
// without ever writing a float distance matrix to HBM.
//
// Replaces essentia ChromaCrossSimilarity (SURVEY.md App. A2-A5; call site
// /root/reference/acoss/algorithms/rqa_serra09.py:60-66).  Results are bit-identical to the
// reference-order arithmetic of k2_exact.cu.  The three sweeps over the cell matrix (row thresholds, column
// thresholds, emit) exist twice and launch_k2_fast picks per call: on the tensor cores (k2_tc.inl: the stacked
// 108-term inner product as an exact integer GEMM, tcgen05.mma kind::i8 over byte-limb planes, items read from
// tensor memory) for lines of TC_MIN_WINDOWS windows or more, and as FFMA2 chains on the CUDA cores (this file)
// for short lines and for features that cannot be quantised inside the error budget.  Everything around the sweeps
// (prep, sampler, selection, candidate lists, exact thresholds, bit patch) is shared.  Structure of the FFMA2 form:
//
//  * The stacked squared distance is a 9-tap diagonal sum of the frame-level dot product
//    e[a][c] = <x_a, y_c> (12 FMAs):  item(i,j) = aa_i + bb_j - 2 * sum_t e[i+t][j+t].
//    A warp sweeps the streamed side (rows a) for a strip of owned columns c kept in REGISTERS
//    (RC columns per lane); the diagonal sum slides: T[a][c] = T[a-1][c-1] + e[a][c] - e[a-9][c-9]
//    (one warp shuffle for the lane boundary, one for the 9-rows-old value from the lane's
//    neighbour's register ring).  e is quantised once to fixed point (float magic-number add), so
//    T is an EXACT integer sliding sum: no drift, identical in every sweep and both orientations.
//  * These approximate items z (|z - exact| <= EPS units, bound in DESIGN.md §4.2) drive two
//    thread-private 64-bin histogram sweeps per orientation (columns: owned = reference; rows:
//    owned = query) that bracket the order statistics floor(k), ceil(k) of every row and column
//    to a handful of cells, and one emit sweep that writes every cell whose membership is certain
//    and appends the few uncertain cells (inside a bracket +- 2 EPS) to per-row / per-column
//    candidate lists.
//  * resolve kernels recompute ONLY the candidate cells in the reference's exact operation order
//    (float32 products, sequential float64 accumulation), pick the exact order statistics, apply
//    essentia's percentile formula and patch the candidate bits.  Consistency checks that make
//    the certain/uncertain split provably exact are evaluated per row/column; a pair that fails
//    one is flagged and re-run by k2_exact.cu.
#include <stdlib.h>

#include <algorithm>

#include "k2_fast.cuh"

namespace {

constexpr int M9 = 9;               // frameStackSize handled by this path
constexpr int HALO = M9 - 1;        // owned columns a strip recomputes (8)
constexpr int NBIN = 64;            // histogram bins per level (+ one underflow and one overflow row)
constexpr int SBIN = 256;           // bins of the per-line sample histogram (select kernel)
constexpr int EPS = 128;            // bound on |z - exact item| in fixed-point units (DESIGN.md §4.2)
constexpr int CAND_CAP = 128;       // candidates per row / column
constexpr int BRACKET_TARGET = 96;  // a bracket holding more cells than this is split by another histogram level
constexpr int WPC = 4;              // warps per CTA in the sweep kernels
constexpr int TC_N = 64;            // streamed windows per tensor-sweep block (MMA N)
constexpr int TC_PAD = 2 * TC_N;    // padding of per-window arrays and byte planes read in whole blocks
constexpr int TC_HUGE = 0x20000000; // norm of a padding window: its items land above every bracket
constexpr int RCV = 4;              // owned frames per lane (register columns) in the sweep kernels
constexpr int HRC = 4;              // register columns per lane of the histogram sweeps
constexpr int MINB = 3;             // CTAs per SM the sweep kernels are compiled for (register cap 168 at 3, 255 at 2)
constexpr int TC_MIN_WINDOWS = 400; // longer side of the matrix from which the tensor sweeps (k2_tc.inl) replace the FFMA2 sweeps

struct PairHdr {                    // per-slot header written by fast_prep_kernel
    int32_t nq, nr, Mx, Nx;         // frames and stacked windows of query / reference
    int32_t fk[2], ck[2];           // 0-based ranks floor(k), ceil(k): [0] rows (L = Nx), [1] columns (L = Mx)
    int32_t quirk[2];               // 1: threshold is forced to 0 (integer k without guard, F1)
    float kf[2];                    // fractional rank (float32, essentia arithmetic)
    int32_t lo1, sh1;               // origin of the pair's item range (fixed point) / shift of a 64-bin split of it
    int32_t hi1;                    // end of the pair's item range
    int32_t dz;                     // tensor sweeps: bound on z' - z (k2_tc.inl), the low-side widening of emit's zones; else 0
};

struct TcShift { int s0, s1, s2; unsigned m0; };       // tensor sweeps (k2_tc.inl): e0, 8 - e0, 16 - e0, 2^e0

struct FastLayout {
    size_t slot_bytes;
    size_t off_hdr, off_rrot, off_aaf, off_bbf, off_aai, off_bbi, off_lo, off_w, off_cb, off_sh, off_cnt,
        off_cand, off_candz, off_zin, off_zout, off_rowpack, off_pool, off_pcnt, off_samp_r, off_samp_c,
        off_lsel, off_wlist, off_wcnt, off_win, off_qpl, off_rpl, off_lsum, off_tcq;
    int max_rows, max_cols, max_frames, lines, pool_cap;
    int plane_frames;                   // frames per byte plane of the tensor sweeps (zero padded past the track end)
    int slog;                           // log2 of the diagonal sampling stride S
    int nst_r, nst_c;                   // sample slots per row (ceil(max_cols / S)) / per column
};

__host__ __device__ inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

FastLayout make_layout(const SlotGeom &g, int max_frames) {
    FastLayout L;
    L.max_rows = g.max_rows; L.max_cols = g.max_cols; L.max_frames = max_frames;
    L.lines = g.max_rows + g.max_cols;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes, 128); return r; };
    L.off_hdr = take(sizeof(PairHdr));
    L.off_rrot = take((size_t)(max_frames + 8) * NBINS * 4);
    L.off_aaf = take((size_t)g.max_rows * 4);
    L.off_bbf = take((size_t)g.max_cols * 4);
    L.off_aai = take((size_t)(g.max_rows + TC_PAD) * 4);       // padded: the tensor sweeps read whole row blocks
    L.off_bbi = take((size_t)(g.max_cols + TC_PAD) * 4);
    L.off_lo = take((size_t)L.lines * 4);
    L.off_w = take((size_t)L.lines * 4);
    L.off_cb = take((size_t)L.lines * 4);
    L.off_sh = take((size_t)L.lines * 4);
    L.off_cnt = take((size_t)L.lines * 4);
    L.off_cand = take((size_t)L.lines * CAND_CAP * 2);
    L.off_candz = take((size_t)L.lines * CAND_CAP * 4);
    L.off_zin = take((size_t)L.lines * 4);
    L.off_zout = take((size_t)L.lines * 4);
    L.off_rowpack = take((size_t)(g.max_rows + TC_PAD) * 16);
    // uncertain cells of the emit sweep, 8 bytes each (i | j << 14, fixed-point item).  A line contributes its
    // bracket cells (a few tens whatever its length), so the fraction of uncertain cells falls with the line
    // length: ~7 % at 500 frames, ~1.7 % at 2k.  Capacity: ~100 cells per line, at most an eighth of the matrix
    // (more -> the pair takes the exact path)
    {
        const int64_t cells = (int64_t)g.max_rows * g.max_cols;
        const int64_t per_line = (int64_t)100 * (g.max_rows + g.max_cols) / 2;
        L.pool_cap = (int)std::min<int64_t>(std::max<int64_t>(4096, std::min(per_line, cells / 8)), (int64_t)1 << 26);
    }
    L.off_pool = take((size_t)L.pool_cap * 8);
    L.off_pcnt = take(4);
    // diagonal sampling stride: the bracket a line gets from n_s samples holds ~2.35 L / sqrt(n_s) cells, which
    // the 64-bin split must bring under BRACKET_TARGET  =>  n_s >= (0.003 L)^2, S = L / n_s <= 1 / (9e-6 L)
    {
        const int Lmax = g.max_rows > g.max_cols ? g.max_rows : g.max_cols;
        const double smax = 1.0 / (9e-6 * (double)(Lmax > 1 ? Lmax : 1));
        L.slog = 5;
        while (L.slog > 2 && (double)(1 << L.slog) > smax) --L.slog;
        // short lines: keep at least 32 samples per line (a bracket from fewer samples is too wide to help;
        // measured at 500 frames: S = 16 or 8 give +30 % pairs/s over S = 32, at 2k frames S = 32 is best)
        while (L.slog > 2 && (Lmax >> L.slog) < 32) --L.slog;
    }
    L.nst_r = ((g.max_cols - 1) >> L.slog) + 1;
    L.nst_c = ((g.max_rows - 1) >> L.slog) + 1;
    L.off_samp_r = take((size_t)L.nst_r * g.max_rows * 4);      // [t = j / S][i]
    L.off_samp_c = take((size_t)L.nst_c * g.max_cols * 4);      // [t = i / S][j]
    L.off_lsel = take((size_t)L.lines * 20);                    // LineSel per line
    L.off_wlist = take((size_t)L.lines * 4 * 8);                // WinCell list: WFLAT_PER_LINE entries per line
    L.off_wcnt = take(4);
    L.off_win = take((size_t)L.lines * 2 * 8 * 4);              // exact items of the window cells: [line][2][WIN_CAP]
    L.plane_frames = max_frames + TC_PAD + 16;
    L.off_qpl = take((size_t)3 * L.plane_frames * 16);          // query byte planes [h, l1, l2][frame][16]
    L.off_rpl = take((size_t)3 * L.plane_frames * 16);          // rotated reference byte planes
    L.off_lsum = take((size_t)2 * L.plane_frames * 4);          // per frame: sum of its h bytes | sum of its l1 bytes << 16 (q, r)
    L.off_tcq = take(4 * 4);                                    // next work item of each tensor sweep (slot 0's copy serves the call)
    L.slot_bytes = align_up(o, 256);
    return L;
}

template <typename T>
__device__ __forceinline__ T *slot_ptr(char *base, const FastLayout &L, int slot, size_t off) {
    return reinterpret_cast<T *>(base + (size_t)slot * L.slot_bytes + off);
}

// Per-row parameters of the emit sweep: {aa_fix, 4 EPS - rowLo, rowW + 4 EPS, aa_fix - rowLo + 2 EPS}.  With ar = z - (rowLo - 2 EPS):
//   ar = .w + bb - T,   row zone <=> (unsigned)ar < .z,   near zero (z < 2 EPS) <=> ar < .y,   rowLo - 2 EPS = 2 EPS - .y
// (the tensor sweeps pass rowLo = lo - dz, rowW = w + dz: their bracket [lo, lo + w) is in z', DESIGN.md 4.2)
__device__ __forceinline__ int4 pack_row(int aa, int lo, int w) { return make_int4(aa, 4 * EPS - lo, w + 4 * EPS, aa - lo + 2 * EPS); }
__device__ __forceinline__ int row_lo_e(const int4 &rp) { return 2 * EPS - rp.y; }

// ------------------------------------------------------------------------------------------------
// Fixed-point frame-level dot product.  2<x, y> is accumulated by TWO fused-multiply-add chains (even and odd
// bins, six steps each) that both start at the float magic constant 2^fx_exp, so every partial sum already sits
// in the fixed-point binade (12 roundings of at most half a unit each: inside the EPS budget, DESIGN.md 4.2).
// The sum of the raw bits of the two chains is the quantised value + 2 * bits(magic).  The sweep kernels run
// the two chains as ONE packed sm_100 instruction stream (fma.rn.f32x2, SASS FFMA2: both halves are IEEE fma
// with round-to-nearest, so they are bit-identical to the scalar chains of dot_fx below, which the sampler, the
// sparse level and the candidate expansion use).  One side is pre-doubled (exact), so which side it is does
// not change a bit.
// ------------------------------------------------------------------------------------------------
typedef unsigned long long u64;

__device__ __forceinline__ u64 pack2(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ u64 ffma2(u64 a, u64 b, u64 c) {
    u64 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
// raw bits of the two half chains, summed (= quantised 2<x, y> + 2 * bits(magic)); x, y: 12 floats each
constexpr int NMAGIC = 2;                           // magic offsets inside one quantised dot product
__device__ __forceinline__ int dot_fx(const float (&x)[NBINS], const float (&y)[NBINS], float magic) {
    float acc[2] = {magic, magic};                  // even bins, odd bins
#pragma unroll
    for (int b = 0; b < NBINS; b += 2)
#pragma unroll
        for (int h = 0; h < 2; ++h) acc[h] = __fmaf_rn(x[b + h], y[b + h], acc[h]);
    // summed in a loop, not as one expression: the compiler then keeps (even + odd) - magic offsets in the callers
    // instead of reassociating it (as one expression the sampler measured 5 % slower on a B200)
    int r = 0;
#pragma unroll
    for (int h = 0; h < 2; ++h) r += __float_as_int(acc[h]);
    return r;
}
__device__ __forceinline__ void load_frame(const float *__restrict__ p, float (&x)[NBINS], float scale) {
    const float4 *q = reinterpret_cast<const float4 *>(p);
    const float4 v0 = __ldg(q), v1 = __ldg(q + 1), v2 = __ldg(q + 2);
    x[0] = scale * v0.x; x[1] = scale * v0.y; x[2] = scale * v0.z; x[3] = scale * v0.w;
    x[4] = scale * v1.x; x[5] = scale * v1.y; x[6] = scale * v1.z; x[7] = scale * v1.w;
    x[8] = scale * v2.x; x[9] = scale * v2.y; x[10] = scale * v2.z; x[11] = scale * v2.w;
}

// ------------------------------------------------------------------------------------------------
// prep: rotated reference copy, exact float32 norms (reference order) + their fixed-point images,
// ranks, level-1 histogram range, zeroed candidate counters
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fast_prep_kernel(TrackSet ts, const int32_t *__restrict__ pairs,
                                                        const int32_t *__restrict__ oti, int64_t first,
                                                        FastLayout L, char *__restrict__ scratch, float qperc,
                                                        int guard, float fx_scale, float q_scale, TcShift sh3) {
    __shared__ int s_max[2];
    __shared__ int s_lmax[4];                                 // largest window sums: h of q, h of r, l1 of q, l1 of r
    const int slot = blockIdx.x;
    const int64_t k = first + slot;
    const int q = pairs[2 * k], r = pairs[2 * k + 1], s = oti[k] % NBINS;
    const int nq = (int)(ts.offsets[q + 1] - ts.offsets[q]), nr = (int)(ts.offsets[r + 1] - ts.offsets[r]);
    const int Mx = nq - M9, Nx = nr - M9;
    const float *Q = ts.frames + ts.offsets[q] * NBINS;
    const float *R = ts.frames + ts.offsets[r] * NBINS;
    float *rrot = slot_ptr<float>(scratch, L, slot, L.off_rrot);
    if (threadIdx.x < 2) s_max[threadIdx.x] = 0;
    if (threadIdx.x < 4) s_lmax[threadIdx.x] = 0;
    for (int idx = threadIdx.x; idx < (nr + 8) * NBINS; idx += blockDim.x) {
        const int f = idx / NBINS, b = idx - f * NBINS;
        rrot[idx] = (f < nr) ? R[f * NBINS + rot_src(b, s)] : 0.f;
    }
    // byte planes of the tensor sweeps: x_q = rint(x * 2^q_exp) < 2^24 as limbs h, l1, l2; 16-byte frames (12 bins + 4 zeros),
    // zero frames past the track end
    uint32_t *lsum = slot_ptr<uint32_t>(scratch, L, slot, L.off_lsum);
    if (q_scale > 0.f) {
        uint4 *qpl = slot_ptr<uint4>(scratch, L, slot, L.off_qpl), *rpl = slot_ptr<uint4>(scratch, L, slot, L.off_rpl);
        for (int idx = threadIdx.x; idx < 2 * L.plane_frames; idx += blockDim.x) {
            const bool isq = idx < L.plane_frames;
            const int f = isq ? idx : idx - L.plane_frames;
            const int nf = isq ? nq : nr;
            uint32_t w[3][4] = {{0u, 0u, 0u, 0u}, {0u, 0u, 0u, 0u}, {0u, 0u, 0u, 0u}};
            if (f < nf) {
#pragma unroll
                for (int b = 0; b < NBINS; ++b) {
                    const float v = isq ? Q[(int64_t)f * NBINS + b] : R[(int64_t)f * NBINS + rot_src(b, s)];
                    const uint32_t xq = (uint32_t)__float2int_rn(v * q_scale);
                    w[0][b >> 2] |= ((xq >> 16) & 255u) << (8 * (b & 3));
                    w[1][b >> 2] |= ((xq >> 8) & 255u) << (8 * (b & 3));
                    w[2][b >> 2] |= (xq & 255u) << (8 * (b & 3));
                }
            }
            uint4 *dst = isq ? qpl : rpl;
#pragma unroll
            for (int pl = 0; pl < 3; ++pl) dst[(size_t)pl * L.plane_frames + f] = make_uint4(w[pl][0], w[pl][1], w[pl][2], 0u);
            uint32_t sh_ = 0u, sl_ = 0u;                      // byte sums (<= 12 * 255 each)
#pragma unroll
            for (int c = 0; c < 3; ++c) { sh_ = __dp4a(w[0][c], 0x01010101u, sh_); sl_ = __dp4a(w[1][c], 0x01010101u, sl_); }
            lsum[idx] = sh_ | (sl_ << 16);
        }
    }
    uint32_t *cnt = slot_ptr<uint32_t>(scratch, L, slot, L.off_cnt);
    for (int i = threadIdx.x; i < L.lines; i += blockDim.x) cnt[i] = 0u;
    if (threadIdx.x == 0) { *slot_ptr<uint32_t>(scratch, L, slot, L.off_pcnt) = 0u; *slot_ptr<uint32_t>(scratch, L, slot, L.off_wcnt) = 0u; }
    if (threadIdx.x < 4) slot_ptr<uint32_t>(scratch, L, slot, L.off_tcq)[threadIdx.x] = 0u;
    __syncthreads();
    float *aaf = slot_ptr<float>(scratch, L, slot, L.off_aaf), *bbf = slot_ptr<float>(scratch, L, slot, L.off_bbf);
    int32_t *aai = slot_ptr<int32_t>(scratch, L, slot, L.off_aai), *bbi = slot_ptr<int32_t>(scratch, L, slot, L.off_bbi);
    int mxa = 0, mxb = 0;
    for (int i = threadIdx.x; i < Mx + Nx; i += blockDim.x) {
        const bool isq = i < Mx;
        const float *src = isq ? Q + (int64_t)i * NBINS : rrot + (int64_t)(i - Mx) * NBINS;
        double acc = 0.0;
        for (int t = 0; t < M9; ++t) {
            const float *fr = src + t * NBINS;
#pragma unroll
            for (int b = 0; b < NBINS; ++b) acc = acc_f32prod(acc, fr[b], fr[b]);
        }
        const float v = (float)acc;
        const int fx = __float2int_rn(v * fx_scale);
        if (isq) { aaf[i] = v; aai[i] = fx; mxa = max(mxa, fx); }
        else { bbf[i - Mx] = v; bbi[i - Mx] = fx; mxb = max(mxb, fx); }
    }
    for (int i = Mx + threadIdx.x; i < L.max_rows + TC_PAD; i += blockDim.x) aai[i] = TC_HUGE;   // padding windows
    for (int i = Nx + threadIdx.x; i < L.max_cols + TC_PAD; i += blockDim.x) bbi[i] = TC_HUGE;
    atomicMax(&s_max[0], mxa);
    atomicMax(&s_max[1], mxb);
    // the bound dz on z' - z of the tensor sweeps (k2_tc.inl): acc2 = l1.l1 + h.l2 + l2.h <= 255 (sum h_X + sum h_Y +
    // min(sum l1_X, sum l1_Y)) over the 108 bytes of the two windows, z' - z <= (acc2 >> (16 - e0)) + 1 (DESIGN.md 4.2)
    if (q_scale > 0.f) {
        int m[4] = {0, 0, 0, 0};
        for (int i = threadIdx.x; i < Mx + Nx; i += blockDim.x) {
            const bool isq = i < Mx;
            const uint32_t *src = lsum + (isq ? i : L.plane_frames + i - Mx);
            uint32_t acc = 0u;                                // (h sum, l1 sum) of the window, no carry between the halves
#pragma unroll
            for (int t = 0; t < M9; ++t) acc += src[t];
            const int sh_ = (int)(acc & 0xffffu), sl_ = (int)(acc >> 16);
            if (isq) { m[0] = max(m[0], sh_); m[2] = max(m[2], sl_); }
            else { m[1] = max(m[1], sh_); m[3] = max(m[3], sl_); }
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) atomicMax(&s_lmax[c], m[c]);
    }
    __syncthreads();
    const int dz = q_scale > 0.f ? ((255 * (s_lmax[0] + s_lmax[1] + min(s_lmax[2], s_lmax[3]))) >> sh3.s2) + 1 : 0;
    PairHdr *h = slot_ptr<PairHdr>(scratch, L, slot, L.off_hdr);
    int lo1 = -2 * EPS, sh1 = 0;
    const long long range1 = (long long)s_max[0] + s_max[1] + 4 * EPS + 1;
    while ((range1 >> sh1) > NBIN - 1) ++sh1;
    int fk2[2], ck2[2], quirk2[2];
    float kf2[2];
    for (int o = 0; o < 2; ++o) {
        const int Ln = (o == 0) ? Nx : Mx;                    // rows see Nx entries, columns see Mx
        const float kf = (Ln > 1) ? __fmul_rn((float)(Ln - 1), qperc) : __fmul_rn((float)Ln, qperc);
        const float fkf = floorf(kf), ckf = ceilf(kf);
        kf2[o] = kf; fk2[o] = (int)fkf; ck2[o] = min((int)ckf, Ln - 1);
        quirk2[o] = (fkf == ckf && !guard) ? 1 : 0;
    }
    if (threadIdx.x == 0) {
        h->nq = nq; h->nr = nr; h->Mx = Mx; h->Nx = Nx;
        for (int o = 0; o < 2; ++o) { h->fk[o] = fk2[o]; h->ck[o] = ck2[o]; h->quirk[o] = quirk2[o]; h->kf[o] = kf2[o]; }
        h->lo1 = lo1; h->sh1 = sh1; h->hi1 = lo1 + (int)range1;
        h->dz = dz;
    }
    // level-1 bracket state for every line; emit-ready defaults for quirk sides (threshold 0)
    int32_t *lo = slot_ptr<int32_t>(scratch, L, slot, L.off_lo), *w = slot_ptr<int32_t>(scratch, L, slot, L.off_w);
    int32_t *cb = slot_ptr<int32_t>(scratch, L, slot, L.off_cb), *sh = slot_ptr<int32_t>(scratch, L, slot, L.off_sh);
    int4 *rowpack = slot_ptr<int4>(scratch, L, slot, L.off_rowpack);
    for (int i = threadIdx.x; i < L.lines; i += blockDim.x) {
        const int side = (i < L.max_rows) ? 0 : 1;
        if (quirk2[side]) { lo[i] = 0; w[i] = 0; cb[i] = 0; sh[i] = -1; }
        else { lo[i] = lo1; w[i] = 0; cb[i] = 0; sh[i] = sh1; }
    }
    for (int i = threadIdx.x; i < L.max_rows + TC_PAD; i += blockDim.x)
        rowpack[i] = pack_row(i < Mx ? aai[i] : TC_HUGE, 0, 0);
}

// ------------------------------------------------------------------------------------------------
// diagonal sampler: fixed-point items of the cells (i, j) with (j - i) % S == 0, i.e. every S-th
// diagonal.  A warp covers 24 consecutive positions of KD such diagonals: lane l computes the
// frame-level dot product of position i0 + l, the 9-tap window sum runs across lanes (4 shuffles).
// Every sample is a sample of its row and of its column: samp_r[j / S][i], samp_c[i / S][j].
// These samples only steer the histogram brackets (select kernel below); exactness never depends
// on them.
// ------------------------------------------------------------------------------------------------
constexpr int SKD = 16;             // diagonals per warp task
constexpr int SPOS = 32 - HALO;     // window sums one warp pass produces per diagonal (24)

__global__ void __launch_bounds__(128) fast_sample_kernel(TrackSet ts, const int32_t *__restrict__ pairs,
                                                          int64_t first, int n, FastLayout L,
                                                          char *__restrict__ scratch, int ngrp_max, int nblk_max,
                                                          float magic) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t task = (int64_t)blockIdx.x * 4 + warp;
    const int per_slot = ngrp_max * nblk_max;
    const int slot = (int)(task / per_slot);
    if (slot >= n) return;
    const int rem = (int)(task - (int64_t)slot * per_slot);
    const int grp = rem / nblk_max, blk = rem - grp * nblk_max;
    const PairHdr *h = slot_ptr<PairHdr>(scratch, L, slot, L.off_hdr);
    if (h->quirk[0] && h->quirk[1]) return;
    const int nq = h->nq, nr = h->nr, Mx = h->Mx, Nx = h->Nx;
    const int slog = L.slog;
    const int i0 = blk * SPOS;
    if (i0 >= Mx) return;
    // diagonals d = S * u, u in [-(Mx-1)/S, (Nx-1)/S]
    const int u_lo = -((Mx - 1) >> slog);
    const int u0 = u_lo + grp * SKD;
    if (((int64_t)u0 << slog) > (int64_t)(Nx - 1) - i0) return;                       // block lies right of the matrix
    if ((((int64_t)u0 + SKD - 1) << slog) + i0 + SPOS - 1 < 0) return;                // ... or left of it
    const int64_t k = first + slot;
    const int q = pairs[2 * k];
    const float *Qf = ts.frames + ts.offsets[q] * NBINS;
    const float *Rf = slot_ptr<float>(scratch, L, slot, L.off_rrot);
    const int32_t *aai = slot_ptr<int32_t>(scratch, L, slot, L.off_aai), *bbi = slot_ptr<int32_t>(scratch, L, slot, L.off_bbi);
    int32_t *samp_r = slot_ptr<int32_t>(scratch, L, slot, L.off_samp_r), *samp_c = slot_ptr<int32_t>(scratch, L, slot, L.off_samp_c);
    const int i = i0 + lane;
    const bool iok = lane < SPOS && i < Mx;
    float x[NBINS];
    load_frame(Qf + (int64_t)min(i, nq - 1) * NBINS, x, 2.f);
    const int aa = iok ? aai[i] : 0;
    const int mbits2 = NMAGIC * __float_as_int(magic);
#pragma unroll
    for (int kd = 0; kd < SKD; ++kd) {
        const int d = (u0 + kd) << slog;
        const int j = i + d;
        float yv[NBINS];
        load_frame(Rf + (int64_t)min(max(j, 0), nr - 1) * NBINS, yv, 1.f);
        const int v = dot_fx(x, yv, magic) - mbits2;
        const int s1 = v + __shfl_down_sync(0xffffffffu, v, 1);
        const int s2 = s1 + __shfl_down_sync(0xffffffffu, s1, 2);
        const int s4 = s2 + __shfl_down_sync(0xffffffffu, s2, 4);
        const int T = s4 + __shfl_down_sync(0xffffffffu, v, 8);
        if (iok && j >= 0 && j < Nx) {
            const int z = aa + bbi[j] - T;
            samp_r[(int64_t)(j >> slog) * L.max_rows + i] = z;
            samp_c[(int64_t)(i >> slog) * L.max_cols + j] = z;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// select: one thread per line.  A private 256-bin histogram of the line's samples (over the pair's
// item range) gives the bins holding the sample ranks mu -+ 4.5 sigma of the wanted order statistic;
// that is the line's first bracket [lo, lo + 64 << sh) for the histogram sweeps.  A wrong bracket
// costs another sweep level, never a wrong result (under / overflow are counted exactly).
// ------------------------------------------------------------------------------------------------
constexpr int SEL_THREADS = 128;
constexpr int MIN_SAMPLES = 24;     // lines with fewer samples start from the whole item range

__global__ void __launch_bounds__(SEL_THREADS) fast_select_kernel(int n, FastLayout L, char *__restrict__ scratch) {
    extern __shared__ uint32_t s_sel_hist[];                 // [SBIN / 2][SEL_THREADS], two 16-bit counters per word
    const int slot = blockIdx.y;
    if (slot >= n) return;
    const PairHdr *h = slot_ptr<PairHdr>(scratch, L, slot, L.off_hdr);
    const int Mx = h->Mx, Nx = h->Nx;
    const int gline = blockIdx.x * SEL_THREADS + threadIdx.x;
    if (blockIdx.x * SEL_THREADS >= Mx + Nx) return;
    uint32_t *hist = s_sel_hist + threadIdx.x;
#pragma unroll 4
    for (int b = 0; b < SBIN / 2; ++b) hist[b * SEL_THREADS] = 0u;
    if (gline >= Mx + Nx) return;
    const bool isrow = gline < Mx;
    const int idx = isrow ? gline : gline - Mx;
    const int side = isrow ? 0 : 1;
    if (h->quirk[side]) return;                               // threshold forced to 0: no selection on this side
    const int line = isrow ? idx : L.max_rows + idx;
    const int slog = L.slog, S = 1 << slog;
    const int Lother = isrow ? Nx : Mx;                       // entries of the line
    const int r0 = idx & (S - 1);                             // first sampled position along the line
    const int ns = (r0 < Lother) ? ((Lother - 1 - r0) >> slog) + 1 : 0;
    const int32_t *samp = isrow ? slot_ptr<int32_t>(scratch, L, slot, L.off_samp_r) : slot_ptr<int32_t>(scratch, L, slot, L.off_samp_c);
    const int64_t pitch = isrow ? L.max_rows : L.max_cols;
    const int lo1 = h->lo1, hi1 = h->hi1;
    int shs = 0;
    while ((((int64_t)hi1 - lo1) >> shs) > SBIN - 1) ++shs;
    for (int t0 = 0; t0 < ns; t0 += 8) {                      // 8 independent loads in flight per thread
        int z[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) z[u] = (t0 + u < ns) ? __ldg(samp + (int64_t)(t0 + u) * pitch + idx) : 0;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            if (t0 + u < ns) {
                const int b = min(max((z[u] - lo1) >> shs, 0), SBIN - 1);
                hist[(b >> 1) * SEL_THREADS] += 1u << (16 * (b & 1));
            }
        }
    }
    // wanted ranks floor(k) .. ceil(k) of Lother entries -> sample ranks mu -+ 4.5 sigma
    const float pq = ((float)h->fk[side] + 0.5f) / (float)Lother;
    const float mu = pq * (float)ns, sg = sqrtf(fmaxf(mu * (1.f - pq), 0.25f));
    const int r_lo = max((int)floorf(mu - 4.5f * sg) - 1, 0);
    const int r_hi = (int)ceilf(mu + 4.5f * sg) + 1;
    int cum = 0, b_lo = -1, b_hi = -1;
    for (int b = 0; b < SBIN / 2; ++b) {
        const uint32_t wv = hist[b * SEL_THREADS];
        const int c0 = wv & 0xffff, c1 = wv >> 16;
        if (b_lo < 0 && cum + c0 > r_lo) b_lo = 2 * b;
        if (b_hi < 0 && cum + c0 > r_hi) b_hi = 2 * b;
        cum += c0;
        if (b_lo < 0 && cum + c1 > r_lo) b_lo = 2 * b + 1;
        if (b_hi < 0 && cum + c1 > r_hi) b_hi = 2 * b + 1;
        cum += c1;
        if (b_hi >= 0) break;                                 // both ranks located (r_lo <= r_hi)
    }
    int lo = lo1, hi = hi1;
    // short lines have too few samples to steer anything: a 64-bin split of the whole item range already
    // isolates their order statistics (a bin then holds ~L / 40 cells)
    if (ns >= MIN_SAMPLES) {
        if (b_lo >= 0) lo = lo1 + (b_lo << shs);
        if (b_hi >= 0) hi = min(hi1, lo1 + ((b_hi + 1) << shs));
    }
    int sh = 0;
    while ((((int64_t)hi - lo) >> sh) > NBIN) ++sh;
    slot_ptr<int32_t>(scratch, L, slot, L.off_lo)[line] = lo;
    slot_ptr<int32_t>(scratch, L, slot, L.off_sh)[line] = sh;
}

// ------------------------------------------------------------------------------------------------
// the sweep: shared by the histogram kernels and the emit kernel
// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// the sweep: shared by the histogram kernels and the emit kernel
// ------------------------------------------------------------------------------------------------
template <int RC>
struct Sweep {
    static constexpr int COLS = 32 * RC;          // owned frames per strip
    static constexpr int OUTW = COLS - HALO;      // output windows per strip
    u64 y[RC][NBINS / 2];                         // owned frames, pre-doubled, as (even, odd) bin pairs
    int ring[M9][RC];                             // raw bits (two magic offsets included) of the last 9 quantised e values
    int T[RC];                                    // fixed-point sliding diagonal sums (of 2e)
    unsigned okm[RC];                             // lane has a left neighbour holding column c-9
    unsigned nz0;                                 // all ones except on lane 0
    u64 magic2;                                   // (magic, magic)
    int mbits2;                                   // NMAGIC * bits(magic) (mod 2^32): the offsets inside one quantised e

    __device__ __forceinline__ void init(const float *__restrict__ Y, int nY, int cb, int lane, float magic_) {
        magic2 = pack2(magic_, magic_);
        mbits2 = NMAGIC * __float_as_int(magic_);
        nz0 = lane ? 0xffffffffu : 0u;
#pragma unroll
        for (int k = 0; k < RC; ++k) {
            const int c = cb + RC * lane + k;
            const float4 *p = reinterpret_cast<const float4 *>(Y + (int64_t)c * NBINS);
            float4 v0 = make_float4(0, 0, 0, 0), v1 = v0, v2 = v0;
            if (c < nY) { v0 = __ldg(p); v1 = __ldg(p + 1); v2 = __ldg(p + 2); }
            y[k][0] = pack2(2.f * v0.x, 2.f * v0.y); y[k][1] = pack2(2.f * v0.z, 2.f * v0.w);
            y[k][2] = pack2(2.f * v1.x, 2.f * v1.y); y[k][3] = pack2(2.f * v1.z, 2.f * v1.w);
            y[k][4] = pack2(2.f * v2.x, 2.f * v2.y); y[k][5] = pack2(2.f * v2.z, 2.f * v2.w);
            T[k] = 0;
            const int kk = ((k - M9) % RC + RC) % RC;
            okm[k] = (lane >= (M9 - k + kk) / RC) ? 0xffffffffu : 0u;
#pragma unroll
            for (int u = 0; u < M9; ++u) ring[u][k] = mbits2;
        }
    }

    // frame-level dot products of one streamed frame (six (even, odd) pairs) with the lane's RC owned frames
    __device__ __forceinline__ void dot(const ulonglong2 &x0, const ulonglong2 &x1, const ulonglong2 &x2, int (&eb)[RC]) const {
        const u64 xs[6] = {x0.x, x0.y, x1.x, x1.y, x2.x, x2.y};
        u64 acc[RC];
#pragma unroll
        for (int t = 0; t < 6; ++t)
#pragma unroll
            for (int k = 0; k < RC; ++k) acc[k] = ffma2(xs[t], y[k][t], t == 0 ? magic2 : acc[k]);
#pragma unroll
        for (int k = 0; k < RC; ++k) eb[k] = (int)(unsigned)(acc[k] & 0xffffffffu) + (int)(unsigned)(acc[k] >> 32);
    }

    // slides the diagonal sums T by one row.  U = a % 9 (static ring slot).
    template <int U>
    __device__ __forceinline__ void finish(const int (&eb)[RC]) {
        int old[RC];
        // e[a-9][c-9]: column c-9 lives dl lanes to the left, in register (k - 9) mod RC of ring slot U
#pragma unroll
        for (int k = 0; k < RC; ++k) {
            const int kk = ((k - M9) % RC + RC) % RC;
            const int dl = (M9 - k + kk) / RC;
            const unsigned v = (unsigned)__shfl_up_sync(0xffffffffu, ring[U][kk], dl);
            old[k] = (int)((v & okm[k]) | ((unsigned)mbits2 & ~okm[k]));
        }
        const int tl = (int)((unsigned)__shfl_up_sync(0xffffffffu, T[RC - 1], 1) & nz0);
#pragma unroll
        for (int k = RC - 1; k >= 1; --k) T[k] = T[k - 1] + eb[k] - old[k];
        T[0] = tl + eb[0] - old[0];
#pragma unroll
        for (int k = 0; k < RC; ++k) ring[U][k] = eb[k];
    }
};

template <int V> struct IC { static constexpr int value = V; };
template <bool V> struct BC { static constexpr bool value = V; };

// ------------------------------------------------------------------------------------------------
// Streamed side of a sweep: per-warp double buffer in shared memory, filled by the TMA engine
// (cp.async.bulk global -> shared, completion on an mbarrier).  A stage holds the 9 streamed frames of one
// round of the register ring (432 B) and the row parameters that go with them; while the warp works on a
// stage the copy of the next one is in flight, so no warp ever waits on an L2 / HBM access for the frames
// (with plain loads every warp of an SM stalled on the same cache line once per 2.7 rows:
// profiles/r2_k2_tma.md).  Reads are warp-uniform LDS.128 broadcasts.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *b, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(unsigned long long *b) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *b, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, unsigned long long *b) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(b))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *b, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LAB_DONE;\n"
        "bra LAB_WAIT;\n"
        "LAB_DONE:\n"
        "}\n" ::"r"(smem_u32(b)),
        "r"(parity)
        : "memory");
}

constexpr int ST_N = 2;                            // stages per warp
template <typename PT>
struct alignas(16) StreamBuf {
    static constexpr int PAL = 16 / (int)sizeof(PT);                   // parameters per 16 bytes (copy granularity)
    static constexpr int PCOPY = (M9 + PAL - 1 + PAL - 1) / PAL * PAL; // parameters copied per stage (start aligned down)
    ulonglong2 x[ST_N][M9][3];                     // 9 frames of 48 B
    PT p[ST_N][PCOPY];
    unsigned long long full[ST_N];
};

// Drives a sweep over streamed frames 0 .. nrows-1 (nrows >= 10 always: Mx >= 2) in rounds of 9 rows = one stage =
// one round of the register ring (static ring slots, immediate shared-memory offsets).  fn(a, param) runs for rows
// a >= HALO, param = P[a - HALO].
template <int RC, typename PT, typename Fn>
__device__ __forceinline__ void run_sweep(Sweep<RC> &sw, const float *__restrict__ X, const PT *__restrict__ P,
                                          int nrows, StreamBuf<PT> *sb, int lane, Fn &&fn) {
    using SB = StreamBuf<PT>;
    const int nchunks = (nrows + M9 - 1) / M9;
    auto pbase = [](int c) { return max(0, c * M9 - HALO) / SB::PAL * SB::PAL; };   // first parameter a stage holds
    auto issue = [&](int c) {                      // one lane: start the copies of round c into stage c & 1
        const int st = c & 1;
        const uint32_t xb = (uint32_t)min(M9, nrows - c * M9) * (NBINS * 4), pb = SB::PCOPY * (uint32_t)sizeof(PT);
        mbar_expect_tx(&sb->full[st], xb + pb);
        bulk_g2s(&sb->x[st][0][0], X + (size_t)c * M9 * NBINS, xb, &sb->full[st]);
        bulk_g2s(&sb->p[st][0], P + pbase(c), pb, &sb->full[st]);
    };
    if (lane == 0) {
        mbar_init(&sb->full[0], 1);
        mbar_init(&sb->full[1], 1);
        mbar_fence_init();
        issue(0);
        if (nchunks > 1) issue(1);
    }
    __syncwarp();
    int a = 0, c = 0;
    const ulonglong2 *xs = nullptr;
    const PT *ps = nullptr;
    auto begin_round = [&]() {
        const int st = c & 1;
        mbar_wait(&sb->full[st], (uint32_t)((c >> 1) & 1));
        xs = &sb->x[st][0][0];
        ps = &sb->p[st][0] + (c * M9 - HALO - pbase(c));          // ps[r] = parameter of row 9c + r
    };
    auto end_round = [&]() {
        __syncwarp();                              // every lane has read the stage
        if (lane == 0 && c + ST_N < nchunks) issue(c + ST_N);
        ++c;
    };
    auto step = [&](auto uc, auto callc) {
        constexpr int U = decltype(uc)::value;     // row within the round = ring slot
        constexpr bool CALL = decltype(callc)::value;
        int eb[RC];
        const ulonglong2 x0 = xs[3 * U], x1 = xs[3 * U + 1], x2 = xs[3 * U + 2];
        sw.dot(x0, x1, x2, eb);
        sw.template finish<U>(eb);
        if (CALL) {
            const PT prm = ps[U];                  // one read of the row's parameters (the callee may store to shared memory)
            fn(a, prm);
        }
        ++a;
    };
    // rows 0..8: the diagonal sums fill up; only row 8 produces a window
    begin_round();
    step(IC<0>{}, BC<false>{}); step(IC<1>{}, BC<false>{}); step(IC<2>{}, BC<false>{});
    step(IC<3>{}, BC<false>{}); step(IC<4>{}, BC<false>{}); step(IC<5>{}, BC<false>{});
    step(IC<6>{}, BC<false>{}); step(IC<7>{}, BC<false>{}); step(IC<8>{}, BC<true>{});
    end_round();
#pragma unroll 1
    while (a + M9 <= nrows) {
        begin_round();
        step(IC<0>{}, BC<true>{}); step(IC<1>{}, BC<true>{}); step(IC<2>{}, BC<true>{});
        step(IC<3>{}, BC<true>{}); step(IC<4>{}, BC<true>{}); step(IC<5>{}, BC<true>{});
        step(IC<6>{}, BC<true>{}); step(IC<7>{}, BC<true>{}); step(IC<8>{}, BC<true>{});
        end_round();
    }
    const int rem = nrows - a;                     // 0..8 rows left, ring slots 0..rem-1
    if (rem > 0) {
        begin_round();
        step(IC<0>{}, BC<true>{});
        if (rem > 1) step(IC<1>{}, BC<true>{});
        if (rem > 2) step(IC<2>{}, BC<true>{});
        if (rem > 3) step(IC<3>{}, BC<true>{});
        if (rem > 4) step(IC<4>{}, BC<true>{});
        if (rem > 5) step(IC<5>{}, BC<true>{});
        if (rem > 6) step(IC<6>{}, BC<true>{});
        if (rem > 7) step(IC<7>{}, BC<true>{});
    }
}

// ------------------------------------------------------------------------------------------------
// Bracket update shared by the dense and the sparse histogram levels.  hist[b * stride] (shifted / masked)
// is the count of bin b: b = 0 items below the bracket, 1..NBIN its bins, NBIN + 1 items above.  The new
// bracket is the run of bins holding ranks fk and ck (the under / overflow "bins" reach to the end of the
// pair's item range, the next level splits them).
// ------------------------------------------------------------------------------------------------
// cells a finished bracket may hold: BRACKET_TARGET on long lines, a sixteenth of the line on short ones (every
// bracket cell is an uncertain cell of the emit sweep, and a short line has few cells to begin with)
__device__ __forceinline__ int bracket_target(int line_len) { return min(BRACKET_TARGET, max(6, line_len >> 4)); }

struct Bracket {
    int lo, w, below, sh;       // new origin, width, exact count of items below lo, shift of the next level
    bool done, miss, bad;
};

template <int STRIDE>
__device__ __forceinline__ Bracket split_bracket(const uint32_t *hp, int hs, uint32_t mask, int fk, int ck, int lo, int sh,
                                                 int rlo, int rhi, int target) {
    int cum = 0, b1 = -2, b2 = -2, cb1 = 0, cend = 0;          // the underflow bin counts every item below the bracket
    for (int b = 0; b < NBIN + 2; ++b) {                      // b - 1 = bin of the bracket; -1 under, NBIN over
        const int c = (int)((hp[b * STRIDE] >> hs) & mask);
        if (b1 < -1 && cum + c > fk) { b1 = b - 1; cb1 = cum; }
        if (b2 < -1 && cum + c > ck) { b2 = b - 1; cend = cum + c; }
        cum += c;
    }
    Bracket r;
    r.bad = (b1 < -1 || b2 < -1);
    const long long nlo = (b1 < 0) ? (long long)rlo : (long long)lo + ((long long)b1 << sh);
    const long long nhi = (b2 >= NBIN) ? (long long)rhi : (b2 < 0) ? (long long)lo : (long long)lo + ((long long)(b2 + 1) << sh);
    r.miss = (b1 < 0) || (b2 >= NBIN);
    const long long range = (nhi > nlo) ? nhi - nlo : 1;
    int sh2 = 0;
    while ((range >> sh2) > NBIN) ++sh2;
    // split again unless the bracket is small enough or cannot shrink
    r.done = !r.miss && ((cend - cb1 <= target) || (sh == 0));
    r.lo = (int)nlo; r.w = (int)range; r.below = cb1; r.sh = sh2;
    return r;
}

constexpr int SPARSE_LEVELS = 3;
constexpr int DENSE2_MIN_LIVE = 16;  // live lines a strip must hold for the second dense level to sweep it

#include "k2_tc.inl"

// ------------------------------------------------------------------------------------------------
// histogram sweep.  ORIENT = 0: owned = reference columns (column thresholds), streamed = query.
//                   ORIENT = 1: owned = query rows (row thresholds), streamed = rotated reference.
// Every live line enters with a bracket [lo, lo + 64 << sh) (first level: from the sample selection).  The
// sweep counts the line's items into 64 bins of the bracket plus an underflow and an overflow bin, so the
// position of the wanted ranks is known exactly whatever the bracket was: inside (bracket shrinks to the
// bins holding floor(k) .. ceil(k)), below or above (bracket moves to that side of the pair's item range
// and the next level splits it).
// ------------------------------------------------------------------------------------------------
template <int RC, int ORIENT>
__global__ void __launch_bounds__(32 * WPC, MINB) fast_hist_kernel(TrackSet ts, const int32_t *__restrict__ pairs,
                                                             int64_t first, int n, FastLayout L,
                                                             char *__restrict__ scratch, int strips_max, float magic,
                                                             uint32_t *__restrict__ status, uint32_t *__restrict__ dbg,
                                                             int min_live, int final_level, uint32_t *__restrict__ glive,
                                                             uint32_t gcap) {
    extern __shared__ uint32_t s_hist[];                      // [WPC][NBIN + 2][RC / 2][32], two 16-bit counters per word
    using SW = Sweep<RC>;
    static_assert(RC % 2 == 0, "histogram packing needs an even number of register columns");
    constexpr int HW = RC / 2;                                // words per (bin, lane)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t task = (int64_t)blockIdx.x * WPC + warp;
    const int slot = (int)(task / strips_max), strip = (int)(task % strips_max);
    if (slot >= n) return;
    const PairHdr *h = slot_ptr<PairHdr>(scratch, L, slot, L.off_hdr);
    if (h->quirk[ORIENT == 0 ? 1 : 0]) return;               // threshold forced to 0: nothing to select
    const int64_t k = first + slot;
    const int q = pairs[2 * k];
    const int nY = (ORIENT == 0) ? h->nr : h->nq, nX = (ORIENT == 0) ? h->nq : h->nr;
    const int My = nY - M9;                                   // owned windows
    const int cb = strip * SW::OUTW;
    if (cb >= My) return;
    const float *Qf = ts.frames + ts.offsets[q] * NBINS;
    const float *Rf = slot_ptr<float>(scratch, L, slot, L.off_rrot);
    const float *Y = (ORIENT == 0) ? Rf : Qf, *X = (ORIENT == 0) ? Qf : Rf;
    const int32_t *xn = slot_ptr<int32_t>(scratch, L, slot, ORIENT == 0 ? L.off_aai : L.off_bbi);
    const int32_t *yn = slot_ptr<int32_t>(scratch, L, slot, ORIENT == 0 ? L.off_bbi : L.off_aai);
    const int line0 = (ORIENT == 0) ? L.max_rows : 0;         // first line index of the owned side
    int32_t *lo_a = slot_ptr<int32_t>(scratch, L, slot, L.off_lo) + line0;
    int32_t *w_a = slot_ptr<int32_t>(scratch, L, slot, L.off_w) + line0;
    int32_t *cb_a = slot_ptr<int32_t>(scratch, L, slot, L.off_cb) + line0;
    int32_t *sh_a = slot_ptr<int32_t>(scratch, L, slot, L.off_sh) + line0;

    // a line is live while its bracket still holds more than BRACKET_TARGET cells and can be split further
    // (shift >= 0 in sh_a; -1 = done).  Strips with nothing left to do return at once, so the extra levels
    // cost nothing on ordinary pairs.
    int ynrel[RC], shf[RC];
    bool valid[RC];
    bool work = false;
#pragma unroll
    for (int kk = 0; kk < RC; ++kk) {
        const int j = cb + RC * lane + kk - HALO;            // owned window of this register column
        valid[kk] = (j >= cb) && (j < My) && (j < cb + SW::OUTW);
        const int shv = valid[kk] ? sh_a[j] : -1;
        if (shv < 0) valid[kk] = false;
        shf[kk] = valid[kk] ? shv : 0;
        // bin index = ((z - lo) >> sh) + 1 clamped to [0, NBIN + 1]: 0 = below the bracket, NBIN + 1 = above
        ynrel[kk] = valid[kk] ? yn[j] - lo_a[j] + (1 << shv) : 0x40000000;   // idle columns land in the overflow bin
        work |= valid[kk];
    }
    if (!__any_sync(0xffffffffu, work)) return;
    int n_live = 0, n_miss = 0, n_left = 0;                  // diagnostics (acoss_debug_counters)
#pragma unroll
    for (int kk = 0; kk < RC; ++kk) n_live += valid[kk] ? 1 : 0;
    const int side = (ORIENT == 0) ? 1 : 0;
    // a line the sparse refinement has to finish goes to the CALL-wide list (lines of all pairs share its warps)
    auto to_sparse = [&](int line) {
        const unsigned pos = atomicAdd(glive, 1u);
        if (pos < gcap) glive[1 + pos] = ((uint32_t)slot << 16) | ((uint32_t)side << 15) | (uint32_t)line;
        else atomicOr(&status[k], PAIR_ST_FALLBACK | 8u);     // reason 8: too many crowded lines in this call
    };
    if (__reduce_add_sync(0xffffffffu, n_live) < min_live) {
        // too few live lines to pay for a dense sweep of the strip: they go to the sparse refinement as they are
#pragma unroll
        for (int kk = 0; kk < RC; ++kk)
            if (valid[kk]) to_sparse(cb + RC * lane + kk - HALO);
        return;
    }
    SW sw;
    sw.init(Y, nY, cb, lane, magic);
    uint32_t *hist = s_hist + (size_t)warp * (NBIN + 2) * HW * 32 + lane;
#pragma unroll 1
    for (int b = 0; b < (NBIN + 2) * HW; ++b) hist[b * 32] = 0u;
    __syncwarp();

    const int nrows = nX - 1;                                 // streamed frames 0 .. nX-2 (F4: last frame unused)
    __shared__ StreamBuf<int> s_stream[WPC];
    run_sweep<RC, int>(sw, X, xn, nrows, &s_stream[warp], lane, [&](int, int xb) {
#pragma unroll
        for (int kk = 0; kk < RC; ++kk) {
            const int zr = xb + ynrel[kk] - sw.T[kk];
            const int idx = __vimin_s32_relu(zr >> shf[kk], NBIN + 1);
            atomicAdd(&hist[(idx * HW + kk / 2) * 32], 1u << (16 * (kk & 1)));   // thread-private bank: conflict-free
        }
    });
    __syncwarp();
    // per-thread scan of its own columns' histograms
    const int fk = h->fk[side], ck = h->ck[side];
    const int rlo = h->lo1, rhi = h->hi1;
#pragma unroll
    for (int kk = 0; kk < RC; ++kk) {
        if (!valid[kk]) continue;
        const int j = cb + RC * lane + kk - HALO;
        const Bracket br = split_bracket<HW * 32>(hist + (kk / 2) * 32, 16 * (kk & 1), 0xffffu, fk, ck, lo_a[j], shf[kk], rlo, rhi,
                                                  bracket_target(nX - M9));
        if (br.bad) {                                         // cannot happen: the bins cover every item of the line
            atomicOr(&status[k], PAIR_ST_FALLBACK | 4u);      // reason 4: rank not found
            sh_a[j] = -1;
            continue;
        }
        lo_a[j] = br.lo;
        w_a[j] = br.w;
        cb_a[j] = br.below;
        sh_a[j] = br.done ? -1 : br.sh;
        n_miss += br.miss ? 1 : 0;
        n_left += br.done ? 0 : 1;
        if (ORIENT == 1) {
            int4 *rowpack = slot_ptr<int4>(scratch, L, slot, L.off_rowpack);
            rowpack[j] = pack_row(yn[j], br.lo, br.w);
        }
        if (!br.done && final_level) to_sparse(j);            // the sparse level refines it
    }
    n_live = __reduce_add_sync(0xffffffffu, n_live);
    n_miss = __reduce_add_sync(0xffffffffu, n_miss);
    n_left = __reduce_add_sync(0xffffffffu, n_left);
    if (lane == 0) {
        atomicAdd(&dbg[0], 1u); atomicAdd(&dbg[1], (unsigned)n_live);
        if (n_miss) atomicAdd(&dbg[2], (unsigned)n_miss);
        if (n_left) atomicAdd(&dbg[3], (unsigned)n_left);
    }
}

// ------------------------------------------------------------------------------------------------
// sparse refinement: the few lines whose bracket is still crowded after the dense level (or whose ranks
// fell outside the sampled bracket).  One lane owns one line: the 9 owned frames of its window stay in
// registers, every streamed frame feeds the 9 rows in flight (acc[(a - t) % 9] += e(a, t)), one row
// completes per step.  The quantised dot products are the same FMA chains as in the sweeps, so the items
// are identical.  A warp repeats the sweep until all its lines are done (at most SPARSE_LEVELS times).
// ------------------------------------------------------------------------------------------------

template <int U>
__device__ __forceinline__ void sparse_step(const float (&y)[M9][NBINS], int (&acc)[M9], const float (&x)[NBINS], float magic) {
#pragma unroll
    for (int t = 0; t < M9; ++t) {
        const int e = dot_fx(x, y[t], magic);
        const int slot = ((U - t) % M9 + M9) % M9;            // row a - t lives in slot (a - t) % 9
        if (t == 0) acc[slot] = e;
        else acc[slot] += e;
    }
}

__global__ void __launch_bounds__(32 * WPC, 2) fast_sparse_kernel(TrackSet ts, const int32_t *__restrict__ pairs,
                                                                  int64_t first, int n, FastLayout L,
                                                                  char *__restrict__ scratch, float magic,
                                                                  uint32_t *__restrict__ status, uint32_t *__restrict__ dbg,
                                                                  const uint32_t *__restrict__ glive, uint32_t gcap) {
    __shared__ uint32_t s_sp[WPC][NBIN + 2][32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t cnt = min(glive[0], gcap);
    const uint32_t e0 = ((uint32_t)blockIdx.x * WPC + warp) * 32u;
    if (e0 >= cnt) return;
    // one lane = one line; the 32 lines of a warp may belong to 32 different pairs (everything below is lane-private)
    bool livel = e0 + lane < cnt;
    const uint32_t ent = glive[1 + (livel ? e0 + lane : e0)];
    const int slot = (int)(ent >> 16), side = (int)((ent >> 15) & 1u), j = (int)(ent & 0x7fffu);   // side 0: rows (owned = query)
    const int64_t k = first + slot;
    const PairHdr *h = slot_ptr<PairHdr>(scratch, L, slot, L.off_hdr);
    const int q = pairs[2 * k];
    const int nY = side ? h->nr : h->nq, nX = side ? h->nq : h->nr;
    const float *Qf = ts.frames + ts.offsets[q] * NBINS;
    const float *Rf = slot_ptr<float>(scratch, L, slot, L.off_rrot);
    const float *Y = side ? Rf : Qf, *X = side ? Qf : Rf;
    const int32_t *xn = slot_ptr<int32_t>(scratch, L, slot, side ? L.off_aai : L.off_bbi);
    const int32_t *yn = slot_ptr<int32_t>(scratch, L, slot, side ? L.off_bbi : L.off_aai);
    const int line0 = side ? L.max_rows : 0;
    int32_t *lo_a = slot_ptr<int32_t>(scratch, L, slot, L.off_lo) + line0;
    int32_t *w_a = slot_ptr<int32_t>(scratch, L, slot, L.off_w) + line0;
    int32_t *cb_a = slot_ptr<int32_t>(scratch, L, slot, L.off_cb) + line0;
    int32_t *sh_a = slot_ptr<int32_t>(scratch, L, slot, L.off_sh) + line0;
    // owned window j: frames j .. j+8, pre-doubled (the sweeps double the owned side too)
    float y[M9][NBINS];
#pragma unroll
    for (int t = 0; t < M9; ++t) load_frame(Y + (int64_t)min(j + t, nY - 1) * NBINS, y[t], 2.f);
    const int ynj = yn[j];
    const int fk = h->fk[side], ck = h->ck[side], rlo = h->lo1, rhi = h->hi1;
    const int mb9 = NMAGIC * M9 * __float_as_int(magic);      // the magic offsets inside a completed sum (mod 2^32)
    uint32_t *hist = &s_sp[warp][0][lane];
    int lo = lo_a[j], sh = sh_a[j];
    if (sh < 0) livel = false;
    const int nrows = nX - 1;                                 // this lane's streamed frames 0 .. nX-2
    const int nrows_w = __reduce_max_sync(0xffffffffu, nrows);
    int n_swept = 0;
    for (int lvl = 0; lvl < SPARSE_LEVELS && __any_sync(0xffffffffu, livel); ++lvl) {
        ++n_swept;
#pragma unroll 1
        for (int b = 0; b < NBIN + 2; ++b) hist[b * 32] = 0u;
        const int shl = max(sh, 0);
        const int yrel = livel ? ynj - lo + (1 << shl) : 0x40000000;   // idle lanes land in the overflow bin
        const float *px = X;
        float xc[NBINS];
        load_frame(px, xc, 1.f);
        int acc[M9];
#pragma unroll
        for (int u = 0; u < M9; ++u) acc[u] = 0;
        int a = 0;
        auto step = [&](auto uc) {
            constexpr int U = decltype(uc)::value;
            sparse_step<U>(y, acc, xc, magic);
            if (a + 1 < nX) px += NBINS;                      // lanes past the end of their track keep their last frame
            load_frame(px, xc, 1.f);
            if (a >= HALO && a < nrows) {                     // row a - 8 is complete (slot (U + 1) % 9)
                const int T = acc[(U + 1) % M9] - mb9;
                const int zr = __ldg(xn + a - HALO) + yrel - T;
                const int idx = __vimin_s32_relu(zr >> shl, NBIN + 1);
                atomicAdd(&hist[idx * 32], 1u);
            }
            ++a;
        };
#pragma unroll 1
        while (a + M9 <= nrows_w) {
            step(IC<0>{}); step(IC<1>{}); step(IC<2>{}); step(IC<3>{}); step(IC<4>{});
            step(IC<5>{}); step(IC<6>{}); step(IC<7>{}); step(IC<8>{});
        }
        const int remr = nrows_w - a;
        if (remr > 0) step(IC<0>{});
        if (remr > 1) step(IC<1>{});
        if (remr > 2) step(IC<2>{});
        if (remr > 3) step(IC<3>{});
        if (remr > 4) step(IC<4>{});
        if (remr > 5) step(IC<5>{});
        if (remr > 6) step(IC<6>{});
        if (remr > 7) step(IC<7>{});
        __syncwarp();
        if (livel) {
            const Bracket br = split_bracket<32>(hist, 0, 0xffffffffu, fk, ck, lo, sh, rlo, rhi, bracket_target(nX - M9));
            if (br.bad) { atomicOr(&status[k], PAIR_ST_FALLBACK | 4u); livel = false; sh_a[j] = -1; }
            else {
                lo = br.lo; sh = br.sh;
                lo_a[j] = br.lo; w_a[j] = br.w; cb_a[j] = br.below; sh_a[j] = br.done ? -1 : br.sh;
                if (side == 0) slot_ptr<int4>(scratch, L, slot, L.off_rowpack)[j] = pack_row(ynj, br.lo, br.w);
                if (br.done) livel = false;
            }
        }
        __syncwarp();
    }
    if (lane == 0) { atomicAdd(&dbg[0], 1u); atomicAdd(&dbg[1], (unsigned)n_swept); }
    const unsigned left = __ballot_sync(0xffffffffu, livel);
    if (lane == 0 && left) atomicAdd(&dbg[2], (unsigned)__popc(left));
}

// ------------------------------------------------------------------------------------------------
// emit sweep (orientation 0: owned = reference columns, streamed = query rows)
//
// One CTA = WPC adjacent strips of one pair = 480 CRP columns = 15 whole CRP words per row, so the CTA owns
// its words: plain stores, no atomics on HBM, no zero-filled CRP to start from.  Per cell the sweep
// classifies: "certainly 1" (one bit shifted into a lane-private accumulator, 4 columns x 8 rows) and
// "uncertain" (inside a row / column bracket widened by 2 EPS, or near zero).  An uncertain cell's record
// (i | j << 14, fixed-point item) goes to a lane-private staging column in shared memory with one predicated
// store.  Every 8 rows the 8 x 8 nibble matrix held by each group of 8 lanes is transposed with three butterfly
// shuffles (lane p then holds the 32 columns of row 7 - p) and OR-ed into a small shared tile at the strip's bit
// offset; the staged records are compacted to the pair's pool (one atomic per warp); after one named barrier the
// CTA's threads store the tile as plain CRP words.
// ------------------------------------------------------------------------------------------------
constexpr int EMIT_ROWS = 8;                       // rows per flush block (8 rows x 4 columns = one 32-bit accumulator)
constexpr int EMIT_TW = 16;                        // tile words per row: word 0 holds only halo bits (always zero)
constexpr int EMIT_CW = WPC * (32 * RCV - HALO) / 32;   // CRP words a CTA owns per row (15)
constexpr int EMIT_STAGE = 4 * EMIT_ROWS;           // staged records per lane and flush block: every cell of the block fits

// 8 x 8 nibble transpose across the 8 lanes of a group: out(lane p) nibble q = in(lane q) nibble p
__device__ __forceinline__ unsigned transpose_nibbles(unsigned x, unsigned selA, unsigned selB, unsigned rotC, unsigned mskC) {
    unsigned y = __shfl_xor_sync(0xffffffffu, x, 4);
    x = __byte_perm(x, y, selA);                           // 16-bit halves
    y = __shfl_xor_sync(0xffffffffu, x, 2);
    x = __byte_perm(x, y, selB);                           // bytes
    y = __shfl_xor_sync(0xffffffffu, x, 1);
    y = __funnelshift_l(y, y, rotC);                       // rotate by +-4 bits, the wrapped nibble is masked off
    return (x & mskC) | (y & ~mskC);                       // nibbles
}

template <int RC>
__global__ void __launch_bounds__(32 * WPC, MINB) fast_emit_kernel(TrackSet ts, const int32_t *__restrict__ pairs,
                                                             int64_t first, int n, FastLayout L,
                                                             char *__restrict__ scratch, int groups, float magic,
                                                             uint32_t *__restrict__ crp_all, int words,
                                                             int64_t crp_words) {
    using SW = Sweep<RC>;
    static_assert(RC == 4 && WPC == 4 && EMIT_CW * 32 == WPC * SW::OUTW, "a CTA must own whole CRP words");
    __shared__ uint32_t s_tile[2][EMIT_ROWS][EMIT_TW + 1];    // [buffer][row][word] (+1: the last strip's empty spill word)
    __shared__ uint2 s_stage[WPC][EMIT_STAGE][32];            // [warp][entry][lane]: lane-private columns, conflict-free
    __shared__ StreamBuf<int4> s_stream[WPC];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = blockIdx.x / groups, grp = blockIdx.x - slot * groups;
    if (slot >= n) return;
    const PairHdr *h = slot_ptr<PairHdr>(scratch, L, slot, L.off_hdr);
    const int64_t k = first + slot;
    const int q = pairs[2 * k];
    const int nY = h->nr, nX = h->nq, My = nY - M9, Mx = nX - M9;
    uint32_t *crp = crp_all + (int64_t)slot * crp_words;
    const int w_first = grp * EMIT_CW;                        // first CRP word of this CTA
    const int cb0 = grp * WPC * SW::OUTW;                     // first CRP column of this CTA
    const int nact = min(WPC, max(0, (My - cb0 + SW::OUTW - 1) / SW::OUTW));   // strips with columns
    if (nact == 0) {
        // nothing to sweep: the CTA's words of the pair's rows are zero (K3 reads the whole row pitch)
        const int nw = min(words, w_first + EMIT_CW) - w_first;
        if (nw <= 0) return;
        for (int e = threadIdx.x; e < Mx * nw; e += blockDim.x) {
            const int i = e / nw, w = w_first + (e - i * nw);
            crp[(int64_t)i * words + w] = 0u;
        }
        return;
    }
    for (int e = threadIdx.x; e < 2 * EMIT_ROWS * (EMIT_TW + 1); e += blockDim.x) (&s_tile[0][0][0])[e] = 0u;
    __syncthreads();
    if (warp >= nact) return;
    const int nthr = 32 * nact;
    const int cb = cb0 + warp * SW::OUTW;
    const float *X = ts.frames + ts.offsets[q] * NBINS;
    const float *Y = slot_ptr<float>(scratch, L, slot, L.off_rrot);
    const int32_t *yn = slot_ptr<int32_t>(scratch, L, slot, L.off_bbi);
    const int4 *rowpack = slot_ptr<int4>(scratch, L, slot, L.off_rowpack);
    const int32_t *lo_c = slot_ptr<int32_t>(scratch, L, slot, L.off_lo) + L.max_rows;
    const int32_t *w_c = slot_ptr<int32_t>(scratch, L, slot, L.off_w) + L.max_rows;
    uint2 *pool = slot_ptr<uint2>(scratch, L, slot, L.off_pool);
    uint32_t *pool_ctr = slot_ptr<uint32_t>(scratch, L, slot, L.off_pcnt);
    const unsigned pool_cap = (unsigned)L.pool_cap;

    SW sw;
    sw.init(Y, nY, cb, lane, magic);
    int ynv[RC], ycl[RC];                                     // bb_fix[j], bb_fix[j] - (colLo - 2 EPS)
    unsigned cw1[RC];                                         // colW + 4 EPS - 1
#pragma unroll
    for (int kk = 0; kk < RC; ++kk) {
        const int j = cb + RC * lane + kk - HALO;
        const bool valid = (j >= cb) && (j < My) && (j < cb + SW::OUTW);
        ynv[kk] = valid ? yn[j] : 0x20000000;                 // invalid: item huge => never in, never uncertain
        ycl[kk] = valid ? yn[j] - (lo_c[j] - 2 * EPS) : 0x20000000;
        cw1[kk] = valid ? (unsigned)(w_c[j] + 4 * EPS - 1) : 0u;
    }
    // Tile placement.  Strip bit t = RC * lane + kk <-> CRP column cb - HALO + t <-> tile bit 32 + (cb - cb0) - HALO + t
    // (tile word 0 = the CRP word before the CTA's first one: only halo bits land there, and they are zero).
    const int tbit0 = 32 + warp * SW::OUTW - HALO;            // tile bit of the strip's first (halo) column
    const int tw0 = (tbit0 >> 5) + (lane >> 3);               // tile word of this lane's 8-lane group
    const int toff = tbit0 & 31;                              // 24, 16, 8, 0 for warps 0..3
    const int grow = 7 - (lane & 7);                          // block row this lane holds after the transpose
    // transpose constants (lane p of a group: bits 4, 2, 1 of p select the half it keeps)
    const unsigned selA = (lane & 4) ? 0x3276u : 0x5410u, selB = (lane & 2) ? 0x3715u : 0x6240u;
    const unsigned rotC = (lane & 1) ? 28u : 4u, mskC = (lane & 1) ? 0xf0f0f0f0u : 0x0f0f0f0fu;
    const unsigned jcol0 = (unsigned)(cb + RC * lane - HALO) << 14;   // column part of a record (+ kk << 14)
    unsigned accI = 0u;
    uint2 *stage = &s_stage[warp][0][lane];
    unsigned ns = 0u;                                         // staged records of this lane in the current block

    auto flush = [&](int blk) {
        const unsigned wi = transpose_nibbles(accI, selA, selB, rotC, mskC);
        accI = 0u;
        uint32_t *ti = &s_tile[blk & 1][grow][tw0];
        const unsigned long long w2 = (unsigned long long)wi << toff;      // branch-free: the word and its spill into the next
        atomicOr(ti, (unsigned)w2);
        atomicOr(ti + 1, (unsigned)(w2 >> 32));
        // staged uncertain cells -> the pair's pool: exclusive prefix of the lanes' counts, one atomic per warp
        if (__any_sync(0xffffffffu, ns != 0u)) {
            const unsigned cnt = ns;
            unsigned incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            unsigned base = 0u;
            if (lane == 31) base = atomicAdd(pool_ctr, incl);
            base = __shfl_sync(0xffffffffu, base, 31) + incl - cnt;
#pragma unroll 1
            for (unsigned e = 0; e < cnt; ++e)
                if (base + e < pool_cap) pool[base + e] = stage[e * 32];
            ns = 0u;
        }
        asm volatile("bar.sync 1, %0;" ::"r"(nthr) : "memory");
        // the CTA's threads store the block: 8 rows x 15 words (tile word 0 is not a CRP word of ours)
#pragma unroll 1
        for (int e = threadIdx.x; e < EMIT_ROWS * EMIT_TW; e += nthr) {
            const int g = e >> 4, tw = e & (EMIT_TW - 1);
            uint32_t *pi = &s_tile[blk & 1][g][tw];
            const uint32_t vi = *pi;
            *pi = 0u;                                          // ready for block blk + 2 (one barrier in between)
            const int i = blk * EMIT_ROWS + g, w = w_first + tw - 1;
            if (tw >= 1 && i < Mx && w < words) crp[(int64_t)i * words + w] = vi;
        }
    };

    const int nrows = nX - 1;
    // Per cell, with z the fixed-point item (sign-bit / unsigned-compare arithmetic):
    //   ar = z - (rowLo - 2 EPS), ac = z - (colLo - 2 EPS)
    //   certainly in  <=> ar < 0 and ac < 0                                  sign(ar & ac)
    //   row zone      <=> 0 <= ar <= rw1 (rw1 = rowW + 4 EPS - 1)            (unsigned)ar <= rw1
    //   near zero     <=> z < 2 EPS  <=>  ar < 4 EPS - rowLo                 (always evaluated exactly: F7's NaN)
    //   uncertain     <=> row zone or column zone or near zero
    // A near-zero cell that is certainly in is emitted as 1 and listed as well: its exact evaluation either
    // confirms a tiny distance or raises the NaN error.
    // (rp by value: a reference into the stage buffer would be re-read after every staging store, which may alias it)
    run_sweep<RC, int4>(sw, X, rowpack, nrows, &s_stream[warp], lane, [&](int a, const int4 rp) {   // rp = pack_row(..)
        const int xr = rp.w, nz = rp.y;
        const unsigned rw1 = (unsigned)(rp.z - 1);
        const int i = a - HALO;                               // CRP row
        const unsigned rec0 = (unsigned)i | jcol0;
#pragma unroll
        for (int kk = RC - 1; kk >= 0; --kk) {
            const int ar = xr + ynv[kk] - sw.T[kk];
            const int ac = rp.x + ycl[kk] - sw.T[kk];
            const bool unc = ((unsigned)ar <= rw1) || ((unsigned)ac <= cw1[kk]) || (ar < nz);
            accI = __funnelshift_l((unsigned)(ar & ac), accI, 1);   // sign bit -> bit 0, earlier cells move up
            if (unc) {
                stage[ns * 32] = make_uint2(rec0 + ((unsigned)kk << 14), (unsigned)ar);
                ++ns;
            }
        }
        if ((i & (EMIT_ROWS - 1)) == EMIT_ROWS - 1) flush(i >> 3);
    });
    if (Mx & (EMIT_ROWS - 1)) {                               // last, partial block: missing rows are zero
        accI <<= 4 * (EMIT_ROWS - (Mx & (EMIT_ROWS - 1)));
        flush(Mx >> 3);
    }
}

// ------------------------------------------------------------------------------------------------
// scatter: the pair's pool of uncertain cells -> per-row / per-column candidate lists (index + fixed-point item).  A
// candidate is flagged "below" when it lies below its line's bracket in the item the histogram levels counted: z (FFMA2
// sweeps) or z' (tensor sweeps, z <= z' <= z + dz).  With ar = z - (lo - dz - 2 EPS): below for ar < 2 EPS, not below for
// ar >= dz + 2 EPS; the cells in between (the band, tensor sweeps only) are queued and their z' recomputed from the byte
// planes once the CTA's records are placed.
// ------------------------------------------------------------------------------------------------
constexpr int SCAT_CHUNK = 4096;    // pool records per CTA

__global__ void __launch_bounds__(256, 4) fast_scatter_kernel(int n, FastLayout L, char *__restrict__ scratch,
                                                           int64_t first, TcShift sh3, uint32_t *__restrict__ status,
                                                           uint32_t *__restrict__ dbg) {
    __shared__ uint32_t s_band[SCAT_CHUNK];                   // record - e0 | row slot << 12 | column slot << 20 (0xff: none)
    __shared__ int s_nband;
    const int slot = blockIdx.y;
    if (slot >= n) return;
    const uint32_t cntv = *slot_ptr<uint32_t>(scratch, L, slot, L.off_pcnt);
    const uint32_t e0 = blockIdx.x * SCAT_CHUNK;
    if (e0 >= cntv && blockIdx.x) return;
    if (threadIdx.x == 0) s_nband = 0;
    __syncthreads();
    const int dz = slot_ptr<PairHdr>(scratch, L, slot, L.off_hdr)->dz;
    if (cntv > (uint32_t)L.pool_cap && blockIdx.x == 0 && threadIdx.x == 0)
        atomicOr(&status[first + slot], PAIR_ST_FALLBACK | 16u);          // reason 16: pool overflow
    const uint32_t m = min(min(cntv, (uint32_t)L.pool_cap), e0 + SCAT_CHUNK);
    const uint2 *pool = slot_ptr<uint2>(scratch, L, slot, L.off_pool);
    uint32_t *cnt = slot_ptr<uint32_t>(scratch, L, slot, L.off_cnt);
    uint16_t *cand = slot_ptr<uint16_t>(scratch, L, slot, L.off_cand);
    int32_t *candz = slot_ptr<int32_t>(scratch, L, slot, L.off_candz);
    const int4 *rowpack = slot_ptr<int4>(scratch, L, slot, L.off_rowpack);
    const int32_t *lo_c = slot_ptr<int32_t>(scratch, L, slot, L.off_lo) + L.max_rows;
    const int32_t *w_c = slot_ptr<int32_t>(scratch, L, slot, L.off_w) + L.max_rows;
    // four records per thread and round: the returning atomics of a round are independent, their latency overlaps
    constexpr int SU = 4;
    for (uint32_t eb = e0 + threadIdx.x; eb < m; eb += SU * blockDim.x) {
        int ii[SU], jj[SU], zz_[SU];
        unsigned pr[SU], pc[SU];
        bool rz[SU], cz[SU], lowr[SU], lowc[SU], bandr[SU], bandc[SU];
#pragma unroll
        for (int u = 0; u < SU; ++u) {
            const uint32_t e = eb + u * blockDim.x;
            rz[u] = cz[u] = false;
            if (e < m) {
                const uint2 rec = pool[e];
                const int i = rec.x & 0x3fff, j = (rec.x >> 14) & 0x3fff;
                const int4 rp = rowpack[i];                   // pack_row(..)
                const int ar = (int)rec.y, z = ar + row_lo_e(rp), ac = z - (lo_c[j] - dz - 2 * EPS);   // the record carries ar = z - (rowLo - 2 EPS)
                const bool zz = z < 2 * EPS;                  // near-zero item: always evaluated exactly
                rz[u] = (ar >= 0 && ar < rp.z) || zz;
                cz[u] = ac >= 0 && ac < w_c[j] + dz + 4 * EPS;
                lowr[u] = ar < 2 * EPS; lowc[u] = ac < 2 * EPS;
                bandr[u] = rz[u] && !lowr[u] && ar < dz + 2 * EPS;
                bandc[u] = cz[u] && !lowc[u] && ac < dz + 2 * EPS;
                ii[u] = i; jj[u] = j; zz_[u] = z;
            }
        }
#pragma unroll
        for (int u = 0; u < SU; ++u) {
            if (rz[u]) pr[u] = atomicAdd(&cnt[ii[u]], 1u);
            if (cz[u]) pc[u] = atomicAdd(&cnt[L.max_rows + jj[u]], 1u);
        }
#pragma unroll
        for (int u = 0; u < SU; ++u) {
            const bool wr = rz[u] && pr[u] < CAND_CAP, wc = cz[u] && pc[u] < CAND_CAP;
            if (wr) {
                cand[(size_t)ii[u] * CAND_CAP + pr[u]] = (uint16_t)(jj[u] | (lowr[u] ? 0x8000 : 0));
                candz[(size_t)ii[u] * CAND_CAP + pr[u]] = zz_[u];
            }
            if (wc) {
                const size_t line = (size_t)(L.max_rows + jj[u]);
                cand[line * CAND_CAP + pc[u]] = (uint16_t)(ii[u] | (lowc[u] ? 0x8000 : 0));
                candz[line * CAND_CAP + pc[u]] = zz_[u];
            }
            const bool br = wr && bandr[u], bc = wc && bandc[u];
            if (br || bc)
                s_band[atomicAdd(&s_nband, 1)] = (eb + u * blockDim.x - e0) | ((br ? pr[u] : 0xffu) << 12) | ((bc ? pc[u] : 0xffu) << 20);
        }
    }
    __syncthreads();
    // the band: z' of the cell (k2_tc.inl: tc_coarse_T), below iff z' < lo  <=>  ar + (z' - z) < dz + 2 EPS
    const int nb = s_nband;
    if (nb) {
        const uint4 *qpl = slot_ptr<uint4>(scratch, L, slot, L.off_qpl), *rpl = slot_ptr<uint4>(scratch, L, slot, L.off_rpl);
        const int32_t *aai = slot_ptr<int32_t>(scratch, L, slot, L.off_aai), *bbi = slot_ptr<int32_t>(scratch, L, slot, L.off_bbi);
        for (int t = threadIdx.x; t < nb; t += blockDim.x) {
            const uint32_t q = s_band[t], pr1 = (q >> 12) & 0xffu, pc1 = q >> 20;
            const uint2 rec = pool[e0 + (q & 0xfffu)];
            const int i = rec.x & 0x3fff, j = (rec.x >> 14) & 0x3fff;
            const int ar = (int)rec.y, z = ar + row_lo_e(rowpack[i]), ac = z - (lo_c[j] - dz - 2 * EPS);
            const int d = aai[i] + bbi[j] - tc_coarse_T(qpl, rpl, L.plane_frames, i, j, sh3) - z;
            if (pr1 != 0xffu && ar + d < dz + 2 * EPS) cand[(size_t)i * CAND_CAP + pr1] |= 0x8000;
            if (pc1 != 0xffu && ac + d < dz + 2 * EPS) cand[(size_t)(L.max_rows + j) * CAND_CAP + pc1] |= 0x8000;
        }
        if (threadIdx.x == 0) atomicAdd(&dbg[26], (unsigned)nb);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&dbg[24], min(cntv, (uint32_t)L.pool_cap));
}

// ------------------------------------------------------------------------------------------------
// resolve: exact order statistics from the candidate lists, thresholds, bit patch
// ------------------------------------------------------------------------------------------------
// acc_f32prod with the float -> double widening done on the integer pipe (exact for normal non-negative
// floats; zero / subnormal products take the conversion instruction).  F2F.F64.F32 issues at 16 lanes/clk/SM
// (profiles/r1_ubench.md), so exact_item alternates the two forms and both pipes share the load.
__device__ __forceinline__ double acc_f32prod_alu(double acc, float a, float b) {
    const float p = __fmul_rn(a, b);
    const uint32_t bts = __float_as_uint(p);
    double w;
    if (bts - 0x00800000u < 0x7f000000u)                      // normal, positive, finite
        w = __hiloint2double((int)((bts >> 3) + 0x38000000u), (int)(bts << 29));
    else
        w = (double)p;
    return __dadd_rn(acc, w);
}

__device__ __forceinline__ float exact_item(const float *__restrict__ Q, const float *__restrict__ R, int i, int j,
                                            float aa, float bb) {
    // 9 consecutive frames of each side = 108 floats = 27 float4 (frames are 48 B, bases 16 B aligned)
    const float4 *a = reinterpret_cast<const float4 *>(Q + (int64_t)i * NBINS);
    const float4 *b = reinterpret_cast<const float4 *>(R + (int64_t)j * NBINS);
    double acc = 0.0;
#pragma unroll 3
    for (int t = 0; t < M9 * NBINS / 4; ++t) {
        const float4 u = __ldg(a + t), v = b[t];
        acc = acc_f32prod(acc, u.x, v.x); acc = acc_f32prod_alu(acc, u.y, v.y);
        acc = acc_f32prod(acc, u.z, v.z); acc = acc_f32prod_alu(acc, u.w, v.w);
    }
    return __fadd_rn(__fsub_rn(aa, __fmul_rn(2.f, (float)acc)), bb);
}

// Thresholds.  32 lines (rows, then columns) per CTA, 8 lanes per line.  The candidates of a line are ALL its
// cells with fixed-point item z in the zone [lo - 2 EPS, lo + w + 2 EPS); the histogram levels counted exactly how
// many cells lie below the zone, so the z-ranks of the wanted order statistics inside the list are known.  Since
// |z - exact item / unit| <= EPS for every cell, the exact order statistic of rank r differs from the z order
// statistic zr of the same rank by at most EPS, every cell attaining it has z within 2 EPS of zr, every cell with
// z < zr - 2 EPS is strictly below it and every cell with z > zr + 2 EPS strictly above.  So only the window
// cells |z - zr| <= 2 EPS (usually one or two) are evaluated in the reference's exact operation order, and the
// exact order statistic is the (r - #cells below the window)-th smallest of them.
constexpr int WIN_CAP = 8;          // window cells per order statistic a line can take; more -> exact path
constexpr int WFLAT_PER_LINE = 4;   // capacity of a pair's window-cell list, per line (average need ~2)

struct LineSel {                    // per line, written by the rank kernel, read by the finalize kernel
    int32_t zf, zc;                 // z order statistics of ranks floor(k), ceil(k)
    int16_t wf, wc;                 // ranks inside the two windows
    int16_t nf, nc;                 // window sizes
    uint32_t bad;                   // fallback reasons found so far (0: fine); 0x80000000: nothing to select (quirk side)
};
static_assert(sizeof(LineSel) == 20, "FastLayout sizes LineSel as 20 bytes");
struct WinCell {                    // one window cell to evaluate exactly
    uint32_t cell;                  // i | j << 14
    uint32_t dst;                   // line << 8 | slot in window 0 (0xf: none) << 4 | slot in window 1 (0xf: none)
};

// rank: 8 lanes per line, 32 lines per CTA, no CTA-wide synchronisation
__global__ void __launch_bounds__(256) fast_rank_kernel(int n, FastLayout L, char *__restrict__ scratch, uint32_t *__restrict__ dbg) {
    __shared__ int s_z[32][CAND_CAP];
    __shared__ int s_zsel[32][2];
    __shared__ int s_wn[32][2];
    const int slot = blockIdx.y;
    if (slot >= n) return;
    const int grp = threadIdx.x >> 3, sub = threadIdx.x & 7;
    const int gline = blockIdx.x * 32 + grp;                  // 0 .. Mx+Nx-1 (rows then columns)
    const PairHdr *h = slot_ptr<PairHdr>(scratch, L, slot, L.off_hdr);
    const int Mx = h->Mx, Nx = h->Nx;
    if (blockIdx.x * 32 >= Mx + Nx) return;
    const bool live = gline < Mx + Nx;
    const bool isrow = gline < Mx;
    const int idx = isrow ? gline : gline - Mx;
    const int line = isrow ? idx : L.max_rows + idx;
    const uint16_t *cand = slot_ptr<uint16_t>(scratch, L, slot, L.off_cand) + (size_t)line * CAND_CAP;
    const int32_t *candz = slot_ptr<int32_t>(scratch, L, slot, L.off_candz) + (size_t)line * CAND_CAP;
    const unsigned gmask = 0xffu << (8 * ((threadIdx.x & 31) >> 3));
    const int side = isrow ? 0 : 1;
    int cnt = 0, nbelow = 0;
    bool over = false;
    if (live) {
        const unsigned c = slot_ptr<uint32_t>(scratch, L, slot, L.off_cnt)[line];
        over = c > CAND_CAP;
        cnt = (int)min(c, (unsigned)CAND_CAP);
    }
    if (sub == 0) { s_wn[grp][0] = 0; s_wn[grp][1] = 0; s_zsel[grp][0] = 0; s_zsel[grp][1] = 0; }
    for (int p = sub; p < cnt; p += 8) {
        s_z[grp][p] = candz[p];
        nbelow += cand[p] >> 15;
    }
    nbelow += __shfl_xor_sync(gmask, nbelow, 1);
    nbelow += __shfl_xor_sync(gmask, nbelow, 2);
    nbelow += __shfl_xor_sync(gmask, nbelow, 4);
    __syncwarp(gmask);
    const int fk = h->fk[side], ck = h->ck[side];
    const bool quirk = h->quirk[side] != 0;
    const int c0 = live ? slot_ptr<int32_t>(scratch, L, slot, L.off_cb)[line] - nbelow : 0;   // cells below every candidate
    const int rfk = fk - c0, rck = ck - c0;
    unsigned bad = over ? 32u : 0u;                           // reason 32: more than CAND_CAP candidates on a line
    const bool sel = live && !quirk;
    if (sel && (rfk < 0 || rck >= cnt || rfk > rck)) bad |= 64u;   // reason 64: ranks not inside the candidate set
    // z order statistics of ranks rfk, rck by counting (ties broken by list position)
    if (sel && !bad) {
        for (int p = sub; p < cnt; p += 8) {
            const int v = s_z[grp][p];
            int rank = 0;
            for (int p2 = 0; p2 < cnt; ++p2) {
                const int v2 = s_z[grp][p2];
                rank += (v2 < v) || (v2 == v && p2 < p);
            }
            if (rank == rfk) s_zsel[grp][0] = v;
            if (rank == rck) s_zsel[grp][1] = v;
        }
    }
    __syncwarp(gmask);
    const int zf = s_zsel[grp][0], zc = s_zsel[grp][1];
    // window cells go to the pair's flat list (evaluated by fast_exact_kernel, one thread per cell: the long
    // exact evaluation runs on full warps); cells below each window are counted
    int nbf = 0, nbc = 0;
    WinCell *wl = slot_ptr<WinCell>(scratch, L, slot, L.off_wlist);
    uint32_t *wcnt = slot_ptr<uint32_t>(scratch, L, slot, L.off_wcnt);
    const uint32_t wcap = (uint32_t)WFLAT_PER_LINE * (uint32_t)L.lines;
    if (sel && !bad) {
        for (int p = sub; p < cnt; p += 8) {
            const int v = s_z[grp][p];
            nbf += (v < zf - 2 * EPS) ? 1 : 0;
            nbc += (v < zc - 2 * EPS) ? 1 : 0;
            const bool inf = (v >= zf - 2 * EPS) && (v <= zf + 2 * EPS), inc = (v >= zc - 2 * EPS) && (v <= zc + 2 * EPS);
            if (inf || inc) {
                const int other = cand[p] & 0x7fff;
                const int i = isrow ? idx : other, j = isrow ? other : idx;
                const int sf = inf ? atomicAdd(&s_wn[grp][0], 1) : 0xf, sc = inc ? atomicAdd(&s_wn[grp][1], 1) : 0xf;
                const uint32_t e = atomicAdd(wcnt, 1u);
                if (e < wcap) {
                    WinCell wc;
                    wc.cell = (uint32_t)i | ((uint32_t)j << 14);
                    wc.dst = ((uint32_t)line << 8) | ((uint32_t)min(sf, 0xf) << 4) | (uint32_t)min(sc, 0xf);
                    wl[e] = wc;
                }
            }
        }
    }
    nbf += __shfl_xor_sync(gmask, nbf, 1); nbf += __shfl_xor_sync(gmask, nbf, 2); nbf += __shfl_xor_sync(gmask, nbf, 4);
    nbc += __shfl_xor_sync(gmask, nbc, 1); nbc += __shfl_xor_sync(gmask, nbc, 2); nbc += __shfl_xor_sync(gmask, nbc, 4);
    __syncwarp(gmask);
    if (!live || sub != 0) return;
    LineSel ls;
    ls.zf = zf; ls.zc = zc;
    ls.nf = (int16_t)min(s_wn[grp][0], 0x7fff); ls.nc = (int16_t)min(s_wn[grp][1], 0x7fff);
    ls.wf = (int16_t)max(min(rfk - nbf, 0x7fff), -1); ls.wc = (int16_t)max(min(rck - nbc, 0x7fff), -1);
    ls.bad = sel ? bad : 0x80000000u;
    slot_ptr<LineSel>(scratch, L, slot, L.off_lsel)[line] = ls;
}

// exact evaluation of the window cells: one thread per cell of the pair's flat list
__global__ void __launch_bounds__(256) fast_exact_kernel(TrackSet ts, const int32_t *__restrict__ pairs, int64_t first, int n,
                                                         FastLayout L, char *__restrict__ scratch,
                                                         uint32_t *__restrict__ status, uint32_t *__restrict__ dbg) {
    const int slot = blockIdx.y;
    if (slot >= n) return;
    const uint32_t wcap = (uint32_t)WFLAT_PER_LINE * (uint32_t)L.lines;
    const uint32_t cntv = *slot_ptr<uint32_t>(scratch, L, slot, L.off_wcnt);
    const uint32_t m = min(cntv, wcap);
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t k = first + slot;
    if (e == 0) {
        if (cntv > wcap) atomicOr(&status[k], PAIR_ST_FALLBACK | 128u);   // reason 128: window-cell list overflow
        if (m) atomicAdd(&dbg[25], m);
    }
    if (e >= m) return;
    const WinCell wc = slot_ptr<WinCell>(scratch, L, slot, L.off_wlist)[e];
    const int i = wc.cell & 0x3fff, j = wc.cell >> 14;
    const int q = pairs[2 * k];
    const float *Q = ts.frames + ts.offsets[q] * NBINS;
    const float *R = slot_ptr<float>(scratch, L, slot, L.off_rrot);
    const float item = exact_item(Q, R, i, j, slot_ptr<float>(scratch, L, slot, L.off_aaf)[i],
                                  slot_ptr<float>(scratch, L, slot, L.off_bbf)[j]);
    if (item != item || item < 0.f) atomicOr(&status[k], PAIR_ST_NAN);   // sqrtf of a negative item is the reference's NaN (F7)
    const uint32_t line = wc.dst >> 8, sf = (wc.dst >> 4) & 0xf, sc = wc.dst & 0xf;
    float *win = slot_ptr<float>(scratch, L, slot, L.off_win) + (size_t)line * 2 * WIN_CAP;
    if (sf < WIN_CAP) win[sf] = item;
    if (sc < WIN_CAP) win[WIN_CAP + sc] = item;
}

// finalize: one thread per line picks the exact order statistics inside the two windows and forms the threshold
__global__ void __launch_bounds__(128) fast_thr_kernel(int64_t first, int n, FastLayout L, char *__restrict__ scratch, int guard,
                                                       double unit, float *__restrict__ thr_q_all,
                                                       float *__restrict__ thr_r_all, uint32_t *__restrict__ status) {
    const int slot = blockIdx.y;
    if (slot >= n) return;
    const PairHdr *h = slot_ptr<PairHdr>(scratch, L, slot, L.off_hdr);
    const int Mx = h->Mx, Nx = h->Nx;
    const int gline = blockIdx.x * blockDim.x + threadIdx.x;
    if (gline >= Mx + Nx) return;
    const bool isrow = gline < Mx;
    const int idx = isrow ? gline : gline - Mx;
    const int line = isrow ? idx : L.max_rows + idx;
    const int side = isrow ? 0 : 1;
    const int64_t k = first + slot;
    const LineSel ls = slot_ptr<LineSel>(scratch, L, slot, L.off_lsel)[line];
    const int32_t lo = slot_ptr<int32_t>(scratch, L, slot, L.off_lo)[line];
    const int32_t w = slot_ptr<int32_t>(scratch, L, slot, L.off_w)[line];
    unsigned bad = ls.bad & 0x7fffffffu;
    float thr = 0.f;
    int zin = -0x40000000, zout = -0x40000000;   // thr = 0 (F1 quirk): only an exact zero distance is in, and near-zero cells are always evaluated exactly
    if (!(ls.bad & 0x80000000u) && !bad) {
        const int nf = ls.nf, nc = ls.nc, wf = ls.wf, wc = ls.wc;
        if (nf > WIN_CAP || nc > WIN_CAP) bad |= 128u;        // reason 128: too many cells within 2 EPS of an order statistic
        else if (wf < 0 || wf >= nf || wc < 0 || wc >= nc) bad |= 256u;   // reason 256: window rank inconsistent
        else {
            const float *win = slot_ptr<float>(scratch, L, slot, L.off_win) + (size_t)line * 2 * WIN_CAP;
            float vf[WIN_CAP], vc[WIN_CAP];
#pragma unroll
            for (int a = 0; a < WIN_CAP; ++a) { vf[a] = (a < nf) ? win[a] : 0.f; vc[a] = (a < nc) ? win[WIN_CAP + a] : 0.f; }
            float ifk = 0.f, ick = 0.f;
#pragma unroll
            for (int a = 0; a < WIN_CAP; ++a) {
                int rf = 0, rc = 0;
#pragma unroll
                for (int b = 0; b < WIN_CAP; ++b) {
                    rf += (b < nf) && ((vf[b] < vf[a]) || (vf[b] == vf[a] && b < a));
                    rc += (b < nc) && ((vc[b] < vc[a]) || (vc[b] == vc[a] && b < a));
                }
                if (a < nf && rf == wf) ifk = vf[a];
                if (a < nc && rc == wc) ick = vc[a];
            }
            // the a-priori bound |z - item / unit| <= EPS, checked on the selected cells (with margin)
            if (fabs((double)ifk / unit - (double)ls.zf) > (double)(2 * EPS) || fabs((double)ick / unit - (double)ls.zc) > (double)(2 * EPS))
                bad |= 512u;                                  // reason 512: fixed-point bound violated
            const float sfk = __fsqrt_rn(ifk), sck = __fsqrt_rn(ick);
            const float kf = h->kf[side];
            const float fkf = floorf(kf), ckf = ceilf(kf);
            if (guard && fkf == ckf) thr = sfk;
            else thr = __fadd_rn(__fmul_rn(sfk, __fsub_rn(ckf, kf)), __fmul_rn(sck, __fsub_rn(kf, fkf)));
            // integer bounds for the bit decisions of resolve_bits: with t2 = thr^2 (exact in double),
            //   item <= t2                => sqrtf(item) <= thr           (sqrt and rounding are monotonic)
            //   item >  t2 (1 + 2^-21)    => sqrtf(item) >= nextafter(thr) > thr
            // and |z - item / unit| <= EPS
            const double t2 = (double)thr * (double)thr;
            const double zi = floor(t2 / unit) - (double)EPS - 1.0, zo = ceil(t2 * (1.0 + 4.76837158203125e-07) / unit) + (double)EPS + 1.0;
            zin = (int)fmax(fmin(zi, 1.0e9), -1.0e9);
            zout = (int)fmax(fmin(zo, 1.0e9), -1.0e9);
            // every cell the sweep emitted as certainly-in has z < lo - dz - 2 EPS, every cell it dropped has z >= lo + w + 2 EPS
            if (zin < lo - h->dz - 2 * EPS - 1 || zout > lo + w + 2 * EPS) bad |= 1024u;   // reason 1024: threshold not between the certain sets
        }
    }
    if (bad) atomicOr(&status[k], PAIR_ST_FALLBACK | bad);
    if (isrow) thr_q_all[(int64_t)slot * L.max_rows + idx] = thr;
    else thr_r_all[(int64_t)slot * L.max_cols + idx] = thr;
    slot_ptr<int32_t>(scratch, L, slot, L.off_zin)[line] = zin;
    slot_ptr<int32_t>(scratch, L, slot, L.off_zout)[line] = zout;
}

// Bits of the listed (uncertain) cells.  A cell is 1 iff thrQ[i] - d >= 0 and thrR[j] - d >= 0.  Each side is decided
// from z and the line's integer bounds when that is certain (z <= zin: in, z >= zout: out); the few cells in between
// (and every near-zero cell, for the NaN rule F7) are evaluated exactly.  A cell listed by its row and its column is
// handled from the row list only.
__global__ void __launch_bounds__(256) fast_resolve_bits_kernel(TrackSet ts, const int32_t *__restrict__ pairs,
                                                                int64_t first, int n, FastLayout L,
                                                                char *__restrict__ scratch,
                                                                const float *__restrict__ thr_q_all,
                                                                const float *__restrict__ thr_r_all,
                                                                uint32_t *__restrict__ crp_all, int words,
                                                                int64_t crp_words, uint32_t *__restrict__ status,
                                                                uint32_t *__restrict__ dbg) {
    const int slot = blockIdx.y;
    if (slot >= n) return;
    const PairHdr *h = slot_ptr<PairHdr>(scratch, L, slot, L.off_hdr);
    const int Mx = h->Mx, Nx = h->Nx;
    const int gline = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;   // 16 lanes per line
    const int sub = threadIdx.x & 15;
    if (gline >= Mx + Nx) return;
    const bool isrow = gline < Mx;
    const int idx = isrow ? gline : gline - Mx;
    const int line = isrow ? idx : L.max_rows + idx;
    const int cnt = (int)min(slot_ptr<uint32_t>(scratch, L, slot, L.off_cnt)[line], (uint32_t)CAND_CAP);
    if (cnt == 0) return;
    const int64_t k = first + slot;
    const uint16_t *cand = slot_ptr<uint16_t>(scratch, L, slot, L.off_cand) + (size_t)line * CAND_CAP;
    const int32_t *candz = slot_ptr<int32_t>(scratch, L, slot, L.off_candz) + (size_t)line * CAND_CAP;
    const int32_t *zin = slot_ptr<int32_t>(scratch, L, slot, L.off_zin), *zout = slot_ptr<int32_t>(scratch, L, slot, L.off_zout);
    const int4 *rowpack = slot_ptr<int4>(scratch, L, slot, L.off_rowpack);
    for (int p = sub; p < cnt; p += 16) {
        const int other = cand[p] & 0x7fff;
        const int z = candz[p];
        const int i = isrow ? idx : other, j = isrow ? other : idx;
        const bool zz = z < 2 * EPS;
        if (!isrow) {                                         // also on the row's list? then the row handles it
            const int4 rp = rowpack[i];
            const int ar = z - row_lo_e(rp);
            if ((ar >= 0 && ar < rp.z) || zz) continue;
        }
        const int lr = i, lc = L.max_rows + j;
        const int zir = zin[lr], zor = zout[lr], zic = zin[lc], zoc = zout[lc];
        const bool in_r = z <= zir, out_r = z >= zor, in_c = z <= zic, out_c = z >= zoc;
        bool one;
        if (!zz && (out_r || out_c)) continue;
        if (!zz && in_r && in_c) one = true;
        else {
            const int q = pairs[2 * k];
            const float *Q = ts.frames + ts.offsets[q] * NBINS;
            const float *R = slot_ptr<float>(scratch, L, slot, L.off_rrot);
            const float item = exact_item(Q, R, i, j, slot_ptr<float>(scratch, L, slot, L.off_aaf)[i],
                                          slot_ptr<float>(scratch, L, slot, L.off_bbf)[j]);
            const float d = __fsqrt_rn(item);
            if (d != d) atomicOr(&status[k], PAIR_ST_NAN);
            const float tq = thr_q_all[(int64_t)slot * L.max_rows + i], tr = thr_r_all[(int64_t)slot * L.max_cols + j];
            one = (__fsub_rn(tq, d) >= 0.f) && (__fsub_rn(tr, d) >= 0.f);
            atomicAdd(&dbg[25], 1u);
        }
        if (one) atomicOr(crp_all + (int64_t)slot * crp_words + (int64_t)i * words + (j >> 5), 1u << (j & 31));
    }
}

__global__ void collect_fallback_kernel(const uint32_t *__restrict__ status, int64_t first, int n,
                                        int32_t *__restrict__ map, int32_t *__restrict__ count) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    if (status[first + t] & PAIR_ST_FALLBACK) map[atomicAdd(count, 1)] = (int32_t)(first + t);
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
bool k2_fast_supported(const acoss_params &p, const SlotGeom &g, const TrackSet &ts) {
    return p.m == M9 && p.tau == 1 && ts.fx_exp > -100 && ts.nonneg && g.max_rows < 16000 && g.max_cols < 16000 &&
           g.max_rows >= 2 && g.max_cols >= 2;
}

size_t k2_fast_slot_bytes(const SlotGeom &g, int max_frames) { return make_layout(g, max_frames).slot_bytes; }

int launch_k2_fast(const TrackSet &ts, const int32_t *pairs, const int32_t *oti, int64_t first, int n,
                   const acoss_params &p, const SlotGeom &g, void *scratch, size_t slot_bytes, uint32_t *crp,
                   float *thr_q, float *thr_r, uint32_t *status, uint32_t *dbg, cudaStream_t st, int64_t *launches,
                   KernelTimer *timer, uint32_t *glive, uint32_t gcap) {
    if (n <= 0) return ACOSS_OK;
    constexpr int RC = RCV;
    const FastLayout L = make_layout(g, ts.max_frames);
    if (L.slot_bytes != slot_bytes) { acoss_set_error("fast path: scratch layout mismatch"); return ACOSS_E_INVALID; }
    char *base = (char *)scratch;
    const float qperc = (float)((double)(p.kappa * 100.f) / 100.);
    // fixed point: 2e < 2^fx_exp, unit = 2^(fx_exp - 23); magic = 2^fx_exp puts 2e in one binade
    const float magic = ldexpf(1.f, ts.fx_exp);
    const double unit = ldexp(1.0, ts.fx_exp - 23);
    const float fx_scale = ldexpf(1.f, 23 - ts.fx_exp);
    CUDA_TRY(cudaMemsetAsync(glive, 0, 4, st));
    auto tb = [&](int id) { if (timer) timer->begin(id); };
    auto te = [&](int id) { if (timer) timer->end(id); };
    tb(K2K_PREP);
    // Sweeps: tensor cores from TC_MIN_WINDOWS windows on the longer side (a work item's fixed costs - operand fill, histogram
    // scan - weigh on short lines; measured against the FFMA2 sweeps before the tensor sweeps became persistent: +17 % pairs/s
    // at 2 000 frames, level at 500), FFMA2 below and whenever the features cannot be quantised within the error budget.  ACOSS_K2_SWEEPS=tc|ffma forces one of them (A/B runs, parity tests of both).
    const char *sweeps_env = getenv("ACOSS_K2_SWEEPS");          // read per call: tests flip it inside one process
    bool use_tc = ts.q_exp >= 0 && std::max(g.max_rows, g.max_cols) >= TC_MIN_WINDOWS;
    if (sweeps_env && sweeps_env[0] == 't') use_tc = ts.q_exp >= 0;
    if (sweeps_env && sweeps_env[0] == 'f') use_tc = false;
    const float q_scale = use_tc ? ldexpf(1.f, ts.q_exp) : 0.f;
    // tensor sweeps: the limb products weigh 2^e0, 2^(e0 - 8), 2^(e0 - 16) fixed-point units (k2_tc.inl), 0 <= e0 <= 6
    const int e0 = 56 - 2 * ts.q_exp - ts.fx_exp;
    const TcShift sh3 = use_tc ? TcShift{e0, 8 - e0, 16 - e0, 1u << e0} : TcShift{0, 0, 0, 0u};
    fast_prep_kernel<<<n, 256, 0, st>>>(ts, pairs, oti, first, L, base, qperc, p.integer_guard, fx_scale, q_scale, sh3);
    CUDA_TRY(cudaGetLastError());
    te(K2K_PREP);
    const int outw = Sweep<RC>::OUTW, houtw = Sweep<HRC>::OUTW;
    const int strips_c = (g.max_cols + outw - 1) / outw;                  // emit strips
    const int hstrips_c = (g.max_cols + houtw - 1) / houtw, hstrips_r = (g.max_rows + houtw - 1) / houtw;
    const size_t smem = (size_t)WPC * (NBIN + 2) * (HRC / 2) * 32 * 4;
    const size_t smem_sel = (size_t)(SBIN / 2) * SEL_THREADS * 4;
    static bool attr_done_dev[64] = {false};                  // function attributes are per device
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    bool &attr_done = attr_done_dev[dev & 63];
    if (!attr_done) {
        CUDA_TRY(cudaFuncSetAttribute(fast_hist_kernel<HRC, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(fast_hist_kernel<HRC, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(fast_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_sel));
        attr_done = true;
    }
    const unsigned gc = (unsigned)(((int64_t)n * hstrips_c + WPC - 1) / WPC), gr = (unsigned)(((int64_t)n * hstrips_r + WPC - 1) / WPC);
    const int lines = g.max_rows + g.max_cols;
    // first brackets from every S-th diagonal (sampler + per-line selection), then up to three histogram
    // levels per orientation; a level returns immediately for strips whose lines are all done
    {
        const int nu_max = ((g.max_rows - 1) >> L.slog) + ((g.max_cols - 1) >> L.slog) + 1;
        const int ngrp = (nu_max + SKD - 1) / SKD, nblk = (g.max_rows + SPOS - 1) / SPOS;
        const int64_t warps = (int64_t)n * ngrp * nblk;
        tb(K2K_SAMPLE);
        fast_sample_kernel<<<(unsigned)((warps + 3) / 4), 128, 0, st>>>(ts, pairs, first, n, L, base, ngrp, nblk, magic);
        CUDA_TRY(cudaGetLastError());
        te(K2K_SAMPLE);
        tb(K2K_SELECT);
        fast_select_kernel<<<dim3((lines + SEL_THREADS - 1) / SEL_THREADS, n), SEL_THREADS, smem_sel, st>>>(n, L, base);
        CUDA_TRY(cudaGetLastError());
        te(K2K_SELECT);
    }
    // two dense levels per orientation: the second sweeps only strips that still hold DENSE2_MIN_LIVE or more live
    // lines (short lines start from the whole item range and need it; ordinary strips skip it at once) and hands
    // every line still live to the sparse refinement
    if (use_tc) {
        // tensor sweeps (k2_tc.inl): one CTA = 128 owned lines; items from tcgen05.mma.kind::i8 over the byte planes
        const int tstrips_c = (g.max_cols + 127) / 128, tstrips_r = (g.max_rows + 127) / 128;
        // (one CTA per SM: it holds all 512 TMEM columns; the requested shared memory keeps a second one off the SM)
        const size_t smem_h = std::max(sizeof(TcSmem<TC_NP_HIST>) + (size_t)(NBIN + 2) * 128 * 4, (size_t)120 * 1024);
        const size_t smem_e = std::max(sizeof(TcSmem<TC_NP_EMIT>) + (size_t)(TC_CONS / 32) * (TC_STAGE * 32 * 8 + 64), (size_t)120 * 1024);
        static bool tc_attr_done[64] = {false};
        if (!tc_attr_done[dev & 63]) {
            CUDA_TRY(cudaFuncSetAttribute(tc_hist_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_h));
            CUDA_TRY(cudaFuncSetAttribute(tc_hist_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_h));
            CUDA_TRY(cudaFuncSetAttribute(tc_emit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_e));
            tc_attr_done[dev & 63] = true;
        }
        // persistent CTAs, one per SM, taking work items from a counter that fast_prep_kernel zeroed (k2_tc.inl)
        static int tc_sms[64] = {0};
        if (!tc_sms[dev & 63]) CUDA_TRY(cudaDeviceGetAttribute(&tc_sms[dev & 63], cudaDevAttrMultiProcessorCount, dev));
        auto tc_grid = [&](int64_t items) { return (unsigned)std::min<int64_t>(items, tc_sms[dev & 63]); };
        // one launch per orientation: an item that still holds DENSE2_MIN_LIVE live lines after its sweep is swept again at once
        tb(K2K_HIST_COL);
        tc_hist_kernel<0><<<tc_grid((int64_t)n * tstrips_c), TC_THREADS, smem_h, st>>>(ts, pairs, first, n, L, base, tstrips_c, sh3, status, dbg,
                                                                                       dbg + 12, glive, gcap);
        te(K2K_HIST_COL);
        tb(K2K_HIST_ROW);
        tc_hist_kernel<1><<<tc_grid((int64_t)n * tstrips_r), TC_THREADS, smem_h, st>>>(ts, pairs, first, n, L, base, tstrips_r, sh3, status,
                                                                                       dbg + 4, dbg + 16, glive, gcap);
        CUDA_TRY(cudaGetLastError());
        te(K2K_HIST_ROW);
        const int64_t warps = ((int64_t)gcap + 31) / 32;
        tb(K2K_SPARSE);
        tc_sparse_kernel<<<(unsigned)((warps + WPC - 1) / WPC), 32 * WPC, 0, st>>>(ts, pairs, first, n, L, base, sh3, status, dbg + 8, glive, gcap);
        CUDA_TRY(cudaGetLastError());
        te(K2K_SPARSE);
        const int groups = std::max(tstrips_c, (g.words + 3) / 4);
        tb(K2K_EMIT);
        tc_emit_kernel<<<tc_grid((int64_t)n * groups), TC_THREADS, smem_e, st>>>(ts, pairs, first, n, L, base, groups, sh3, crp, g.words,
                                                                                 g.crp_words);
        CUDA_TRY(cudaGetLastError());
        te(K2K_EMIT);
    } else {
    tb(K2K_HIST_COL);
    fast_hist_kernel<HRC, 0><<<gc, 32 * WPC, smem, st>>>(ts, pairs, first, n, L, base, hstrips_c, magic, status, dbg, 1, 0, glive, gcap);
    te(K2K_HIST_COL);
    tb(K2K_HIST_ROW);
    fast_hist_kernel<HRC, 1><<<gr, 32 * WPC, smem, st>>>(ts, pairs, first, n, L, base, hstrips_r, magic, status, dbg + 4, 1, 0, glive, gcap);
    te(K2K_HIST_ROW);
    tb(K2K_HIST_COL2);
    fast_hist_kernel<HRC, 0><<<gc, 32 * WPC, smem, st>>>(ts, pairs, first, n, L, base, hstrips_c, magic, status, dbg + 12, DENSE2_MIN_LIVE, 1, glive, gcap);
    te(K2K_HIST_COL2);
    tb(K2K_HIST_ROW2);
    fast_hist_kernel<HRC, 1><<<gr, 32 * WPC, smem, st>>>(ts, pairs, first, n, L, base, hstrips_r, magic, status, dbg + 16, DENSE2_MIN_LIVE, 1, glive, gcap);
    CUDA_TRY(cudaGetLastError());
    te(K2K_HIST_ROW2);
    {
        // the crowded lines of ALL pairs of the call, one lane each (warps that find nothing past the list's end return)
        const int64_t warps = ((int64_t)gcap + 31) / 32;
        tb(K2K_SPARSE);
        fast_sparse_kernel<<<(unsigned)((warps + WPC - 1) / WPC), 32 * WPC, 0, st>>>(ts, pairs, first, n, L, base, magic, status, dbg + 8,
                                                                                     glive, gcap);
        CUDA_TRY(cudaGetLastError());
        te(K2K_SPARSE);
    }
    {
        // one CTA per group of WPC strips (EMIT_CW whole CRP words per row); the groups also cover the row pitch padding
        const int groups = std::max((strips_c + WPC - 1) / WPC, (g.words + EMIT_CW - 1) / EMIT_CW);
        tb(K2K_EMIT);
        fast_emit_kernel<RC><<<(unsigned)((int64_t)n * groups), 32 * WPC, 0, st>>>(ts, pairs, first, n, L, base, groups, magic, crp,
                                                                                g.words, g.crp_words);
        CUDA_TRY(cudaGetLastError());
        te(K2K_EMIT);
    }
    }
    tb(K2K_SCATTER);
    fast_scatter_kernel<<<dim3((L.pool_cap + SCAT_CHUNK - 1) / SCAT_CHUNK, n), 256, 0, st>>>(n, L, base, first, sh3, status, dbg);
    CUDA_TRY(cudaGetLastError());
    te(K2K_SCATTER);
    tb(K2K_THR);
    fast_rank_kernel<<<dim3((lines + 31) / 32, n), 256, 0, st>>>(n, L, base, dbg);
    te(K2K_THR);
    tb(K2K_EXACT);
    fast_exact_kernel<<<dim3((WFLAT_PER_LINE * lines + 255) / 256, n), 256, 0, st>>>(ts, pairs, first, n, L, base, status, dbg);
    te(K2K_EXACT);
    tb(K2K_FINAL);
    fast_thr_kernel<<<dim3((lines + 127) / 128, n), 128, 0, st>>>(first, n, L, base, p.integer_guard, unit, thr_q, thr_r, status);
    CUDA_TRY(cudaGetLastError());
    te(K2K_FINAL);
    tb(K2K_BITS);
    fast_resolve_bits_kernel<<<dim3((lines * 16 + 255) / 256, n), 256, 0, st>>>(ts, pairs, first, n, L, base, thr_q, thr_r, crp,
                                                                                      g.words, g.crp_words, status, dbg);
    CUDA_TRY(cudaGetLastError());
    te(K2K_BITS);
    // kernels launched above: prep, sample, select, sparse, emit, scatter, rank, exact, thr, bits + the histogram sweeps (one
    // launch per orientation on the tensor cores, two with the FFMA2 sweeps)
    if (launches) *launches += 10 + (use_tc ? 2 : 4);
    return ACOSS_OK;
}

int k2_fast_collect_fallback(const uint32_t *status, int64_t first, int n, int32_t *map_dev, int32_t *count_dev,
                             int *count_host, cudaStream_t st) {
    if (count_host) *count_host = 0;
    if (n <= 0) return ACOSS_OK;
    CUDA_TRY(cudaMemsetAsync(count_dev, 0, 4, st));
    collect_fallback_kernel<<<(n + 255) / 256, 256, 0, st>>>(status, first, n, map_dev, count_dev);
    CUDA_TRY(cudaGetLastError());
    if (count_host) {                                         // synchronous variant (single-pair debug dumps)
        int32_t c = 0;
        CUDA_TRY(cudaMemcpyAsync(&c, count_dev, 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        *count_host = c;
    }
    return ACOSS_OK;
}
