"""Thin host wrapper over the C ABI: one Engine = one acoss_ctx on one CUDA device.

PyTorch appears only as an optional way to hand over device memory (``data_ptr()``); all
arithmetic runs in the CUDA kernels of libacoss_b200.so.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import ALIGN_DMAX, ALIGN_DMAX_PLAIN, ALIGN_QMAX, ALIGN_SW, AcossError, Params, check, default_params  # noqa: F401
from ._lib import SimpleParams, simple_default_params  # noqa: F401

__all__ = ["Engine", "AcossError", "default_params", "pack_tracks", "check_snf_args"]


def pack_tracks(tracks):
    """list of (n_i, 12) arrays -> (frames float32 [sum n_i, 12] C-contiguous, offsets int64)."""
    lens = [int(t.shape[0]) for t in tracks]
    for t in tracks:
        if t.ndim != 2 or t.shape[1] != 12:
            raise ValueError("every track must be (n_frames, 12); got %r" % (t.shape,))
    offsets = np.zeros(len(tracks) + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    frames = np.empty((int(offsets[-1]), 12), dtype=np.float32)
    for t, o in zip(tracks, offsets[:-1]):
        frames[o:o + t.shape[0]] = t            # handles the reference's transposed views
    return frames, offsets


def check_snf_args(n_mats: int, n: int, K: int, niters: int = 0):
    """The arguments acoss_snf refuses, as ValueError: n_mats outside 2..16 (the reference divides by n_mats - 1 and
    returns NaN for one matrix), K outside 1..63, K + 1 >= n (np.partition raises ValueError), niters < 0."""
    if not 2 <= n_mats <= _lib.SNF_MAX_MATS:
        raise ValueError("similarity fusion needs 2..%d score matrices, got %d" % (_lib.SNF_MAX_MATS, n_mats))
    if not 1 <= K <= _lib.SNF_MAX_K:
        raise ValueError("K = %d outside 1..%d" % (K, _lib.SNF_MAX_K))
    if K + 1 >= n:
        raise ValueError("kth(=%d) out of bounds (%d): K + 1 must be smaller than the number of tracks" % (K + 1, n))
    if n > 65535:
        raise ValueError("n = %d tracks; at most 65535 supported" % n)
    if niters < 0:
        raise ValueError("niters = %d < 0" % niters)


class Engine:
    def __init__(self, device: int = 0, workspace_bytes: int | None = None):
        self._lib = _lib.load()
        self._ctx = C.c_void_p()
        check(self._lib.acoss_create(C.byref(self._ctx), int(device)))
        self.device = int(device)
        self.n_tracks = 0
        self.offsets = None
        self._keepalive = None
        if workspace_bytes is not None:
            check(self._lib.acoss_set_workspace_limit(self._ctx, int(workspace_bytes)))

    # -- lifetime -------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self._lib.acoss_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- tracks ---------------------------------------------------------------------------------
    def set_tracks(self, frames, offsets):
        """frames: float32 (total, 12) numpy array (host) or CUDA torch tensor (adopted, not copied)."""
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n = len(offsets) - 1
        if hasattr(frames, "data_ptr"):                       # torch tensor hand-off
            if not frames.is_cuda or frames.dtype.__str__() != "torch.float32" or not frames.is_contiguous():
                raise ValueError("device frames must be a contiguous float32 CUDA tensor")
            if frames.numel() != int(offsets[-1]) * 12:
                raise ValueError("frames size does not match offsets")
            self._keepalive = frames
            check(self._lib.acoss_set_tracks(self._ctx, frames.data_ptr(), offsets.ctypes.data, n, 1))
        else:
            frames = np.ascontiguousarray(frames, dtype=np.float32)
            if frames.size != int(offsets[-1]) * 12:
                raise ValueError("frames size does not match offsets")
            self._keepalive = None
            check(self._lib.acoss_set_tracks(self._ctx, frames.ctypes.data, offsets.ctypes.data, n, 0))
        self.n_tracks = n
        self.offsets = offsets

    def set_tracks_raw(self, raw_frames, raw_offsets, downsample_fac: int) -> np.ndarray:
        """Raw (not yet downsampled) chroma frames -> GPU median downsampling (acoss_set_tracks_raw, the
        aggregation of rqa_serra09.py:47-53) -> resident track set.  Returns the downsampled offsets."""
        raw_offsets = np.ascontiguousarray(raw_offsets, dtype=np.int64)
        raw_frames = np.ascontiguousarray(raw_frames, dtype=np.float32)
        n = len(raw_offsets) - 1
        if raw_frames.size != int(raw_offsets[-1]) * 12:
            raise ValueError("frames size does not match offsets")
        out_off = np.zeros(n + 1, dtype=np.int64)
        check(self._lib.acoss_set_tracks_raw(self._ctx, raw_frames.ctypes.data, raw_offsets.ctypes.data, n,
                                             int(downsample_fac), out_off.ctypes.data))
        self._keepalive = None
        self.n_tracks = n
        self.offsets = out_off
        return out_off

    def set_tracks_pooled(self, raw_frames, raw_offsets, win: int = 200, skip: int = 100,
                          keep_partial: bool = False) -> np.ndarray:
        """Raw chroma frames -> GPU mean pooling (acoss_set_tracks_pooled, the pooling of simple_silva.py:38-41) ->
        resident track set.  keep_partial is switch S5.  Returns the pooled offsets."""
        raw_offsets = np.ascontiguousarray(raw_offsets, dtype=np.int64)
        raw_frames = np.ascontiguousarray(raw_frames, dtype=np.float32)
        n = len(raw_offsets) - 1
        if raw_frames.size != int(raw_offsets[-1]) * 12:
            raise ValueError("frames size does not match offsets")
        out_off = np.zeros(n + 1, dtype=np.int64)
        check(self._lib.acoss_set_tracks_pooled(self._ctx, raw_frames.ctypes.data, raw_offsets.ctypes.data, n,
                                                int(win), int(skip), int(bool(keep_partial)), out_off.ctypes.data))
        self._keepalive = None
        self.n_tracks = n
        self.offsets = out_off
        return out_off

    def get_tracks(self) -> np.ndarray:
        """The resident (post-downsampling) frames, float32 (total, 12)."""
        total = int(self.offsets[-1])
        out = np.empty((total, 12), dtype=np.float32)
        check(self._lib.acoss_get_tracks(self._ctx, out.ctypes.data, total))
        return out

    # -- scoring --------------------------------------------------------------------------------
    def score_pairs(self, pairs, params: Params | None = None) -> np.ndarray:
        """Host in / host out (the end-to-end path): pairs (K, 2) int -> scores float32 (K,)."""
        params = params or default_params()
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        out = np.empty(len(pairs), dtype=np.float32)
        check(self._lib.acoss_score_pairs(self._ctx, pairs.ctypes.data, len(pairs), C.byref(params),
                                          out.ctypes.data))
        return out

    def score_pairs_chen(self, pairs, params: Params | None = None):
        """ChenFusion flavour: (qmax, dmax) float32 arrays of the same CRPs (acoss_score_pairs_chen)."""
        params = params or default_params()
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        q = np.empty(len(pairs), dtype=np.float32)
        d = np.empty(len(pairs), dtype=np.float32)
        check(self._lib.acoss_score_pairs_chen(self._ctx, pairs.ctypes.data, len(pairs), C.byref(params),
                                               q.ctypes.data, d.ctypes.data))
        return q, d

    def score_pairs_device(self, pairs_ptr: int, n_pairs: int, scores_ptr: int, params: Params | None = None):
        """Device in / device out, asynchronous on the engine stream; call sync()."""
        params = params or default_params()
        check(self._lib.acoss_score_pairs_device(self._ctx, pairs_ptr, int(n_pairs), C.byref(params), scores_ptr))

    def score_pairs_chen_device(self, pairs_ptr: int, n_pairs: int, qmax_ptr: int, dmax_ptr: int,
                                params: Params | None = None):
        """ChenFusion flavour of score_pairs_device (acoss_score_pairs_chen_device): Qmax and Dmax of the same CRPs
        into two device buffers, asynchronous on the engine stream; call sync()."""
        params = params or default_params()
        check(self._lib.acoss_score_pairs_chen_device(self._ctx, pairs_ptr, int(n_pairs), C.byref(params), qmax_ptr,
                                                      dmax_ptr))

    def sync(self):
        check(self._lib.acoss_sync(self._ctx))

    @property
    def stream_ptr(self) -> int:
        return int(self._lib.acoss_stream(self._ctx) or 0)

    def oti_pairs(self, pairs, noti: int = 12) -> np.ndarray:
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        out = np.empty(len(pairs), dtype=np.int32)
        check(self._lib.acoss_oti_pairs(self._ctx, pairs.ctypes.data, len(pairs), int(noti), out.ctypes.data))
        return out

    def dump_pair(self, q: int, r: int, params: Params | None = None):
        """-> dict(oti, crp uint8 (M', N'), thr_q, thr_r, score) for one pair (debug API)."""
        params = params or default_params()
        incr = (params.m - 1) * params.tau if params.f4_keep_last else params.m * params.tau   # F4
        M = int(self.offsets[q + 1] - self.offsets[q]) - incr
        N = int(self.offsets[r + 1] - self.offsets[r]) - incr
        if M < 2 or N < 2:
            # let the library produce the reference-shaped error
            check(self._lib.acoss_dump_pair(self._ctx, q, r, C.byref(params), None, None, None, None, None))
        W = (N + 31) // 32
        oti = C.c_int32(0)
        score = C.c_float(0)
        bits = np.zeros((M, W), dtype=np.uint32)
        tq = np.zeros(M, dtype=np.float32)
        tr = np.zeros(N, dtype=np.float32)
        check(self._lib.acoss_dump_pair(self._ctx, q, r, C.byref(params), C.addressof(oti), bits.ctypes.data,
                                        tq.ctypes.data, tr.ctypes.data, C.addressof(score)))
        crp = np.unpackbits(bits.view(np.uint8), axis=1, bitorder="little")[:, :N]
        return dict(oti=int(oti.value), crp=crp, bits=bits, thr_q=tq, thr_r=tr, score=float(score.value))

    def dp_bytes(self, mats, mode: int = ALIGN_SW, gamma_o: float = 0.5, gamma_e: float = 0.5) -> np.ndarray:
        """Batched alignment DP over binary uint8 matrices (K3 only)."""
        mats = [np.ascontiguousarray(m) for m in mats]
        for m in mats:
            if m.ndim != 2:
                raise ValueError("matrices must be 2-D")
        # values other than 0/1 must reach the kernel's validation: clip into uint8 keeping >1 as 2
        conv = []
        for m in mats:
            if m.dtype != np.uint8:
                mm = np.where(m == 0, 0, np.where(m == 1, 1, 2)).astype(np.uint8)
            else:
                mm = m
            conv.append(mm)
        shapes = np.array([m.shape for m in conv], dtype=np.int32).reshape(-1, 2)
        sizes = np.array([m.size for m in conv], dtype=np.int64)
        offs = np.zeros(len(conv), dtype=np.int64)
        if len(conv) > 1:
            offs[1:] = np.cumsum(sizes)[:-1]
        buf = np.concatenate([m.ravel() for m in conv]) if conv else np.zeros(0, np.uint8)
        if buf.size == 0:
            buf = np.zeros(1, np.uint8)
        out = np.zeros(len(conv), dtype=np.float32)
        check(self._lib.acoss_dp_bytes(self._ctx, buf.ctypes.data, offs.ctypes.data, shapes.ctypes.data,
                                       len(conv), int(mode), float(gamma_o), float(gamma_e), out.ctypes.data))
        return out

    def set_profiling(self, on: bool = True):
        check(self._lib.acoss_set_profiling(self._ctx, int(bool(on))))

    def stage_ms(self) -> dict:
        """Accumulated CUDA-event milliseconds per pipeline stage since set_profiling(True)."""
        ms = np.zeros(4, dtype=np.float64)
        check(self._lib.acoss_stage_ms(self._ctx, ms.ctypes.data))
        return dict(k1_oti=float(ms[0]), k2_crp=float(ms[1]), k3_dp=float(ms[2]), k2_emit=float(ms[3]))

    K2_KERNELS = ("prep", "sample", "select", "hist_col", "hist_row", "hist_col2", "hist_row2", "sparse", "emit",
                  "scatter", "rank", "bits", "exact", "thr")

    def kernel_ms(self) -> dict:
        """Accumulated CUDA-event milliseconds of every kernel of the fast K2 path since set_profiling(True)."""
        ms = np.zeros(16, dtype=np.float64)
        check(self._lib.acoss_kernel_ms(self._ctx, ms.ctypes.data))
        return {k: float(ms[i]) for i, k in enumerate(self.K2_KERNELS)}

    def debug_counters(self) -> dict:
        """Diagnostic counters of the last scoring call (acoss_debug_counters): dense histogram level per
        orientation (strips, live lines, bracket misses, lines left), sparse refinement (warps, sweeps,
        lines left), listed uncertain cells, exact candidates, band cells whose coarse item was recomputed."""
        d = np.zeros(32, dtype=np.int64)
        check(self._lib.acoss_debug_counters(self._ctx, d.ctypes.data))
        lv = {"col_dense": tuple(int(x) for x in d[0:4]), "row_dense": tuple(int(x) for x in d[4:8]),
              "sparse": tuple(int(x) for x in d[8:11]),
              "col_dense2": tuple(int(x) for x in d[12:16]), "row_dense2": tuple(int(x) for x in d[16:20])}
        lv["uncertain_cells"] = int(d[24]); lv["exact_candidates"] = int(d[25]); lv["band_cells"] = int(d[26])
        return lv

    def last_stats(self) -> dict:
        st = np.zeros(8, dtype=np.int64)
        check(self._lib.acoss_last_stats(self._ctx, st.ctypes.data))
        return dict(pairs=int(st[0]), fallback_pairs=int(st[1]), launches=int(st[2]), cells=int(st[3]),
                    exact_cells=int(st[4]), status_or=int(st[5]), chunks=int(st[6]))

    # -- Simple (SiMPle) pair scoring ----------------------------------------------------------------
    def simple_score_pairs(self, pairs, params: SimpleParams | None = None) -> np.ndarray:
        """pairs (K, 2) int -> float32 (K,): the values Simple.similarity stores (acoss_simple_score_pairs)."""
        params = params or simple_default_params()
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        out = np.empty(len(pairs), dtype=np.float32)
        check(self._lib.acoss_simple_score_pairs(self._ctx, pairs.ctypes.data, len(pairs), C.byref(params),
                                                 out.ctypes.data))
        return out

    def simple_score_pairs_device(self, pairs_ptr: int, n_pairs: int, scores_ptr: int,
                                  params: SimpleParams | None = None):
        """Device in / device out, asynchronous on the engine stream; call sync()."""
        params = params or simple_default_params()
        check(self._lib.acoss_simple_score_pairs_device(self._ctx, pairs_ptr, int(n_pairs), C.byref(params),
                                                        scores_ptr))

    def simple_dump_pair(self, q: int, r: int, params: SimpleParams | None = None) -> dict:
        """-> dict(oti, profile float64 (n_q - m + 1,), index int32, score float32) of one pair."""
        params = params or simple_default_params()
        rows = max(int(self.offsets[q + 1] - self.offsets[q]) - int(params.m) + 1, 0)
        oti = C.c_int32(0)
        score = C.c_float(0)
        prof = np.zeros(max(rows, 1), dtype=np.float64)
        idx = np.zeros(max(rows, 1), dtype=np.int32)
        check(self._lib.acoss_simple_dump_pair(self._ctx, int(q), int(r), C.byref(params), C.addressof(oti),
                                               prof.ctypes.data, idx.ctypes.data, C.addressof(score)))
        return dict(oti=int(oti.value), profile=prof[:rows], index=idx[:rows], score=np.float32(score.value))

    # -- EarlyFusion pair scoring ---------------------------------------------------------------
    EF_KINDS = ("mfccs", "ssms", "chromas", "early")

    def ef_set_tracks(self, feats):
        """feats: one dict per track with the keys EarlyFusion.load_features returns
        (earlyfusion_traile.py:66-155): 'mfccs', 'ssms', 'chromas' (n_blocks, d) and 'chroma_med' (12,).
        float32 features (the reference's dtype) are uploaded as they are; anything else as float64."""
        n = len(feats)
        kinds = ("mfccs", "ssms", "chromas")
        f32 = all(np.asarray(f[k]).dtype == np.float32 for f in feats for k in kinds)
        dt = np.float32 if f32 else np.float64
        lens = [int(np.asarray(f["mfccs"]).shape[0]) for f in feats]
        offsets = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(lens, out=offsets[1:])
        bufs, dims = [], []
        for k in kinds:
            d = int(np.asarray(feats[0][k]).shape[1])
            for f, ln in zip(feats, lens):
                a = np.asarray(f[k])
                if a.ndim != 2 or a.shape != (ln, d):
                    raise ValueError("'%s' must be (n_blocks, %d) with the same n_blocks for every kind; got %r"
                                     % (k, d, a.shape))
            bufs.append(np.ascontiguousarray(np.concatenate([np.asarray(f[k], dtype=dt) for f in feats], axis=0)))
            dims.append(d)
        cmed = np.ascontiguousarray(np.stack([np.asarray(f["chroma_med"], dtype=np.float64).reshape(12)
                                              for f in feats]))
        check(self._lib.acoss_ef_set_tracks(self._ctx, bufs[0].ctypes.data, dims[0], bufs[1].ctypes.data, dims[1],
                                            bufs[2].ctypes.data, dims[2], cmed.ctypes.data, offsets.ctypes.data, n,
                                            4 if f32 else 8))
        self.ef_offsets = offsets
        self.ef_h2d_bytes = int(sum(b.nbytes for b in bufs) + cmed.nbytes + offsets.nbytes)

    def ef_score_pairs(self, pairs, kappa: float = 0.1, K: int = 10) -> np.ndarray:
        """pairs (n, 2) int -> float32 (4, n): rows 'mfccs', 'ssms', 'chromas', 'early' — the four values
        EarlyFusion.similarity stores per pair (acoss_ef_score_pairs)."""
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        out = np.zeros((4, len(pairs)), dtype=np.float32)
        check(self._lib.acoss_ef_score_pairs(self._ctx, pairs.ctypes.data, len(pairs), float(kappa), int(K),
                                             out.ctypes.data))
        return out

    def ef_dump_pair(self, q: int, r: int, kappa: float = 0.1, K: int = 10) -> dict:
        """-> dict(oti, csms float64 (4, M, N), bins uint8 (4, M, N), scores float32 (4,)) of one pair."""
        M = int(self.ef_offsets[q + 1] - self.ef_offsets[q])
        N = int(self.ef_offsets[r + 1] - self.ef_offsets[r])
        W = (N + 31) // 32
        oti = C.c_int32(0)
        csms = np.zeros((4, M, N), dtype=np.float64)
        bits = np.zeros((4, M, W), dtype=np.uint32)
        scores = np.zeros(4, dtype=np.float32)
        check(self._lib.acoss_ef_dump_pair(self._ctx, int(q), int(r), float(kappa), int(K), C.addressof(oti),
                                           csms.ctypes.data, bits.ctypes.data, scores.ctypes.data))
        bins = np.unpackbits(bits.view(np.uint8), axis=2, bitorder="little")[:, :, :N]
        return dict(oti=int(oti.value), csms=csms, bins=bins, scores=scores)

    def ef_stage_ms(self) -> dict:
        ms = np.zeros(5, dtype=np.float64)
        check(self._lib.acoss_ef_stage_ms(self._ctx, ms.ctypes.data))
        return dict(csm=float(ms[0]), knn=float(ms[1]), sw=float(ms[2]), radii=float(ms[3]), fuse=float(ms[4]))

    def ef_last_stats(self) -> dict:
        st = np.zeros(4, dtype=np.int64)
        check(self._lib.acoss_ef_last_stats(self._ctx, st.ctypes.data))
        return dict(pairs=int(st[0]), cells=int(st[1]), launches=int(st[2]), chunks=int(st[3]))

    # -- similarity-network fusion -------------------------------------------------------------------
    def snf(self, Ds, K: int = 5, niters: int = 20, reg_diag: float = 1.0, reg_neighbs: float = 0.5,
            jacobi: bool = False, want_W: bool = False, want_PS: bool = False) -> dict:
        """doSimilarityFusion of the n x n score matrices Ds on the GPU (acoss_snf): dict(fused float64 (n, n)), plus
        W float32 (n_mats, n, n) when want_W, and P float32 (n_mats, n, n), S_idx int32 / S_val float32
        (n_mats, n, K) when want_PS.  jacobi is switch L1."""
        mats = [np.ascontiguousarray(D, dtype=np.float32) for D in Ds]
        n = int(mats[0].shape[0]) if mats else 0
        for D in mats:
            if D.ndim != 2 or D.shape != (n, n):
                raise ValueError("score matrices must all be square and of one size; got %r" % (D.shape,))
        check_snf_args(len(mats), n, int(K), int(niters))
        ptrs = (C.c_void_p * len(mats))(*[D.ctypes.data for D in mats])
        out = dict(fused=np.empty((n, n), dtype=np.float64))
        if want_W:
            out["W"] = np.empty((len(mats), n, n), dtype=np.float32)
        if want_PS:
            out["P"] = np.empty((len(mats), n, n), dtype=np.float32)
            out["S_idx"] = np.empty((len(mats), n, int(K)), dtype=np.int32)
            out["S_val"] = np.empty((len(mats), n, int(K)), dtype=np.float32)
        ptr = lambda k: out[k].ctypes.data if k in out else None
        check(self._lib.acoss_snf(self._ctx, ptrs, len(mats), n, int(K), int(niters), float(reg_diag),
                                  float(reg_neighbs), int(bool(jacobi)), ptr("fused"), ptr("W"), ptr("P"),
                                  ptr("S_idx"), ptr("S_val")))
        return out

    def snf_stage_ms(self) -> dict:
        """Accumulated device milliseconds of the fusion stages since set_profiling(True)."""
        ms = np.zeros(4, dtype=np.float64)
        check(self._lib.acoss_snf_stage_ms(self._ctx, ms.ctypes.data))
        return dict(h2d=float(ms[0]), affinity=float(ms[1]), diffusion=float(ms[2]), average_d2h=float(ms[3]))
