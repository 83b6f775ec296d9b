"""Drop-in ``EarlyFusion`` plugin (reference: /root/reference/acoss/algorithms/earlyfusion_traile.py:20-198
and the in-tree kernels it calls, utils/cross_recurrence.py, utils/similarity_fusion.py:38-54,
utils/alignment_tools.py).

``similarity(idxs)`` scores a whole batch of pairs in ONE GPU call (``acoss_ef_score_pairs``): per pair the
Euclidean cross-similarity matrices of the mfcc and ssm blocks, the blocked-OTI cosine matrix of the chroma
blocks, the "early" fusion exp(-sum of getWCSM(CSM, K, K)), and
``smith_waterman_constrained(csm_to_binary(., kappa))`` of all four — ``Ds['mfccs' | 'ssms' | 'chromas' |
'early'][i, j]`` exactly as earlyfusion_traile.py:166-198 fills them.  The block features of every track are
uploaded once (``acoss_ef_set_tracks``) and stay resident in HBM; no matrix crosses PCIe.

Out of scope (SURVEY.md §8f rank 4 covers the pair scoring only): the beat-synchronous block-feature
on-ramp of ``load_features`` (madmom onsets, skimage resize — absent from this image).  ``load_features``
therefore returns precomputed block features exactly as the reference's returns them (keys 'mfccs', 'ssms',
'chromas', 'chroma_med', 'label'), from memory or from the reference's own cache file layout.
``do_late_fusion`` (N x N similarity-network fusion of finished score matrices) is delegated to the
reference's function when the ``acoss`` package is importable; ``impl="gpu"`` runs it on the GPU
(``acoss_b200.fusion``, k7_snf.cu).

``sw_of_csms`` scores caller-supplied float64 cross-similarity matrices on the GPU (``acoss_knn_sw``).  There is
no host (numpy) implementation of any stage in this package: without the CUDA library every call raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _lib
from .algorithm_template import CoverAlgorithm, _load_feature_file
from .engine import Engine

__all__ = ["EarlyFusion", "nneighbs", "sw_of_csms"]


def nneighbs(kappa, n_cols: int) -> int:
    """Neighbours per row of csm_to_binary (cross_recurrence.py:151-155): kappa == 0 -> all (-1),
    kappa < 1 -> int(np.round(kappa * n_cols)) (banker's rounding), else kappa."""
    if kappa == 0:
        return -1
    if kappa < 1:
        return int(np.round(kappa * n_cols))
    return int(kappa)


def sw_of_csms(engine: Engine, csms, kappa, want_bits=False):
    """scores[k] = smith_waterman_constrained(csm_to_binary(csms[k], kappa)) for a batch of float64
    cross-similarity matrices, on the GPU (acoss_knn_sw)."""
    csms = [np.ascontiguousarray(c, dtype=np.float64) for c in csms]
    n = len(csms)
    shapes = np.array([c.shape for c in csms], dtype=np.int32).reshape(-1, 2)
    sizes = np.array([c.size for c in csms], dtype=np.int64)
    offs = np.zeros(n, dtype=np.int64)
    if n > 1:
        offs[1:] = np.cumsum(sizes)[:-1]
    nn = np.array([nneighbs(kappa, c.shape[1]) for c in csms], dtype=np.int32)
    buf = np.concatenate([c.ravel() for c in csms]) if n else np.zeros(1)
    scores = np.zeros(n, dtype=np.float32)
    bits = None
    if want_bits:
        bits = np.zeros(int(sum(c.shape[0] * ((c.shape[1] + 31) // 32) for c in csms)), dtype=np.uint32)
    _lib.check(engine._lib.acoss_knn_sw(engine._ctx, buf.ctypes.data, offs.ctypes.data, shapes.ctypes.data,
                                        nn.ctypes.data, n, scores.ctypes.data,
                                        bits.ctypes.data if bits is not None else None))
    if not want_bits:
        return scores
    mats, o = [], 0
    for c in csms:
        M, N = c.shape
        W = (N + 31) // 32
        w = bits[o:o + M * W].reshape(M, W)
        mats.append(np.unpackbits(w.view(np.uint8), axis=1, bitorder="little")[:, :N])
        o += M * W
    return scores, mats


class EarlyFusion(CoverAlgorithm):
    """Constructor signature of the reference class (earlyfusion_traile.py:44-58) plus ``device``,
    ``features`` (in-memory block features) and ``cachedir``.  Score types: 'mfccs', 'ssms', 'chromas',
    'early' (earlyfusion_traile.py:58)."""

    def __init__(self, dataset_csv, datapath, chroma_type='hpcp', shortname='benchmark', blocksize=20,
                 mfccs_per_block=50, ssm_res=50, chromas_per_block=40, kappa=0.1, K=10, niters=5,
                 log_times=False, device=0, features=None, cachedir="cache", engine=None):
        self.chroma_type = chroma_type
        self.blocksize = blocksize
        self.mfccs_per_block = mfccs_per_block
        self.ssm_res = ssm_res
        self.chromas_per_block = chromas_per_block
        self.kappa = kappa
        self.K = K
        self.niters = niters
        self.log_times = log_times
        if log_times:
            self.times = {'features': [], 'raw': []}
        self.device = device
        self.all_block_feats = {}
        self._engine = engine
        self._resident = False
        self.tile_pairs = 1 << 15
        CoverAlgorithm.__init__(self, dataset_csv, name="EarlyFusionTraile", datapath=datapath,
                                shortname=shortname, cachedir=cachedir,
                                similarity_types=["mfccs", "ssms", "chromas", "early"], features=features)

    def get_cacheprefix(self):
        return "%s/%s_%s_%s" % (self.cachedir, self.name, self.shortname, self.chroma_type)

    def load_features(self, i):
        """Precomputed block features of song i (what the reference's load_features returns,
        earlyfusion_traile.py:66-155); records the clique as a side effect.  Lookup order of the reference
        (:84-97): the in-memory cache, then the per-song cache file ``<cacheprefix>_<i>.h5`` the reference
        writes after computing the blocks (read through deepdish when importable, else the same dictionary as
        ``<cacheprefix>_<i>.npz``), then the feature dictionary of the song itself, which must already hold the
        block features (the beat-synchronous block computation is not part of this package)."""
        if i in self.all_block_feats:
            return self.all_block_feats[i]
        cached = "%s_%i.h5" % (self.get_cacheprefix(), i)
        feats = None
        if self._features is None and (os.path.exists(cached) or os.path.exists(cached[:-3] + ".npz")):
            feats = _load_feature_file(cached)
            CoverAlgorithm.load_features(self, i)               # clique info as a side effect (:95-96)
        else:
            feats = CoverAlgorithm.load_features(self, i)
        missing = [k for k in ("mfccs", "ssms", "chromas", "chroma_med") if k not in feats]
        if missing:
            raise KeyError("song %d has no precomputed block features %r; compute them with the reference's "
                           "EarlyFusion.load_features (madmom / skimage on-ramp) first" % (i, missing))
        self.all_block_feats[i] = feats
        return feats

    def engine(self) -> Engine:
        if self._engine is None:
            self._engine = Engine(self.device)
        return self._engine

    def _ensure_resident(self):
        """Upload every track's block features once (the per-process cache all_block_feats of the
        reference becomes the HBM-resident feature set)."""
        if not self._resident:
            self.engine().ef_set_tracks([self.load_features(i) for i in range(self.N)])
            self._resident = True

    def similarity(self, idxs):
        """Ds[s][i, j] for s in mfccs / ssms / chromas / early and every (i, j) row of idxs
        (earlyfusion_traile.py:157-198), one batched GPU call."""
        import time
        idxs = np.asarray(idxs).reshape(-1, 2)
        if len(idxs) == 0:
            return
        self._ensure_resident()
        tic = time.time()
        scores = self.engine().ef_score_pairs(idxs.astype(np.int32), self.kappa, self.K)
        if self.log_times:
            self.times['raw'].append((time.time() - tic) / len(idxs))
        for k, s in enumerate(Engine.EF_KINDS):
            self.Ds[s][idxs[:, 0], idxs[:, 1]] = scores[k]

    def all_pairwise(self, parallel=0, n_cores=12, symmetric=False, precomputed=False):
        """algorithm_template.py:142-192 with the pair fan-out batched for the GPU: tiles of ``tile_pairs``
        pairs per ``similarity`` call instead of the reference's 45 joblib chunks (``parallel`` / ``n_cores`` are
        accepted and ignored: a CUDA context must not be forked)."""
        h5filename = "%s_Ds.h5" % self.get_cacheprefix()
        if precomputed:
            self.Ds = self._load_Ds(h5filename)
            self.get_all_clique_ids()
            return
        all_pairs = self._pair_array(symmetric)
        self._ensure_resident()                    # loads every song => cliques are complete
        for k0 in range(0, len(all_pairs), self.tile_pairs):
            self.similarity(all_pairs[k0:k0 + self.tile_pairs])
        if symmetric:
            for similarity_type in self.Ds:
                self.Ds[similarity_type] += self.Ds[similarity_type].T
        self._save_Ds(h5filename)

    # -- hooks of acoss_b200.distributed.all_pairwise_distributed (one process per GPU) -----------------
    def pair_weights(self, pairs):
        """Work of a pair = cells of its cross-similarity matrices (blocks_i x blocks_j)."""
        pairs = np.asarray(pairs).reshape(-1, 2)
        nb = np.array([np.asarray(self.load_features(i)["mfccs"]).shape[0] for i in range(self.N)], dtype=np.int64)
        return nb[pairs[:, 0]] * nb[pairs[:, 1]]

    def score_pairs(self, pairs):
        """float32 (4, n): rows in Ds key order (mfccs, ssms, chromas, early)."""
        pairs = np.asarray(pairs).reshape(-1, 2)
        if len(pairs) == 0:
            return np.zeros((4, 0), dtype=np.float32)
        self._ensure_resident()
        return self.engine().ef_score_pairs(pairs.astype(np.int32), self.kappa, self.K)

    def do_late_fusion(self, impl="reference"):
        """earlyfusion_traile.py:200-206 — SNF of the finished N x N score matrices.  impl="reference" calls the
        reference's own doSimilarityFusion (NotImplementedError when the acoss package is not importable);
        impl="gpu" runs both fusions on this plugin's GPU (acoss_b200.fusion) with the same keys and dtypes."""
        if impl == "gpu":
            from .fusion import fuse
            def doSimilarityFusion(Scores, K, niters, reg_diag):
                return None, fuse(Scores, K=K, niters=niters, reg_diag=reg_diag, engine=self.engine())["fused"]
        elif impl == "reference":
            try:
                from acoss.algorithms.utils.similarity_fusion import doSimilarityFusion
            except Exception as e:
                raise NotImplementedError(
                    "do_late_fusion is the reference's N x N similarity-network fusion (similarity_fusion.py); "
                    "install the reference package to use it, or pass impl='gpu'") from e
        else:
            raise ValueError("impl must be 'reference' or 'gpu', got %r" % (impl,))
        self.Ds["late"] = doSimilarityFusion([1.0 / (1.0 + self.Ds[s]) for s in ["chromas", "ssms", "mfccs"]],
                                             K=20, niters=20, reg_diag=1)[1]
        self.Ds["early+late"] = doSimilarityFusion(
            [1.0 / (1.0 + self.Ds[s]) for s in ["chromas", "ssms", "mfccs", "early"]], K=20, niters=20, reg_diag=1)[1]

    def close(self):
        if self._engine is not None:
            self._engine.close()
            self._engine = None
            self._resident = False
