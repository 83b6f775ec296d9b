"""Drop-in ``ChenFusion`` plugin (reference: /root/reference/acoss/algorithms/latefusion_chen.py:18-91).

Same constructor arguments, attributes and methods as the reference class.  ``similarity(idxs)``
builds ONE binary cross-recurrence plot per pair on the GPU (K1 OTI -> K2 CRP, shared with
``Serra09``) and runs both alignments over it: Qmax (``Ds["qmax"]``) and Dmax (``Ds["dmax"]``),
where the reference calls essentia three times per pair (latefusion_chen.py:63-73).

``do_late_fusion`` is the reference's N x N similarity-network fusion of the two finished score
matrices (acoss/algorithms/utils/similarity_fusion.py).  By default it is delegated to the reference's
own function when the ``acoss`` package is importable and refused otherwise; ``impl="gpu"`` runs it on
the GPU (``acoss_b200.fusion``, k7_snf.cu).
"""
from __future__ import annotations

import numpy as np

from .engine import Engine
from .serra09 import Serra09

__all__ = ["ChenFusion"]


class ChenFusion(Serra09):
    def __init__(self, dataset_csv, datapath, chroma_type='hpcp', shortname='benchmark',
                 oti=True, kappa=0.095, tau=1, m=9, downsample_fac=40, **kw):
        Serra09.__init__(self, dataset_csv, datapath, chroma_type=chroma_type, shortname=shortname, oti=oti,
                         kappa=kappa, tau=tau, m=m, downsample_fac=downsample_fac,
                         _name="LateFusionChen", _similarity_types=("qmax", "dmax"), **kw)

    def score_pairs(self, pairs):
        """pairs (n, 2) int -> float32 (2, n): the Qmax and Dmax rows, in Ds key order, of one batched GPU call.
        The scoring hook of all_pairwise_distributed; there is no pair_weights, so the distributed run keeps the
        list-free triangle shard of Serra09."""
        pairs = np.asarray(pairs).reshape(-1, 2).astype(np.int32)
        return np.stack(self.engine().score_pairs_chen(pairs, self.params()))

    def similarity(self, idxs):
        """Ds["qmax"][i, j], Ds["dmax"][i, j] for every (query i, reference j) row of idxs
        (latefusion_chen.py:58-73), one batched GPU call."""
        idxs = np.asarray(idxs).reshape(-1, 2)
        if len(idxs) == 0:
            return
        qmax, dmax = self.score_pairs(idxs)
        self.Ds["qmax"][idxs[:, 0], idxs[:, 1]] = qmax
        self.Ds["dmax"][idxs[:, 0], idxs[:, 1]] = dmax

    def normalize_by_length(self):
        """Ds[i, j] = sqrt(n_frames_j) / Ds[i, j] (latefusion_chen.py:75-85): scores become distances;
        float64 quotient, float32 store; a zero score gives inf exactly as numpy does in the reference."""
        fac = np.sqrt(np.array([self.load_features(j).shape[0] for j in range(self.N)], dtype=np.int64))
        for key in self.Ds.keys():
            D = np.asarray(self.Ds[key]).astype(np.float64)
            with np.errstate(divide="ignore"):
                self.Ds[key][:, :] = (fac[None, :] / D).astype(np.float32)

    def do_late_fusion(self, impl="reference"):
        """latefusion_chen.py:87-91 — SNF of the two distance matrices, then the sign flip.  impl="reference" calls the
        reference's doSimilarityFusion (NotImplementedError when the acoss package is not importable); impl="gpu"
        runs the fusion on this plugin's GPU (acoss_b200.fusion) with the same keys, signs and dtypes."""
        if impl == "gpu":
            from .fusion import fuse
            if self._engine is None:             # the fusion needs a device, not the resident tracks of engine()
                self._engine = Engine(self.device)
            DLate = fuse([self.Ds[s] for s in self.Ds], K=20, niters=20, reg_diag=1, engine=self._engine)["fused"]
        elif impl == "reference":
            try:
                from acoss.algorithms.utils.similarity_fusion import doSimilarityFusion
            except Exception as e:  # the reference package (and its heavy imports) is not installed
                raise NotImplementedError(
                    "do_late_fusion is the reference's N x N similarity-network fusion (similarity_fusion.py); "
                    "install the reference package to use it, or pass impl='gpu'") from e
            DLate = doSimilarityFusion([self.Ds[s] for s in self.Ds], K=20, niters=20, reg_diag=1)[1]
        else:
            raise ValueError("impl must be 'reference' or 'gpu', got %r" % (impl,))
        for key in self.Ds:
            self.Ds[key] *= -1                    # switch back to larger scores being closer
        self.Ds["Late"] = DLate
