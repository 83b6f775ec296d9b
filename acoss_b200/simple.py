"""Drop-in ``Simple`` plugin (SiMPle; reference: acoss/algorithms/simple_silva.py:17-126).

Per pair the score is the median of the SiMPle matrix profile of the query against the reference: every length-m
subsequence of pooled chroma frames of the query is matched to its nearest length-m subsequence of the (transposed)
reference.  ``similarity(idxs)`` scores a whole batch in one GPU call (acoss_simple_score_pairs, k6_simple.cu) and
``all_pairwise`` walks the pair space in tiles.  Parity is unpinned against the reference and pinned against the
restatement in DESIGN.md §2 (switches S1-S5, checked by oracle/simple_np.py); the default subsequence length (S1,
m = 10 pooled frames, about 12 s) is not confirmed against the reference.
"""
from __future__ import annotations

import numpy as np

from . import _lib
from .algorithm_template import CoverAlgorithm
from .engine import Engine, pack_tracks

__all__ = ["Simple"]


class Simple(CoverAlgorithm):
    """
    Attributes: chroma_type, oti, subsequence_length, win, skip, all_feats (the pooled chroma per song).
    Extra keyword arguments: ``device`` (CUDA ordinal), ``features`` (in-memory feature dicts), ``cachedir``,
    ``engine``, ``tile_pairs``; the switches ``keep_partial`` (S5), ``squared`` (S2), ``positive`` (S3) and
    ``roll_first`` (S4), all off by default.
    """

    def __init__(self, dataset_csv, datapath, chroma_type='hpcp', shortname='benchmark', oti=True,
                 subsequence_length=10, win=200, skip=100, keep_partial=False, squared=False, positive=False,
                 roll_first=False, device=0, features=None, cachedir="cache", engine=None, tile_pairs=1 << 16):
        self.chroma_type = chroma_type
        self.oti = oti
        self.subsequence_length = int(subsequence_length)
        self.win = int(win)
        self.skip = int(skip)
        self.keep_partial = bool(keep_partial)
        self.squared = bool(squared)
        self.positive = bool(positive)
        self.roll_first = bool(roll_first)
        self.device = device
        self.tile_pairs = int(tile_pairs)
        self.all_feats = {}
        self._engine = engine
        self._resident = False
        CoverAlgorithm.__init__(self, dataset_csv=dataset_csv, name="Simple", datapath=datapath,
                                shortname=shortname, cachedir=cachedir, features=features,
                                similarity_types=["main"])

    def load_features(self, i):
        """Pooled chroma of song i, (n_pooled, 12) float32 (simple_silva.py:38-41).  The pooling runs on the GPU
        for the whole data set at once (acoss_set_tracks_pooled) and is mirrored into ``all_feats``."""
        if i not in self.all_feats:
            self.engine()
        return self.all_feats[i]

    def params(self) -> _lib.SimpleParams:
        return _lib.simple_default_params(m=self.subsequence_length, oti=bool(self.oti), s2_squared=self.squared,
                                          s3_positive=self.positive, s4_roll_first=self.roll_first)

    def engine(self) -> Engine:
        """The CUDA engine with every song's pooled frames resident in HBM (raw frames uploaded once)."""
        if self._engine is None:
            self._engine = Engine(self.device)
        if not self._resident:
            raws = [np.asarray(CoverAlgorithm.load_features(self, i)[self.chroma_type], dtype=np.float32)
                    for i in range(self.N)]                          # also fills self.cliques
            frames, offsets = pack_tracks(raws)
            out_off = self._engine.set_tracks_pooled(frames, offsets, self.win, self.skip, self.keep_partial)
            pooled = self._engine.get_tracks()
            for i in range(self.N):
                self.all_feats.setdefault(i, pooled[out_off[i]:out_off[i + 1]])
            self._resident = True
        return self._engine

    def similarity(self, idxs):
        """Ds["main"][i, j] for every (query i, reference j) row of idxs, in one batched GPU call."""
        idxs = np.asarray(idxs).reshape(-1, 2)
        if len(idxs) == 0:
            return
        self.Ds["main"][idxs[:, 0], idxs[:, 1]] = self.score_pairs(idxs)

    def all_pairwise(self, parallel=0, n_cores=12, symmetric=False, precomputed=False):
        """algorithm_template.py:142-192 with the pair fan-out batched for the GPU (``parallel`` / ``n_cores`` are
        accepted and ignored: a CUDA context must not be forked)."""
        h5filename = "%s_Ds.h5" % self.get_cacheprefix()
        if precomputed:
            self.Ds = self._load_Ds(h5filename)
            self.get_all_clique_ids()
            return
        all_pairs = self._pair_array(symmetric)
        self.engine()                              # loads every song => cliques are complete
        for k0 in range(0, len(all_pairs), self.tile_pairs):
            self.similarity(all_pairs[k0:k0 + self.tile_pairs])
        if symmetric:
            for similarity_type in self.Ds:
                self.Ds[similarity_type] += self.Ds[similarity_type].T
        self._save_Ds(h5filename)

    # -- hooks of acoss_b200.distributed.all_pairwise_distributed (one process per GPU) -----------------
    def pair_weights(self, pairs):
        """Work of a pair = cells of its join, (n_i - m + 1)(n_j - m + 1)."""
        pairs = np.asarray(pairs).reshape(-1, 2)
        lens = np.array([self.load_features(i).shape[0] for i in range(self.N)], dtype=np.int64)
        cells = np.maximum(lens - self.subsequence_length + 1, 0)
        return cells[pairs[:, 0]] * cells[pairs[:, 1]]

    def score_pairs(self, pairs):
        """float32 (n,) scores of the pairs."""
        pairs = np.asarray(pairs).reshape(-1, 2)
        if len(pairs) == 0:
            return np.zeros(0, dtype=np.float32)
        return self.engine().simple_score_pairs(pairs.astype(np.int32), self.params())

    def close(self):
        if self._engine is not None:
            self._engine.close()
            self._engine = None
            self._resident = False
