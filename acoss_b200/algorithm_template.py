"""Host-side mirror of the reference's plugin base class ``CoverAlgorithm``
(/root/reference/acoss/algorithms/algorithm_template.py:17-290).

Same attribute names (``filepaths``, ``cliques``, ``Ds``, ``N``, ``name``, ``shortname``,
``cachedir``), same method names, argument meanings and side effects (NxN float32 memmap score
matrices under ``cachedir``; ``results_<shortname>_<name>.csv`` appended by ``getEvalStatistics``),
so code written against the reference class runs against this one.  Written from the interface,
not from the reference's code: pair enumeration is array-based (no 112 M-tuple Python list,
algorithm_template.py:168-169), and the evaluation is vectorised while returning exactly the
numbers the reference loop returns (tests/test_plugin_cpu.py checks it against golden vectors the
reference produced).

Feature files: the reference reads deepdish ``.h5`` dictionaries (algorithm_template.py:90).
deepdish/HDF5 are absent from this image, so ``load_features`` reads ``<path>.h5`` through deepdish
when it is importable, else the same dictionary stored as ``<path minus .h5>.npz``; synthetic runs
pass ``features=[{...}, ...]`` and skip files entirely.
"""
from __future__ import annotations

import csv
import os
import warnings

import numpy as np

__all__ = ["CoverAlgorithm", "create_dataset_filepaths"]


def create_dataset_filepaths(dataset_csv, root_audio_dir, file_format=".h5"):
    """``root_audio_dir + work_id + "/" + track_id + file_format`` per CSV row
    (acoss/utils.py:87-102; note: no separator is inserted after root_audio_dir)."""
    with open(dataset_csv, newline="") as f:
        rd = csv.DictReader(f)
        keys = rd.fieldnames or []
        for k in keys:
            if k not in ("work_id", "track_id"):
                raise IOError("Wrong input dataset csv annotation file '%s'. Expected a csv file with the "
                              "columns of key 'work_id', 'track_id'" % dataset_csv)
        return [root_audio_dir + row["work_id"] + "/" + row["track_id"] + file_format for row in rd]


def _load_feature_file(path):
    try:
        import deepdish as dd
        return dd.io.load(path)
    except ImportError:
        alt = path[:-3] + ".npz" if path.endswith(".h5") else path + ".npz"
        with np.load(alt, allow_pickle=False) as z:
            out = {k: z[k] for k in z.files}
        if "label" in out:
            out["label"] = str(out["label"])
        return out


def _zeroed_memmap(path, shape):
    """What ``np.memmap(path, mode="w+")`` gives (a zero float32 matrix backed by ``path``), without its window in
    which the file is 0 bytes long: ranks that construct on the same cache prefix at once would otherwise fail to
    map a file another rank has just truncated."""
    nbytes = int(np.prod(shape)) * 4
    fd = os.open(path, os.O_RDWR | os.O_CREAT, 0o666)
    try:
        size = os.fstat(fd).st_size
        if size != nbytes:
            os.ftruncate(fd, nbytes)
    finally:
        os.close(fd)
    mm = np.memmap(path, mode="r+", dtype="float32", shape=shape)
    if size:                                                 # a file that existed keeps old scores: clear them
        mm[:] = 0
    return mm


class CoverAlgorithm(object):
    """
    Attributes
    ----------
    filepaths: list(string)   paths of all feature files of the dataset
    cliques: {string: set}    cover cliques, indices into filepaths
    Ds: {similarity type: ndarray(N, N) float32 memmap}   pairwise score matrices
    """

    def __init__(self, dataset_csv, name="Serra09", datapath="features_benchmark", shortname="full",
                 cachedir="cache", similarity_types=["main"], features=None):
        self.name = name
        self.shortname = shortname
        self.cachedir = cachedir
        self._features = features
        if features is not None:
            self.filepaths = ["<memory>/%d" % i for i in range(len(features))]
        else:
            self.filepaths = create_dataset_filepaths(dataset_csv, root_audio_dir=datapath, file_format=".h5")
        self.cliques = {}
        self.N = len(self.filepaths)
        os.makedirs(cachedir, exist_ok=True)                  # (several ranks of one box may construct at once)
        self.Ds = {}
        for s in similarity_types:
            self.Ds[s] = _zeroed_memmap("%s_%s_dmat" % (self.get_cacheprefix(), s), (self.N, self.N))
        print("Initialized %s algorithm on %i songs in dataset %s" % (name, self.N, shortname))

    def get_cacheprefix(self):
        return "%s/%s_%s" % (self.cachedir, self.name, self.shortname)

    def load_features(self, i):
        """Feature dictionary of song i; records its clique in ``self.cliques`` as a side effect
        (algorithm_template.py:71-95)."""
        feats = self._features[i] if self._features is not None else _load_feature_file(self.filepaths[i])
        label = feats["label"]
        if label not in self.cliques:
            self.cliques[label] = set([])
        self.cliques[label].add(i)
        return feats

    def get_all_clique_ids(self, verbose=False):
        """Fill ``self.cliques`` for every song, cached in ``<prefix>_clique_info.txt``
        (algorithm_template.py:97-119)."""
        filepath = "%s_clique_info.txt" % self.get_cacheprefix()
        if not os.path.exists(filepath):
            with open(filepath, "w") as fout:
                for i in range(len(self.filepaths)):
                    feats = CoverAlgorithm.load_features(self, i)
                    if verbose:
                        print(i)
                    fout.write("%i,%s\n" % (i, feats["label"]))
        else:
            with open(filepath) as fin:
                for line in fin.readlines():
                    i, label = line.split(",")
                    label = label.strip()
                    if label not in self.cliques:
                        self.cliques[label] = set([])
                    self.cliques[label].add(int(i))

    def similarity(self, idxs):
        """Template: score 0 for every (i, j) row of idxs (algorithm_template.py:121-140)."""
        idxs = np.asarray(idxs)
        for i, j in idxs:
            self.Ds["main"][i, j] = 0.0

    # ------------------------------------------------------------------------------------------
    def _pair_array(self, symmetric):
        n = len(self.filepaths)
        if symmetric:
            i, j = np.triu_indices(n, k=1)                  # itertools.combinations order
            return np.stack([i, j], axis=1).astype(np.int64)
        i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
        keep = i != j                                        # itertools.permutations order
        return np.stack([i[keep], j[keep]], axis=1).astype(np.int64)

    def _save_Ds(self, h5filename):
        try:
            import deepdish as dd
            dd.io.save(h5filename, self.Ds)
        except ImportError:
            np.savez(h5filename[:-3] + ".npz", **{k: np.asarray(v) for k, v in self.Ds.items()})

    def _load_Ds(self, h5filename):
        try:
            import deepdish as dd
            return dd.io.load(h5filename)
        except ImportError:
            with np.load(h5filename[:-3] + ".npz") as z:
                return {k: z[k] for k in z.files}

    def all_pairwise(self, parallel=0, n_cores=12, symmetric=False, precomputed=False):
        """All pairwise comparisons (algorithm_template.py:142-192).  The base implementation walks
        the reference's 45 chunks serially; GPU plugins override the fan-out.  ``parallel`` /
        ``n_cores`` are accepted for signature compatibility."""
        h5filename = "%s_Ds.h5" % self.get_cacheprefix()
        if precomputed:
            self.Ds = self._load_Ds(h5filename)
            self.get_all_clique_ids()
            return
        all_pairs = self._pair_array(symmetric)
        for chunk in np.array_split(all_pairs, 45):
            if len(chunk):
                self.similarity(chunk)
        if parallel == 1:
            self.get_all_clique_ids()
        if symmetric:
            for similarity_type in self.Ds:
                self.Ds[similarity_type] += self.Ds[similarity_type].T
        self._save_Ds(h5filename)

    def cleanup_memmap(self):
        """Remove the memmap files.  (The reference calls shutil.rmtree on a *file*, which always
        fails and prints 'Could not clean-up automatically.' — algorithm_template.py:194-203; the
        files are actually removed here.)"""
        for s in list(self.Ds):
            path = "%s_%s_dmat" % (self.get_cacheprefix(), s)
            try:
                mm = self.Ds[s]
                if isinstance(mm, np.memmap):
                    mm.flush()
                if os.path.exists(path):
                    os.remove(path)
            except OSError:
                print("Could not clean-up automatically.")

    # ------------------------------------------------------------------------------------------
    def getEvalStatistics(self, similarity_type, topsidx=[1, 10, 100, 1000]):
        """MR, MRR, MDR, MAP and Top-k of ``self.Ds[similarity_type]``; appends a row to
        ``results_<shortname>_<name>.csv`` (algorithm_template.py:205-290).  Vectorised per clique,
        numerically identical to the reference loop (same ``np.argsort(-D, 1)`` call, so tie order
        matches too)."""
        MR, MRR, MDR, MAP, tops, ranks = eval_statistics(np.asarray(self.Ds[similarity_type]), self.cliques,
                                                         topsidx)
        print(ranks)
        print("%s %s STATS\n-------------------------\nMR = %.3g\nMRR = %.3g\nMDR = %.3g\nMAP = %.3g"
              % (self.name, similarity_type, MR, MRR, MDR, MAP))
        for t, v in zip(topsidx, tops):
            print("Top-%i: %i" % (t, v))
        resultsfile = "results_%s_%s.csv" % (self.shortname, self.name)
        if not os.path.exists(resultsfile):
            with open(resultsfile, "w") as fout:
                fout.write("name, MR, MRR, MDR, MAP")
                for t in topsidx:
                    fout.write(",Top-%i" % t)
                fout.write("\n")
        with open(resultsfile, "a") as fout:
            fout.write("%s_%s," % (self.name, similarity_type))
            fout.write("%.3g, %.3g, %.3g, %.3g" % (MR, MRR, MDR, MAP))
            for t in tops:
                fout.write(", %.3g" % t)
            fout.write("\n")
        return MR, MRR, MDR, MAP, tops


def eval_statistics(D, cliques, topsidx=(1, 10, 100, 1000), row_block=2048):
    """Vectorised evaluation with the reference's exact semantics:

    * cliques are laid out contiguously in descending size (``np.argsort(-Ks)`` order), members in
      set-iteration order; rows/columns of D are permuted accordingly;
    * the diagonal is -inf; ``np.argsort(-D, 1)`` ranks every row (same call => same tie order);
    * per query in a clique of size K >= 2: the 1-based ranks of the K clique members in ascending
      order with the LAST one dropped (the reference assumes it is the query itself);
    * evaluation stops at the first clique of size < 2 (descending order => all the rest);
    * MRR divides by N = all tracks including singletons (algorithm_template.py:266).
    """
    D = np.array(D, dtype=np.float32)
    N = D.shape[0]
    groups = [list(cliques[s]) for s in cliques]
    Ks = np.array([len(c) for c in groups])
    order = np.argsort(-Ks)
    Ks = Ks[order]
    groups = [groups[i] for i in order]
    perm = np.fromiter((x for c in groups for x in c), dtype=np.int64, count=int(Ks.sum()))
    D = D[perm, :][:, perm]
    np.fill_diagonal(D, -np.inf)
    starts = np.concatenate([[0], np.cumsum(Ks)[:-1]])
    ranks = np.full(N, np.nan)
    allmap = np.full(N, np.nan)
    n_eval = int(Ks[Ks >= 2].sum()) if (Ks >= 2).any() else 0
    # rows are evaluated in order until the first clique with fewer than 2 members
    first_small = np.nonzero(Ks < 2)[0]
    n_groups = int(first_small[0]) if len(first_small) else len(Ks)
    n_eval = int(Ks[:n_groups].sum())
    clique_of_row = np.repeat(np.arange(len(Ks)), Ks)
    stop = False
    for r0 in range(0, n_eval, row_block):
        r1 = min(n_eval, r0 + row_block)
        srt = np.argsort(-D[r0:r1], 1)
        pos = np.empty_like(srt)
        rows = np.arange(r1 - r0)[:, None]
        pos[rows, srt] = np.arange(1, N + 1)[None, :]        # pos[i, col] = 1-based rank of col in row i
        for i in range(r0, r1):
            g = clique_of_row[i]
            K = int(Ks[g])
            member_ranks = np.sort(pos[i - r0, starts[g]:starts[g] + K])[:-1]
            if len(member_ranks) == 0:
                warnings.warn("Recalling 0 songs for clique of size %i at song index %i" % (K, i))
                stop = True
                break
            ranks[i] = member_ranks[0]
            allmap[i] = np.mean(np.arange(1, K, dtype=np.float64) / member_ranks.astype(np.float64))
        if stop:
            break
    MAP = np.nanmean(allmap)
    ranks = ranks[~np.isnan(ranks)]
    MR = np.mean(ranks)
    MRR = 1.0 / N * (np.sum(1.0 / ranks))
    MDR = np.median(ranks)
    tops = np.zeros(len(topsidx))
    for i, t in enumerate(topsidx):
        tops[i] = np.sum(ranks <= t)
    return MR, MRR, MDR, MAP, tops, ranks
