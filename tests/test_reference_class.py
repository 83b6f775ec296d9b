"""The drop-in boundary under the reference's OWN classes (VERDICT r1, "prove the boundary against the real class").

With ``ACOSS_REFERENCE`` naming a checkout of the original acoss (github.com/furkanyesiler/acoss): the unmodified
``acoss.algorithms.rqa_serra09.Serra09`` (on its unmodified ``CoverAlgorithm`` base, imported through the SURVEY
App. C shims) is subclassed by the INTEGRATION.md section B binding (``acoss_b200.integration.bind_serra09``) and runs
the ``coverid.benchmark`` sequence (``acoss/coverid.py:57-70``) with the reference's own ``all_pairwise`` /
``normalize_by_length`` / ``getEvalStatistics``.  The binding talks to a CPU stand-in of the same C ABI backed by the
oracle (``oracle/abi_stub.c``, test infrastructure).  The resulting score matrix and metrics are the committed golden
``tests/golden/refclass_tiny_golden.npz``.

Without the reference, the same binding on this package's mirror base class must reproduce that golden bit for bit:
on the CPU stand-in, and on the real ``libacoss_b200.so`` together with ``acoss_b200.serra09.Serra09``."""
import ctypes as C
import os
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("ACOSS_REFERENCE", "")                # checkout of the original acoss (optional)
GOLDEN = os.path.join(ROOT, "tests", "golden", "refclass_tiny_golden.npz")
TOPS = [1, 10]


def _tiny():
    from acoss_b200 import synthetic
    tracks, labels = synthetic.config_dataset("tiny")
    return tracks, ["w%d" % l for l in labels]


def _install_shims():
    """SURVEY Appendix C: stub modules so the untouched reference package imports; deepdish reads the .npz
    dictionaries this test writes, librosa.util.sync is the median aggregation restated in oracle/onramp_np.py."""
    from oracle.onramp_np import median_sync

    def mk(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    def dd_load(path, *a, **k):
        with np.load(path, allow_pickle=False) as z:
            return {key: (str(z[key]) if z[key].ndim == 0 else z[key]) for key in z.files}
    dd = mk("deepdish")
    io = mk("deepdish.io", load=dd_load, save=lambda *a, **k: None)
    dd.io = io; dd.load = io.load; dd.save = io.save

    class Bar:
        def __init__(self, *a, **k): pass
        def next(self): pass
        def finish(self): pass
    pr = mk("progress"); pr.bar = mk("progress.bar", Bar=Bar)
    es = mk("essentia", Pool=object, array=np.array, run=lambda *a: None)
    es.standard = mk("essentia.standard", ChromaCrossSimilarity=object, CoverSongSimilarity=object)

    def sync(data, idx, aggregate=None, **k):              # librosa.util.sync(chroma.T, arange(0, n, fac), np.median)
        assert aggregate is np.median
        idx = np.asarray(idx)
        fac = int(idx[1] - idx[0]) if len(idx) > 1 else int(data.shape[1])
        return median_sync(np.ascontiguousarray(data.T), fac).T
    lr = mk("librosa")
    lr.util = mk("librosa.util", sync=sync, normalize=None)
    lr.filters = mk("librosa.filters", get_window=None)
    if REF not in sys.path:
        sys.path.insert(0, REF)
    sys.dont_write_bytecode = True


def _write_dataset(tmp, tracks, labels):
    """dataset csv (work_id, track_id) + one feature dictionary per track where create_dataset_filepaths points."""
    feat = os.path.join(tmp, "features") + os.sep
    rows = ["work_id,track_id"]
    for t, (x, lab) in enumerate(zip(tracks, labels)):
        os.makedirs(os.path.join(feat, lab), exist_ok=True)
        with open(os.path.join(feat, lab, "t%03d.h5" % t), "wb") as f:      # the name the reference builds
            np.savez(f, hpcp=x, label=np.array(lab))
        rows.append("%s,t%03d" % (lab, t))
    csv = os.path.join(tmp, "tiny.csv")
    with open(csv, "w") as f:
        f.write("\n".join(rows) + "\n")
    return csv, feat


@pytest.fixture()
def shimmed_reference():
    """Installs the shims and removes them (and the imported reference package) again afterwards, so no other test
    sees stub modules."""
    before = set(sys.modules)
    path = list(sys.path)
    _install_shims()
    yield
    for name in set(sys.modules) - before:
        del sys.modules[name]
    sys.path[:] = path


@pytest.mark.skipif(not os.path.isdir(REF), reason="ACOSS_REFERENCE names no checkout of acoss: the committed golden stands in")
def test_binding_under_the_reference_classes(tmp_path, monkeypatch, shimmed_reference):
    monkeypatch.chdir(tmp_path)                              # the reference writes cache/ and results_*.csv into the CWD
    from acoss.algorithms.algorithm_template import CoverAlgorithm as RefCoverAlgorithm
    from acoss.algorithms.rqa_serra09 import Serra09 as RefSerra09
    assert RefSerra09.__mro__[1] is RefCoverAlgorithm and RefSerra09.__module__ == "acoss.algorithms.rqa_serra09"
    from acoss_b200.integration import bind_serra09
    from oracle import build as obuild
    stub = C.CDLL(obuild.build_stub())
    tracks, labels = _tiny()
    csv, feat = _write_dataset(str(tmp_path), tracks, labels)
    Bound = bind_serra09(RefSerra09, lib=stub)
    assert Bound.all_pairwise is RefCoverAlgorithm.all_pairwise                # the reference's own driver,
    assert Bound.normalize_by_length is RefSerra09.normalize_by_length        # normalisation
    assert Bound.getEvalStatistics is RefCoverAlgorithm.getEvalStatistics     # and evaluation
    alg = Bound(dataset_csv=csv, datapath=feat, chroma_type="hpcp", shortname="tiny", downsample_fac=1)
    # the sequence of coverid.benchmark (coverid.py:57-70)
    alg.all_pairwise(0, n_cores=1, symmetric=True)
    raw = np.array(alg.Ds["main"])
    alg.normalize_by_length()
    Dn = np.array(alg.Ds["main"])
    MR, MRR, MDR, MAP, tops = alg.getEvalStatistics("main", topsidx=TOPS)
    alg.release()
    metrics = np.array([MR, MRR, MDR, MAP] + list(tops), dtype=np.float64)
    assert MAP > 0.9 and raw.max() > 50
    if os.environ.get("ACOSS_REGEN_GOLDEN") or not os.path.exists(GOLDEN):
        np.savez_compressed(GOLDEN, raw=raw, normalized=Dn, metrics=metrics, tops=np.array(TOPS))
    g = np.load(GOLDEN)
    assert np.array_equal(g["raw"], raw) and np.array_equal(g["normalized"], Dn)
    assert np.array_equal(g["metrics"], metrics)
    # and the mirror base class of this package gives the same numbers from the same scores
    from oracle import evalstats_np as ev
    assert np.array_equal(ev.normalize_by_length(raw, [len(t) for t in tracks]), Dn)


def _run_sequence(alg):
    alg.all_pairwise(0, n_cores=1, symmetric=True)
    raw = np.array(alg.Ds["main"])
    alg.normalize_by_length()
    Dn = np.array(alg.Ds["main"])
    MR, MRR, MDR, MAP, tops = alg.getEvalStatistics("main", topsidx=TOPS)
    return raw, Dn, np.array([MR, MRR, MDR, MAP] + list(tops), dtype=np.float64)


def _serial_serra09():
    from acoss_b200.serra09 import Serra09

    class SerialSerra09(Serra09):                            # the reference's serial driver: one pair per call
        def all_pairwise(self, parallel=0, n_cores=12, symmetric=False, precomputed=False):
            for i, j in self._pair_array(symmetric):
                self.similarity(np.array([[i, j]]))
            if symmetric:
                for key in self.Ds:
                    self.Ds[key] += self.Ds[key].T
    return SerialSerra09


def _bound_sequence(lib=None):
    """The INTEGRATION.md section B binding on the mirror base class, one pair per similarity() call."""
    from acoss_b200.algorithm_template import CoverAlgorithm
    from acoss_b200.integration import bind_serra09
    Bound = bind_serra09(_serial_serra09(), lib=lib)
    assert issubclass(Bound, CoverAlgorithm)
    tracks, labels = _tiny()
    feats = [dict(hpcp=t, label=l) for t, l in zip(tracks, labels)]
    alg = Bound(None, None, features=feats, downsample_fac=1, shortname="tinyb")
    raw, Dn, metrics = _run_sequence(alg)
    alg.release()
    return raw, Dn, metrics


def test_binding_on_the_cpu_abi_stub_reproduces_the_reference_class_golden(tmp_path, monkeypatch):
    """The binding on the CPU stand-in of the C ABI == the golden produced under the reference's own classes."""
    monkeypatch.chdir(tmp_path)
    from oracle import build as obuild
    raw, Dn, metrics = _bound_sequence(C.CDLL(obuild.build_stub()))
    g = np.load(GOLDEN)
    assert np.array_equal(g["raw"], raw) and np.array_equal(g["normalized"], Dn)
    assert np.array_equal(g["metrics"], metrics)


@pytest.mark.gpu
def test_gpu_plugin_reproduces_the_reference_class_golden(tmp_path, monkeypatch):
    """acoss_b200.serra09.Serra09 (batched GPU path) == the golden produced under the reference's own classes."""
    monkeypatch.chdir(tmp_path)
    from acoss_b200.serra09 import Serra09
    tracks, labels = _tiny()
    feats = [dict(hpcp=t, label=l) for t, l in zip(tracks, labels)]
    alg = Serra09(None, None, features=feats, downsample_fac=1, shortname="tiny")
    raw, Dn, metrics = _run_sequence(alg)
    alg.close()
    g = np.load(GOLDEN)
    assert np.array_equal(g["raw"], raw) and np.array_equal(g["normalized"], Dn)
    assert np.array_equal(g["metrics"], metrics)


@pytest.mark.gpu
def test_gpu_binding_reproduces_the_reference_class_golden(tmp_path, monkeypatch):
    """The INTEGRATION.md section B binding on the real libacoss_b200.so, one pair per similarity() call through the
    base class's serial all_pairwise (the mirror base here; the reference's base in the CPU test above)."""
    monkeypatch.chdir(tmp_path)
    raw, Dn, metrics = _bound_sequence()
    g = np.load(GOLDEN)
    assert np.array_equal(g["raw"], raw) and np.array_equal(g["normalized"], Dn)
    assert np.array_equal(g["metrics"], metrics)
