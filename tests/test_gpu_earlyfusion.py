"""GPU parity of the full EarlyFusion pair scoring (acoss_ef_set_tracks / acoss_ef_score_pairs /
acoss_ef_dump_pair through the ctypes binding and the EarlyFusion plugin) against

* the golden vectors the reference's own ``EarlyFusion.similarity`` produced
  (tests/golden/make_golden_earlyfusion_full.py), and
* the pinned numpy oracle (oracle/earlyfusion_np.py) on seeded inputs.

Bars: OTI exact; float64 matrices within 1e-11 relative of the oracle's (different summation order of the
same float64 contraction); binary matrices bit-identical; Smith-Waterman scores identical as float32."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KINDS = ("mfccs", "ssms", "chromas", "early")
EF_FULL_CASES = [
    ("f64_small", [2, 2, 1], 70, 301, dict(mfccs=60, ssms=45, chromas=48), "float64", 0.1, 10),
    ("f64_full", [2, 1], 90, 302, None, "float64", 0.1, 10),
    ("f64_k5", [3], 55, 303, dict(mfccs=40, ssms=28, chromas=24), "float64", 0.15, 5),
    ("f32_full", [2, 1], 90, 302, None, "float32", 0.1, 10),
    ("f64_count", [2, 1, 1], 45, 304, dict(mfccs=30, ssms=21, chromas=36), "float64", 6, 4),
    ("f32_small", [3, 1], 60, 305, dict(mfccs=50, ssms=36, chromas=60), "float32", 0.2, 12),
    ("f64_ragged", [2, 2], 80, 306, dict(mfccs=24, ssms=15, chromas=12), "float64", 0.05, 8),
]
EF_JITTER = {"f64_ragged": 0.6}


@pytest.fixture(scope="module")
def eng():
    from acoss_b200 import Engine
    with Engine(0) as e:
        yield e


@pytest.fixture(scope="module")
def gfull(golden_dir):
    return np.load(os.path.join(golden_dir, "earlyfusion_full_golden.npz"))


def _all_pairs(n):
    i, j = np.triu_indices(n, k=1)
    return np.stack([i, j], axis=1).astype(np.int32)


@pytest.mark.parametrize("case", EF_FULL_CASES, ids=[c[0] for c in EF_FULL_CASES])
def test_scores_match_reference_golden(eng, gfull, case):
    """Device scores == what the reference's EarlyFusion.similarity stored in Ds (float32), all pairs."""
    from acoss_b200 import synthetic
    name, cliques, nb, seed, dims, dtype, kappa, K = case
    feats = synthetic.ef_dataset(cliques, nb, seed, dims=dims, dtype=np.dtype(dtype), jitter=EF_JITTER.get(name, 0.15))
    eng.ef_set_tracks(feats)
    pairs = _all_pairs(len(feats))
    got = eng.ef_score_pairs(pairs, kappa, K)
    for k, s in enumerate(KINDS):
        want = gfull["%s_D_%s" % (name, s)][pairs[:, 0], pairs[:, 1]]
        assert np.array_equal(got[k], want), (name, s, got[k], want)
    # first pair: OTI and the four binary matrices, bit for bit
    d = eng.ef_dump_pair(0, 1, kappa, K)
    assert d["oti"] == int(gfull["%s_oti01" % name])
    for k, s in enumerate(KINDS):
        want = np.unpackbits(gfull["%s_bin01_%s" % (name, s)], axis=1, bitorder="little")[:, :d["bins"].shape[2]]
        assert np.array_equal(d["bins"][k], want), (name, s)
    E = gfull["%s_early01" % name]
    got_e = d["csms"][3] if name != "f64_full" else d["csms"][3][::7, ::5]
    assert np.allclose(got_e, E, rtol=(1e-11 if dtype == "float64" else 1e-4), atol=0)
    assert np.array_equal(d["scores"], got[:, 0])


ORACLE_DIMS = dict(mfccs=200, ssms=231, chromas=96)
# chroma blocks padded to 2 064 doubles: wider than the rolled-column map of the chroma contraction (2 048)
WIDE_CHROMA_DIMS = dict(mfccs=200, ssms=231, chromas=2052)


@pytest.mark.parametrize("dtype,dims", [("float32", ORACLE_DIMS), ("float64", ORACLE_DIMS), ("float32", WIDE_CHROMA_DIMS)],
                         ids=["float32", "float64", "float32-wide_chroma"])
def test_matrices_match_oracle(eng, dtype, dims):
    """Every stage of one pair against the oracle: OTI, three CSMs, fused matrix, binarisations, scores;
    ragged shapes (rows != columns, neither a multiple of the 64-wide tile)."""
    from acoss_b200 import synthetic
    from oracle import earlyfusion_np as ef
    feats = synthetic.ef_dataset([2, 1, 1], 150, 411, dims=dims, dtype=np.dtype(dtype), jitter=0.4)
    eng.ef_set_tracks(feats)
    for q, r in [(0, 1), (1, 0), (0, 2), (3, 1)]:
        d = eng.ef_dump_pair(q, r, 0.1, 10)
        scores, mats, bins = ef.similarity_pair(feats[q], feats[r], 0.1, 10, want_matrices=True)
        assert d["oti"] == ef.get_oti(feats[q]["chroma_med"], feats[r]["chroma_med"])
        for k, s in enumerate(KINDS):
            assert d["csms"][k].shape == mats[s].shape
            assert np.allclose(d["csms"][k], mats[s], rtol=1e-11, atol=1e-13), (q, r, s)
            assert np.array_equal(d["bins"][k], bins[s]), (q, r, s)
            assert d["scores"][k] == np.float32(scores[s]), (q, r, s)


def test_euclidean_csm_symmetry_full_dims(eng):
    """Size-independent property at the reference's full block dimensions (1000 / 1225 / 480): the Euclidean
    matrices of (i, j) and (j, i) are exact transposes (sequential-k FMA contraction is symmetric in its
    operands), every entry is finite and >= 0, and a track against itself has an exactly zero diagonal in
    the cosine-free kinds' squared form up to rounding (<= 1e-6)."""
    from acoss_b200 import synthetic
    feats = synthetic.ef_dataset([2, 1], 300, 512, jitter=0.2)
    eng.ef_set_tracks(feats)
    a = eng.ef_dump_pair(0, 2, 0.1, 10)
    b = eng.ef_dump_pair(2, 0, 0.1, 10)
    for k in (0, 1):
        assert np.array_equal(a["csms"][k], b["csms"][k].T)
        assert np.isfinite(a["csms"][k]).all() and (a["csms"][k] >= 0).all()
    s = eng.ef_dump_pair(1, 1, 0.1, 10)
    for k in (0, 1):
        assert np.abs(np.diag(s["csms"][k])).max() <= 1e-5
    assert np.abs(np.diag(s["csms"][2])).max() <= 1e-12          # cosine distance of a block to itself
    assert s["oti"] == 0
    # exactly nn ones per row in every binary matrix (csm_to_binary, cross_recurrence.py:156-160)
    nn = int(np.round(0.1 * a["bins"].shape[2]))
    assert (a["bins"].sum(axis=2) == nn).all()


def test_kappa_and_k_variants(eng):
    from acoss_b200 import synthetic
    from acoss_b200.engine import AcossError
    from oracle import earlyfusion_np as ef
    feats = synthetic.ef_dataset([2, 1], 60, 77, dims=dict(mfccs=33, ssms=21, chromas=36), dtype=np.float64)
    eng.ef_set_tracks(feats)
    pairs = _all_pairs(len(feats))
    for kappa, K in [(0, 10), (7, 3), (0.25, 20), (0.1, 1), (0.1, 17)]:
        got = eng.ef_score_pairs(pairs, kappa, K)
        for n, (i, j) in enumerate(pairs):
            want = ef.similarity_pair(feats[i], feats[j], kappa, K)
            for k, s in enumerate(KINDS):
                assert got[k, n] == np.float32(want[s]), (kappa, K, i, j, s)
    n_min = min(f["mfccs"].shape[0] for f in feats)
    with pytest.raises(AcossError):                      # np.partition(CSM, K, ...) raises in the reference
        eng.ef_score_pairs(pairs, 0.1, n_min)
    with pytest.raises(AcossError):
        eng.ef_score_pairs(pairs, 0.1, 0)
    with pytest.raises(AcossError):
        eng.ef_score_pairs(np.array([[0, 99]]), 0.1, 5)
    assert eng.ef_score_pairs(np.zeros((0, 2), np.int32), 0.1, 5).shape == (4, 0)


def test_short_tracks(eng):
    """Fewer than 4 blocks on either side: smith_waterman_constrained returns 0.0 (alignment_tools.py:34-35)."""
    from oracle import earlyfusion_np as ef
    rng = np.random.default_rng(5)
    feats = []
    for nb in (3, 4, 5, 40):
        c = rng.random((nb, 24))
        feats.append(dict(mfccs=rng.normal(size=(nb, 10)), ssms=rng.normal(size=(nb, 6)), chromas=c,
                          chroma_med=np.median(c.reshape(-1, 12), axis=0), label="x"))
    eng.ef_set_tracks(feats)
    pairs = np.array([(0, 1), (1, 0), (0, 3), (3, 0), (1, 2), (2, 3), (3, 2), (1, 3)], dtype=np.int32)
    got = eng.ef_score_pairs(pairs, 0.3, 2)
    for n, (i, j) in enumerate(pairs):
        want = ef.similarity_pair(feats[i], feats[j], 0.3, 2)
        for k, s in enumerate(KINDS):
            assert got[k, n] == np.float32(want[s]), (i, j, s)
    assert (got[:, 0] == 0).all() and (got[:, 2] == 0).all()


def test_chunked_equals_single(eng):
    """A small workspace forces several slot chunks; the scores do not depend on the chunking."""
    from acoss_b200 import Engine, synthetic
    feats = synthetic.ef_dataset([3] * 5 + [1] * 9, 110, 99, dims=dict(mfccs=48, ssms=32, chromas=24))
    pairs = _all_pairs(len(feats))
    eng.ef_set_tracks(feats)
    one = eng.ef_score_pairs(pairs, 0.1, 10)
    assert eng.ef_last_stats()["chunks"] == 1
    with Engine(0, workspace_bytes=64 << 20) as small:
        small.ef_set_tracks(feats)
        many = small.ef_score_pairs(pairs, 0.1, 10)
        st = small.ef_last_stats()
    assert st["chunks"] > 1 and st["pairs"] == len(pairs)
    assert np.array_equal(one, many)
    # covers score higher than non-covers on every kind (sanity of the synthetic cliques)
    lab = np.array([f["label"] for f in feats])
    same = lab[pairs[:, 0]] == lab[pairs[:, 1]]
    for k in range(4):
        assert one[k][same].min() > one[k][~same].max()


def test_plugin_all_pairwise_and_stats(tmp_path, monkeypatch):
    """EarlyFusion drop-in: all_pairwise -> four symmetric score matrices equal to the oracle's per-pair
    scores -> getEvalStatistics of the reference on each."""
    monkeypatch.chdir(tmp_path)
    from acoss_b200 import synthetic
    from acoss_b200.earlyfusion import EarlyFusion
    from oracle import earlyfusion_np as ef
    feats = synthetic.ef_dataset([3, 2, 2, 1, 1], 48, 2024, dims=dict(mfccs=40, ssms=36, chromas=48))
    e = EarlyFusion(None, None, features=feats, shortname="efgpu", cachedir=str(tmp_path / "cache"))
    assert list(e.Ds) == ["mfccs", "ssms", "chromas", "early"] and e.name == "EarlyFusionTraile"
    e.all_pairwise(parallel=0, n_cores=1, symmetric=True)
    n = len(feats)
    for i in range(n):
        for j in range(i + 1, n):
            want = ef.similarity_pair(feats[i], feats[j], 0.1, 10)
            for s in KINDS:
                assert e.Ds[s][i, j] == np.float32(want[s]) and e.Ds[s][j, i] == np.float32(want[s]), (i, j, s)
    assert len(e.cliques) == 5
    for s in KINDS:
        MR, MRR, MDR, MAP, tops = e.getEvalStatistics(s, topsidx=[1, 5])
        assert MAP == 1.0 and MR == 1.0
    e.cleanup_memmap()
    e.close()


def test_tile_edges_and_long_tracks(eng):
    """Block counts on and around the 64-wide tile / 32-row quadrant / 8-wide MMA edges, and one track longer
    than the 1 024 columns the warp-per-row k-NN kernel keeps in registers (falls back to the CTA kernel)."""
    from oracle import earlyfusion_np as ef
    rng = np.random.default_rng(77)
    sizes = [64, 65, 63, 32, 33, 8, 9, 127, 128, 1100]
    feats = []
    for nb in sizes:
        z = np.cumsum(rng.normal(0, 0.4, size=(nb, 4)), axis=0)
        c = np.abs(np.tanh(z @ rng.normal(size=(4, 24)))) + 0.1 * rng.random((nb, 24))
        feats.append(dict(mfccs=(z @ rng.normal(size=(4, 17)) + 0.2 * rng.normal(size=(nb, 17))).astype(np.float32),
                          ssms=(z @ rng.normal(size=(4, 30)) + 0.2 * rng.normal(size=(nb, 30))).astype(np.float32),
                          chromas=c.astype(np.float32),
                          chroma_med=np.median(c.astype(np.float32).reshape(-1, 12), axis=0), label="x"))
    eng.ef_set_tracks(feats)
    pairs = np.array([(0, 1), (1, 0), (2, 3), (4, 0), (5, 6), (6, 5), (7, 8), (8, 2), (3, 7), (9, 0), (1, 9), (9, 8)],
                     dtype=np.int32)
    got = eng.ef_score_pairs(pairs, 0.1, 5)
    for n, (i, j) in enumerate(pairs):
        want = ef.similarity_pair(feats[i], feats[j], 0.1, 5)
        for k, s in enumerate(KINDS):
            assert got[k, n] == np.float32(want[s]), (sizes[i], sizes[j], s, got[k, n], want[s])
    # one pair across the long track, matrix level
    d = eng.ef_dump_pair(8, 9, 0.1, 5)
    _, mats, bins = ef.similarity_pair(feats[8], feats[9], 0.1, 5, want_matrices=True)
    for k, s in enumerate(KINDS):
        assert np.allclose(d["csms"][k], mats[s], rtol=1e-11, atol=1e-13), s
        assert np.array_equal(d["bins"][k], bins[s]), s


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5, 6])
def test_randomised_shapes(eng, seed):
    """Seeded random block counts, dimensions, kappa and K: all four scores of all pairs equal the oracle's."""
    from acoss_b200 import synthetic
    from oracle import earlyfusion_np as ef
    rng = np.random.default_rng(1000 + seed)
    dims = dict(mfccs=int(rng.integers(5, 130)), ssms=int(rng.integers(5, 130)), chromas=12 * int(rng.integers(1, 9)))
    feats = synthetic.ef_dataset([2, 1, 1], int(rng.integers(30, 180)), 500 + seed, dims=dims, jitter=0.5,
                                 dtype=np.float32 if seed % 2 else np.float64)
    kappa = float(rng.choice([0.05, 0.1, 0.2]))
    K = int(rng.integers(2, 14))
    eng.ef_set_tracks(feats)
    pairs = np.array([(i, j) for i in range(len(feats)) for j in range(len(feats)) if i != j], dtype=np.int32)
    got = eng.ef_score_pairs(pairs, kappa, K)
    for n, (i, j) in enumerate(pairs):
        want = ef.similarity_pair(feats[i], feats[j], kappa, K)
        for k, s in enumerate(KINDS):
            assert got[k, n] == np.float32(want[s]), (seed, i, j, s, got[k, n], want[s])
