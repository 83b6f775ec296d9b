"""GPU similarity-network fusion (k7_snf.cu, acoss_snf) against the numpy oracle (oracle/snf_np.py): the affinity W,
P and S recomputed from the GPU's own W, the diffusion from the GPU's P and S bit for bit, the end-to-end fused
matrix and its evaluation statistics, the NaN pattern of a zero score, the two plugins' late fusion, the refusals."""
import numpy as np
import pytest

from oracle import snf_np as snf
from oracle.evalstats_np import eval_statistics

pytestmark = pytest.mark.gpu

# (N, n_mats, jacobi, niters, reg_diag, reg_neighbs, K): N not a multiple of the 32 / 128 tiles; every n_mats with
# each L1 value, each niters, both regularisation settings; K = 20 as the plugins, 5 and 40 for both selection widths
CASES = [
    (50, 2, 0, 0, 1.0, 0.5, 20),
    (50, 3, 1, 20, 0.0, 0.0, 5),
    (50, 4, 0, 1, 1.0, 0.5, 20),
    (257, 2, 1, 1, 1.0, 0.0, 20),
    (257, 3, 0, 20, 1.0, 0.5, 40),
    (257, 4, 1, 20, 0.0, 0.5, 20),
    (1000, 2, 0, 20, 1.0, 0.5, 20),
    (1000, 3, 1, 1, 0.0, 0.0, 20),
    (1000, 4, 0, 1, 1.0, 0.5, 5),
]


@pytest.fixture(scope="module")
def engine():
    from acoss_b200 import Engine
    with Engine(0) as eng:
        yield eng


def _ulps(a, b):
    """float32 distance in units in the last place (NaN only against NaN)."""
    assert np.array_equal(np.isnan(a), np.isnan(b))
    ok = ~np.isnan(a)
    return np.abs(a[ok].view(np.int32).astype(np.int64) - b[ok].view(np.int32).astype(np.int64))


@pytest.mark.parametrize("case", CASES, ids=lambda c: "N%d-m%d-jac%d-it%d-reg%g_%g-K%d" % c)
def test_snf_against_oracle(engine, case):
    n, n_mats, jacobi, niters, reg_diag, reg_neighbs, K = case
    Ds, lab = snf.clique_distances(n, n_mats, seed=n + n_mats)
    got = engine.snf(Ds, K, niters, reg_diag, reg_neighbs, jacobi=bool(jacobi), want_W=True, want_PS=True)
    # 1. W: expf and the summation order of the K+1 mean are the only differences
    Wo = [snf.getW(D, K) for D in Ds]
    for m in range(n_mats):
        np.testing.assert_allclose(got["W"][m], Wo[m], rtol=1e-5, atol=0)
    # 2. P and S recomputed from the GPU's W: same neighbours, values within 1 ulp
    Ss = []
    for m in range(n_mats):
        W = got["W"][m]
        assert _ulps(got["P"][m], snf.getP(W)).max() <= 1
        J, V = snf.getS(W, K)
        assert np.array_equal(got["S_idx"][m], J)
        assert _ulps(got["S_val"][m], V).max() <= 1
        Ss.append((got["S_idx"][m], got["S_val"][m]))
    # 3. the diffusion from the GPU's P and S is bit-identical
    want = snf.diffuse(list(got["P"]), Ss, niters, reg_diag, reg_neighbs, bool(jacobi))
    assert np.array_equal(got["fused"], want, equal_nan=True)
    # 4. end to end: the oracle's neighbour lists are the GPU's, fused within 1e-4, identical evaluation statistics
    for m in range(n_mats):
        assert np.array_equal(snf.getS(Wo[m], K)[0], got["S_idx"][m])
    _, fo = snf.doSimilarityFusion(Ds, K, niters, reg_diag, reg_neighbs, bool(jacobi))
    np.testing.assert_allclose(got["fused"], fo, rtol=1e-4, atol=0)
    cliques = {}
    for i, c in enumerate(lab):
        cliques.setdefault(int(c), set()).add(i)
    a, b = eval_statistics(got["fused"], cliques), eval_statistics(fo, cliques)
    for x, y in zip(a, b):
        assert np.array_equal(np.asarray(x), np.asarray(y))


def test_snf_zero_score_nan_pattern(engine):
    """ChenFusion input with zero scores (inf distances after normalize_by_length): NaN where the oracle has NaN."""
    n, K = 257, 20
    Ds, _ = snf.clique_distances(n, 2, seed=11)
    Ds[0][5, 90] = np.inf
    Ds[1][200, 3] = np.inf
    got = engine.snf(Ds, K, 20, 1, 0.5, want_W=True)
    Ws, fo = snf.doSimilarityFusion(Ds, K, 20, 1, 0.5)
    for m in range(2):
        assert np.array_equal(np.isnan(got["W"][m]), np.isnan(Ws[m]))
    assert np.isnan(fo).any() and np.array_equal(np.isnan(got["fused"]), np.isnan(fo))
    ok = ~np.isnan(fo)
    np.testing.assert_allclose(got["fused"][ok], fo[ok], rtol=1e-4, atol=0)


def test_plugins_late_fusion(engine, tmp_path, monkeypatch):
    """ChenFusion / EarlyFusion do_late_fusion(impl="gpu"): the reference's keys, signs and dtypes, values of
    fusion.doSimilarityFusion and of the oracle."""
    from acoss_b200 import fusion
    from acoss_b200.chenfusion import ChenFusion
    from acoss_b200.earlyfusion import EarlyFusion
    monkeypatch.chdir(tmp_path)
    (tmp_path / "cache").mkdir()
    n = 120
    Ds, _ = snf.clique_distances(n, 4, seed=7)
    c = ChenFusion(None, None, downsample_fac=1,
                   features=[dict(hpcp=np.zeros((20, 12), np.float32), label="x") for _ in range(n)])
    c._engine = engine
    c.Ds["qmax"][:] = Ds[0]
    c.Ds["dmax"][:] = Ds[1]
    c.do_late_fusion(impl="gpu")
    assert list(c.Ds) == ["qmax", "dmax", "Late"] and c.Ds["Late"].dtype == np.float64
    assert np.array_equal(np.asarray(c.Ds["qmax"]), -Ds[0]) and np.array_equal(np.asarray(c.Ds["dmax"]), -Ds[1])
    _, want = fusion.doSimilarityFusion(Ds[:2], K=20, niters=20, reg_diag=1, engine=engine)
    assert np.array_equal(c.Ds["Late"], want)
    np.testing.assert_allclose(c.Ds["Late"], snf.doSimilarityFusion(Ds[:2], 20, 20, 1)[1], rtol=1e-4, atol=0)

    sims = [np.float32(1) / (np.float32(1) + D) for D in Ds]          # EarlyFusion scores are similarities
    e = EarlyFusion(None, None, features=[dict(label="x") for _ in range(n)], shortname="snf", engine=engine)
    for k, s in zip(("mfccs", "ssms", "chromas", "early"), sims):
        e.Ds[k][:] = s
    e.do_late_fusion(impl="gpu")
    assert list(e.Ds)[-2:] == ["late", "early+late"]
    for key, kinds in (("late", ["chromas", "ssms", "mfccs"]), ("early+late", ["chromas", "ssms", "mfccs", "early"])):
        assert e.Ds[key].dtype == np.float64
        inputs = [1.0 / (1.0 + e.Ds[s]) for s in kinds]
        assert np.array_equal(e.Ds[key], fusion.doSimilarityFusion(inputs, K=20, niters=20, reg_diag=1, engine=engine)[1])
        np.testing.assert_allclose(e.Ds[key], snf.doSimilarityFusion(inputs, 20, 20, 1)[1], rtol=1e-4, atol=0)
    with pytest.raises(ValueError):
        c.do_late_fusion(impl="cpu")


def test_snf_refusals(engine):
    """ValueError for K + 1 >= N and for fewer than two matrices; the C ABI itself refuses them (ACOSS_E_INVALID)."""
    import ctypes as C
    from acoss_b200 import _lib
    Ds, _ = snf.clique_distances(30, 2, seed=1)
    with pytest.raises(ValueError):
        engine.snf(Ds, K=29)
    with pytest.raises(ValueError):
        engine.snf(Ds[:1], K=5)
    fused = np.zeros((30, 30))
    ptrs = (C.c_void_p * 2)(*[D.ctypes.data for D in Ds])
    for n_mats, K in ((2, 29), (1, 5), (2, 64)):
        rc = engine._lib.acoss_snf(engine._ctx, ptrs, n_mats, 30, K, 20, 1.0, 0.5, 0, fused.ctypes.data,
                                   None, None, None, None)
        assert rc == _lib.E_INVALID
