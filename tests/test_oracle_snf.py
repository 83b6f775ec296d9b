"""CPU checks of the similarity-network-fusion oracle (oracle/snf_np.py) and of the refusals of acoss_b200.fusion,
which happen before any device is touched."""
import numpy as np
import pytest

from oracle import snf_np as snf


def _mats(n, n_mats, seed):
    return snf.clique_distances(n, n_mats, seed=seed)[0]


def test_slot_order_spmm_matches_scipy():
    """The slot-order sparse products (the form the GPU repeats) against the reference's scipy CSR products."""
    Ws = [snf.getW(D, 6) for D in _mats(90, 3, 1)]
    Ps = [snf.getP(W) for W in Ws]
    Ss = [snf.getS(W, 6) for W in Ws]
    for jacobi in (False, True):
        a = snf.diffuse(Ps, Ss, 4, 1, 0.5, jacobi, spmm=snf.spmm_slots)
        b = snf.diffuse(Ps, Ss, 4, 1, 0.5, jacobi, spmm=snf.spmm_scipy)
        assert np.max(np.abs(a - b) / np.abs(b)) <= 1e-13


def test_w_p_s_per_cell():
    """getW, getP and getS against their per-cell definitions."""
    K, n = 3, 12
    D = _mats(n, 1, 2)[0]
    W = snf.getW(D, K)
    P = snf.getP(W)
    J, V = snf.getS(W, K)
    assert W.dtype == P.dtype == V.dtype == np.float32
    ds = np.zeros((n, n))
    for r in range(n):
        for c in range(n):
            ds[r, c] = 0.0 if r == c else 0.5 * (float(D[r, c]) + float(D[c, r]))
    md = np.array([np.sort(ds[r])[:K + 1].mean() * (K + 1) / K for r in range(n)])
    for r in range(n):
        for c in range(n):
            eps = (md[r] + md[c] + ds[r, c]) / 3
            den = 2 * (0.5 * eps) ** 2
            assert W[r, c] == pytest.approx(np.exp(-ds[r, c] ** 2 / (den if den else 1.0)), rel=1e-5)
    assert np.allclose(P, W / W.astype(np.float64).sum(1)[:, None], rtol=1e-6)
    for r in range(n):
        order = sorted(range(n), key=lambda c: (-W[r, c], c))[:K]
        assert list(J[r]) == sorted(order)
        assert np.allclose(V[r], W[r, sorted(order)] / W[r, sorted(order)].astype(np.float64).sum(), rtol=1e-6)


def test_switch_l1():
    """Iteration 1 reads P either way; from iteration 2 the reference's aliasing (Gauss-Seidel) differs from Jacobi."""
    Ws = [snf.getW(D, 5) for D in _mats(40, 3, 3)]
    Ps = [snf.getP(W) for W in Ws]
    Ss = [snf.getS(W, 5) for W in Ws]
    lit, jac = [], []
    snf.diffuse(Ps, Ss, 2, 1, 0.5, False, keep=lit)
    snf.diffuse(Ps, Ss, 2, 1, 0.5, True, keep=jac)
    assert all(np.array_equal(a, b) for a, b in zip(lit[0], jac[0]))
    assert np.array_equal(lit[1][0], jac[1][0])          # matrix 0 reads only last iteration's values either way
    assert not np.array_equal(lit[1][1], jac[1][1])
    assert not np.array_equal(lit[1][2], jac[1][2])


def test_zero_score_nan_pattern():
    """A zero ChenFusion score becomes an inf distance (normalize_by_length): W is NaN (inf / inf) at that cell and its
    mirror, the two rows of P are NaN, and the NaN spreads through the diffusion identically in both product forms."""
    n, K = 30, 4
    Ds = _mats(n, 2, 4)
    Ds[0][5, 9] = np.inf
    Ws = [snf.getW(D, K) for D in Ds]
    assert set(zip(*np.nonzero(np.isnan(Ws[0])))) == {(5, 9), (9, 5)} and not np.isnan(Ws[1]).any()
    P = snf.getP(Ws[0])
    assert set(np.nonzero(np.isnan(P).any(1))[0]) == {5, 9} and np.isnan(P[[5, 9]]).all()
    J, V = snf.getS(Ws[0], K)
    assert np.isfinite(V).all() and 9 not in J[5] and 5 not in J[9]
    a = snf.doSimilarityFusionWs(Ws, K, 3)
    b = snf.doSimilarityFusionWs(Ws, K, 3, spmm=snf.spmm_scipy)
    assert np.isnan(a).any() and not np.isnan(a).all()
    assert np.array_equal(np.isnan(a), np.isnan(b))


def test_refusals():
    """np.partition raises ValueError for K + 1 >= N; the GPU mirror refuses that, fewer than two matrices (the
    reference returns all NaN), the animation and K above 63 before it opens a device."""
    from acoss_b200 import fusion
    Ds = _mats(10, 2, 5)
    with pytest.raises(ValueError):
        snf.getW(Ds[0], 9)
    with np.errstate(invalid="ignore", divide="ignore"):
        assert np.isnan(snf.doSimilarityFusion(Ds[:1], 3, 2)[1]).all()
    for kw in (dict(Scores=Ds, K=9), dict(Scores=Ds[:1], K=3), dict(Scores=Ds, K=3, do_animation=True),
               dict(Scores=_mats(80, 2, 6), K=64)):
        with pytest.raises(ValueError):
            fusion.doSimilarityFusion(**kw)
