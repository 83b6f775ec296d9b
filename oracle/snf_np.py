"""numpy restatement of similarity-network fusion (TEST INFRASTRUCTURE).

Restates acoss/algorithms/utils/similarity_fusion.py as published: getW, getP, getS, doSimilarityFusionWs and
doSimilarityFusion, operation for operation, with the reference's float32 / float64 dtypes.  Two points are pinned
here rather than in the reference:

* Selection ties.  getW's ``np.partition`` and getS's ``np.argpartition`` pick among equal values in introselect's
  order.  Here equal values are taken lowest column first (a stable sort, NaN after +inf), and the K values of a row
  of S are summed in ascending column order: the order of the CSR row ``coo_matrix.tocsr()`` builds.
* Switch L1.  ``Pts = nextPts`` binds both names to one list, so from the second iteration on matrix i reads the
  Pts[k] already updated in the same iteration for k < i (Gauss-Seidel).  ``jacobi=True`` copies instead: every
  iteration reads the previous one, as in the SNF paper.

The sparse products are written twice: ``spmm_slots`` (``R += V[:, t] * Y[J[:, t]]`` for each slot t, a multiply and
an add per term, which is scipy's csr_matvecs ``y += a * x``) and ``spmm_scipy`` (the reference's csr_matrix.dot).
"""
from __future__ import annotations

import numpy as np
from scipy import sparse

__all__ = ["getW", "getP", "getS", "spmm_slots", "spmm_scipy", "diffuse", "doSimilarityFusionWs",
           "doSimilarityFusion"]


def getW(D, K, Mu=0.5):
    """Affinity: DSym = 0.5 (D + D.T) with a zero diagonal, Eps from the mean of the K+1 smallest per row."""
    DSym = 0.5 * (D + D.T)
    np.fill_diagonal(DSym, 0)
    Neighbs = np.partition(DSym, K + 1, 1)[:, 0:K + 1]
    MeanDist = np.mean(Neighbs, 1) * float(K + 1) / float(K)
    Eps = MeanDist[:, None] + MeanDist[None, :] + DSym
    Eps = Eps / 3
    Denom = (2 * (Mu * Eps) ** 2)
    Denom[Denom == 0] = 1
    with np.errstate(invalid="ignore", over="ignore"):
        W = np.exp(-DSym ** 2 / Denom)
    return W


def getP(W):
    """Transition matrix W / row sum (a zero row sum replaced by 1); no diagonal regularisation."""
    RowSum = np.sum(W, 1)
    RowSum[RowSum == 0] = 1
    return W / RowSum[:, None]


def getS(W, K):
    """The K largest W of each row as (J int32 (N, K) ascending per row, V float32 (N, K)): V = W / sum of the row's
    K kept values (a zero sum replaced by 1).  Ties: lowest column; NaN after every number."""
    J = np.argsort(-W, axis=1, kind="stable")[:, :K]
    J = np.sort(J, axis=1).astype(np.int32)
    V = np.take_along_axis(W, J, axis=1)
    VSum = np.sum(V, 1)
    VSum[VSum == 0] = 1
    return J, V / VSum[:, None]


def to_csr(J, V, N):
    """The reference's CSR form of S: coo_matrix((V, (I, J))).tocsr()."""
    I = np.tile(np.arange(J.shape[0])[:, None], (1, J.shape[1]))
    return sparse.coo_matrix((V.flatten(), (I.flatten(), J.flatten())), shape=(J.shape[0], N)).tocsr()


def spmm_slots(S, Y):
    """S . Y for S = (J, V), as scipy computes it: R = 0, then R += V[:, t] * Y[J[:, t]] slot by slot."""
    J, V = S
    R = np.zeros((J.shape[0], Y.shape[1]))
    for t in range(J.shape[1]):
        R += V[:, t, None].astype(np.float64) * Y[J[:, t], :]
    return R


def spmm_scipy(S, Y):
    """S . Y through the reference's scipy CSR matrix."""
    J, V = S
    return to_csr(J, V, Y.shape[0]).dot(Y)


def diffuse(Ps, Ss, niters=20, reg_diag=1, reg_neighbs=0.5, jacobi=False, spmm=spmm_slots, keep=None):
    """doSimilarityFusionWs after getP / getS: the cross-diffusion of the P matrices through the S matrices, then
    the average.  keep (a list) receives a copy of Pts after every iteration."""
    Pts = [np.array(P) for P in Ps]
    nextPts = [np.zeros(P.shape) for P in Pts]
    N = len(Pts)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        for it in range(niters):
            for i in range(N):
                nextPts[i] *= 0
                for k in range(N):
                    if i == k:
                        continue
                    nextPts[i] += Pts[k]
                nextPts[i] /= float(N - 1)
                A = spmm(Ss[i], nextPts[i].T)
                nextPts[i] = spmm(Ss[i], A.T)
                if reg_diag > 0:
                    nextPts[i] += reg_diag * np.eye(nextPts[i].shape[0])
                if reg_neighbs > 0:
                    arr = np.arange(nextPts[i].shape[0])
                    [I, J] = np.meshgrid(arr, arr)
                    nextPts[i][np.abs(I - J) == 1] += reg_neighbs
            Pts = [np.array(P) for P in nextPts] if jacobi else nextPts
            if keep is not None:
                keep.append([np.array(P) for P in Pts])
        FusedScores = np.zeros(Pts[0].shape)
        for Pt in Pts:
            FusedScores += Pt
        return FusedScores / N


def doSimilarityFusionWs(Ws, K=5, niters=20, reg_diag=1, reg_neighbs=0.5, jacobi=False, spmm=spmm_slots):
    Ps = [getP(W) for W in Ws]
    Ss = [getS(W, K) for W in Ws]
    return diffuse(Ps, Ss, niters, reg_diag, reg_neighbs, jacobi, spmm)


def doSimilarityFusion(Scores, K=5, niters=20, reg_diag=1, reg_neighbs=0.5, jacobi=False, spmm=spmm_slots):
    """(Ws, fused) as the reference returns them."""
    Ws = [getW(D, K) for D in Scores]
    return Ws, doSimilarityFusionWs(Ws, K, niters, reg_diag, reg_neighbs, jacobi, spmm)


def clique_distances(n, n_mats, clique=4, seed=0):
    """Seeded clique-structured float32 distance matrices (the shape of finished cover-song scores): labels
    i // clique, distance 1 + U(0, 1) across cliques and 0.25 + U(0, 0.5) within, an inf diagonal (a zero score
    normalised by length).  -> (list of (n, n) float32, labels int)."""
    rng = np.random.default_rng(seed)
    lab = np.arange(n) // clique
    same = lab[:, None] == lab[None, :]
    Ds = []
    for _ in range(n_mats):
        D = np.where(same, 0.25 + 0.5 * rng.random((n, n)), 1.0 + rng.random((n, n))).astype(np.float32)
        np.fill_diagonal(D, np.inf)
        Ds.append(D)
    return Ds, lab
