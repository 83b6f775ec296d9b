"""Similarity-network fusion of finished N x N score matrices on the GPU (acoss/algorithms/utils/similarity_fusion.py).

``doSimilarityFusion`` has the reference function's signature and return value, ``(Ws, fused)``: the float32 affinity
matrices of getW and the float64 fused matrix.  It is the late-fusion step of ``ChenFusion.do_late_fusion`` and
``EarlyFusion.do_late_fusion``.  Every stage runs in k7_snf.cu (``acoss_snf``); DESIGN.md §2 and §4.7 give the
parity status (switch L1) and the kernels.

Differences from the reference: fewer than two matrices are refused (the reference returns all NaN, dividing by
``n_mats - 1 == 0``), as are ``do_animation`` and K above 63.  Equal values in the neighbour selections are taken
lowest column first; the reference takes them in introselect's order.
"""
from __future__ import annotations

import numpy as np

from .engine import Engine, check_snf_args

__all__ = ["doSimilarityFusion", "fuse"]


def fuse(Scores, K=5, niters=20, reg_diag=1, reg_neighbs=0.5, *, jacobi=False, engine=None, want_W=False):
    """The GPU fusion of the score matrices Scores: dict(fused float64 (N, N)) plus W float32 (n_mats, N, N) when
    want_W.  jacobi is switch L1 (default: the reference's Gauss-Seidel aliasing from the second iteration on).
    engine: an Engine to run on (default: a new one on device 0, closed afterwards)."""
    Scores = list(Scores)
    n = int(np.shape(Scores[0])[0]) if Scores else 0
    check_snf_args(len(Scores), n, int(K), int(niters))
    eng = engine if engine is not None else Engine(0)
    try:
        return eng.snf(Scores, K=K, niters=niters, reg_diag=reg_diag, reg_neighbs=reg_neighbs, jacobi=jacobi,
                       want_W=want_W)
    finally:
        if engine is None:
            eng.close()


def doSimilarityFusion(Scores, K=5, niters=20, reg_diag=1, reg_neighbs=0.5, do_animation=False, PlotNames=[],
                       PlotExtents=None, *, engine=None):
    """similarity_fusion.py doSimilarityFusion: (Ws, fused), Ws a list of float32 (N, N) affinity matrices, fused the
    float64 (N, N) fusion.  PlotNames / PlotExtents only serve the animation, which is refused."""
    if do_animation:
        raise ValueError("do_animation is not supported: the fusion runs on the GPU without plotting")
    out = fuse(Scores, K, niters, reg_diag, reg_neighbs, engine=engine, want_W=True)
    return list(out["W"]), out["fused"]
