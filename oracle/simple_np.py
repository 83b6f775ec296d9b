"""numpy restatement of the SiMPle pair score of ``Simple`` (TEST INFRASTRUCTURE).

Reference followed: acoss/algorithms/simple_silva.py:17-126 (pooling :38-41, OTI :45-54, the
FFT-based join ``simple_sim`` :68-118).  The reference's source is not available where this package is built and
tested, so this module restates the published SiMPle (Silva, Yeh, Batista, Keogh, ISMIR 2016) with every uncertain
point as a switch (DESIGN.md §2, S1-S5).  Parity: unpinned against the reference, pinned against this restatement.

* ``pool``            mean pooling, np.mean arithmetic (sequential float32 sum, one float32 division); S5.
* ``oti``             float64 global chroma, first argmax of the circular correlation; S4 picks the rolled song.
* ``join_d2``         the direct float64 join in the order the CUDA kernel evaluates it (sequential over t, then b).
* ``score_pair``      profile (S2), index, median, polarity (S3): what Ds["main"][i, j] holds.
* ``simple_fast_profile``  SiMPle-Fast as the reference computes it (fftconvolve for the first row and column,
  then sliding dot-product updates).  Not bit-exact; checked against ``join_d2`` to 1e-9 and used as the timed CPU
  baseline (tools/time_simple.py).
"""
from __future__ import annotations

import numpy as np

__all__ = ["DEFAULT_M", "pool", "pool_count", "global_chroma", "oti", "roll_pair", "join_d2", "profile",
           "median", "score_pair", "simple_fast_profile", "score_pair_fast"]

DEFAULT_M = 10          # S1: subsequence length in pooled frames (unconfirmed against the reference)
WIN, SKIP = 200, 100


def pool_count(n: int, win: int = WIN, skip: int = SKIP, keep_partial: bool = False) -> int:
    if not keep_partial:
        if n < win:
            raise ValueError("track has %d raw frames, fewer than win = %d" % (n, win))
        return (n - win) // skip + 1
    if n <= win:
        return 1 if n > 0 else 0
    return (n - win + skip - 1) // skip + 1


def pool(X, win: int = WIN, skip: int = SKIP, keep_partial: bool = False) -> np.ndarray:
    """Pooled frame k = mean of raw frames [k*skip, min(k*skip + win, n)), float32 (n, 12) -> float32."""
    X = np.ascontiguousarray(X, dtype=np.float32)
    n = X.shape[0]
    K = pool_count(n, win, skip, keep_partial)
    out = np.empty((K, X.shape[1]), dtype=np.float32)
    for k in range(K):
        blk = X[k * skip:min(k * skip + win, n)]
        acc = np.zeros(X.shape[1], dtype=np.float32)
        for row in blk:                                  # sequential float32 sum in frame order
            acc = acc + row
        out[k] = acc / np.float32(len(blk))
    return out


def global_chroma(X) -> np.ndarray:
    """float64 sequential frame sum per bin."""
    g = np.zeros(X.shape[1], dtype=np.float64)
    for row in np.asarray(X, dtype=np.float64):
        g = g + row
    return g


def oti(A, B, roll_first: bool = False) -> int:
    """First argmax over s of sum_b g_A[b] g_B[(b - s) % 12] (S4 = 0) or sum_b g_A[(b - s) % 12] g_B[b] (S4 = 1),
    products and sums rounded one by one in float64."""
    ga, gb = global_chroma(A), global_chroma(B)
    best, best_s = -np.inf, 0
    for s in range(12):
        ra, rb = (np.roll(ga, s), gb) if roll_first else (ga, np.roll(gb, s))
        acc = 0.0
        for b in range(12):
            acc = acc + float(ra[b]) * float(rb[b])
        if acc > best:
            best, best_s = acc, s
    return best_s


def roll_pair(A, B, use_oti: bool = True, roll_first: bool = False):
    """-> (oti, A', B') with the rolled song rolled along the bin axis (np.roll)."""
    s = oti(A, B, roll_first) if use_oti else 0
    A = np.asarray(A, dtype=np.float32)
    B = np.asarray(B, dtype=np.float32)
    return (s, np.roll(A, s, axis=1), B) if roll_first else (s, A, np.roll(B, s, axis=1))


def join_d2(A, B, m: int) -> np.ndarray:
    """(n_a - m + 1, n_b - m + 1) float64: sum_{t<m} sum_b (A[i+t][b] - B[j+t][b])^2, sequential over t then b,
    every subtraction, product and sum rounded (numpy never contracts)."""
    A = np.asarray(A, dtype=np.float64)
    B = np.asarray(B, dtype=np.float64)
    La, Lb = A.shape[0] - m + 1, B.shape[0] - m + 1
    if La < 1 or Lb < 1:
        raise ValueError("a track is shorter than m = %d" % m)
    acc = np.zeros((La, Lb), dtype=np.float64)
    for t in range(m):
        for b in range(A.shape[1]):
            d = A[t:t + La, b][:, None] - B[t:t + Lb, b][None, :]
            acc += d * d
    return acc


def profile(d2, squared: bool = False):
    """-> (P float64, I int32): row minimum of d = sqrt(d2) (S2 = 1: d2) and the lowest column attaining it."""
    d = d2 if squared else np.sqrt(d2)
    return d.min(axis=1), d.argmin(axis=1).astype(np.int32)


def median(P) -> float:
    """np.median: the mean (a + b) / 2 of the two middle values when the length is even."""
    return float(np.median(np.asarray(P, dtype=np.float64)))


def score_pair(A, B, m: int = DEFAULT_M, use_oti: bool = True, squared: bool = False, positive: bool = False,
               roll_first: bool = False) -> dict:
    """Everything Simple stores or dumps for the pair (query A, reference B): oti, profile, index, score (float32)."""
    s, A2, B2 = roll_pair(A, B, use_oti, roll_first)
    P, I = profile(join_d2(A2, B2, m), squared)
    med = median(P)
    return dict(oti=s, profile=P, index=I, score=np.float32(med if positive else -med))


def simple_fast_profile(A, B, m: int, squared: bool = False):
    """SiMPle-Fast restatement (the reference's arithmetic shape): d2(i, j) = |A_i|^2 + |B_j|^2 - 2 QT(i, j) with the
    sliding dot products QT of the 12-dimensional windows; the first row and column come from scipy's fftconvolve,
    the rest from QT(i, j) = QT(i-1, j-1) - <A[i-1], B[j-1]> + <A[i+m-1], B[j+m-1]>.  Returns (P, I)."""
    from scipy.signal import fftconvolve
    A = np.asarray(A, dtype=np.float64)
    B = np.asarray(B, dtype=np.float64)
    La, Lb = A.shape[0] - m + 1, B.shape[0] - m + 1

    def sliding(q, T):                     # <q (m x 12), T[j:j+m]> for every j, by FFT
        return sum(fftconvolve(T[:, b], q[::-1, b], mode="valid") for b in range(T.shape[1]))

    def win_norms(X, L):
        c = np.concatenate([[0.0], np.cumsum((X * X).sum(axis=1))])
        return c[m:m + L] - c[:L]

    na, nb = win_norms(A, La), win_norms(B, Lb)
    row0 = sliding(A[:m], B)               # QT(0, j)
    col0 = sliding(B[:m], A)               # QT(i, 0)
    fa = A[:-1]
    P = np.empty(La)
    I = np.empty(La, dtype=np.int32)
    qt = row0.copy()
    for i in range(La):
        if i > 0:
            qt[1:] = qt[:-1] - (fa[i - 1] * B[:Lb - 1]).sum(axis=1) + (A[i + m - 1] * B[m:m + Lb - 1]).sum(axis=1)
            qt[0] = col0[i]
        d2 = np.maximum(na[i] + nb - 2.0 * qt, 0.0)
        d = d2 if squared else np.sqrt(d2)
        j = int(np.argmin(d))
        P[i], I[i] = d[j], j
    return P, I


def score_pair_fast(A, B, m: int = DEFAULT_M, use_oti: bool = True, squared: bool = False, positive: bool = False,
                    roll_first: bool = False) -> np.float32:
    s, A2, B2 = roll_pair(A, B, use_oti, roll_first)
    P, _ = simple_fast_profile(A2, B2, m, squared)
    med = median(P)
    return np.float32(med if positive else -med)
