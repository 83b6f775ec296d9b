"""The coarse item of the tensor-core histogram sweeps (k2_tc.inl, DESIGN.md 4.2).

The histogram sweeps and the sparse level bin the coarse item z' = aa + bb - T' of the two high byte limbs,
T' = acc0 * 2^e0 + ((acc1 * 256) >> (16 - e0)), while the emit sweep lists cells by the item z = aa + bb - T of all three
(T adds acc2 = l1.l1 + h.l2 + l2.h below the shift).  Exactness rests on 0 <= z' - z <= dz, with the per-pair bound dz that
fast_prep_kernel derives from the largest window sums of the h and l1 bytes:
    dz = ((255 * (max sum h_Q + max sum h_R + min(max sum l1_Q, max sum l1_R))) >> (16 - e0)) + 1.
The CPU part checks that bound against brute-force limb products; the GPU part (marked gpu) runs pairs whose order statistics
fall into the widened low band of emit's zones and requires the scores, CRP bits and thresholds of the exact path and of the
C oracle."""
import numpy as np
import pytest


def limbs(xq):
    return xq >> 16, (xq >> 8) & 255, xq & 255


def windows(frames_q):
    """Stacked 9-frame windows (108 bytes) of a quantised track (n frames x 12), as the sweeps see them (F4: n - 9 windows)."""
    n = len(frames_q) - 9
    return np.stack([frames_q[i:i + 9].ravel() for i in range(n)])


def items(Xq, Yq, e0):
    """T and T' for every (window of X, window of Y), from brute-force limb products."""
    xh, xl1, xl2 = limbs(Xq)
    yh, yl1, yl2 = limbs(Yq)
    a0 = xh @ yh.T
    a1 = xh @ yl1.T + xl1 @ yh.T
    a2 = xl1 @ yl1.T + xh @ yl2.T + xl2 @ yh.T
    assert (a1 * 256 + a2).max() < 2 ** 32 and a0.max() < 2 ** 31
    s2 = 16 - e0
    T = a0 * (1 << e0) + ((a1 * 256 + a2) >> s2)
    Tc = a0 * (1 << e0) + ((a1 * 256) >> s2)
    assert np.array_equal(Tc, a0 * (1 << e0) + (a1 >> (8 - e0)))           # tc_item_coarse's single shift
    return T, Tc, a2


def prep_dz(Xq, Yq, e0):
    """fast_prep_kernel's bound."""
    xh, xl1, _ = limbs(Xq)
    yh, yl1, _ = limbs(Yq)
    s = 255 * (int(xh.sum(1).max()) + int(yh.sum(1).max()) + min(int(xl1.sum(1).max()), int(yl1.sum(1).max())))
    return (s >> (16 - e0)) + 1


def check(fq, fr, e0):
    Xq, Yq = windows(fq), windows(fr)
    T, Tc, a2 = items(Xq, Yq, e0)
    dz = prep_dz(Xq, Yq, e0)
    d = T - Tc                                                               # = z' - z
    assert d.min() >= 0 and d.max() <= dz
    assert np.all(d <= (a2 >> (16 - e0)) + 1)                                # the per-cell bound
    return d, dz


def hpcp_q(rng, n, q=23):
    f = rng.random((n, 12)) ** 3
    f /= f.max(axis=1, keepdims=True)
    return np.minimum(np.rint(f.astype(np.float32).astype(np.float64) * 2.0 ** q), 2 ** 24 - 1).astype(np.int64)


@pytest.mark.parametrize("e0", [0, 3, 5, 6])
def test_bound_on_hpcp_like_tracks(e0):
    rng = np.random.default_rng(11 + e0)
    d, dz = check(hpcp_q(rng, 160), hpcp_q(rng, 190), e0)
    assert dz <= ((3 * 108 * 255 * 255) >> (16 - e0)) + 1                    # never looser than the flat bound
    assert d.max() > 0


def test_bound_all_ff_limbs_is_tight():
    """Every limb 0xFF: acc2 = 3 * 108 * 255^2 in every cell, the bound equals the flat bound and is reached up to the floor."""
    fq = np.full((30, 12), 2 ** 24 - 1, dtype=np.int64)
    for e0 in (0, 6):
        d, dz = check(fq, fq, e0)
        flat = ((3 * 108 * 255 * 255) >> (16 - e0)) + 1
        assert dz == flat and d.min() >= flat - 1


@pytest.mark.parametrize("pattern", ["h_only", "l1_only", "l2_only", "h_l2", "mixed_zero_rows"])
def test_bound_adversarial_limbs(pattern):
    rng = np.random.default_rng(3)
    n = 40

    def make(seed):
        r = np.random.default_rng(seed)
        h = r.integers(0, 256, size=(n, 12))
        l1 = r.integers(0, 256, size=(n, 12))
        l2 = r.integers(0, 256, size=(n, 12))
        if pattern == "h_only":
            l1[:] = 0; l2[:] = 0
        elif pattern == "l1_only":
            h[:] = 0; l2[:] = 0
        elif pattern == "l2_only":
            h[:] = 0; l1[:] = 0
        elif pattern == "h_l2":
            h[:] = 255; l1[:] = 0; l2[:] = 255
        else:
            zero = r.random(n) < 0.5
            h[zero] = 0; l1[zero] = 255; l2[zero] = 255
        return (h << 16) | (l1 << 8) | l2

    for e0 in (0, 6):
        check(make(rng.integers(1 << 30)), make(rng.integers(1 << 30)), e0)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: pairs whose order statistics fall into the widened band
# ---------------------------------------------------------------------------------------------------------------------
def _hpcp_tracks(lens, seed):
    from acoss_b200 import synthetic
    base, _ = synthetic.config_dataset("C3", max_tracks=13)                # ~2k-frame synthetic tracks
    return [np.ascontiguousarray(base[(i + seed) % len(base)][:n]) for i, n in enumerate(lens)]


def _wide_band_tracks(lens, seed):
    """HPCP-like tracks whose middle limb is 255 in every bin: x = (h 2^16 + 255 2^8 + l2) / 2^24 (exact in float32, quantised
    back to these limbs).  Every window's l1 sum is at its maximum, so dz is about 60 % of the flat bound (HPCP-like tracks:
    about 30 %), z' - z is large in every cell and the wanted order statistics of many lines sit in the low band of emit's
    widened zone."""
    out = []
    for t in _hpcp_tracks(lens, seed):
        h = np.rint(t.astype(np.float64) * 254.0).astype(np.int64)             # largest feature < 1: q_exp = 24
        l2 = np.random.default_rng(seed).integers(0, 256, size=t.shape)
        xq = (h << 16) | (255 << 8) | l2
        out.append(np.ascontiguousarray((xq.astype(np.float64) / 2.0 ** 24).astype(np.float32)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["hpcp", "wide_band"])
def test_band_cells_exact(monkeypatch, kind):
    from acoss_b200 import Engine, default_params, pack_tracks
    from acoss_b200._lib import CRP_EXACT
    from oracle import serra09_c as oc
    lens = [700, 90, 1500, 420, 1100, 130]
    tracks = _hpcp_tracks(lens, 2) if kind == "hpcp" else _wide_band_tracks(lens, 4)
    frames, offs = pack_tracks(tracks)
    pairs = np.array([(i, j) for i in range(len(lens)) for j in range(len(lens)) if i != j], dtype=np.int32)
    dump = [(0, 2), (2, 4), (1, 3), (5, 0)]
    with Engine(0) as eng:
        eng.set_tracks(frames, offs)
        monkeypatch.setenv("ACOSS_K2_SWEEPS", "tc")
        got = eng.score_pairs(pairs)
        st = eng.last_stats()
        counters = eng.debug_counters()
        dumps = {(q, r): eng.dump_pair(q, r) for q, r in dump}
        monkeypatch.delenv("ACOSS_K2_SWEEPS")
        exact = eng.score_pairs(pairs, default_params(crp_path=CRP_EXACT))
    assert counters["band_cells"] > 0                                        # cells whose coarse item scatter recomputed
    assert st["fallback_pairs"] == 0
    assert np.array_equal(got, exact)
    op = oc.params(hoist_norms=True)
    assert np.array_equal(got, oc.pairs(frames, offs, pairs, op, nthreads=8))
    for (q, r), d in dumps.items():
        s, dbg = oc.pair(tracks[q], tracks[r], op, want_debug=True)
        assert d["score"] == s and np.array_equal(d["crp"], dbg["crp"])
        assert np.array_equal(d["thr_q"], dbg["thr_q"]) and np.array_equal(d["thr_r"], dbg["thr_r"])
