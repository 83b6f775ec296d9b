"""GPU: the second dense level of the tensor histogram sweeps, taken through the re-queue.

An item (pair, 128-line strip) that still holds DENSE2_MIN_LIVE or more live lines after its first dense level is re-queued
and swept again by the same persistent CTAs once every item has had its first level (k2_tc.inl).  Short tracks start
their lines from the whole item range, so a call of many short and a few long tracks sends hundreds of items through the
re-queue.  The scores must match the exact path and the C oracle, and the dense-level counters (items, live lines,
misses, lines left, per level and orientation) must match those of the build that ran both levels back to back in one
CTA: a line gets at most two dense levels, and the same lines reach the sparse level with the same brackets."""
import json
import os

import numpy as np
import pytest

LENS = [40, 75, 120, 150, 200, 260, 330, 420, 520, 700, 60, 90, 1500, 180, 1900, 110, 300, 950, 136, 240]
GOLDEN = "tc_requeue_counts.json"
COUNTERS = ("col_dense", "row_dense", "col_dense2", "row_dense2", "sparse")   # sparse: (warps, lines left)


def dataset():
    """Slices of the ~2k-frame synthetic C3 tracks at the lengths of LENS, and every ordered pair of them."""
    from acoss_b200 import synthetic
    base, _ = synthetic.config_dataset("C3", max_tracks=13)
    tracks = []
    for i, n in enumerate(LENS):
        t = base[i % len(base)]
        a = min(7 * i, len(t) - n)
        tracks.append(np.ascontiguousarray(t[a:a + n]))
        assert len(tracks[-1]) == n
    pairs = np.array([(i, j) for i in range(len(LENS)) for j in range(len(LENS)) if i != j], dtype=np.int32)
    return tracks, pairs


def tc_run(eng, tracks, pairs):
    """Scores and debug counters of one call with the tensor sweeps forced."""
    from acoss_b200 import pack_tracks
    frames, offs = pack_tracks(tracks)
    eng.set_tracks(frames, offs)
    old = os.environ.get("ACOSS_K2_SWEEPS")
    os.environ["ACOSS_K2_SWEEPS"] = "tc"
    try:
        got = eng.score_pairs(pairs)
        st = eng.last_stats()
        counters = eng.debug_counters()
    finally:
        if old is None:
            del os.environ["ACOSS_K2_SWEEPS"]
        else:
            os.environ["ACOSS_K2_SWEEPS"] = old
    # (the sparse level's sweep count depends on which lines share a warp, i.e. on the order of its call-wide list)
    out = {k: list(counters[k]) for k in COUNTERS}
    out["sparse"] = [out["sparse"][0], out["sparse"][2]]
    return frames, offs, got, st, out


@pytest.mark.gpu
def test_requeued_second_levels(golden_dir):
    from acoss_b200 import Engine, default_params
    from acoss_b200._lib import CRP_EXACT
    from oracle import serra09_c as oc
    tracks, pairs = dataset()
    with Engine(0) as eng:
        frames, offs, got, st, counters = tc_run(eng, tracks, pairs)
        exact = eng.score_pairs(pairs, default_params(crp_path=CRP_EXACT))
    assert st["fallback_pairs"] == 0
    assert np.array_equal(got, exact)
    # hundreds of items take the second level: more than one per CTA of a 148-SM launch, in both orientations
    assert counters["col_dense2"][0] > 148 and counters["row_dense2"][0] > 148
    assert counters["sparse"][0] > 0
    sel = np.random.default_rng(11).permutation(len(pairs))[:48]
    want_scores = oc.pairs(frames, offs, pairs[sel], oc.params(hoist_norms=True), nthreads=os.cpu_count() or 1)
    assert np.array_equal(got[sel], want_scores)
    with open(os.path.join(golden_dir, GOLDEN)) as f:
        want = json.load(f)["counters"]
    assert counters == want
