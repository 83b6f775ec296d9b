"""GPU: the persistent tensor-core sweeps hand out their work items correctly.

The three tensor sweeps (k2_tc.inl) run one CTA per SM; each CTA walks the work items (pair, 128-line strip) of the call,
skips those with nothing to do (quirk sides, strips past a short track's end, strips whose lines are all done) and keeps its
mbarrier phases running from one item to the next.  These cases put few items, many items, skipped items, quirk sides and
lines that need the second dense level or the sparse level through the sweeps, with the tensor sweeps forced, and require
the CRP bits, thresholds and scores of the exact path and of the C oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from acoss_b200 import Engine
    e = Engine(0)
    yield e
    e.close()


def _tracks(lens, seed=0):
    from acoss_b200 import synthetic
    base, _ = synthetic.config_dataset("C3", max_tracks=13)                # ~2k-frame synthetic tracks
    out = []
    for i, n in enumerate(lens):
        t = base[(i + seed) % len(base)]
        a = min(5 * i, len(t) - n)
        out.append(np.ascontiguousarray(t[a:a + n]))
        assert len(out[-1]) == n
    return out


def _tc_scores(monkeypatch, eng, tracks, pairs, dump=()):
    from acoss_b200 import default_params, pack_tracks
    from acoss_b200._lib import CRP_EXACT
    frames, offs = pack_tracks(tracks)
    eng.set_tracks(frames, offs)
    monkeypatch.setenv("ACOSS_K2_SWEEPS", "tc")
    got = eng.score_pairs(pairs)
    st = eng.last_stats()
    counters = eng.debug_counters()
    dumps = {(int(q), int(r)): eng.dump_pair(int(q), int(r)) for q, r in dump}
    monkeypatch.setenv("ACOSS_K2_SWEEPS", "ffma")
    ffma = eng.score_pairs(pairs)
    st_ffma = eng.last_stats()
    monkeypatch.delenv("ACOSS_K2_SWEEPS")
    # the tensor sweeps ran: one histogram launch per orientation and chunk instead of the FFMA2 sweeps' two (pairs that
    # take the exact path add launches of their own)
    if st["fallback_pairs"] == 0 and st_ffma["fallback_pairs"] == 0:
        assert st["chunks"] == st_ffma["chunks"] and st["launches"] == st_ffma["launches"] - 2 * st["chunks"]
    exact = eng.score_pairs(pairs, default_params(crp_path=CRP_EXACT))
    assert np.array_equal(got, exact) and np.array_equal(ffma, exact)
    return frames, offs, got, st["fallback_pairs"], counters, dumps


def _against_oracle(tracks, frames, offs, pairs, got, dumps):
    from oracle import serra09_c as oc
    op = oc.params(hoist_norms=True)
    want = oc.pairs(frames, offs, pairs, op, nthreads=8)
    assert np.array_equal(got, want)
    for (q, r), d in dumps.items():
        s, dbg = oc.pair(tracks[q], tracks[r], op, want_debug=True)
        assert d["score"] == s and np.array_equal(d["crp"], dbg["crp"])
        assert np.array_equal(d["thr_q"], dbg["thr_q"]) and np.array_equal(d["thr_r"], dbg["thr_r"])


@pytest.mark.parametrize("npairs", [1, 3])
def test_fewer_items_than_sms(monkeypatch, eng, npairs):
    """1 and 3 pairs of ~700 frames: 5 strips per orientation and pair, so most CTAs of a launch get one item or none."""
    tracks = _tracks([700, 650, 720, 690])
    pairs = np.array([(0, 1), (2, 3), (1, 2)], dtype=np.int32)[:npairs]
    frames, offs, got, fallback, counters, dumps = _tc_scores(monkeypatch, eng, tracks, pairs, pairs)
    assert fallback == 0 and counters["col_dense"][0] > 0 and counters["row_dense"][0] > 0
    _against_oracle(tracks, frames, offs, pairs, got, dumps)


def test_many_items_per_cta(monkeypatch, eng):
    """96 pairs of ~2k frames: about 1 500 items per orientation, ten per CTA on a 148-SM B200; against the exact path."""
    from acoss_b200 import synthetic
    tracks, _ = synthetic.config_dataset("C3", max_tracks=16)
    pairs = synthetic.all_pairs_upper(len(tracks))
    pairs = pairs[np.random.default_rng(5).permutation(len(pairs))[:96]].astype(np.int32)
    _, _, got, fallback, counters, _ = _tc_scores(monkeypatch, eng, tracks, pairs)
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert fallback == 0
    assert counters["col_dense"][0] > sms and counters["row_dense"][0] > sms   # swept items: more than one per CTA


def test_short_and_long_tracks_mixed(monkeypatch, eng):
    """Tracks below 128 windows (their strips past the end are skipped, and their lines start from the whole item range, so
    they take the second dense level and the sparse level) in one call with long ones."""
    lens = [40, 90, 136, 1500, 60, 1100, 120, 1800]
    tracks = _tracks(lens, seed=3)
    pairs = np.array([(i, j) for i in range(len(lens)) for j in range(len(lens)) if i != j], dtype=np.int32)
    dump = [(0, 3), (3, 0), (4, 7), (6, 5), (1, 2)]
    frames, offs, got, _, counters, dumps = _tc_scores(monkeypatch, eng, tracks, pairs, dump)
    assert counters["col_dense2"][0] + counters["row_dense2"][0] > 0   # some items ran the second dense level
    assert counters["sparse"][0] > 0                                   # and some lines went on to the sparse level
    _against_oracle(tracks, frames, offs, pairs, got, dumps)


def test_quirk_sides(monkeypatch, eng):
    """A track of 210 frames has 201 windows: k = 200 * 0.095 rounds to exactly 19 in float32, so with the default
    parameters (no integer guard) its side's thresholds are forced to 0 and the sweeps skip every item of that side."""
    from acoss_b200 import default_params
    p = default_params()
    assert not p.integer_guard and np.float32(200) * np.float32(p.kappa) == np.float32(19)
    tracks = _tracks([210, 900, 210, 1300, 600])
    pairs = np.array([(0, 1), (1, 0), (0, 2), (3, 0), (2, 4), (4, 3)], dtype=np.int32)
    frames, offs, got, _, _, dumps = _tc_scores(monkeypatch, eng, tracks, pairs, pairs)
    # the quirk sides: the 210-frame track's columns as query, its rows as reference, both in (0, 2)
    for (q, r), side in [((0, 1), "thr_r"), ((1, 0), "thr_q"), ((0, 2), "thr_q"), ((0, 2), "thr_r"), ((3, 0), "thr_q")]:
        assert not np.any(dumps[(q, r)][side]), (q, r, side)
    assert np.all(dumps[(0, 1)]["thr_q"] > 0) and np.all(dumps[(4, 3)]["thr_q"] > 0)   # the other sides are selected
    _against_oracle(tracks, frames, offs, pairs, got, dumps)
