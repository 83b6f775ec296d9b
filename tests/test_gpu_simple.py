"""GPU checks of the Simple (SiMPle) path: pooling on-ramp, OTI, join / profile / median (k6_simple.cu) against the
numpy restatement (oracle/simple_np.py), bit for bit."""
import numpy as np
import pytest

from acoss_b200 import AcossError, Engine, pack_tracks
from acoss_b200 import _lib
from oracle import simple_np as sp

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    with Engine(0) as e:
        yield e


def _chroma(rng, n):
    X = rng.random((n, 12)).astype(np.float32)
    return X / X.max(axis=1, keepdims=True)


def _load(eng, tracks):
    frames, offs = pack_tracks(tracks)
    eng.set_tracks(frames, offs)


def test_pooling_bit_identical(eng):
    rng = np.random.default_rng(0)
    lens = [200, 300, 1000, 537, 12345, 201, 299]
    raws = [rng.random((n, 12)).astype(np.float32) for n in lens]
    frames, offs = pack_tracks(raws)
    for keep in (False, True):
        out_off = eng.set_tracks_pooled(frames, offs, keep_partial=keep)
        got = eng.get_tracks()
        for t, X in enumerate(raws):
            assert np.array_equal(got[out_off[t]:out_off[t + 1]], sp.pool(X, keep_partial=keep)), (t, keep)
    eng.set_tracks_pooled(frames, offs, win=37, skip=11)
    got = eng.get_tracks()
    assert np.array_equal(got[:sp.pool_count(200, 37, 11)], sp.pool(raws[0], 37, 11))
    short = pack_tracks([raws[0], raws[0][:150]])
    with pytest.raises(AcossError) as ei:
        eng.set_tracks_pooled(*short)
    assert ei.value.code == _lib.E_TOO_SHORT


def test_oti_exact(eng):
    rng = np.random.default_rng(1)
    base = [_chroma(rng, int(n)) for n in rng.integers(20, 60, size=12)]
    tracks = base + [np.roll(t, s, axis=1) for t, s in zip(base, rng.integers(0, 12, size=12))]
    _load(eng, tracks)
    pairs = np.array([(i, j) for i in range(24) for j in range(24)])[::2]
    for rf in (0, 1):
        p = _lib.simple_default_params(m=3, s4_roll_first=rf)
        for i, j in pairs[:: 3]:
            want = sp.oti(tracks[i], tracks[j], bool(rf))
            assert eng.simple_dump_pair(int(i), int(j), p)["oti"] == want, (i, j, rf)
    for k in range(12):                                         # planted transpositions
        d = eng.simple_dump_pair(k, 12 + k)
        assert np.all(d["profile"] == 0.0) and d["oti"] == sp.oti(tracks[k], tracks[12 + k])


def _check_pairs(eng, tracks, pairs, **sw):
    p = _lib.simple_default_params(**sw)
    got = eng.simple_score_pairs(pairs, p)
    kw = dict(m=p.m, use_oti=bool(p.oti), squared=bool(p.s2_squared), positive=bool(p.s3_positive),
              roll_first=bool(p.s4_roll_first))
    for k, (i, j) in enumerate(pairs):
        want = sp.score_pair(tracks[i], tracks[j], **kw)
        assert got[k] == want["score"], (i, j, sw)
    i, j = pairs[0]
    d = eng.simple_dump_pair(int(i), int(j), p)
    want = sp.score_pair(tracks[i], tracks[j], **kw)
    assert np.array_equal(d["profile"], want["profile"]) and np.array_equal(d["index"], want["index"])
    assert d["oti"] == want["oti"] and d["score"] == want["score"]


@pytest.mark.parametrize("m", [1, 5, 10, 32, 128])
def test_scores_identical(eng, m):
    rng = np.random.default_rng(m)
    lens = [max(m, n) for n in (20, 33, 64, 205, 700, 131)]
    tracks = [_chroma(rng, n) for n in lens]
    tracks.append(np.roll(tracks[3][5:150], 4, axis=1))          # a transposed, shifted excerpt
    _load(eng, tracks)
    pairs = np.array([(i, j) for i in range(len(tracks)) for j in range(len(tracks)) if i != j])
    _check_pairs(eng, tracks, pairs, m=m)
    sub = pairs[::5]
    for sw in (dict(s2_squared=1), dict(s3_positive=1), dict(s4_roll_first=1), dict(oti=0)):
        _check_pairs(eng, tracks, sub, m=m, **sw)


def test_fallback_rows_identical(eng):
    """Constant and repeated-window tracks list more candidates per row than the kernel holds."""
    rng = np.random.default_rng(7)
    const = np.full((120, 12), 0.5, np.float32)
    loop = np.tile(_chroma(rng, 4), (40, 1))
    silent = np.zeros((90, 12), np.float32)
    tracks = [const, loop, silent, _chroma(rng, 100)]
    _load(eng, tracks)
    pairs = np.array([(i, j) for i in range(4) for j in range(4)])
    for m in (1, 6, 10):
        _check_pairs(eng, tracks, pairs, m=m)


def test_host_device_and_chunking(eng):
    import torch
    rng = np.random.default_rng(9)
    tracks = [_chroma(rng, int(n)) for n in rng.integers(30, 300, size=20)]
    _load(eng, tracks)
    pairs = np.array([(i, j) for i in range(20) for j in range(20) if i != j], dtype=np.int32)
    host = eng.simple_score_pairs(pairs)
    dp = torch.from_numpy(pairs).cuda()
    ds = torch.zeros(len(pairs), dtype=torch.float32, device="cuda")
    eng.simple_score_pairs_device(dp.data_ptr(), len(pairs), ds.data_ptr())
    eng.sync()
    assert np.array_equal(ds.cpu().numpy(), host)
    with Engine(0, workspace_bytes=64 << 20) as small:            # 64 MiB: several chunks of pairs
        _load(small, tracks)
        big = np.concatenate([pairs] * 200)
        got = small.simple_score_pairs(big)
        assert np.array_equal(got, np.tile(host, 200))


def test_errors(eng):
    rng = np.random.default_rng(11)
    _load(eng, [_chroma(rng, 40), _chroma(rng, 9)])
    with pytest.raises(AcossError) as ei:
        eng.simple_score_pairs(np.array([[0, 1]]))                 # m = 10 > 9 frames
    assert ei.value.code == _lib.E_TOO_SHORT
    for m in (0, 129):
        with pytest.raises(AcossError) as ei:
            eng.simple_score_pairs(np.array([[0, 1]]), _lib.simple_default_params(m=m))
        assert ei.value.code == _lib.E_INVALID
    assert eng.simple_score_pairs(np.array([[0, 1]]), _lib.simple_default_params(m=9)).shape == (1,)


def test_plugin_eval_matches_oracle(tmp_path, monkeypatch):
    from acoss_b200.simple import Simple
    monkeypatch.chdir(tmp_path)                                    # getEvalStatistics appends to a results file in cwd
    rng = np.random.default_rng(12)
    feats, labels = [], []
    for c in range(6):
        base = _chroma(rng, 4000)
        for v in range(3):
            n = int(rng.integers(2600, 4000))
            X = np.roll(base[:n], int(rng.integers(0, 12)), axis=1) + 0.05 * rng.random((n, 12)).astype(np.float32)
            feats.append(dict(hpcp=X.astype(np.float32), label=str(c)))
    alg = Simple(None, None, features=feats, cachedir=str(tmp_path / "c"))
    alg.all_pairwise(symmetric=True)
    got = alg.getEvalStatistics("main")
    N = len(feats)
    pooled = [sp.pool(f["hpcp"]) for f in feats]
    D = np.zeros((N, N), np.float32)
    for i in range(N):
        for j in range(i + 1, N):
            D[i, j] = sp.score_pair(pooled[i], pooled[j])["score"]
    D = D + D.T
    assert np.array_equal(np.asarray(alg.Ds["main"]), D)
    alg2 = Simple(None, None, features=feats, shortname="oracle", cachedir=str(tmp_path / "c2"))
    alg2.get_all_clique_ids()
    alg2.Ds["main"][:, :] = D
    want = alg2.getEvalStatistics("main")
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    alg.close()
