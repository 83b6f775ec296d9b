"""CPU checks of the SiMPle restatement (oracle/simple_np.py) and of the Simple plugin's host logic."""
import os
import socket
import sys

import numpy as np
import pytest

from oracle import simple_np as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _track(rng, n):
    return rng.random((n, 12)).astype(np.float32)


@pytest.mark.parametrize("n,keep", [(200, False), (537, False), (600, False), (537, True), (600, True), (150, True)])
def test_pool_is_np_mean(n, keep):
    X = np.random.default_rng(n).random((n, 12)).astype(np.float32)
    got = sp.pool(X, keep_partial=keep)
    assert got.shape[0] == sp.pool_count(n, keep_partial=keep)
    for k in range(got.shape[0]):
        want = np.mean(X[k * 100:k * 100 + 200], axis=0)
        assert want.dtype == np.float32 and np.array_equal(got[k], want), k


def test_pool_rejects_short_track():
    with pytest.raises(ValueError):
        sp.pool(np.zeros((199, 12), np.float32))
    assert sp.pool_count(450, keep_partial=True) == 4 and sp.pool_count(450) == 3
    assert sp.pool_count(400, keep_partial=True) == 3


@pytest.mark.parametrize("m", [1, 5, 10])
@pytest.mark.parametrize("squared", [False, True])
def test_direct_matches_simple_fast(m, squared):
    rng = np.random.default_rng(10 * m + squared)
    A, B = _track(rng, 57), _track(rng, 41)
    P, I = sp.profile(sp.join_d2(A, B, m), squared)
    Pf, If = sp.simple_fast_profile(A, B, m, squared)
    np.testing.assert_allclose(Pf, P, rtol=1e-9, atol=1e-9)
    assert np.mean(If == I) > 0.95                         # the index may differ only at near-ties


def test_identical_tracks_zero_profile():
    A = _track(np.random.default_rng(1), 30)
    r = sp.score_pair(A, A, m=5)
    assert r["oti"] == 0 and np.all(r["profile"] == 0.0) and np.array_equal(r["index"], np.arange(26))
    assert r["score"] == 0.0


@pytest.mark.parametrize("s", [1, 5, 11])
def test_rolled_track_oti(s):
    A = _track(np.random.default_rng(s), 40)
    B = np.roll(A, s, axis=1)
    r = sp.score_pair(A, B, m=4)
    assert r["oti"] == (12 - s) % 12 and np.all(r["profile"] == 0.0)
    r1 = sp.score_pair(A, B, m=4, roll_first=True)          # S4: rolling the query by s aligns it with B
    assert r1["oti"] == s and np.all(r1["profile"] == 0.0)


def test_time_shift_zero_on_overlap():
    rng = np.random.default_rng(2)
    X = _track(rng, 60)
    k, m = 7, 5
    A, B = X[k:], X                                         # A[i] = B[i + k]
    r = sp.score_pair(A, B, m=m, use_oti=False)
    assert np.all(r["profile"] == 0.0) and np.array_equal(r["index"], np.arange(len(A) - m + 1) + k)


def test_hand_computed_three_frames():
    A = np.zeros((3, 12), np.float32)
    B = np.zeros((3, 12), np.float32)
    A[:, 0] = [1, 2, 3]
    B[:, 0] = [0, 2, 5]
    d2 = sp.join_d2(A, B, 2)                                # windows (1,2),(2,3) vs (0,2),(2,5)
    assert np.array_equal(d2, [[1.0, 10.0], [5.0, 4.0]])
    r = sp.score_pair(A, B, m=2, use_oti=False)
    assert np.array_equal(r["profile"], [1.0, 2.0]) and np.array_equal(r["index"], [0, 1])
    assert r["score"] == np.float32(-1.5)


def test_median_even_and_odd():
    assert sp.median([3.0, 1.0, 2.0]) == 2.0
    assert sp.median([4.0, 1.0, 3.0, 2.0]) == 2.5


def test_switches():
    rng = np.random.default_rng(5)
    A, B = _track(rng, 30), np.roll(_track(rng, 30), 3, axis=1)
    base = sp.score_pair(A, B, m=4)
    sq = sp.score_pair(A, B, m=4, squared=True)              # S2
    assert np.allclose(sq["profile"], base["profile"] ** 2)
    pos = sp.score_pair(A, B, m=4, positive=True)            # S3
    assert pos["score"] == -base["score"] and base["score"] < 0
    first = sp.score_pair(A, B, m=4, roll_first=True)        # S4
    assert first["oti"] == (12 - base["oti"]) % 12
    noti = sp.score_pair(A, B, m=4, use_oti=False)
    assert noti["oti"] == 0
    X = _track(rng, 450)
    assert sp.pool(X).shape[0] == 3 and sp.pool(X, keep_partial=True).shape[0] == 4     # S5


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _tracks17():
    rng = np.random.default_rng(3)
    return [rng.random((int(n), 12)).astype(np.float32) for n in rng.integers(12, 40, size=17)]


def _oracle_scores(pairs, tracks):
    return np.array([sp.score_pair(tracks[i], tracks[j], m=6)["score"] for i, j in np.asarray(pairs)], np.float32)


def _worker(rank, world, port, tmp, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    os.chdir(tmp)
    import torch.distributed as dist
    from acoss_b200.distributed import all_pairwise_distributed
    from acoss_b200.simple import Simple
    dist.init_process_group("gloo", rank=rank, world_size=world)
    tracks = _tracks17()
    feats = [dict(hpcp=t, label=str(i // 3)) for i, t in enumerate(tracks)]
    alg = Simple(None, None, features=feats, subsequence_length=6, shortname="r%d" % rank, cachedir="cache%d" % rank)
    alg.all_feats = dict(enumerate(tracks))                  # pooled features pre-filled: no device needed
    all_pairwise_distributed(alg, symmetric=True, score_fn=lambda p: _oracle_scores(p, tracks))
    q.put((rank, np.array(alg.Ds["main"])))
    dist.destroy_process_group()


def test_distributed_simple_matches_single_process(tmp_path):
    import torch.multiprocessing as mp
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, str(tmp_path), q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    tracks = _tracks17()
    n = len(tracks)
    i, j = np.triu_indices(n, k=1)
    want = np.zeros((n, n), np.float32)
    want[i, j] = _oracle_scores(np.stack([i, j], 1), tracks)
    want = want + want.T
    for _, D in res:
        assert np.array_equal(D, want)


def test_pair_weights(tmp_path):
    from acoss_b200.simple import Simple
    tracks = _tracks17()
    alg = Simple(None, None, features=[dict(hpcp=t, label="0") for t in tracks], subsequence_length=6,
                 cachedir=str(tmp_path / "cache"))
    alg.all_feats = dict(enumerate(tracks))
    w = alg.pair_weights(np.array([[0, 1], [2, 3]]))
    assert list(w) == [(len(tracks[0]) - 5) * (len(tracks[1]) - 5), (len(tracks[2]) - 5) * (len(tracks[3]) - 5)]
