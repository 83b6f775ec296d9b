"""gloo tests of the row contract of all_pairwise_distributed: ChenFusion's two score rows on the triangle shard, a
tile with the wrong number of rows failing on every rank (also when a shard is empty), and a four-row plugin on a
world with an empty shard."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _fake_two(pairs):
    p = np.asarray(pairs, dtype=np.int64)
    q = ((p[:, 0] * 131 + p[:, 1] * 7) % 1000).astype(np.float32) / 8.0
    d = ((p[:, 0] * 17 + p[:, 1] * 53) % 777).astype(np.float32) / 4.0 + 0.25
    return np.stack([q, d])


def _fake_four(pairs):
    p = np.asarray(pairs, dtype=np.int64)
    base = ((p[:, 0] * 37 + p[:, 1] * 11) % 500).astype(np.float32)
    return np.stack([base + 0.1 * k for k in range(4)]).astype(np.float32)


def _chen_feats(n_tracks, seed=3):
    rng = np.random.default_rng(seed)
    return [dict(hpcp=rng.random((int(n), 12)).astype(np.float32), label=str(i // 3))
            for i, n in enumerate(rng.integers(20, 200, size=n_tracks))]


def _init(rank, world, port, tmp):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    os.chdir(tmp)
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    return dist


def _worker_chen(rank, world, port, tmp, q):
    dist = _init(rank, world, port, tmp)
    from acoss_b200.chenfusion import ChenFusion
    from acoss_b200.distributed import all_pairwise_distributed

    class FakeChen(ChenFusion):                             # the GPU scoring hook replaced by a two-row fake
        def score_pairs(self, pairs):
            return _fake_two(pairs)
    feats = _chen_feats(17)
    alg = FakeChen(None, None, features=feats, downsample_fac=1, shortname="c%d" % rank, cachedir="cachec%d" % rank)
    bounds = all_pairwise_distributed(alg, symmetric=True)
    q.put((rank, {k: np.array(v) for k, v in alg.Ds.items()}, bounds, [len(f["hpcp"]) for f in feats]))
    dist.destroy_process_group()


def _worker_one_row(rank, world, port, tmp, n_tracks, q):
    dist = _init(rank, world, port, tmp)
    from acoss_b200.chenfusion import ChenFusion
    from acoss_b200.distributed import all_pairwise_distributed
    alg = ChenFusion(None, None, features=_chen_feats(n_tracks), downsample_fac=1, shortname="o%d" % rank,
                     cachedir="cacheo%d" % rank)
    try:
        all_pairwise_distributed(alg, symmetric=True, score_fn=lambda p: _fake_two(p)[0])
        q.put((rank, "ok"))
    except (ValueError, RuntimeError) as e:
        q.put((rank, "%s: %s" % (type(e).__name__, e)))
        dist.destroy_process_group()
        sys.exit(3)
    dist.destroy_process_group()


def _worker_four_empty(rank, world, port, tmp, q):
    dist = _init(rank, world, port, tmp)
    from acoss_b200.distributed import all_pairwise_distributed
    from acoss_b200.earlyfusion import EarlyFusion
    feats = [dict(mfccs=np.zeros((n, 4), np.float32), ssms=np.zeros((n, 3), np.float32),
                  chromas=np.zeros((n, 12), np.float32), chroma_med=np.zeros(12), label=str(i))
             for i, n in enumerate((14, 23))]
    alg = EarlyFusion(None, None, features=feats, shortname="e%d" % rank, cachedir="cachee%d" % rank)
    bounds = all_pairwise_distributed(alg, symmetric=True, score_fn=_fake_four)
    q.put((rank, {k: np.array(v) for k, v in alg.Ds.items()}, bounds))
    dist.destroy_process_group()


def _spawn(target, world, tmp_path, *args):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=target, args=(r, world, port, str(tmp_path), *args, q)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        res = [q.get(timeout=120) for _ in procs]
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.kill()
                p.join()
    return res, [p.exitcode for p in procs]


def _upper(n, scores):
    i, j = np.triu_indices(n, k=1)
    D = np.zeros((n, n), np.float32)
    D[i, j] = scores
    return D + D.T


@pytest.mark.parametrize("world", [2, 3])
def test_chenfusion_two_rows_triangle_shard(tmp_path, world):
    """Each of Ds["qmax"] and Ds["dmax"] is its own score row, symmetrised (not a copy of row 0), and the shard is
    the list-free triangle split weighted by the stacked-window counts (frames - m tau = frames - 9)."""
    from acoss_b200.distributed import triangle_shard
    res, codes = _spawn(_worker_chen, world, tmp_path)
    assert codes == [0] * world
    n = 17
    i, j = np.triu_indices(n, k=1)
    want = _fake_two(np.stack([i, j], 1))
    for rank, Ds, bounds, lens in res:
        assert list(Ds) == ["qmax", "dmax"]
        assert np.array_equal(Ds["qmax"], _upper(n, want[0]))
        assert np.array_equal(Ds["dmax"], _upper(n, want[1]))
        assert not np.array_equal(Ds["qmax"], Ds["dmax"])
        assert np.array_equal(bounds, triangle_shard(np.array(lens) - 9, world, rank)[0])


@pytest.mark.parametrize("n_tracks", [17, 2], ids=["every_shard_scored", "one_shard_empty"])
def test_one_row_for_two_keys_fails_on_every_rank(tmp_path, n_tracks):
    """A two-key plugin scored with one row per pair is a scoring failure: every rank raises before the gather,
    including a rank whose shard is empty (2 tracks = 1 pair on 2 ranks), and no rank is left waiting."""
    world = 2
    res, codes = _spawn(_worker_one_row, world, tmp_path, n_tracks)
    msgs = dict(res)
    assert codes == [3] * world, msgs
    assert all(m.startswith(("ValueError", "RuntimeError")) for m in msgs.values()), msgs
    assert any("shape" in m for m in msgs.values()), msgs


def test_four_rows_with_an_empty_shard(tmp_path):
    """Four score rows (EarlyFusion-shaped) on 3 ranks and 1 pair: the empty shards contribute (4, 0) and every
    rank gathers the same sizes, so all four keys are filled."""
    world = 3
    res, codes = _spawn(_worker_four_empty, world, tmp_path)
    assert codes == [0] * world
    sc = _fake_four(np.array([[0, 1]]))
    for rank, Ds, bounds in res:
        assert (np.diff(bounds) == 0).sum() == world - 1
        assert list(Ds) == ["mfccs", "ssms", "chromas", "early"]
        for k, key in enumerate(Ds):
            assert np.array_equal(Ds[key], _upper(2, sc[k])), key
