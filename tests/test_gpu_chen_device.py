"""GPU: ChenFusion's device-resident entry point (acoss_score_pairs_chen_device) against the host entry and the C
oracle, and ChenFusion through all_pairwise_distributed (world 1, and two NCCL ranks when two GPUs are visible)."""
import ctypes as C
import os
import socket
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32


def hp(rng, n):
    X = rng.random((n, 12)).astype(F32)
    return (X / X.max(1, keepdims=True)).astype(F32)


@pytest.fixture(scope="module")
def eng():
    from acoss_b200 import Engine
    e = Engine(0)
    yield e
    e.close()


def _slices(lens):
    """Ragged slices of ~2k-frame synthetic C3 tracks."""
    from acoss_b200 import synthetic
    base, _ = synthetic.config_dataset("C3", max_tracks=13)
    return [np.ascontiguousarray(base[i % len(base)][7 * i:7 * i + n]) for i, n in enumerate(lens)]


def _tie_heavy():
    """The tracks and pairs of test_many_flagged_pairs_deferred_fallback: 91 pairs of tracks made of runs of 40
    identical frames (rows with hundreds of tied distances) mixed with 150 ordinary pairs."""
    rng = np.random.default_rng(77)
    tracks = [hp(rng, int(n)) for n in rng.integers(60, 260, size=40)]
    nt = 14
    for k in range(nt):
        tracks.append(np.repeat(hp(rng, 5 + k % 3), 40, axis=0))
    n = len(tracks)
    ti, tj = np.triu_indices(nt, k=1)
    tied = np.stack([40 + ti, 40 + tj], 1)
    other = np.stack([rng.integers(0, n, 150), rng.integers(0, n, 150)], 1)
    pairs = np.concatenate([tied, other]).astype(np.int32)
    return tracks, pairs[rng.permutation(len(pairs))]


def _case(name):
    if name == "tie_heavy":
        return _tie_heavy()
    if name == "ffma_sweeps":                    # every track below 400 stacked windows (409 frames)
        lens = [73, 74, 137, 138, 200, 265, 266, 329, 380, 408]
    else:                                        # tensor sweeps: the longest side reaches 400 windows and more
        lens = [73, 137, 200, 266, 329, 408, 409, 410, 521, 700, 1033]
    tracks = _slices(lens)
    pairs = np.array([(i, j) for i in range(len(lens)) for j in range(len(lens)) if i != j], dtype=np.int32)
    return tracks, pairs


@pytest.mark.parametrize("case", ["ffma_sweeps", "tensor_sweeps", "tie_heavy"])
def test_chen_device_equals_host_and_oracle(eng, case):
    import torch
    from acoss_b200 import pack_tracks
    from oracle import serra09_c as oc
    tracks, pairs = _case(case)
    frames, offs = pack_tracks(tracks)
    eng.set_tracks(frames, offs)
    hq, hd = eng.score_pairs_chen(pairs)
    st_host = eng.last_stats()
    dp = torch.from_numpy(pairs).cuda()
    dq = torch.full((len(pairs),), -1.0, dtype=torch.float32, device="cuda")
    dd = torch.full((len(pairs),), -1.0, dtype=torch.float32, device="cuda")
    eng.score_pairs_chen_device(dp.data_ptr(), len(pairs), dq.data_ptr(), dd.data_ptr())
    eng.sync()
    st_dev = eng.last_stats()
    wq, wd = oc.chen_pairs(frames, offs, pairs, oc.params(hoist_norms=True), nthreads=8)
    assert np.array_equal(dq.cpu().numpy(), hq) and np.array_equal(dd.cpu().numpy(), hd)
    assert np.array_equal(hq, wq) and np.array_equal(hd, wd)
    assert not np.array_equal(hq, hd)
    assert st_dev["fallback_pairs"] == st_host["fallback_pairs"]
    if case == "tie_heavy":
        assert st_host["fallback_pairs"] > 64, st_host    # the in-call rounds and the acoss_sync remainder both ran


def test_chen_device_refusals(eng):
    """NULL pointers, bad parameters and too-short tracks: the device entry returns the host entry's code."""
    import torch
    from acoss_b200 import default_params, pack_tracks
    from acoss_b200._lib import E_INVALID, E_TOO_SHORT, OK
    rng = np.random.default_rng(3)
    frames, offs = pack_tracks([hp(rng, 80), hp(rng, 120)])
    eng.set_tracks(frames, offs)
    lib = eng._lib
    pairs = np.array([[0, 1], [1, 0]], np.int32)
    dp = torch.from_numpy(pairs).cuda()
    dq = torch.zeros(2, dtype=torch.float32, device="cuda")
    dd = torch.zeros(2, dtype=torch.float32, device="cuda")
    hq = np.zeros(2, F32)
    hd = np.zeros(2, F32)
    good, bad_m, long_win = default_params(), default_params(m=0), default_params(m=64, tau=64)
    P = lambda p: C.byref(p) if p is not None else None
    cases = [  # (ctx, pointers present (pairs, qmax, dmax), n, params, code)
        (eng._ctx, (0, 1, 1), 2, good, E_INVALID),
        (eng._ctx, (1, 0, 1), 2, good, E_INVALID),
        (eng._ctx, (1, 1, 0), 2, good, E_INVALID),
        (None, (1, 1, 1), 2, good, E_INVALID),
        (eng._ctx, (1, 1, 1), 2, None, E_INVALID),
        (eng._ctx, (1, 1, 1), 2, bad_m, E_INVALID),
        (eng._ctx, (0, 0, 0), 0, good, OK),
        (eng._ctx, (0, 0, 0), 0, bad_m, E_INVALID),
        (eng._ctx, (0, 0, 0), -1, None, E_INVALID),
        (eng._ctx, (0, 0, 0), 0, long_win, E_TOO_SHORT),
    ]
    for ctx, (hp_, hq_, hd_), n, p, code in cases:
        rc_dev = lib.acoss_score_pairs_chen_device(ctx, dp.data_ptr() if hp_ else None, n, P(p),
                                                   dq.data_ptr() if hq_ else None, dd.data_ptr() if hd_ else None)
        rc_host = lib.acoss_score_pairs_chen(ctx, pairs.ctypes.data if hp_ else None, n, P(p),
                                             hq.ctypes.data if hq_ else None, hd.ctypes.data if hd_ else None)
        assert rc_dev == rc_host == code, (ctx, (hp_, hq_, hd_), n, code, rc_dev, rc_host)
    eng.sync()


def _chen(tmp, name, tracks, labels, device=0):
    from acoss_b200.chenfusion import ChenFusion
    feats = [dict(hpcp=t, label="w%d" % l) for t, l in zip(tracks, labels)]
    return ChenFusion(None, None, features=feats, downsample_fac=1, shortname=name, cachedir=os.path.join(tmp, name),
                      device=device, tile_pairs=64)


def _dataset():
    from acoss_b200 import synthetic
    return synthetic.config_dataset("tiny")


@pytest.fixture(scope="module")
def world1(tmp_path_factory):
    """all_pairwise_distributed(ChenFusion) without a process group (world 1)."""
    from acoss_b200.distributed import all_pairwise_distributed
    tmp = str(tmp_path_factory.mktemp("chen_w1"))
    tracks, labels = _dataset()
    c = _chen(tmp, "w1", tracks, labels)
    all_pairwise_distributed(c, symmetric=True)
    out = {k: np.array(v) for k, v in c.Ds.items()}
    c.cleanup_memmap()
    c.close()
    return out


def test_distributed_world1_chenfusion(world1, tmp_path):
    """Ds["qmax"] and Ds["dmax"] of the distributed path equal ChenFusion.all_pairwise and the oracle, and differ
    from each other (the distributed path once wrote the Qmax row into every key)."""
    from acoss_b200 import pack_tracks, synthetic
    from oracle import evalstats_np as ev
    from oracle import serra09_c as oc
    tracks, labels = _dataset()
    c = _chen(str(tmp_path), "ap", tracks, labels)
    c.all_pairwise(symmetric=True)
    frames, offs = pack_tracks(tracks)
    pairs = synthetic.all_pairs_upper(len(tracks))
    want = dict(zip(("qmax", "dmax"), oc.chen_pairs(frames, offs, pairs, nthreads=8)))
    assert list(world1) == ["qmax", "dmax"]
    for key in ("qmax", "dmax"):
        D = np.zeros((len(tracks), len(tracks)), np.float32)
        D[pairs[:, 0], pairs[:, 1]] = want[key]
        assert np.array_equal(world1[key], np.array(c.Ds[key])), key
        assert np.array_equal(world1[key], ev.symmetrize(D)), key
    assert not np.array_equal(world1["qmax"], world1["dmax"])
    c.cleanup_memmap()
    c.close()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker_nccl(rank, world, port, tmp, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from acoss_b200.distributed import all_pairwise_distributed
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        tracks, labels = _dataset()
        c = _chen(tmp, "n%d" % rank, tracks, labels, device=rank)
        bounds = all_pairwise_distributed(c, symmetric=True)
        q.put((rank, {k: np.array(v) for k, v in c.Ds.items()}, [int(b) for b in bounds]))
        c.cleanup_memmap()
        c.close()
    finally:
        dist.destroy_process_group()


def test_distributed_nccl_two_ranks_chenfusion(world1, tmp_path):
    """Two NCCL ranks give the world-1 matrices bit for bit on both ranks."""
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker_nccl, args=(r, world, port, str(tmp_path), q)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        res = [q.get(timeout=300) for _ in procs]
    finally:
        for p in procs:
            p.join(timeout=120)
            if p.is_alive():
                p.kill()
                p.join()
    assert [p.exitcode for p in procs] == [0] * world
    for rank, Ds, bounds in res:
        assert 0 < bounds[1] < bounds[2]                    # both ranks scored pairs
        for key in ("qmax", "dmax"):
            assert np.array_equal(Ds[key], world1[key]), (rank, key)
