"""Multi-GPU all-pairs scoring: one process per GPU (torch.distributed), pair space sharded by
work, no data-path collective, one gather of the per-rank score tiles at the end.

The reference's only parallelism is a single-host joblib fan-out of 45 pair chunks whose workers
write disjoint cells of a shared memmap (/root/reference/acoss/algorithms/algorithm_template.py:
172-177).  Here every rank holds all track features (<= 1.5 GB at 15 000 tracks), scores its own
contiguous slice of the pair list — cut so that every rank gets the same number of DP cells, not
the same number of pairs, because track lengths vary — and the score slices are exchanged with one
all_gather (NCCL over NVLink on GPUs; gloo in the CPU tests).
"""
from __future__ import annotations

import numpy as np

__all__ = ["shard_bounds", "triangle_shard", "gather_scores", "all_pairwise_distributed"]


def shard_bounds(weights, world: int) -> np.ndarray:
    """Cut points b[0..world] of a contiguous split of len(weights) items into `world` shards of
    (nearly) equal total weight.  Deterministic, identical on every rank."""
    w = np.asarray(weights, dtype=np.float64)
    n = len(w)
    if world <= 1 or n == 0:
        return np.array([0, n] + [n] * max(0, world - 1), dtype=np.int64)[:world + 1]
    c = np.concatenate([[0.0], np.cumsum(w)])
    targets = c[-1] * np.arange(1, world) / world
    cuts = np.searchsorted(c, targets, side="left")
    b = np.concatenate([[0], cuts, [n]]).astype(np.int64)
    return np.maximum.accumulate(b)


def triangle_shard(a, world: int, rank: int):
    """The same split for the upper-triangle pair list (i < j, row-major = itertools.combinations order) with product
    weights w_ij = a_i a_j, WITHOUT building the list: at 15 000 tracks the list has 1.1e8 pairs and every rank would
    spend seconds and gigabytes on pairs it never scores.  Row i holds N-1-i pairs of weight a_i * (a_{i+1} + ...): the
    cut points are located by row, then inside the row.  Returns (bounds[0..world], this rank's pairs as (n, 2) int64);
    the bounds equal shard_bounds(weights of the full list, world)."""
    a = np.asarray(a, dtype=np.float64)
    n = len(a)
    cnt = np.arange(n - 1, -1, -1, dtype=np.int64)                     # pairs per row
    start = np.concatenate([[0], np.cumsum(cnt)])                      # first pair index of each row
    total_pairs = int(start[-1])
    suffix = np.concatenate([np.cumsum(a[::-1])[::-1][1:], [0.0]])     # a_{i+1} + ... + a_{n-1}
    roww = a * suffix
    crow = np.concatenate([[0.0], np.cumsum(roww)])                    # weight before each row

    def cum_at(k):                                                     # weight of the first k pairs, as np.cumsum accumulates it
        i = int(np.searchsorted(start, k, side="right") - 1)
        i = min(i, n - 1)
        return i, k - int(start[i])

    if world <= 1 or total_pairs == 0:
        bounds = np.array([0, total_pairs] + [total_pairs] * max(0, world - 1), dtype=np.int64)[:world + 1]
    else:
        targets = crow[-1] * np.arange(1, world) / world
        cuts = []
        for t in targets:
            i = int(np.searchsorted(crow, t, side="right") - 1)       # row holding the cut
            i = max(0, min(i, n - 2))
            inrow = crow[i] + a[i] * np.concatenate([[0.0], np.cumsum(a[i + 1:])])
            off = int(np.searchsorted(inrow, t, side="left"))
            cuts.append(int(start[i]) + min(off, int(cnt[i])))
        bounds = np.maximum.accumulate(np.array([0] + cuts + [total_pairs], dtype=np.int64))
    k0, k1 = int(bounds[rank]), int(bounds[rank + 1])
    if k1 <= k0:
        return bounds, np.zeros((0, 2), dtype=np.int64)
    (i0, o0), (i1, o1) = cum_at(k0), cum_at(k1 - 1)
    rows = np.arange(i0, i1 + 1, dtype=np.int64)
    first = np.where(rows == i0, o0, 0)
    last = np.where(rows == i1, o1 + 1, cnt[rows])
    lens = last - first
    ii = np.repeat(rows, lens)
    within = np.arange(lens.sum(), dtype=np.int64) - np.repeat(np.cumsum(lens) - lens, lens)
    jj = ii + 1 + np.repeat(first, lens) + within
    return bounds, np.stack([ii, jj], axis=1)


def gather_scores(local_scores, bounds, rank: int, world: int, device=None):
    """all_gather of variable-length per-rank score slices -> the full score vector (every rank).
    `local_scores`: torch tensor (CUDA for NCCL, CPU for gloo) of length bounds[rank+1]-bounds[rank]."""
    import torch
    import torch.distributed as dist
    n = int(bounds[-1])
    if world == 1:
        return local_scores
    sizes = np.diff(bounds)
    pad = int(sizes.max())
    buf = torch.zeros(pad, dtype=torch.float32, device=local_scores.device)
    buf[:local_scores.numel()] = local_scores
    out = torch.empty(world * pad, dtype=torch.float32, device=local_scores.device)
    dist.all_gather_into_tensor(out, buf)
    full = torch.empty(n, dtype=torch.float32, device=local_scores.device)
    for r in range(world):
        full[int(bounds[r]):int(bounds[r + 1])] = out[r * pad:r * pad + int(sizes[r])]
    return full


def _tile_store(checkpoint_dir, rank, world, n_pairs, tile, bounds):
    """Per-rank tile files + manifest for resuming an interrupted all-pairs run (the reference can only reload a
    COMPLETE run: `precomputed=True`, algorithm_template.py:163-166).  Returns (load, save) closures or (None, None)."""
    if not checkpoint_dir:
        return None, None
    import json
    import os
    os.makedirs(checkpoint_dir, exist_ok=True)
    manifest = dict(world=int(world), n_pairs=int(n_pairs), tile=int(tile), bounds=[int(b) for b in bounds])
    mpath = os.path.join(checkpoint_dir, "manifest_rank%d.json" % rank)
    valid = False
    if os.path.exists(mpath):
        try:
            with open(mpath) as f:
                valid = json.load(f) == manifest
        except Exception:
            valid = False
    if not valid:                                           # different job: forget its tiles
        for fn in os.listdir(checkpoint_dir):
            if fn.startswith("rank%d_tile" % rank):
                os.remove(os.path.join(checkpoint_dir, fn))
        with open(mpath, "w") as f:
            json.dump(manifest, f)

    def path(t):
        return os.path.join(checkpoint_dir, "rank%d_tile%06d.npy" % (rank, t))

    def load(t, n_expected):
        if os.path.exists(path(t)):
            try:
                a = np.load(path(t))
                if a.shape[-1] == n_expected:
                    return a
            except Exception:
                pass
        return None

    def save(t, a):
        tmp = path(t) + ".tmp.npy"
        np.save(tmp, a)
        os.replace(tmp, path(t))                            # a tile file is either complete or absent
    return load, save


def all_pairwise_distributed(alg, symmetric=True, score_fn=None, fill_on=None, checkpoint_dir=None, timings=None):
    """Distributed `all_pairwise` for a plugin `alg`.  Every rank calls this; on return every rank's
    `alg.Ds[key]` holds the full (symmetrised) score matrix of every key (`fill_on=r`: only rank r's, the other
    ranks skip the assembly — what a benchmark run that evaluates on one rank wants).

    Serra09-style plugins (`_pair_array`, `load_features`, `Ds`, `N`, `m`, `tau`) are balanced by DP cells
    (n_q - m tau)(n_r - m tau) over the list-free triangle shard.  Those with several scores per pair (ChenFusion:
    'qmax', 'dmax') provide `score_pairs(pairs)` and keep that shard.  Other plugins with several scores per pair
    (EarlyFusion: 'mfccs', 'ssms', 'chromas', 'early') also provide `pair_weights(pairs)`.
    Row contract: every scoring call returns float32 (len(alg.Ds), n) with rows in `alg.Ds` key order (a plugin
    with one key may return (n,)); an empty shard contributes (rows, 0); a tile of any other shape is a scoring
    failure.  All score rows travel in ONE gather.
    `score_fn(pairs)` overrides the scoring call (CPU tests).  The shard is scored in tiles of `alg.tile_pairs`;
    with `checkpoint_dir` every finished tile is saved per rank and an interrupted run resumes from the tiles it
    finds (same world size, pair list and tile size).  `timings` (a dict) receives the seconds of each phase."""
    import time
    import torch
    import torch.distributed as dist
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    t0 = time.perf_counter()
    pairs = None                                            # the full pair list: built lazily (only the assembling rank needs it)
    if symmetric and not hasattr(alg, "pair_weights"):
        # Serra09-style plugin, upper triangle: product weights -> the shard is computed without the 1e8-pair list
        lens = np.array([alg.load_features(i).shape[0] for i in range(alg.N)], dtype=np.int64)
        incr = int(alg.m) * int(alg.tau)
        bounds, mine = triangle_shard(lens - incr, world, rank)
        n_pairs = int(bounds[-1])
    else:
        pairs = alg._pair_array(symmetric)
        if hasattr(alg, "pair_weights"):
            cells = np.asarray(alg.pair_weights(pairs), dtype=np.float64)
        else:
            lens = np.array([alg.load_features(i).shape[0] for i in range(alg.N)], dtype=np.int64)
            incr = int(alg.m) * int(alg.tau)
            cells = (lens[pairs[:, 0]] - incr) * (lens[pairs[:, 1]] - incr)
        bounds = shard_bounds(cells, world)
        del cells
        mine = pairs[bounds[rank]:bounds[rank + 1]]
        n_pairs = len(pairs)
    keys = list(alg.Ds.keys())
    rows = len(keys)

    def tile_rows(got, n):                                  # the row contract: (rows, n); (n,) only for one key
        got = np.asarray(got, dtype=np.float32)
        if rows == 1 and got.ndim == 1:
            got = got.reshape(1, -1)
        if got.shape != (rows, n):
            raise ValueError("a tile of %d pairs was scored as shape %r; the score types %r need (%d, %d)"
                             % (n, got.shape, keys, rows, n))
        return got
    tile = int(getattr(alg, "tile_pairs", 1 << 16))
    if score_fn is not None:
        score_tile = lambda p: np.asarray(score_fn(p), dtype=np.float32)
    elif hasattr(alg, "score_pairs"):
        score_tile = lambda p: np.asarray(alg.score_pairs(p), dtype=np.float32)
    else:
        eng = alg.engine()
        score_tile = lambda p: eng.score_pairs(p.astype(np.int32), alg.params())
    load, save = _tile_store(checkpoint_dir, rank, world, n_pairs, tile, bounds)
    backend = dist.get_backend() if dist.is_initialized() else "none"
    # staging device: the plugin's own device (alg.device), not whatever torch's current device happens to be —
    # with one process per GPU every rank must stage on ITS GPU or NCCL deadlocks
    if backend == "nccl":
        dev = torch.device("cuda", int(getattr(alg, "device", torch.cuda.current_device())))
        torch.cuda.set_device(dev)
    else:
        dev = torch.device("cpu")
    t1 = time.perf_counter()
    parts, resumed = [], 0
    failure = None
    try:
        for t, k in enumerate(range(0, len(mine), tile)):
            p = mine[k:k + tile]
            got = load(t, len(p)) if load else None
            if got is None:
                got = score_tile(p)
                if save:
                    save(t, got)
            else:
                resumed += 1
            parts.append(tile_rows(got, len(p)))
    except Exception as e:                                  # noqa: BLE001 - reported to every rank below
        failure = e
    # A rank whose scoring failed must not leave the others waiting in the gather: agree on the outcome first (one
    # tiny all_reduce), then every rank raises - the launcher sees non-zero exit codes instead of a hang.
    if world > 1:
        flag = torch.tensor([0 if failure is None else 1], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        if int(flag.item()) and failure is None:
            raise RuntimeError("all_pairwise_distributed: scoring failed on another rank (rank %d had finished its shard)" % rank)
    if failure is not None:
        raise RuntimeError("all_pairwise_distributed: scoring failed on rank %d: %s" % (rank, failure)) from failure
    local = np.concatenate(parts, axis=1) if parts else np.zeros((rows, 0), np.float32)
    t2 = time.perf_counter()
    # one gather for all score rows: rank r contributes rows x (bounds[r+1] - bounds[r]) floats, row-major
    flat = np.ascontiguousarray(local).ravel()
    full = gather_scores(torch.from_numpy(flat).to(dev), bounds * rows, rank, world)
    if dev.type == "cuda":
        torch.cuda.synchronize(dev)
    t3 = time.perf_counter()
    if fill_on is None or fill_on == rank:
        fill_score_matrices(alg, pairs, full, bounds, rows, keys, symmetric, world)
    t4 = time.perf_counter()
    if timings is not None:
        timings.update(shard_s=t1 - t0, score_s=t2 - t1, gather_s=t3 - t2, fill_s=t4 - t3, resumed_tiles=resumed,
                       tiles=len(parts))
    return bounds


def fill_score_matrices(alg, pairs, full, bounds, rows, keys, symmetric, world):
    """Gathered score vector -> alg.Ds[key].  The (N, N) matrix is assembled in a PRIVATE buffer — on the
    staging device when that is a GPU (one index_put_ + one transposed add, then ONE contiguous device-to-host
    copy), in a private ndarray otherwise — and then written to alg.Ds[key] by a plain, idempotent assignment.
    Ranks of one box that were constructed with the same cache prefix map the same memmap file: an in-place
    `Ds += Ds.T` on the shared file would symmetrise twice (scores doubled); a plain assignment of the finished
    matrix cannot.  `pairs=None`: the full upper triangle in combinations order (indices generated on the staging device)."""
    import torch
    N = int(alg.N)
    n_pairs = len(pairs) if pairs is not None else N * (N - 1) // 2
    # rank r's slice holds its rows back to back (row-major rows x n_r): un-interleave into (rows, n_pairs)
    if rows == 1:
        per_key = full.reshape(1, -1)
    else:
        per_key = torch.empty((rows, n_pairs), dtype=torch.float32, device=full.device)
        for r in range(world):
            a, b = int(bounds[r]), int(bounds[r + 1])
            per_key[:, a:b] = full[a * rows:b * rows].reshape(rows, b - a)
    if pairs is None:
        pi, pj = torch.triu_indices(N, N, offset=1, device=full.device)      # row-major: itertools.combinations order
    else:
        pi = torch.from_numpy(np.ascontiguousarray(pairs[:, 0]).astype(np.int64)).to(full.device)
        pj = torch.from_numpy(np.ascontiguousarray(pairs[:, 1]).astype(np.int64)).to(full.device)
    for k, key in enumerate(keys):
        D = torch.zeros((N, N), dtype=torch.float32, device=full.device)
        D.index_put_((pi, pj), per_key[k if rows > 1 else 0])
        if symmetric:
            D = D + D.T                                    # out of place: no aliasing between D and its transpose
        alg.Ds[key][:, :] = D.cpu().numpy()
