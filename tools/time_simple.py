#!/usr/bin/env python
"""Throughput of the Simple (SiMPle) pair scoring (acoss_simple_score_pairs_device, k6_simple.cu) on one B200, with
the CPU oracle's SiMPle-Fast (oracle/simple_np.py: scipy fftconvolve + sliding updates, the reference's arithmetic
shape) timed on a sample of the same pairs over all host threads, and a parity check on that sample.

    python tools/time_simple.py [--tracks 15000] [--pairs 2000000] [--cpu-pairs 256] [--m 10] [--out f.json]

Workload: Da-TACOS-shaped, the C4s clique layout (1000 cliques of 13 + 2000 singletons = 15 000 tracks) with pooled
lengths drawn from 154..256 frames (3-5 min at 86 raw frames/s pooled by SKIP = 100).  The pooled frames are
generated directly (the on-ramp is timed separately as `pool_s`).  The timed pairs are a uniform sample of the
upper triangle; pairs/s is device-resident (CUDA events around the device entry point, after a warm-up call).
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _cpu_score(args):
    A, B, m = args
    from oracle import simple_np as sp
    return float(sp.score_pair_fast(A, B, m))


def _card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl, clk = [x.strip() for x in out.split(",")]
        return name, pl, float(clk.split()[0])
    except Exception as e:                                   # noqa: BLE001 - reported, not hidden
        return "unknown (%s)" % e, "unknown", float("nan")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tracks", type=int, default=15000)
    ap.add_argument("--pairs", type=int, default=2000000)
    ap.add_argument("--cpu-pairs", type=int, default=256)
    ap.add_argument("--m", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_simple_time.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_simple.py measures the GPU: no CUDA device")
    from acoss_b200 import Engine, pack_tracks, synthetic
    from acoss_b200._lib import simple_default_params
    from oracle import simple_np as sp

    cliques = [13] * 1000 + [1] * 2000
    out, tot = [], 0
    for s in cliques:
        if tot + s > a.tracks:
            break
        out.append(s)
        tot += s
    tracks, _ = synthetic.make_dataset(out, 205, 20246, length_jitter=0.25)
    n = len(tracks)
    lens = np.array([t.shape[0] for t in tracks], dtype=np.int64)
    rng = np.random.default_rng(0)
    total_pairs = n * (n - 1) // 2
    k = rng.choice(total_pairs, size=min(a.pairs, total_pairs), replace=False)
    k.sort()
    iu, ju = np.triu_indices(n, k=1)
    pairs = np.stack([iu[k], ju[k]], axis=1).astype(np.int32)
    del iu, ju
    cells_per = (lens[pairs[:, 0]] - a.m + 1) * (lens[pairs[:, 1]] - a.m + 1)
    cells = int(cells_per.sum())
    L = lens - a.m + 1
    full_cells = float((L.sum() ** 2 - (L * L).sum()) / 2)

    p = simple_default_params(m=a.m)
    name, plimit, clk = _card()
    with Engine(0) as eng:
        # on-ramp: raw frames of the first 200 tracks at 100x the pooled length, pooled on the GPU
        raws = [np.repeat(t, 100, axis=0) for t in tracks[:200]]
        rf, ro = pack_tracks(raws)
        t0 = time.perf_counter()
        eng.set_tracks_pooled(rf, ro)
        pool_s = time.perf_counter() - t0
        frames, offs = pack_tracks(tracks)
        eng.set_tracks(frames, offs)
        dp = torch.from_numpy(pairs).cuda()
        ds = torch.zeros(len(pairs), dtype=torch.float32, device="cuda")
        stream = torch.cuda.ExternalStream(eng.stream_ptr)
        warm = min(len(pairs), 20000)
        eng.simple_score_pairs_device(dp.data_ptr(), warm, ds.data_ptr(), p)
        eng.sync()
        times = []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            eng.simple_score_pairs_device(dp.data_ptr(), len(pairs), ds.data_ptr(), p)
            e1.record(stream)
            eng.sync()
            times.append(e0.elapsed_time(e1) / 1e3)
        gpu_scores = ds.cpu().numpy()
    t = float(np.median(times))

    # CPU baseline and parity on a sample
    cs = rng.choice(len(pairs), size=min(a.cpu_pairs, len(pairs)), replace=False)
    work = [(tracks[pairs[c, 0]], tracks[pairs[c, 1]], a.m) for c in cs]
    threads = os.cpu_count() or 1
    t0 = time.perf_counter()
    with ProcessPoolExecutor(threads) as ex:
        cpu_fast = np.array(list(ex.map(_cpu_score, work, chunksize=4)), dtype=np.float64)
    cpu_s = time.perf_counter() - t0
    exact_n = min(16, len(cs))
    exact_ok = all(gpu_scores[c] == sp.score_pair(tracks[pairs[c, 0]], tracks[pairs[c, 1]], a.m)["score"]
                   for c in cs[:exact_n])
    fast_rel = float(np.max(np.abs(cpu_fast - gpu_scores[cs]) / np.maximum(np.abs(cpu_fast), 1e-30)))

    fp32_per_cell = 2 * 24          # two filter sweeps, 12 FSUB + 12 FFMA per frame item
    fma_per_cell = 12               # one 12-term frame dot per cell: the least FP32 work a cell needs
    peak_lane_ops = 148 * 128 * clk * 1e6          # FP32 lanes x max SM clock (one op per lane per clock)
    res = dict(
        tool="time_simple", card=name, power_limit=plimit, max_sm_clock_mhz=clk, tracks=n, m=a.m,
        pooled_len_min=int(lens.min()), pooled_len_max=int(lens.max()), pooled_len_mean=float(lens.mean()),
        pairs=int(len(pairs)), cells=cells, gpu_s=t, gpu_s_reps=times, pairs_per_s=len(pairs) / t,
        cells_per_s=cells / t, fp32_fma_fraction=fma_per_cell * cells / t / peak_lane_ops,
        fp32_pipe_fraction=fp32_per_cell * cells / t / peak_lane_ops,
        full_set_pairs=total_pairs, full_set_cells=full_cells, full_set_est_s=full_cells / (cells / t),
        cpu_pairs=len(cs), cpu_threads=threads, cpu_s=cpu_s, cpu_pairs_per_s=len(cs) / cpu_s,
        speedup=(len(pairs) / t) / (len(cs) / cpu_s), parity_exact_pairs=exact_n, parity_exact_ok=bool(exact_ok),
        parity_fast_max_rel=fast_rel, onramp_tracks=200, onramp_raw_frames=int(ro[-1]), pool_s=pool_s)
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")
    if not exact_ok:
        raise SystemExit("GPU scores differ from the oracle on the parity sample")


if __name__ == "__main__":
    main()
