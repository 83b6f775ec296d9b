#!/usr/bin/env python
"""Device-resident pair rates of ChenFusion (Qmax + Dmax over one CRP per pair, acoss_score_pairs_chen_device) and
Serra09 (Qmax, acoss_score_pairs_device) on one GPU, on a C3 slice (~2 000 frames per track) and a C4s slice (~500).

    python tools/time_chen.py [--c3-tracks 120] [--c4s-tracks 1000] [--reps 3] [--out profiles/r6_chen_time.json]

Each slice's upper-triangle pairs are scored with the pairs and the scores in HBM: CUDA events on the engine stream
around one call, then acoss_sync (which also finishes any deferred exact fallback), after a warm-up call of both entry
points.  The two entry points alternate, `--reps` times each; the median is reported.  A separate profiled call of
each gives the K1 / K2 / K3 device milliseconds.  ChenFusion's Qmax row must equal Serra09's scores bit for bit.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl = [x.strip() for x in out.split(",")]
        return name, pl
    except Exception as e:                                   # noqa: BLE001 - reported, not hidden
        return "unknown (%s)" % e, "unknown"


def time_slice(config, max_tracks, reps):
    import torch
    from acoss_b200 import Engine, pack_tracks, synthetic
    tracks, _ = synthetic.config_dataset(config, max_tracks=max_tracks)
    frames, offs = pack_tracks(tracks)
    pairs = synthetic.all_pairs_upper(len(tracks))
    cells = int(synthetic.pair_cells([len(t) for t in tracks], pairs))
    n = len(pairs)
    with Engine(0) as eng:
        eng.set_tracks(frames, offs)
        stream = torch.cuda.ExternalStream(eng.stream_ptr)
        dp = torch.from_numpy(pairs.astype(np.int32)).cuda()
        s = torch.zeros(n, dtype=torch.float32, device="cuda")
        q = torch.zeros(n, dtype=torch.float32, device="cuda")
        d = torch.zeros(n, dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        run = dict(serra09=lambda: eng.score_pairs_device(dp.data_ptr(), n, s.data_ptr()),
                   chen=lambda: eng.score_pairs_chen_device(dp.data_ptr(), n, q.data_ptr(), d.data_ptr()))
        warm = min(n, 4096)
        eng.score_pairs_device(dp.data_ptr(), warm, s.data_ptr())
        eng.score_pairs_chen_device(dp.data_ptr(), warm, q.data_ptr(), d.data_ptr())
        eng.sync()
        times = {k: [] for k in run}
        fallback = {}
        for _ in range(reps):
            for k, fn in run.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                fn()
                e1.record(stream)
                eng.sync()
                times[k].append(e0.elapsed_time(e1) / 1e3)
                fallback[k] = eng.last_stats()["fallback_pairs"]
        stages = {}
        for k, fn in run.items():
            eng.set_profiling(True)
            fn()
            eng.sync()
            stages[k] = eng.stage_ms()
            eng.set_profiling(False)
        qmax_equals_serra09 = bool(torch.equal(q, s))
    res = dict(config=config, tracks=len(tracks), mean_frames=float(np.mean([len(t) for t in tracks])), pairs=n,
               cells=cells, qmax_equals_serra09=qmax_equals_serra09)
    for k in run:
        t = float(np.median(times[k]))
        res[k] = dict(s=t, s_reps=times[k], pairs_per_s=n / t, gcups=cells / t / 1e9, fallback_pairs=fallback[k],
                      stage_ms=stages[k])
    res["chen_over_serra09"] = res["chen"]["s"] / res["serra09"]["s"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c3-tracks", type=int, default=120)
    ap.add_argument("--c4s-tracks", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_chen_time.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_chen.py measures the GPU: no CUDA device")
    name, plimit = _card()
    out = dict(tool="time_chen", card=name, power_limit=plimit, reps=a.reps,
               slices=[time_slice("C3", a.c3_tracks, a.reps), time_slice("C4s", a.c4s_tracks, a.reps)])
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")
    if not all(s["qmax_equals_serra09"] for s in out["slices"]):
        raise SystemExit("ChenFusion's Qmax differs from Serra09's scores")


if __name__ == "__main__":
    main()
