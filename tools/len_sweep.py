#!/usr/bin/env python
"""Tensor-core vs FFMA2 sweeps by track length (ACOSS_K2_SWEEPS forced, host-to-host score_pairs on slices of the C3 tracks):
the crossover behind TC_MIN_WINDOWS.  Scores of the two runs must be identical."""
import os, sys, time, json
import numpy as np
sys.path.insert(0, os.getcwd())
from acoss_b200 import Engine, pack_tracks, synthetic
base, _ = synthetic.config_dataset("C3", max_tracks=200)
res = {}
for L in (300, 700, 1000, 1400):
    tracks = [np.ascontiguousarray(t[:L + (7 * i) % 60]) for i, t in enumerate(base)]
    frames, offs = pack_tracks(tracks)
    pairs = synthetic.all_pairs_upper(len(tracks))
    npairs = int(min(len(pairs), 3.0e10 / (L * L)))
    pairs = pairs[np.random.default_rng(1).permutation(len(pairs))[:npairs]].astype(np.int32)
    for mode in ("tc", "ffma"):
        os.environ["ACOSS_K2_SWEEPS"] = mode
        e = Engine(0); e.set_tracks(frames, offs)
        e.score_pairs(pairs[:256])
        t0 = time.perf_counter(); s = e.score_pairs(pairs); dt = time.perf_counter() - t0
        res[(L, mode)] = (len(pairs) / dt, s)
        e.close()
    same = np.array_equal(res[(L, "tc")][1], res[(L, "ffma")][1])
    print("L=%d pairs=%d  tc %.0f pairs/s  ffma %.0f pairs/s  ratio %.3f  identical %s" % (L, len(pairs), res[(L, "tc")][0], res[(L, "ffma")][0], res[(L, "tc")][0] / res[(L, "ffma")][0], same))
