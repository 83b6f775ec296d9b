"""GPU box: time the Serra09 pair pipeline of the library build on a synthetic configuration.

    python tools/k2_time.py [--config C3] [--tracks 400] [--pairs 8192] [--reps 3] [--check]

Prints one JSON line: pairs/s, GCUPS, per-stage device ms (CUDA events), fallback pairs, diagnostic counters.
--check compares the scores of the first 256 pairs with the exact CRP path."""
import argparse, json, os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from acoss_b200 import Engine, pack_tracks, synthetic, default_params
from acoss_b200._lib import CRP_EXACT, LIB_PATH

ap = argparse.ArgumentParser()
ap.add_argument("--config", default="C3")
ap.add_argument("--tracks", type=int, default=400)
ap.add_argument("--pairs", type=int, default=8192)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--check", action="store_true")
ap.add_argument("--tag", default="")
a = ap.parse_args()
tracks, labels = synthetic.config_dataset(a.config, max_tracks=a.tracks)
frames, offs = pack_tracks(tracks)
pairs = synthetic.all_pairs_upper(len(tracks))
rng = np.random.default_rng(7)
pairs = pairs[rng.permutation(len(pairs))[:a.pairs]].astype(np.int32)
lens = np.diff(offs)
cells = int(((lens[pairs[:, 0]] - 9) * (lens[pairs[:, 1]] - 9)).sum())
with Engine(0) as eng:
    eng.set_tracks(frames, offs)
    eng.score_pairs(pairs[:512])                       # warm-up (allocations, module load)
    eng.score_pairs(pairs)
    eng.set_profiling(True)
    t0 = time.time()
    for _ in range(a.reps):
        s = eng.score_pairs(pairs)
    dt = (time.time() - t0) / a.reps
    ms = {k: v / a.reps for k, v in eng.stage_ms().items()}
    kms = {k: round(v / a.reps, 3) for k, v in eng.kernel_ms().items()}
    st = eng.last_stats()
    out = dict(tag=a.tag or os.path.basename(LIB_PATH), config=a.config, pairs=len(pairs), cells=cells, pairs_per_s=len(pairs) / dt,
               gcups=cells / dt / 1e9, stage_ms=ms, kernel_ms=kms, fallback=st["fallback_pairs"], chunks=st["chunks"],
               dbg=eng.debug_counters())
    if a.check:
        se = eng.score_pairs(pairs[:256], default_params(crp_path=CRP_EXACT))
        out["mismatch_vs_exact"] = int((se != s[:256]).sum())
print(json.dumps(out))
