"""Write tc_requeue_counts.json: the dense-level debug counters of tests/test_gpu_tc_requeue.py's call (needs a B200).

Generated with the build that ran an item's second dense level straight after its first one inside the same CTA
(git e6744ff); the re-queue must count the same items and lines.
usage: python tests/golden/make_tc_requeue_counts.py [OUT]"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

import test_gpu_tc_requeue as t  # noqa: E402
from acoss_b200 import Engine  # noqa: E402

out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, t.GOLDEN)
tracks, pairs = t.dataset()
with Engine(0) as eng:
    _, _, got, st, counters = t.tc_run(eng, tracks, pairs)
with open(out, "w") as f:
    json.dump({"note": "acoss_debug_counters of test_gpu_tc_requeue.dataset() with ACOSS_K2_SWEEPS=tc: per orientation "
                       "and dense level (items, live lines, bracket misses, lines left), sparse (warps, lines left)",
               "fallback_pairs": int(st["fallback_pairs"]), "counters": counters}, f, indent=1)
print(out, counters)
