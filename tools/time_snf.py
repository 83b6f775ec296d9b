#!/usr/bin/env python
"""Time the similarity-network fusion (acoss_snf, k7_snf.cu) on one B200 at the benchmark's size, and the numpy
oracle on the host for the CPU comparison.

    python tools/time_snf.py [--n 15000] [--cpu-n 4000] [--niters 20] [--out profiles/r5_snf_time.json]

Inputs: seeded clique-structured float32 distance matrices (oracle/snf_np.py clique_distances), K = 20, reg_diag = 1,
reg_neighbs = 0.5, the reference's aliasing (L1 default).  Shapes: two matrices (ChenFusion's Ds["Late"]), three and
four (EarlyFusion's "late" and "early+late").  Each shape is run once to warm up, then timed with the library's CUDA
events: H2D of the score matrices, affinity (DSym, W, P, S), diffusion (per iteration and per step, one step being
one matrix of one iteration), final average plus D2H of the fused matrix.  Two models from the shapes, per step:
HBM bytes (n_mats + 4) * 8 * N^2 over 7.7 TB/s, and bytes gathered from L2 by the two sparse products, 2 * K * 8 * N^2.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BPS = 7.7e12


def _card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl, clk = [x.strip() for x in out.split(",")]
        return name, pl, clk
    except Exception as e:                                   # noqa: BLE001 - reported, not hidden
        return "unknown (%s)" % e, "unknown", "unknown"


def cpu_oracle(n, K, seed=0):
    """One affinity pass and one diffusion iteration of the numpy oracle over two matrices, host seconds."""
    from oracle import snf_np as snf
    Ds, _ = snf.clique_distances(n, 2, seed=seed)
    t = time.perf_counter()
    Ws = [snf.getW(D, K) for D in Ds]
    Ps = [snf.getP(W) for W in Ws]
    Ss = [snf.getS(W, K) for W in Ws]
    t_aff = time.perf_counter() - t
    t = time.perf_counter()
    snf.diffuse(Ps, Ss, 1)
    return dict(n=n, n_mats=2, affinity_s=t_aff, iteration_s=time.perf_counter() - t, host_cpus=os.cpu_count())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=15000)
    ap.add_argument("--cpu-n", type=int, default=4000)
    ap.add_argument("--niters", type=int, default=20)
    ap.add_argument("--K", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_snf_time.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("time_snf.py measures the GPU: no CUDA device")
    from acoss_b200 import Engine
    from oracle import snf_np as snf

    name, power_limit, max_sm_clock = _card()
    n, K = a.n, a.K
    Ds, _ = snf.clique_distances(n, 4, seed=1)
    res = dict(card=name, power_limit=power_limit, max_sm_clock=max_sm_clock, n=n, K=K, niters=a.niters,
               shapes=[])
    with Engine(0) as eng:
        for n_mats in (2, 3, 4):
            mats = Ds[:n_mats]
            eng.snf(mats, K, 1)                                # warm-up of this shape
            eng.set_profiling(True)
            t = time.perf_counter()
            out = eng.snf(mats, K, a.niters, 1, 0.5)
            wall = time.perf_counter() - t
            ms = eng.snf_stage_ms()
            eng.set_profiling(False)
            step_ms = ms["diffusion"] / (a.niters * n_mats)
            hbm = (n_mats + 4) * 8.0 * n * n
            l2 = 2.0 * K * 8.0 * n * n
            row = dict(n_mats=n_mats, wall_s=wall, h2d_ms=ms["h2d"], affinity_ms=ms["affinity"],
                       diffusion_ms=ms["diffusion"], iteration_ms=ms["diffusion"] / a.niters, step_ms=step_ms,
                       average_d2h_ms=ms["average_d2h"], hbm_bytes_per_step=hbm,
                       hbm_model_ms_per_step=hbm / HBM_BPS * 1e3, hbm_share_of_step=hbm / HBM_BPS * 1e3 / step_ms,
                       l2_gather_bytes_per_step=l2, l2_gather_tb_s=l2 / (step_ms * 1e-3) / 1e12,
                       fused_finite=bool(np.isfinite(out["fused"]).all()))
            row["binds"] = ("HBM" if row["hbm_share_of_step"] > 0.7 else
                            "not HBM (%.0f %% of the step); the L2 gathers run at %.1f TB/s"
                            % (100 * row["hbm_share_of_step"], row["l2_gather_tb_s"]))
            res["shapes"].append(row)
            print(json.dumps(row), flush=True)
    res["cpu_oracle"] = cpu_oracle(a.cpu_n, K)
    print(json.dumps(res["cpu_oracle"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
