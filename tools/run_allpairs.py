#!/usr/bin/env python
"""Full all-pairs Serra09 or ChenFusion run of a synthetic BASELINE config on 1..8 GPUs (one process per GPU).

    python tools/run_allpairs.py --config C4s [--algorithm chen]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29511 \
        tools/run_allpairs.py --config C4 [--checkpoint-dir DIR]

The coverid.benchmark sequence (coverid.py:57-70): all_pairwise(symmetric) -> normalize_by_length ->
getEvalStatistics, through the product path acoss_b200.distributed.all_pairwise_distributed: pair list sharded
across ranks by DP cells, one NCCL all_gather of the score slices, matrix assembly and evaluation on rank 0.  A random
sample of pairs is re-scored by the CPU oracle (rank 0) as the parity check at sizes the oracle cannot cover in
full.  --checkpoint-dir saves every finished tile per rank; a re-run with the same arguments resumes from them.
--algorithm chen runs ChenFusion the same way (Qmax and Dmax rows of one CRP per pair, one gather), checks both keys
against the oracle, and adds ChenFusion's late fusion on the GPU (do_late_fusion(impl="gpu")) before evaluating
'qmax', 'dmax' and 'Late'.  Prints one JSON line, with the card's name and power limit.
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _card(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl = [x.strip() for x in out.split(",")]
        return name, pl
    except Exception as e:                                   # noqa: BLE001 - reported, not hidden
        return "unknown (%s)" % e, "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C4s")
    ap.add_argument("--algorithm", default="serra09", choices=["serra09", "chen"],
                    help="Serra09 (Qmax, key 'main') or ChenFusion (keys 'qmax', 'dmax', then the late fusion 'Late')")
    ap.add_argument("--max-tracks", type=int, default=None)
    ap.add_argument("--oracle-sample", type=int, default=256, help="pairs re-scored by the CPU oracle (0 = skip)")
    ap.add_argument("--tile", type=int, default=1 << 18, help="pairs per engine call")
    ap.add_argument("--no-eval", action="store_true")
    ap.add_argument("--checkpoint-dir", default=None)
    ap.add_argument("--align", default="qmax", choices=["qmax", "sw"],
                    help="alignment over the CRPs: Serra09's Qmax, or smith_waterman_constrained (BASELINE configs[1], C2)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    import torch
    import torch.distributed as dist
    from acoss_b200 import synthetic
    from acoss_b200.chenfusion import ChenFusion
    from acoss_b200.distributed import all_pairwise_distributed
    from acoss_b200.engine import ALIGN_QMAX, ALIGN_SW
    from acoss_b200.serra09 import Serra09
    chen = args.algorithm == "chen"
    if chen and args.align != "qmax":
        ap.error("--align applies to Serra09 only (ChenFusion scores Qmax and Dmax)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    t0 = time.perf_counter()
    tracks, labels = synthetic.config_dataset(args.config, max_tracks=args.max_tracks)
    t_gen = time.perf_counter() - t0
    N = len(tracks)
    lens = np.array([len(t) for t in tracks], dtype=np.int64)

    class Plugin(Serra09):                                    # the alignment switch of the C2 configuration
        def params(self, **kw):
            return Serra09.params(self, align=ALIGN_SW if args.align == "sw" else ALIGN_QMAX, **kw)
    if chen:
        Plugin = ChenFusion

    with contextlib.redirect_stdout(sys.stderr):
        # ranks of one box may share the cache prefix: the matrix reaches Ds by a plain assignment on rank 0 only
        alg = Plugin(None, None, features=[dict(hpcp=t, label=str(l)) for t, l in zip(tracks, labels)],
                     downsample_fac=1, shortname="%s_r%d" % (args.config, rank), device=local,
                     cachedir="/tmp/acoss_allpairs_%d" % rank, tile_pairs=args.tile)
    t0 = time.perf_counter()
    alg.engine()
    t_upload = time.perf_counter() - t0

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    sync_all()
    tm = {}
    t0 = time.perf_counter()
    bounds = all_pairwise_distributed(alg, symmetric=True, fill_on=0, checkpoint_dir=args.checkpoint_dir, timings=tm)
    sync_all()
    t_total = time.perf_counter() - t0
    tt = torch.tensor([tm["score_s"], tm["gather_s"], tm["fill_s"], tm["shard_s"]], dtype=torch.float64, device="cuda:%d" % local)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    if rank == 0:
        pairs = alg._pair_array(True)
        cells = int(((lens[pairs[:, 0]] - 9) * (lens[pairs[:, 1]] - 9)).sum())
        out = dict(config=args.config, algorithm=args.algorithm, align=args.align, n_gpus=world, tracks=N,
                   pairs=int(len(pairs)), cells=cells, mean_frames=float(lens.mean()), t_generate_s=t_gen, t_upload_s=t_upload,
                   t_all_pairwise_s=t_total, t_shard_s=float(tt[3]), t_score_s=float(tt[0]), t_gather_s=float(tt[1]),
                   t_fill_s=float(tt[2]), pairs_per_s=len(pairs) / t_total, gcups=cells / t_total / 1e9,
                   pairs_per_s_scoring=len(pairs) / float(tt[0]), gcups_scoring=cells / float(tt[0]) / 1e9,
                   resumed_tiles=tm["resumed_tiles"], tiles_rank0=tm["tiles"], shard_pairs=[int(x) for x in np.diff(bounds)])
        out["card"], out["power_limit"] = _card(local)
        if args.oracle_sample:
            from acoss_b200 import pack_tracks
            from oracle import serra09_c as oc
            frames, offs = pack_tracks(tracks)
            sel = np.random.default_rng(3).permutation(len(pairs))[:args.oracle_sample]
            t0 = time.perf_counter()
            if chen:                                            # both keys, before normalisation
                want = dict(zip(("qmax", "dmax"), oc.chen_pairs(frames, offs, pairs[sel], oc.params(hoist_norms=True),
                                                                 nthreads=os.cpu_count() or 1)))
            elif args.align == "sw":                           # oracle CRP of each sampled pair -> oracle SW
                from oracle import earlyfusion_np as ef
                want = np.array([ef.smith_waterman_constrained_x10(
                    oc.pair(tracks[a], tracks[b], want_debug=True)[1]["crp"]) / 10.0 for a, b in pairs[sel]], np.float32)
            else:
                want = oc.pairs(frames, offs, pairs[sel], oc.params(hoist_norms=True), nthreads=os.cpu_count() or 1)
            if not chen:
                want = dict(main=want)
            same = {k: bool(np.array_equal(w, np.asarray(alg.Ds[k])[pairs[sel, 0], pairs[sel, 1]])) for k, w in want.items()}
            out["oracle_sample"] = dict(pairs=int(len(sel)), identical=all(same.values()),
                                        cpu_s=time.perf_counter() - t0, cores=os.cpu_count())
            if chen:
                out["oracle_sample"]["identical_per_key"] = same
        if not args.no_eval:
            t0 = time.perf_counter()
            alg.normalize_by_length()
            out["t_normalize_s"] = time.perf_counter() - t0

            def evaluate(key):
                t0 = time.perf_counter()
                with contextlib.redirect_stdout(sys.stderr):
                    MR, MRR, MDR, MAP, tops = alg.getEvalStatistics(key)
                return time.perf_counter() - t0, dict(MR1=float(MR), MRR=float(MRR), MDR=float(MDR), MAP=float(MAP),
                                                      tops=[float(x) for x in tops])
            if chen:
                t0 = time.perf_counter()
                alg.do_late_fusion(impl="gpu")
                out["t_fusion_s"] = time.perf_counter() - t0
                out["late_nonfinite"] = int((~np.isfinite(alg.Ds["Late"])).sum())
                out["t_eval_s"], out["eval"] = {}, {}
                for key in ("qmax", "dmax", "Late"):
                    out["t_eval_s"][key], out["eval"][key] = evaluate(key)
            else:
                out["t_eval_s"], out["eval"] = evaluate("main")
        print(json.dumps(out), flush=True)
    alg.cleanup_memmap()
    alg.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
