#!/usr/bin/env python
"""bench.py — all-pairs Serra09 scoring throughput (alignments/s, GCUPS) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch P] [--impl reference]

Workload (BASELINE.json configs[2], "C3"): synthetic 1 000-track Da-TACOS-shaped slice, 12-bin
HPCP, ~2k frames/track, 499 500 unique (i<j) pairs.  A *step* is one pass of the hot path
(K1 OTI -> K2 CRP -> K3 Qmax) over one batch of P consecutive pairs of that pair list; at N>1 the
pair list is sharded across ranks (weak scaling: every rank does K steps of P pairs of its own
shard, no data-path collective) and the per-rank score tiles are gathered with one NCCL
all_gather at the end of the timed region.

Output: ONE JSON line on rank 0 (contract in the task statement), with
  value        device-resident throughput (pairs and scores in HBM, CUDA events, max over ranks)
  e2e          the same metric through the product path at every N: all_pairwise_distributed(Serra09) over the
               WHOLE C3 pair list (strong scaling): host pair tiles in, host score tiles out, NCCL gather of the
               score slices at N > 1, N x N matrix assembled and symmetrised; rank-0 tail timed separately
  roofline     dominant kernel (the emit sweep: tc_emit_kernel) against measured HBM bandwidth (contract view) and, in
               `roofline.binding`, against the instruction-issue roofline that binds it; DRAM traffic and
               lane-instructions per cell come from the committed ncu capture of this build
               (profiles/k2_constants.json); `roofline_alu` keeps the per-stage / per-kernel breakdown
  gather_parity (N > 1) every rank re-scores 64 pairs of another rank's shard against the gathered vector
  cpu_baseline the oracle's plain-C port of the reference CPU path (oracle/serra09_c.c), all host
               threads, on a bounded sample of the same pairs; `hoisted` = the same with the norms hoisted
  c4s          (N=1 only, informational) the pipeline at the realistic ~500-frame track length
  earlyfusion  (N=1 only, informational, after the timed region) the EarlyFusion pair scoring on a covers80-shaped
               slice (BASELINE.json configs[1]): its own e2e, tensor roofline of the float64 DMMA kernel and numpy
               oracle sample (DESIGN.md §4.5); `--no-earlyfusion` skips it
`--impl reference` times that CPU port alone (the reference's essentia path cannot be installed:
DESIGN.md §5) on the same config/metric/unit.
`--dump-outputs DIR` writes the scores of the last timed step to DIR/scores.npy (float32), so that two builds run
with the same arguments, hence on the same pairs, can be compared output for output.
"""
import argparse
import contextlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                                 # the tree bench.py runs from may be read-only
DUMP_LIMIT = 64 << 20                                          # bytes written by --dump-outputs

# Per-pair constants of the dominant kernel (the emit sweep) measured by the committed `ncu --set full` capture of
# THIS build: DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) and executed warp instructions
# (smsp__inst_executed.sum) of one launch divided by its pairs.  profiles/make_constants.py writes the file from the
# .ncu-rep kept beside it; it records the git hash it was taken at.
CONSTANTS_FILE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "k2_constants.json")


def load_constants():
    try:
        with open(CONSTANTS_FILE) as f:
            return json.load(f)
    except Exception:
        return None

METRIC = "all-pairs alignments/sec"
UNIT = "pairs/s"
WORKLOAD = "C3: Serra09 all-pairs, 1000 synthetic tracks x ~2k HPCP frames (499500 unique pairs)"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d.get("hbm_gbs", 6650.0)), "measured", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback", 1965.0


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_dataset():
    from acoss_b200 import pack_tracks, synthetic
    tracks, labels = synthetic.config_dataset("C3")
    frames, offs = pack_tracks(tracks)
    pairs = synthetic.all_pairs_upper(len(tracks))
    lens = np.diff(offs)
    return tracks, labels, frames, offs, pairs, lens


def algorithmic_bytes(lens, pairs, incr=9):
    """SURVEY §8d: 48(n_q+n_r) frames in + M'N'/8 CRP out (K2) + M'N'/8 CRP in (K3) + 4 score."""
    nq = lens[pairs[:, 0]].astype(np.int64); nr = lens[pairs[:, 1]].astype(np.int64)
    cells = (nq - incr) * (nr - incr)
    k2 = 48 * (nq + nr) + cells // 8
    k3 = cells // 8 + 4
    return int(cells.sum()), int(k2.sum()), int(k3.sum())


def earlyfusion_leg(eng, sm_mhz):
    """Secondary, informational leg: the full EarlyFusion pair scoring (acoss_ef_score_pairs: float64 DMMA
    cross-similarity matrices -> getWCSM fusion -> k-NN binarisation -> Smith-Waterman, four scores per pair) on a
    covers80-shaped slice (96 tracks x ~400 beat-synchronous blocks, the reference's block dimensions), host pair
    list in / host scores out, with the numpy oracle timed on a few of the same pairs.  DESIGN.md 4.5."""
    from acoss_b200 import synthetic
    from oracle import earlyfusion_np as ef
    feats = synthetic.ef_dataset([2] * 48, 400, 20242)
    n = len(feats)
    i, j = np.triu_indices(n, k=1)
    pairs = np.stack([i, j], axis=1).astype(np.int32)
    nb = np.array([f["mfccs"].shape[0] for f in feats], dtype=np.int64)
    cells = int((nb[pairs[:, 0]] * nb[pairs[:, 1]]).sum())
    dsum = sum(feats[0][k].shape[1] for k in ("mfccs", "ssms", "chromas"))
    eng.ef_set_tracks(feats)
    eng.ef_score_pairs(pairs[:64])
    eng.ef_score_pairs(pairs)
    eng.set_profiling(True)
    reps, times = 3, []
    for _ in range(reps):
        t0 = time.perf_counter()
        got = eng.ef_score_pairs(pairs)
        times.append(time.perf_counter() - t0)
    ms = eng.ef_stage_ms()
    st = eng.ef_last_stats()
    eng.set_profiling(False)
    csm_tflops = 2.0 * cells * dsum / (ms["csm"] / reps * 1e-3) / 1e12
    peak_tflops = 148 * 64 * 2 * sm_mhz * 1e6 / 1e12            # 64 float64 FMA / clk / SM (DFMA and DMMA alike)
    sel = np.random.default_rng(2).choice(len(pairs), size=6, replace=False)
    t0 = time.perf_counter()
    same = True
    for k in sel:
        w = ef.similarity_pair(feats[pairs[k, 0]], feats[pairs[k, 1]])
        same &= all(got[q, k] == np.float32(w[s]) for q, s in enumerate(("mfccs", "ssms", "chromas", "early")))
    tc = time.perf_counter() - t0
    return {"workload": "EarlyFusion pair scoring: %d tracks x ~400 blocks, dims 1000/1225/480 float32, %d pairs per call"
                        % (n, len(pairs)),
            "e2e": {"value": len(pairs) / min(times), "unit": UNIT, "h2d_bytes_per_step": int(pairs.nbytes),
                    "d2h_bytes_per_step": int(got.nbytes), "api": "Engine.ef_score_pairs (acoss_ef_score_pairs), host buffers"},
            "device_ms_per_call": {k: v / reps for k, v in ms.items()}, "gpu_launches_per_call": st["launches"],
            "roofline": {"bound": "tensor", "kernel": "ef_csm3_kernel (float64 DMMA cross-similarity contraction)",
                         "achieved": csm_tflops, "peak": peak_tflops, "unit": "TFLOP/s", "frac": csm_tflops / peak_tflops,
                         "peak_kind": "nominal float64 rate (64 FMA/clk/SM x 148 SMs) at the sampled SM clock",
                         "traffic": None, "note": "achieved counts 2*M*N*d flops of the pair matrices only (tile padding excluded)"},
            "cpu_baseline": {"value": len(sel) / tc, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                             "sample": "%d pairs through the numpy oracle (BLAS threads), %.1f s" % (len(sel), tc),
                             "parity_on_sample": bool(same)}}


def c4s_leg(device):
    """Informational: the pair pipeline on C4s-shaped tracks (the Da-TACOS clique layout at ~500 frames per track, what
    the x40 median downsampling of a 4-minute song gives: SURVEY 8d), 1 000 tracks, 131 072 random pairs per call, host
    pair list in / host scores out, with a parity sample against the C oracle."""
    from acoss_b200 import Engine, pack_tracks, synthetic
    from oracle import serra09_c as oc
    tracks, labels = synthetic.config_dataset("C4s", max_tracks=1000)
    frames, offs = pack_tracks(tracks)
    pairs = synthetic.all_pairs_upper(len(tracks))
    pairs = pairs[np.random.default_rng(3).permutation(len(pairs))[:131072]].astype(np.int32)
    lens = np.diff(offs)
    cells = int(((lens[pairs[:, 0]] - 9) * (lens[pairs[:, 1]] - 9)).sum())
    with Engine(device) as e2:
        e2.set_tracks(frames, offs)
        e2.score_pairs(pairs[:4096])
        e2.score_pairs(pairs)
        e2.set_profiling(True)
        reps, times = 3, []
        for _ in range(reps):
            t0 = time.perf_counter()
            got = e2.score_pairs(pairs)
            times.append(time.perf_counter() - t0)
        st = e2.last_stats()
        stage = {k: v / reps for k, v in e2.stage_ms().items()}
        kms = {k: v / reps for k, v in e2.kernel_ms().items()}
    sel = np.random.default_rng(4).permutation(len(pairs))[:256]
    want = oc.pairs(frames, offs, pairs[sel], oc.params(hoist_norms=True), nthreads=os.cpu_count() or 1)
    dt = min(times)
    return {"workload": "C4s: Da-TACOS-shaped cliques at ~500 frames per track, 1000 tracks, %d pairs per call" % len(pairs),
            "e2e": {"value": len(pairs) / dt, "unit": UNIT, "h2d_bytes_per_step": int(pairs.nbytes), "d2h_bytes_per_step": int(got.nbytes),
                    "api": "Engine.score_pairs (acoss_score_pairs), host buffers"},
            "gcups": cells / dt / 1e9, "stage_ms_per_call": stage, "k2_kernel_ms_per_call": kms,
            "fallback_pairs": st["fallback_pairs"], "parity_on_sample": bool(np.array_equal(got[sel], want))}


def dump_outputs(dirname, scores):
    """Scores of the last timed step as DIR/scores.npy; above DUMP_LIMIT a fixed, seeded sample of them."""
    scores = np.asarray(scores, dtype=np.float32).reshape(-1)
    if scores.nbytes > DUMP_LIMIT:
        scores = scores[np.sort(np.random.default_rng(0).choice(scores.size, DUMP_LIMIT // 4, replace=False))]
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "scores.npy"), scores)


def run_reference(args, rank, world):
    """--impl reference: the CPU port of the reference path, all host threads, bounded steps."""
    if rank != 0:
        return
    from oracle import serra09_c as oc
    tracks, labels, frames, offs, pairs, lens = build_dataset()
    cores = os.cpu_count() or 1
    per_step = 4 * max(cores, 8)                               # a few seconds of CPU per step
    rng = np.random.default_rng(1234)
    sel = rng.permutation(len(pairs))
    p = oc.params()
    k0 = 0
    for _ in range(max(1, min(args.warmup, 1))):
        oc.pairs(frames, offs, pairs[sel[k0:k0 + per_step]], p, nthreads=cores); k0 += per_step
    t0 = time.perf_counter()
    ncell = 0
    for _ in range(args.steps):
        idx = pairs[sel[k0:k0 + per_step]]; k0 += per_step
        scores = oc.pairs(frames, offs, idx, p, nthreads=cores)
        ncell += algorithmic_bytes(lens, idx)[0]
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, scores)
    val = args.steps * per_step / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "gcups": ncell / dt / 1e9,
            "config": {"workload": WORKLOAD, "pairs_per_step": per_step,
                       "note": "plain-C port of the reference CPU path (essentia ChromaCrossSimilarity + "
                               "CoverSongSimilarity restated; essentia itself is not installable), pthreads over pairs"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d random C3 pairs per step, %d steps" % (per_step, args.steps)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=0, help="pairs per step (0 = auto)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=0, help="pairs in the cpu_baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-earlyfusion", action="store_true", help="skip the secondary EarlyFusion leg")
    ap.add_argument("--crp-path", default="auto", choices=["auto", "exact"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the scores of the last timed step to DIR/scores.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist
    from acoss_b200 import Engine, default_params
    from acoss_b200._lib import CRP_AUTO, CRP_EXACT
    from acoss_b200.serra09 import Serra09
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    hbm_peak, peak_kind, sm_max = load_peaks()

    tracks, labels, frames, offs, pairs, lens = build_dataset()
    P = args.batch or (8192 if args.crp_path == "exact" else 32768)
    total_steps = args.warmup + args.steps
    # shard: rank r owns a contiguous region of a fixed random permutation of the pair list
    perm = np.random.default_rng(99).permutation(len(pairs))
    need = total_steps * P
    if need * world > len(perm):
        perm = np.concatenate([perm] * (need * world // len(perm) + 1))
    mine = pairs[perm[rank * need:(rank + 1) * need]]
    params = default_params(crp_path=CRP_EXACT if args.crp_path == "exact" else CRP_AUTO)

    eng = Engine(local)
    t0 = time.perf_counter()
    eng.set_tracks(frames, offs)
    setup_s = time.perf_counter() - t0
    stream = torch.cuda.ExternalStream(eng.stream_ptr, device=torch.device("cuda", local))
    d_pairs = torch.from_numpy(mine.astype(np.int32)).cuda(local)
    d_scores = torch.zeros(need, dtype=torch.float32, device="cuda:%d" % local)
    gathered = torch.zeros(world * need, dtype=torch.float32, device="cuda:%d" % local) if world > 1 else None

    def step(k):
        eng.score_pairs_device(d_pairs[k * P:(k + 1) * P].data_ptr(), P, d_scores[k * P:(k + 1) * P].data_ptr(), params)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing --------------------------------------------------------------
    for k in range(args.warmup):
        step(k)
    eng.sync()
    eng.set_profiling(True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    try:
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches = 0
        with torch.cuda.stream(stream):
            ev0.record(stream)
            for k in range(args.warmup, total_steps):
                step(k)
                launches += eng.last_stats()["launches"]
            if world > 1:
                dist.all_gather_into_tensor(gathered, d_scores)      # NCCL gather of the per-rank score tiles
            ev1.record(stream)
        eng.sync()
        barrier()
    finally:
        clocks = sampler.stop() if rank == 0 else None           # the sampler process must not outlive a failed run
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        last = slice((total_steps - 1) * P, total_steps * P)
        dump_outputs(args.dump_outputs, (gathered.view(world, need)[:, last] if world > 1 else d_scores[last]).cpu().numpy())
    stage = eng.stage_ms()
    kernel_ms_timed = eng.kernel_ms()
    k2_debug = eng.debug_counters()                            # of the last timed step
    fallback_timed = eng.last_stats()["fallback_pairs"]
    eng.set_profiling(False)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda:%d" % local)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    timed = mine[args.warmup * P: total_steps * P]
    cells, bytes_k2, bytes_k3 = algorithmic_bytes(lens, timed)
    value = world * args.steps * P / (ms_max / 1e3)
    gcups = world * cells / (ms_max / 1e3) / 1e9

    # ---- gather parity (N > 1): every rank re-scores a sample of ANOTHER rank's shard ----------------------
    gather_parity = None
    if world > 1:
        other = (rank + 1) % world
        theirs = pairs[perm[other * need:(other + 1) * need]]
        sel = args.warmup * P + np.random.default_rng(100 + rank).permutation(args.steps * P)[:64]
        mine_of_theirs = eng.score_pairs(theirs[sel].astype(np.int32), params)
        got = gathered[other * need:(other + 1) * need].cpu().numpy()[sel]
        ok = torch.tensor([1 if np.array_equal(mine_of_theirs, got) else 0], dtype=torch.int32, device="cuda:%d" % local)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        gather_parity = bool(int(ok.item()))

    # ---- end to end: the product path, all_pairwise_distributed over the WHOLE C3 pair list (strong scaling) -----
    # host pair tiles in, host score tiles out (acoss_score_pairs), NCCL gather of the score slices, assembly of the
    # N x N matrix and its symmetrisation; then the reference's tail on rank 0 (normalize_by_length, getEvalStatistics)
    from acoss_b200.distributed import all_pairwise_distributed
    feats = [dict(hpcp=t_, label=str(l)) for t_, l in zip(tracks, labels)]
    workdir = tempfile.mkdtemp(prefix="acoss_bench_")          # score memmap and results csv of the plugin
    with contextlib.redirect_stdout(sys.stderr):               # keep stdout to the one JSON line
        alg = Serra09(None, None, features=feats, downsample_fac=1, shortname="bench%d" % rank, device=local,
                      cachedir=os.path.join(workdir, "cache"), engine=eng, tile_pairs=P)
    alg._resident = True                                       # tracks already resident in this engine
    alg.crp_path = params.crp_path
    alg.similarity(pairs[:4096].astype(np.int64))              # warm-up of the host path (pinned staging, allocations)
    alg.Ds["main"][:, :] = 0
    barrier()
    te0 = time.perf_counter()
    all_pairwise_distributed(alg, symmetric=True)
    torch.cuda.synchronize()
    te = time.perf_counter() - te0
    t = torch.tensor([te], dtype=torch.float64, device="cuda:%d" % local)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    e2e_val = len(pairs) / e2e_s
    tail = None
    if rank == 0:
        with contextlib.redirect_stdout(sys.stderr), contextlib.chdir(workdir):   # results csv goes to the CWD
            tt0 = time.perf_counter()
            alg.normalize_by_length()
            tt1 = time.perf_counter()
            MR, MRR, MDR, MAP, tops = alg.getEvalStatistics("main")
            tt2 = time.perf_counter()
        tail = {"normalize_by_length_s": tt1 - tt0, "getEvalStatistics_s": tt2 - tt1, "MAP": float(MAP), "MR1": float(MR)}
    alg.cleanup_memmap()
    shutil.rmtree(workdir, ignore_errors=True)

    # ---- roofline of the dominant kernel (the emit sweep, which writes the bit-packed CRP) ---------------------------
    k2_ms = stage["k2_crp"]
    k3_ms = stage["k3_dp"]
    emit_ms = stage.get("k2_emit", 0.0)
    emit_launches = max(1, eng.last_stats().get("chunks", 1)) * args.steps
    # Algorithmic bytes of one launch (DESIGN.md 4.2): 48 (n_q + n_r) frame bytes in + M'N'/8 CRP bytes out per pair.
    ach_gbs = bytes_k2 / (emit_ms / 1e3) / 1e9 if emit_ms > 0 else None
    sm_mhz = (clocks or {}).get("sm_mhz") or sm_max
    issue_peak = 148 * 128 * sm_mhz * 1e6                      # lane-instructions / s: 4 schedulers x 32 lanes x 148 SMs
    fp32_peak = 2 * issue_peak                                 # flop / s: one FMA per lane and clock
    pairs_per_launch = args.steps * P / emit_launches
    consts = load_constants() or {}
    ce = consts.get("emit", {})
    emit_s = emit_ms / 1e3
    traffic = int(ce["dram_bytes_per_pair"] * pairs_per_launch) if "dram_bytes_per_pair" in ce else None
    lane_inst = ce.get("lane_inst_per_cell")
    binding = None
    if emit_s > 0:
        # tensor view of the same launch: 30 tcgen05.mma (M 128 x N 64 x K 32 bytes, u8 x u8 -> s32) per block of 128 x 64 cells
        int8_ops_per_cell = 30 * 2 * 32
        int8_peak = 4.5e15                                       # nominal dense int8 (B200_PROFILING.md has no measured int8 figure)
        binding = {"kind": "instruction issue of the consumer warps (per cell: item from three TMEM accumulators, two zone "
                           "tests, one ballot; the items themselves come from the tensor cores: `tensor` view)",
                   "tensor": {"int8_ops_per_cell": int8_ops_per_cell, "achieved_tops": int8_ops_per_cell * cells / emit_s / 1e12,
                              "peak_tops": int8_peak / 1e12, "frac": int8_ops_per_cell * cells / emit_s / int8_peak,
                              "peak_kind": "nominal dense int8; an N = 64 MMA takes ~51 cycles against a 32-cycle pipe floor "
                                           "(profiles/r2_umma_probe.md), so ~0.6 of it is reachable at this tile shape"},
                   "achieved_lane_inst_per_s": (lane_inst * cells / emit_s) if lane_inst else None,
                   "peak_lane_inst_per_s": issue_peak,
                   "frac": (lane_inst * cells / emit_s / issue_peak) if lane_inst else None,
                   "lane_inst_per_cell": lane_inst,
                   "fp32": {"flop_per_cell": 30, "achieved_tflops": 30 * cells / emit_s / 1e12,
                            "peak_tflops": fp32_peak / 1e12, "frac": 30 * cells / emit_s / fp32_peak,
                            "peak_kind": "nominal: 148 SMs x 128 lanes x 2 flop at the sampled SM clock (no measured FP32 peak)"},
                   "constants_from": consts.get("source"), "constants_git": consts.get("git")}
    roofline = {"bound": "hbm", "kernel": ce.get("kernel", "tc_emit_kernel") + " (K2 emit sweep)", "achieved": ach_gbs, "peak": hbm_peak,
                "unit": "GB/s", "frac": (ach_gbs / hbm_peak) if ach_gbs else None,
                "traffic": traffic,
                "traffic_source": consts.get("source"),
                "peak_kind": peak_kind + " (MEASURED_PEAKS.json hbm_gbs, sustained copy)" if peak_kind == "measured" else peak_kind,
                "algorithmic_bytes_per_launch": int(bytes_k2 / emit_launches),
                "launches": emit_launches, "ms_per_launch": emit_ms / emit_launches,
                "k2_stage_ms_per_step": k2_ms / args.steps, "emit_share_of_step": emit_ms / ms,
                "binding": binding,
                "note": "no float CSM ever reaches HBM, so the HBM fraction is small by design; `binding` is the roofline that binds"}
    roofline_alu = {"k2_cells_per_s": cells / (k2_ms / 1e3) if k2_ms > 0 else None,
                    "k3_cells_per_s": cells / (k3_ms / 1e3) if k3_ms > 0 else None,
                    "issue_peak_lane_ops_per_s": issue_peak,
                    "k2_lane_ops_per_cell_at_peak": issue_peak / (cells / (k2_ms / 1e3)) if k2_ms > 0 else None,
                    "k3_frac_of_5op_int_roofline": (5 * cells / (k3_ms / 1e3)) / issue_peak if k3_ms > 0 else None,
                    "emit_cells_per_s": cells / (emit_ms / 1e3) if emit_ms > 0 else None,
                    "k2_kernel_ms_per_step": {k: v / args.steps for k, v in kernel_ms_timed.items()},
                    "stage_share": {"k1": stage["k1_oti"] / ms, "k2": k2_ms / ms, "k3": k3_ms / ms,
                                    "k2_emit": emit_ms / ms}}

    # ---- CPU baseline (rank 0, N=1): bounded sample of the same pairs --------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import serra09_c as oc
        cores = os.cpu_count() or 1
        n_s = args.cpu_sample or max(cores, 8) * 10              # about 10-15 s of CPU work
        idx = timed[np.random.default_rng(5).permutation(len(timed))[:n_s]]
        tc0 = time.perf_counter()
        ref_scores = oc.pairs(frames, offs, idx, oc.params(), nthreads=cores)
        tc = time.perf_counter() - tc0
        # parity spot check on the sample: GPU scores must equal the oracle's
        got = eng.score_pairs(idx.astype(np.int32), params)
        # the same port with the norms hoisted out of the cell loop (essentia re-evaluates a.a and b.b for every cell;
        # hoisting them is the first thing a CPU optimiser would do): reported beside the essentia-shaped number
        n_h = max(cores, 8) * 4
        th0 = time.perf_counter()
        hs = oc.pairs(frames, offs, idx[:n_h], oc.params(hoist_norms=True), nthreads=cores)
        th = time.perf_counter() - th0
        cpu = {"value": n_s / tc, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "%d random pairs of the timed C3 batches, %.1f s of CPU" % (n_s, tc),
               "gcups": algorithmic_bytes(lens, idx)[0] / tc / 1e9,
               "parity_on_sample": bool(np.array_equal(got, ref_scores)),
               "hoisted": {"value": n_h / th, "unit": UNIT, "gcups": algorithmic_bytes(lens, idx[:n_h])[0] / th / 1e9,
                           "sample": "%d of the same pairs, norms hoisted, %.1f s" % (n_h, th),
                           "same_scores": bool(np.array_equal(hs, ref_scores[:n_h]))}}

    # ---- secondary workload: the realistic track length (C4s: ~500 frames = a 4-minute song after the x40 median) ----
    c4s_line = None
    if rank == 0 and world == 1:
        try:
            c4s_line = c4s_leg(local)
        except Exception as e:
            c4s_line = {"error": "%s: %s" % (type(e).__name__, e)}

    # ---- secondary workload (not the headline): EarlyFusion pair scoring, BASELINE.json configs[1] shape ----
    ef_line = None
    if rank == 0 and world == 1 and not args.no_earlyfusion:
        try:
            ef_line = earlyfusion_leg(eng, (clocks or {}).get("sm_mhz") or sm_max)
        except Exception as e:                                  # never let the extra leg break the headline line
            ef_line = {"error": "%s: %s" % (type(e).__name__, e)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32+s16x2", "data": "synthetic",
                "gcups": gcups,
                "config": {"workload": WORKLOAD, "pairs_per_step": P, "crp_path": args.crp_path,
                           "sharding": "pair list sharded across ranks, NCCL all_gather of score tiles" if world > 1 else "single GPU",
                           "l2": "inputs larger than L2: each step streams >= %.1f GB of CRP scratch" % (bytes_k2 / args.steps / 1e9),
                           "track_upload_s": setup_s},
                "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(P * 8), "d2h_bytes_per_step": int(P * 4),
                        "api": "acoss_b200.distributed.all_pairwise_distributed(Serra09) over the whole C3 pair list: host pair "
                               "tiles of %d in / host score tiles out (acoss_score_pairs), score slices gathered (NCCL at N > 1), "
                               "N x N matrix assembled and symmetrised into Ds" % P,
                        "scaling": "strong", "pairs": int(len(pairs)), "seconds": e2e_s,
                        "rank0_tail": tail},
                "gather_parity": gather_parity,
                "gpu_launches": int(launches),
                "clocks": clocks, "roofline": roofline, "roofline_alu": roofline_alu, "cpu_baseline": cpu,
                "fallback_pairs": fallback_timed, "k2_debug": k2_debug,
                "c4s": c4s_line, "earlyfusion": ef_line}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if gather_parity is False:
        raise SystemExit("gather parity FAILED: a rank's re-scored sample differs from the gathered score vector")


if __name__ == "__main__":
    main()
