#!/usr/bin/env python3
"""Benchmark of the one hot path: HC path tracking of the trifocal_2op1p_30x30 RANSAC round.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--hyp H] [--abort] [--dump-outputs DIR]

One "step" = one RANSAC round: H hypotheses x 312 homotopy paths tracked in one launch per GPU
(BASELINE.json configs[1]: the full default run — H = 100 = NUM_OF_RANSAC_ITERATIONS, 80 max steps, 3 corrections,
no early abort, positive-depth pruning on as in the reference GPU kernels; dataset file 000, sampler seed 0).
N > 1 (torchrun, one process per GPU): every rank tracks its own 100 hypotheses of a 100*N-hypothesis round,
sharded contiguously exactly like sub_RANSAC_iters (reference GPU_HC_Solver.cpp:85-88) -> weak scaling.  At every N a step is
track -> device-side scoring of the round (hcb200_score_tracks) -> one 128-byte best-pose record per GPU -> gather of those
records -> arg-max (hcb200_reduce_pose_records): the only exchange is that gather (NCCL all_gather; the host-side alternative
is timed beside it and reported under `gather`).  Extra legs in the same JSON line: `strong_scaling` (ONE 10 000- and one
100 000-hypothesis round split over the N GPUs), `host_class` (the C++ GPU_HC_Solver with Num_Of_GPUs = N in one process,
flags checked against the committed golden), `ref_gpu` (the reference's own GPU kernels on the same GPU, N = 1).

Prints ONE JSON line (rank 0).  `value` = hypotheses/s with inputs resident in HBM, timed with CUDA events on the
launch stream; `e2e` = the same through host buffers (H2D of the parameters + launch + D2H of every end point and flag,
what GPU_HC_Solver::Solve_by_GPU_HC does, reference GPU_HC_Solver.cpp:335-362,449-460).
`--impl reference` times the reference's own CPU-HC (oracle/_ref, built from /root/reference) on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_PRED_STAGE = 91312.0     # SURVEY.md §8(d): lerp + Hx + Ht + 30x30 complex solve + update
FLOPS_CORR_STAGE = 90874.0     #                   Hx + H + solve + update
NOMINAL_FP32_TFLOPS = 74.4     # 148 SMs x 128 lanes x 2 flop x 1.965 GHz

# Executed FP32 work of the FINAL kernel, from its ncu capture (profiles/ncu_r2.md): thread-level FFMA/FMUL/FADD executed per HC stage
# (smsp__sass_thread_inst_executed_op_f{fma,mul,add}_pred_on.sum / stages; an FMA counts 2 flop) — what the FP32 pipe really did,
# beside the dense-LU model above, which also counts the structural zeros the kernel skips.
EXEC_FLOP_PER_STAGE = 54772.0
EXEC_SOURCE = "profiles/ncu_r2.md: executed FP32 thread instructions of the final kernel per HC stage (FMA = 2 flop), x stages / kernel time"
TRAFFIC_BYTES_H100 = 821760
TRAFFIC_SOURCE = ("dram__bytes_read.sum + dram__bytes_write.sum of one tracker launch of the default round, ncu --set full capture of the final "
                  "kernel (profiles/ncu_r2.md); the 7.8 MB of results stay in the 126 MB L2, so traffic < algorithmic bytes")


def _rank_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        load = [s for s, p in zip(sm, power) if p >= 0.5 * max(power)] or sm
        return {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": float(max(power))}


def reference_arm(args):
    """Reference CPU-HC (unmodified sources, oracle/_ref) on all host cores; bounded sample per step."""
    rank, _, world = _rank_env()
    if rank != 0:
        return 0
    from oracle import pyoracle
    from trifocal_pose_estimation_using_improved_gpuhc_b200 import fixtures
    cores = os.cpu_count() or 1
    sample = args.ref_hyp
    line = {"impl": "reference", "metric": "RANSAC hypotheses/s (312 HC paths each)", "unit": "hypotheses/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "c64", "data": "synthetic",
            "config": {"workload": "trifocal_2op1p_30x30 default RANSAC round: 100 hypotheses x 312 paths per GPU, 80 max steps, "
                                   "3 corrections, pruning on, early abort off, dataset Synthetic/000, seed 0",
                       "sample_hypotheses_per_step": sample,
                       "note": "bounded sample of that round; the reference CPU-HC has no path pruning (SURVEY.md App. E-8)"}}
    try:
        ref = pyoracle.ReferenceCPU()
        kind = "reference"
    except (FileNotFoundError, OSError):
        ref = None
        kind = "port"
    with tempfile.TemporaryDirectory() as tmp:
        times = []
        if ref is not None:
            bindir = fixtures.materialize_tree(tmp, files=[0])
            for i in range(args.warmup + args.steps):
                _, _, _, _, sec = ref.run(bindir, sample, seed=0, dataset_index=0, n_cores=cores)
                if i >= args.warmup:
                    times.append(sec)
        else:
            prob, rs = fixtures.load_problem(), fixtures.load_ransac(0)
            orc = pyoracle.Oracle(prob)
            tgt, dif, _ = orc.prepare_target_params(0, sample, rs["locations"], rs["tangents"])
            for i in range(args.warmup + args.steps):
                t0 = time.perf_counter()
                orc.track(tgt, dif, prune=False, n_threads=cores)
                if i >= args.warmup:
                    times.append(time.perf_counter() - t0)
    t = float(np.mean(times))
    v = sample / t
    line.update({"value": v, "ms_per_step": t * 1e3, "paths_per_s": v * 312,
                 "cpu_baseline": {"value": v, "unit": "hypotheses/s", "cores": cores, "kind": kind,
                                  "sample": "first %d hypotheses of the seed-0 round, OpenMP over paths, %d threads" % (sample, cores)},
                 "e2e": {"value": v, "unit": "hypotheses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                 "gpu_launches": 0})
    print(json.dumps(line))
    return 0


def cpu_baseline_leg(sample_hyp):
    from oracle import pyoracle
    from trifocal_pose_estimation_using_improved_gpuhc_b200 import fixtures
    cores = os.cpu_count() or 1
    try:
        ref = pyoracle.ReferenceCPU()
        with tempfile.TemporaryDirectory() as tmp:
            bindir = fixtures.materialize_tree(tmp, files=[0])
            _, _, _, _, sec = ref.run(bindir, sample_hyp, seed=0, dataset_index=0, n_cores=cores)
        kind = "reference"
    except (FileNotFoundError, OSError):
        prob, rs = fixtures.load_problem(), fixtures.load_ransac(0)
        orc = pyoracle.Oracle(prob)
        tgt, dif, _ = orc.prepare_target_params(0, sample_hyp, rs["locations"], rs["tangents"])
        t0 = time.perf_counter()
        orc.track(tgt, dif, prune=False, n_threads=cores)
        sec = time.perf_counter() - t0
        kind = "port"
    return {"value": sample_hyp / sec, "unit": "hypotheses/s", "cores": cores, "kind": kind, "seconds": sec,
            "sample": "first %d hypotheses of the seed-0 round (%d paths), no pruning (reference CPU-HC), %d threads"
                      % (sample_hyp, sample_hyp * 312, cores)}


def ref_gpu_leg(prob, rs, target, diff, H, abort):
    """The reference's own GPU-HC++ kernel (unmodified sources compiled for sm_100a with a MAGMA shim, SURVEY.md App. D.3) on the
    same round, same GPU, timed launch->sync with CUDA events like multi_GPUs_time; tracks are re-loaded outside the timing."""
    import torch
    from oracle import pyoracle
    if not os.path.exists(pyoracle.REF_GPU_SO):
        return None
    ref = pyoracle.ReferenceGPU(prob, device="cuda:%d" % torch.cuda.current_device())
    ref.setup(target, diff, rs["locations"], rs["K"])
    ts = []
    for i in range(5):
        ref.reload()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ref.track_abort() if abort else ref.track()
        b.record()
        b.synchronize()
        if i >= 2:
            ts.append(a.elapsed_time(b))
    tr, cv, inf = ref.results()
    ms = float(np.mean(ts))
    return {"what": "reference GPU-HC++ kernel (…TrunPaths%s.cu) built for sm_100a, same inputs" % ("_TrunRANSAC" if abort else ""),
            "ms_per_step": ms, "value": H / (ms * 1e-3), "unit": "hypotheses/s",
            "result": {"converged": int(cv.sum()), "infinity": int(inf.sum())}}


def host_class_leg(n_gpus, abort):
    """GPU_HC_Solver (C++ host class, lib/libhcb200_host.so) with Num_Of_GPUs = n_gpus in ONE process: the reference's own multi-GPU
    scheme (GPU_HC_Solver.cpp:85-88, 390-506).  The default round's stacked flags must equal the committed 1-GPU oracle golden."""
    from trifocal_pose_estimation_using_improved_gpuhc_b200 import fixtures
    from trifocal_pose_estimation_using_improved_gpuhc_b200.host_solver import HostSolver
    out = {"n_gpus": n_gpus}
    with tempfile.TemporaryDirectory() as tmp:
        fixtures.materialize_tree(tmp, files=[0])
        s = HostSolver(tmp, "Num_Of_GPUs=%d%s" % (n_gpus, ";Abort_RANSAC_by_Good_Sol=true" if abort else ""))
        r = s.round()                      # warm-up round (module load, allocations)
        secs = []
        for _ in range(3):
            r = s.round()
            secs.append(r["seconds"])
        s.close()
        out.update({"hypotheses": int(r["H"]), "multi_GPUs_time_ms": float(np.mean(secs)) * 1e3,
                    "value": r["H"] / float(np.mean(secs)), "unit": "hypotheses/s",
                    "totals_conv_real_inf": [int(v) for v in r["totals"]], "selected_path": int(r["selected_path"]),
                    "selected_support": [int(v) for v in r["selected_support"]], "pose_found": int(r["pose_found"])})
        gpath = os.path.join(ROOT, "tests", "golden", "oracle_seed0_h100_prune.npz")
        if not abort and os.path.exists(gpath) and r["H"] == 100:
            g = np.load(gpath)
            out["flags_equal_1gpu_golden"] = bool(np.array_equal(np.packbits(r["conv"]), g["converged_bits"]) and
                                                  np.array_equal(np.packbits(r["inf"]), g["infinity_bits"]))
        # the same class on a 10 000-hypothesis round split over the GPUs (results stay on the host side of the class)
        s = HostSolver(tmp, "Num_Of_GPUs=%d;Num_Of_RANSAC_Iterations=10000" % n_gpus)
        r = s.round(fetch=False)
        r = s.round(fetch=False)
        s.close()
        out["h10000"] = {"multi_GPUs_time_ms": r["seconds"] * 1e3, "value": 10000 / r["seconds"], "unit": "hypotheses/s"}
        if n_gpus > 1:
            # early abort on a 10 000-hypothesis round: the reference's per-GPU flag against the flag shared over NVLink peer mappings
            ab = {}
            for key, ov in (("per_gpu_flag", ""), ("shared_flag", ";Abort_Across_GPUs=true")):
                s = HostSolver(tmp, "Num_Of_GPUs=%d;Num_Of_RANSAC_Iterations=10000;Abort_RANSAC_by_Good_Sol=true%s" % (n_gpus, ov))
                s.round(fetch=False)
                secs = [s.round(fetch=False)["seconds"] for _ in range(3)]
                r = s.round(fetch=False)
                s.close()
                ab[key] = {"ms": float(np.mean(secs)) * 1e3, "pose_found": int(r["pose_found"]), "first_passing_path": int(r["best"][1]),
                           "paths_converged_before_stop": int(r["totals"][0])}
            out["abort_h10000"] = ab
    return out


def abort_compare_leg(trk, prob, rs, H, prune):
    """BASELINE.json configs[2]: Abort_RANSAC_by_Good_Sol = true.  Both kernels, same inputs: sampler seed 0 (the ground-truth pose sits in
    hypothesis 0) and a late-hit seed (first passing hypothesis around 30 of 100, profiles/abort_seeds_r1.txt)."""
    import torch
    from oracle import pyoracle
    from trifocal_pose_estimation_using_improved_gpuhc_b200 import hc
    out = {}
    for seed in (0, 13):
        picked = hc.sample_hypotheses(seed, H, rs["locations"].shape[0])
        target, diff = hc.target_params_from_picks(picked, rs["locations"], rs["tangents"], prob["start_params"])
        trk.upload_params(target, diff)
        ts = []
        for i in range(5):
            a, b = _events(torch, 2)
            a.record(); trk.track_abort(H, prune=prune); b.record(); b.synchronize()
            if i >= 2:
                ts.append(a.elapsed_time(b))
        best = trk.d_best.cpu().numpy()
        ours = {"ms": float(np.mean(ts)), "found": int(best[0]), "first_passing_path": int(best[1]), "inliers": [int(best[2]), int(best[3])]}
        ref = pyoracle.ReferenceGPU(prob, device="cuda:%d" % torch.cuda.current_device())
        ref.setup(target, diff, rs["locations"], rs["K"])
        tr = []
        for i in range(4):
            ref.reload(); torch.cuda.synchronize()
            a, b = _events(torch, 2)
            a.record(); ref.track_abort(); b.record(); b.synchronize()
            if i >= 1:
                tr.append(a.elapsed_time(b))
        ref.results()
        idx = ref.d_found_index.cpu().numpy()
        hits = idx[idx >= 0]
        out["seed%d" % seed] = {"ours": ours, "reference": {"ms": float(np.mean(tr)), "found": int(bool(ref.d_found.cpu()[0])),
                                                           "first_passing_path": int(hits.min()) if len(hits) else -1},
                                "speedup": float(np.mean(tr)) / ours["ms"]}
    return out


def _events(torch, n):
    return [torch.cuda.Event(enable_timing=True) for _ in range(n)]


DUMP_BYTES = 63 * 1000 * 1000      # per-path arrays of all ranks together; leaves room under 64 MB for the pose record and .npy headers


def dump_outputs(out_dir, rank, world, tracks, conv, inf, stats, support, rec):
    """What the last timed step handed its caller, as DIR/<name>.npy (float32 / float64, values exact): per path the end point
    (re, im of the 31 entries), converged / infinity flags, the step counters and, when scored, the (inliers21, inliers31) support;
    and the round's selected pose record.  Inputs are seeded, so two builds can be compared file for file.  With N GPUs every rank
    writes its own shard as <name>_rank<k>.npy and rank 0 alone the pose record, which all ranks share.  Above DUMP_BYTES / N per rank
    the per-path arrays are a fixed (seed 0) sample of the rank's paths, in path order; path_index holds the path ids either way."""
    n = tracks.shape[0]
    per_path = 31 * 2 * 4 + 4 + 4 + stats.shape[1] * 8 + 8 + (2 * 4 if support is not None else 0)
    keep = DUMP_BYTES // world // per_path
    idx = np.arange(n) if n <= keep else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    arrays = {"path_index": idx.astype(np.float64),
              "tracks": np.stack([tracks[idx].real, tracks[idx].imag], -1).astype(np.float32),
              "converged": conv[idx].astype(np.float32), "infinity": inf[idx].astype(np.float32),
              "stats": stats[idx].astype(np.float64)}
    if support is not None:
        arrays["support"] = support[idx].astype(np.float32)
    suffix = "" if world == 1 else "_rank%d" % rank
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)
    if rank == 0:
        pose = [rec["found"], rec["inliers21"], rec["inliers31"], rec["n_candidates"], rec["abort_flag"], rec["rank"], rec["path_id"]]
        np.save(os.path.join(out_dir, "round_pose.npy"), np.concatenate([np.array(pose, np.float64), rec["R21"].reshape(-1), rec["t21"],
                                                                        rec["R31"].reshape(-1), rec["t31"]]).astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--hyp", type=int, default=100, help="hypotheses per GPU per step (100 = default RANSAC round)")
    ap.add_argument("--abort", action="store_true", help="Abort_RANSAC_by_Good_Sol = true (configs[2])")
    ap.add_argument("--no-prune", action="store_true")
    ap.add_argument("--ref-hyp", type=int, default=8, help="hypotheses per step of the reference CPU arm (--impl reference)")
    ap.add_argument("--cpu-baseline-hyp", type=int, default=40, help="hypotheses of the cpu_baseline sample (about 15 s on 16 cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip timing the reference GPU-HC++ kernels (oracle/_ref/libref_gpuhc.so)")
    ap.add_argument("--strong-hyp", type=int, default=10000, help="strong-scaling leg: ONE round of this many hypotheses split over the GPUs (0 = skip)")
    ap.add_argument("--strong-hyp-large", type=int, default=100000, help="second strong-scaling point (0 = skip)")
    ap.add_argument("--no-host-class", action="store_true", help="skip the C++ GPU_HC_Solver leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of --impl ours computed to DIR/<name>.npy "
                                                          "(at most 64 MB in all); not available with --impl reference")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        return reference_arm(args)

    import torch
    from trifocal_pose_estimation_using_improved_gpuhc_b200 import fixtures, hc

    rank, local_rank, world = _rank_env()
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local_rank)
    dist, cpu_group = None, None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")      # host-side waits (a spinning NCCL barrier would occupy the GPUs)
    dev = torch.device("cuda", local_rank)

    def host_barrier():
        if world > 1:
            dist.barrier(group=cpu_group)

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    prob = fixtures.load_problem()
    rs = fixtures.load_ransac(0)
    H = args.hyp
    prune = not args.no_prune
    n_edgels = rs["locations"].shape[0]
    # one rand() stream for the whole (multi-GPU) round, consumed in GPU-major order (GPU_HC_Solver.cpp:263-271)
    picked_all = hc.sample_hypotheses(0, H * world, n_edgels)
    offs = hc.shard_offsets(H * world, world)
    picked = picked_all[offs[rank]:offs[rank + 1]]
    target, diff = hc.target_params_from_picks(picked, rs["locations"], rs["tangents"], prob["start_params"])

    trk = hc.Tracker(device=dev, problem=prob, stats=True)
    trk.reserve(H)
    trk.set_edgels(rs["locations"], rs["K"])
    n_paths = H * hc.NUM_TRACKS

    # pinned host staging for the e2e leg (what GPU_HC_Solver keeps in h_Target_Params / h_GPU_HC_Track_Sols)
    h_target = torch.view_as_real(torch.from_numpy(target)).contiguous().pin_memory()
    h_diff = torch.view_as_real(torch.from_numpy(diff)).contiguous().pin_memory()
    h_tracks = torch.empty((n_paths, 31, 2), dtype=torch.float32).pin_memory()
    h_conv = torch.empty(n_paths, dtype=torch.uint8).pin_memory()
    h_inf = torch.empty(n_paths, dtype=torch.uint8).pin_memory()
    h_rec = torch.zeros(32, dtype=torch.float32).pin_memory()
    gathered = torch.zeros((world, 32), dtype=torch.float32, device=dev)       # one 128-byte record per GPU
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2

    def launch(n_hyp=H):
        if args.abort:
            trk.track_abort(n_hyp, prune=prune)
        else:
            trk.track(n_hyp, prune=prune)

    def exchange(n_hyp, hyp_offset, ev_mid=None):
        """score the round on the device -> 128-byte record -> gather -> arg-max (all on the launch stream)."""
        if not args.abort:
            trk.score_tracks_async(n_hyp)
        rec = trk.make_pose_record(hyp_offset * hc.NUM_TRACKS, rank, abort=args.abort)
        if ev_mid is not None:
            ev_mid.record()
        if world > 1:
            dist.all_gather_into_tensor(gathered.view(-1), rec)
        else:
            gathered[0].copy_(rec)
        trk.reduce_pose_records(gathered, world)

    def step_device(ev_track=None, ev_mid=None):
        launch()
        if ev_track is not None:
            ev_track.record()
        exchange(H, offs[rank], ev_mid)

    trk.upload_params(target, diff)
    for _ in range(args.warmup):
        step_device()
    torch.cuda.synchronize()

    # ---- device-timed leg ------------------------------------------------------------------------------------
    host_barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = trk.launches
    ev = [_events(torch, 4) for _ in range(args.steps)]
    for a, t, m, b in ev:
        flush.fill_(1.0)            # L2 flush between timed iterations (outside the event pair)
        a.record()
        step_device(t, m)
        b.record()
    torch.cuda.synchronize()
    launches = trk.launches - l0
    host_barrier()
    dev_ms = max_over_ranks(sum(a.elapsed_time(b) for a, t, m, b in ev))
    track_ms = max_over_ranks(sum(a.elapsed_time(t) for a, t, m, b in ev)) / args.steps
    score_ms = max_over_ranks(sum(t.elapsed_time(m) for a, t, m, b in ev)) / args.steps
    gather_ms = max_over_ranks(sum(m.elapsed_time(b) for a, t, m, b in ev)) / args.steps
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = dev_ms / args.steps
    round_record = hc.decode_pose_record(trk.d_round_record.cpu().numpy())

    # per-path stage counters of the last step -> algorithmic flops of one launch
    tracks, conv, inf, stats = trk.results(H)
    n_pred, n_corr = float(stats[:, 1].sum()), float(stats[:, 2].sum())
    flops_launch = FLOPS_PRED_STAGE * n_pred + FLOPS_CORR_STAGE * n_corr
    counts = hc.count_solutions(tracks, conv, inf, H)
    if args.dump_outputs:
        support = None if args.abort else trk.d_support[:n_paths].cpu().numpy()
        dump_outputs(args.dump_outputs, rank, world, tracks, conv, inf, stats, support, round_record)

    # ---- the gather itself: NCCL all_gather of the 128-byte records vs D2H + host (gloo) exchange -------------------
    gather_cmp = None
    if world > 1:
        reps = 50
        e0, e1 = _events(torch, 2)
        torch.cuda.synchronize(); host_barrier()
        e0.record()
        for _ in range(reps):
            dist.all_gather_into_tensor(gathered.view(-1), trk.d_pose_record)
        e1.record(); torch.cuda.synchronize()
        nccl_us = max_over_ranks(e0.elapsed_time(e1)) / reps * 1e3
        h_all = [torch.zeros(32, dtype=torch.float32) for _ in range(world)]
        host_barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            h_rec.copy_(trk.d_pose_record, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            dist.all_gather(h_all, h_rec, group=cpu_group)
        host_us = max_over_ranks(time.perf_counter() - t0) / reps * 1e6
        gather_cmp = {"nccl_all_gather_us": nccl_us, "host_d2h_plus_gloo_us": host_us, "used": "nccl",
                      "bytes_per_rank": 128, "note": "device-timed back-to-back all_gather vs pinned D2H + stream sync + gloo all_gather, max over ranks"}

    # ---- e2e leg: host buffers in, host buffers out, every step --------------------------------------------
    def step_e2e():
        trk.d_target[:H].copy_(h_target, non_blocking=True)
        trk.d_diff[:H].copy_(h_diff, non_blocking=True)
        launch()
        exchange(H, offs[rank])
        h_tracks.copy_(trk.d_tracks[:n_paths], non_blocking=True)
        h_conv.copy_(trk.d_conv[:n_paths], non_blocking=True)
        h_inf.copy_(trk.d_inf[:n_paths], non_blocking=True)
        h_rec.copy_(trk.d_round_record, non_blocking=True)
        torch.cuda.synchronize()
        return int(h_conv.sum())     # device -> host read of the step's result

    for _ in range(2):
        step_e2e()
    host_barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    h2d = h_target.numel() * 4 + h_diff.numel() * 4
    d2h = h_tracks.numel() * 4 + h_conv.numel() + h_inf.numel() + 128

    # ---- like-for-like with the reference CPU-HC, which never prunes: the same round with pruning off --------------------
    noprune_ms = None
    if world == 1 and not args.abort and prune:
        for i in range(4):
            if i == 1:
                e0, e1 = _events(torch, 2); e0.record()
            trk.track(H, prune=False)
        e1.record(); torch.cuda.synchronize()
        noprune_ms = e0.elapsed_time(e1) / 3
        trk.track(H, prune=True)

    # ---- strong scaling: ONE big round split over the GPUs (BASELINE.json configs[4]) -----------------------------------------
    def strong_leg(h_total, reps, warm):
        pk = hc.sample_hypotheses(0, h_total, n_edgels)
        so = hc.shard_offsets(h_total, world)
        mine = pk[so[rank]:so[rank + 1]]
        tg, df = hc.target_params_from_picks(mine, rs["locations"], rs["tangents"], prob["start_params"])
        hr = mine.shape[0]
        trk.upload_params(tg, df)
        def one():
            launch(hr)
            exchange(hr, so[rank])
        for _ in range(warm):
            one()
        torch.cuda.synchronize(); host_barrier()
        ts = []
        for _ in range(reps):
            e0, e1 = _events(torch, 2)
            e0.record(); one(); e1.record(); torch.cuda.synchronize()
            ts.append(max_over_ranks(e0.elapsed_time(e1)))
        rec = hc.decode_pose_record(trk.d_round_record.cpu().numpy())
        ms = float(np.mean(ts))
        return {"hypotheses_total": h_total, "hypotheses_per_gpu": [so[g + 1] - so[g] for g in range(world)], "ms_per_round": ms,
                "value": h_total / (ms * 1e-3), "unit": "hypotheses/s", "paths_per_s": h_total * 312 / (ms * 1e-3), "timed_rounds": reps,
                "selected_global_path": rec["path_id"], "selected_inliers": [rec["inliers21"], rec["inliers31"]]}

    strong = {}
    if args.strong_hyp > 0:
        strong["h%d" % args.strong_hyp] = strong_leg(args.strong_hyp, 2, 1)
    if args.strong_hyp_large > 0:
        strong["h%d" % args.strong_hyp_large] = strong_leg(args.strong_hyp_large, 1, 0)
    trk.upload_params(target, diff)

    # ---- the C++ host class with Num_Of_GPUs = N in ONE process (rank 0; the other ranks wait on the host) ---------------------
    host_class = None
    host_barrier()
    if rank == 0 and not args.no_host_class and torch.cuda.device_count() >= world:
        try:
            host_class = host_class_leg(world, args.abort)
        except Exception as e:                          # the leg must never take the headline down with it
            host_class = {"error": repr(e)}
    host_barrier()

    if rank == 0:
        fp32_peak = trk.ffma_probe()
        hyp_per_s = H * world / (ms_per_step * 1e-3)
        achieved = flops_launch / (track_ms * 1e-3) / 1e12
        executed = (EXEC_FLOP_PER_STAGE * (n_pred + n_corr)) / (track_ms * 1e-3) / 1e12
        info = trk.kernel_info(abort=args.abort)
        alg_bytes = H * (2 * 34 * 8) + n_paths * (31 * 8 + 2)
        line = {
            "metric": "RANSAC hypotheses/s (312 HC paths each)", "value": hyp_per_s, "unit": "hypotheses/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "c64", "data": "synthetic",
            "paths_per_s": hyp_per_s * hc.NUM_TRACKS,
            "config": {"workload": "trifocal_2op1p_30x30 default RANSAC round: %d hypotheses x 312 paths per GPU, 80 max steps, "
                                   "3 corrections, pruning %s, early abort %s, dataset Synthetic/000, seed 0; step = track + device scoring "
                                   "+ 128-byte best-pose record per GPU + gather + arg-max"
                                   % (H, "on" if prune else "off", "on" if args.abort else "off"),
                       "hypotheses_per_gpu": H, "paths_per_gpu": n_paths, "sharding": "contiguous hypotheses (sub_RANSAC_iters)",
                       "l2": "256 MB L2 flush between timed iterations (outside the event pair)",
                       "kernel": info},
            "step_breakdown_ms": {"track": track_ms, "score_and_record": score_ms, "gather_and_argmax": gather_ms},
            "round_result": {"selected_global_path": round_record["path_id"], "inliers": [round_record["inliers21"], round_record["inliers31"]],
                             "candidates": round_record["n_candidates"], "abort_flag": round_record["abort_flag"], "owner_rank": round_record["rank"]},
            "e2e": {"value": H * world / (e2e_s / args.steps), "unit": "hypotheses/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_s / args.steps * 1e3},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"bound": "fp32", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                         "frac": achieved / fp32_peak if fp32_peak else None,
                         "kernel": "hc_track_kernel (%.3f of %.3f ms per step)" % (track_ms, ms_per_step),
                         "executed_tflops": executed, "executed_frac": executed / fp32_peak if fp32_peak else None,
                         "executed_source": EXEC_SOURCE,
                         "traffic": TRAFFIC_BYTES_H100 if (H == 100 and prune and not args.abort) else None, "traffic_source": TRAFFIC_SOURCE,
                         "hbm": {"algorithmic_bytes_per_launch": alg_bytes, "achieved_gbs": alg_bytes / (track_ms * 1e-3) / 1e9,
                                 "peak_gbs": 6553.0, "peak_source": "MEASURED_PEAKS.json hbm_gbs",
                                 "note": "the path is not HBM-bound: 78 KB and ~8 Gflop (model) per hypothesis"},
                         "peak_source": "FFMA probe kernel timed live on this GPU (MEASURED_PEAKS.json has no FP32 entry); "
                                        "nominal 148x128x2x1.965GHz = %.1f" % NOMINAL_FP32_TFLOPS,
                         "frac_of_nominal": achieved / NOMINAL_FP32_TFLOPS,
                         "flops_per_launch": flops_launch, "model": "91312*pred_stages + 90874*corr_stages (dense-LU model, SURVEY §8d)",
                         "stages_per_path": (n_pred + n_corr) / n_paths},
            "result": {"converged": int(counts[:, 0].sum()), "infinity": int(counts[:, 1].sum()), "real": int(counts[:, 2].sum())},
        }
        if strong:
            line["strong_scaling"] = strong
        if gather_cmp:
            line["gather"] = gather_cmp
        if host_class is not None:
            line["host_class"] = host_class
        if world == 1 and not args.no_ref_gpu:
            rg = ref_gpu_leg(prob, rs, target, diff, H, args.abort)
            if rg:
                rg["speedup_ours_vs_ref_gpu"] = rg["ms_per_step"] / track_ms
                line["ref_gpu"] = rg
                if not args.abort:               # configs[2] beside the headline: both kernels with Abort_RANSAC_by_Good_Sol, same inputs
                    line["ref_gpu_abort"] = abort_compare_leg(trk, prob, rs, H, prune)
        if not args.no_cpu_baseline and world == 1:
            cb = cpu_baseline_leg(args.cpu_baseline_hyp)
            line["cpu_baseline"] = cb
            if noprune_ms:
                line["like_for_like_cpu"] = {"ours_noprune_ms_per_round": noprune_ms, "ours_noprune_hyp_per_s": H / (noprune_ms * 1e-3),
                                             "reference_cpu_hyp_per_s": cb["value"], "ratio": H / (noprune_ms * 1e-3) / cb["value"],
                                             "note": "both WITHOUT path pruning (the reference CPU-HC has none): same work on both sides"}
        print(json.dumps(line))
    host_barrier()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
