#!/usr/bin/env python3
"""Early-abort rounds of several image triplets ("problems"): K sequential hcb200_track_abort launches against one
hcb200_track_abort_batched launch, on the same stacked inputs (100 hypotheses per problem, pruning on).

Each sample is one CUDA-event window around `--reps` repetitions of the whole sequence (reset of the flags and found indices + the
launches); the two ways alternate `--alternations` times after a warm-up of each.  Also times K = 1 (the batched launch with one problem
against hcb200_track_abort), which is the cost of the variant itself, and records the card's name, power limit and maximum SM clock.
Usage: python tools/time_batched_abort.py [--out FILE]"""
import argparse
import ctypes
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from trifocal_pose_estimation_using_improved_gpuhc_b200 import fixtures, hc

H = 100
T = hc.NUM_TRACKS
SETS = [("dataset 0, seeds {0,1,3,7,11,15} (first hit in hypothesis 0-1)", [(0, s) for s in (0, 1, 3, 7, 11, 15)]),
        ("dataset 0, seeds {4,5,9,13,14} (first hit in hypothesis 27-31)", [(0, s) for s in (4, 5, 9, 13, 14)]),
        ("dataset 0, seeds 0-15", [(0, s) for s in range(16)]),
        ("datasets 0-3 x seeds 0-3", [(d, s) for d in range(4) for s in range(4)])]


def p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def setup(trk, problems, data, start_params):
    ts, ds = [], []
    for d, seed in problems:
        rs = data[d]
        picked = hc.sample_hypotheses(seed, H, rs["locations"].shape[0])
        t, df = hc.target_params_from_picks(picked, rs["locations"], rs["tangents"], start_params)
        ts.append(t)
        ds.append(df)
    trk.upload_params(np.concatenate(ts), np.concatenate(ds))
    trk.set_edgel_batch([data[d]["locations"] for d, _ in problems], [data[d]["K"] for d, _ in problems])
    trk.reset_abort_batched(len(problems), H)


def sequential(trk, K):
    """Problem after problem: reset its flag and found indices, then hcb200_track_abort on its slice."""
    L = H * T
    off = trk.batch_offsets
    for k in range(K):
        s = slice(k * L, (k + 1) * L)
        trk.d_found_batch[k].zero_()
        trk.d_found_index[s].fill_(-1)
        rc = trk.lib.hcb200_track_abort(trk._stream(), H, int(off[k + 1] - off[k]), trk.max_steps, trk.max_corr, trk.dt_inc, hc.FLAG_PRUNE_PATHS,
                                        p(trk.d_start_sols), p(trk.d_start_params), p(trk.d_target[k * H:]), p(trk.d_diff[k * H:]),
                                        p(trk.d_edgels_batch[int(off[k]):]), p(trk.d_K_batch[k]), p(trk.d_tracks[s]), p(trk.d_conv[s]),
                                        p(trk.d_inf[s]), p(trk.d_found_batch[k:]), p(trk.d_found_index[s]), p(trk.d_best_batch[k]),
                                        p(trk.d_stats[s]), p(trk.d_ws))
        hc._check(rc, "hcb200_track_abort")


def batched(trk, K):
    trk.track_abort_batched(K, H, prune=True)


def window(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def summary(trk, K):
    recs = trk.batch_records(K)
    ran = ((trk.d_stats[:K * H * T, 3] >> 16) != 4).sum().item()
    return [r["path_id"] if r["found"] else -1 for r in recs], ran


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--alternations", type=int, default=3)
    args = ap.parse_args()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    say("# nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv")
    for ln in smi.stdout.strip().splitlines():
        say("#   " + ln)
    say("# %d hypotheses per problem, pruning on; one sample = CUDA events around %d repetitions of the whole sequence (reset + launches),"
        % (H, args.reps))
    say("# per-sequence ms; sequential (K x hcb200_track_abort) and batched (1 x hcb200_track_abort_batched) alternate %d times after a warm-up"
        % args.alternations)
    problem = fixtures.load_problem()
    data = {d: fixtures.load_ransac(d) for d in range(4)}
    trk = hc.Tracker(problem=problem, stats=True)
    for name, problems in SETS:
        K = len(problems)
        setup(trk, problems, data, problem["start_params"])
        modes = [("sequential", lambda: sequential(trk, K)), ("batched", lambda: batched(trk, K))]
        info = {}
        for m, fn in modes:                                   # warm-up, and the first hit / work of each way
            fn()
            info[m] = summary(trk, K)
        times = {m: [] for m, _ in modes}
        for _ in range(args.alternations):
            for m, fn in modes:
                times[m].append(window(fn, args.reps))
        say()
        say("%s: K = %d" % (name, K))
        for m, _ in modes:
            say("  %-10s %s ms   paths tracked %7d   best local path per problem %s"
                % (m, " ".join("%8.3f" % t for t in times[m]), info[m][1], info[m][0]))
        say("  gain: sequential / batched = %.2fx (medians %.3f / %.3f ms)"
            % (np.median(times["sequential"]) / np.median(times["batched"]), np.median(times["sequential"]), np.median(times["batched"])))

    say()
    say("K = 1: hcb200_track_abort_batched with one problem against hcb200_track_abort (Tracker.track_abort), dataset 0")
    for seed in (0, 13):
        setup(trk, [(0, seed)], data, problem["start_params"])
        trk.set_edgels(data[0]["locations"], data[0]["K"])
        modes = [("track_abort", lambda: trk.track_abort(H, prune=True)), ("batched", lambda: batched(trk, 1))]
        for _, fn in modes:
            fn()
        times = {m: [] for m, _ in modes}
        for _ in range(args.alternations):
            for m, fn in modes:
                times[m].append(window(fn, args.reps))
        say("  seed %2d: %s" % (seed, "   ".join("%s %s ms" % (m, " ".join("%7.3f" % t for t in times[m])) for m, _ in modes)))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
