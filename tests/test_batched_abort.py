"""hcb200_track_abort_batched: the early-abort rounds of many image triplets in one launch, each with its own flag, edgels, K and best record.

The reference of every GPU test is the no-abort hcb200_track on the same stacked parameters (bit-identical to the oracle, test_gpu_parity.py)
plus the oracle's scoring (oracle.score) with each problem's own edgels and K."""
import ctypes
import os
import re

import numpy as np
import pytest

from trifocal_pose_estimation_using_improved_gpuhc_b200 import fixtures, hc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "trifocal_pose_estimation_using_improved_gpuhc_b200", "lib")
PROBLEMS = sorted(os.listdir(os.path.join(ROOT, "problems")))
T = hc.NUM_TRACKS
INVALID_VALUE, NOT_SUPPORTED = 1, 801


# ---------------------------------------------------------------------------------------------------------------------
# CPU: workspace size and argument validation (all before any CUDA call)

def test_batch_workspace_bytes_formula():
    lib = hc.load_library()
    for n in (1, 2, 16, 1000, hc.BATCH_MAX_PROBLEMS):
        assert lib.hcb200_batch_workspace_bytes(n) == 256 + 16 * (n + 1)
    assert lib.hcb200_batch_workspace_bytes(hc.BATCH_MAX_PROBLEMS) == 256 + 65536
    text = open(os.path.join(ROOT, "include", "hcb200.h")).read()
    assert int(re.search(r"#define HCB200_BATCH_MAX_PROBLEMS (\d+)", text).group(1)) == hc.BATCH_MAX_PROBLEMS


def _call(lib, n_problems=2, n_hyp=3, offsets=(0, 10, 25), max_corr=3, null=None):
    """hcb200_track_abort_batched with fake (never dereferenced) device pointers; `null` names the buffer passed as NULL."""
    names = ["start_sols", "start_params", "target", "diff", "edgels", "K", "tracks", "conv", "inf", "found", "found_index", "best",
             "stats", "ws"]
    bufs = [None if n == null else ctypes.c_void_p(0x1000 * (i + 1)) for i, n in enumerate(names)]
    off = None if offsets is None else np.ascontiguousarray(offsets, np.int32)
    return lib.hcb200_track_abort_batched(None, n_problems, n_hyp, None if off is None else off.ctypes.data_as(ctypes.c_void_p),
                                          80, max_corr, 4, hc.FLAG_PRUNE_PATHS, *bufs)


@pytest.mark.parametrize("null", ["start_sols", "start_params", "target", "diff", "edgels", "K", "tracks", "conv", "inf", "found",
                                  "found_index", "ws", "offsets"])
def test_batched_abort_refuses_null_buffers(null):
    lib = hc.load_library()
    if null == "offsets":
        assert _call(lib, offsets=None) == INVALID_VALUE
    else:
        assert _call(lib, null=null) == INVALID_VALUE


@pytest.mark.parametrize("case", ["no_problems", "negative_problems", "too_many_problems", "negative_hyp", "path_ids_overflow",
                                  "no_correction_steps", "first_offset", "empty_problem", "decreasing_offsets", "too_many_edgels",
                                  "empty_last_problem"])
def test_batched_abort_refuses_bad_counts(case):
    """Each case returns cudaErrorInvalidValue on a machine without a GPU too: the check runs before any CUDA call."""
    lib = hc.load_library()
    m = hc.BATCH_MAX_PROBLEMS
    kw = {"no_problems": dict(n_problems=0, offsets=(0,)),
          "negative_problems": dict(n_problems=-1),
          "too_many_problems": dict(n_problems=m + 1, offsets=np.arange(m + 2)),
          "negative_hyp": dict(n_hyp=-1),
          "path_ids_overflow": dict(n_hyp=0x7fffffff // (T * 2) // 2 + 1),
          "no_correction_steps": dict(max_corr=0),
          "first_offset": dict(offsets=(1, 10, 25)),
          "empty_problem": dict(offsets=(0, 0, 25)),
          "decreasing_offsets": dict(offsets=(0, 30, 25)),
          "too_many_edgels": dict(offsets=(0, 10, 10 + 65536)),
          "empty_last_problem": dict(offsets=(0, 10, 10))}[case]
    assert _call(lib, **kw) == INVALID_VALUE


def test_compiled_problem_libraries_do_not_support_batched_abort():
    from trifocal_pose_estimation_using_improved_gpuhc_b200 import problem as pm
    built = [name for name in PROBLEMS if os.path.exists(pm.library_path(name))]
    if not built:
        pytest.skip("no compiled-problem library built (make problem PROBLEM_DIR=problems/<name>)")
    for name in built:
        lib = ctypes.CDLL(pm.library_path(name))
        lib.hcb200_track_abort_batched.restype = ctypes.c_int
        lib.hcb200_track_abort_batched.argtypes = hc.load_library().hcb200_track_abort_batched.argtypes
        lib.hcb200_batch_workspace_bytes.restype = ctypes.c_size_t
        lib.hcb200_batch_workspace_bytes.argtypes = [ctypes.c_int]
        assert _call(lib) == NOT_SUPPORTED, name
        assert lib.hcb200_batch_workspace_bytes(3) == 256 + 64


# ---------------------------------------------------------------------------------------------------------------------
# GPU

def _bit_equal(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    av, bv = a.view(np.uint32), b.view(np.uint32)
    both_nan = np.isnan(a.view(np.float32)) & np.isnan(b.view(np.float32))
    return bool(np.all((av == bv) | both_nan))


def _targets(problem, specs, n_hyp):
    """specs: [(locations, tangents, sampler seed)] -> stacked problem-major (target, diff) [len(specs) * n_hyp, 34]."""
    ts, ds = [], []
    for loc, tan, seed in specs:
        picked = hc.sample_hypotheses(seed, n_hyp, loc.shape[0])
        t, d = hc.target_params_from_picks(picked, loc, tan, problem["start_params"])
        ts.append(t)
        ds.append(d)
    return np.concatenate(ts), np.concatenate(ds)


def _run(problem, specs, edgels, Ks, n_hyp):
    """No-abort reference and batched abort launch on the same stacked parameters.  Returns (reference, batched, records, found index)."""
    trk = hc.Tracker(problem=problem, stats=True)
    target, diff = _targets(problem, specs, n_hyp)
    trk.upload_params(target, diff)
    trk.track(len(specs) * n_hyp, prune=True)
    ref = trk.results(len(specs) * n_hyp)
    trk.set_edgel_batch(edgels, Ks)
    trk.track_abort_batched(len(specs), n_hyp, prune=True)
    got = trk.results(len(specs) * n_hyp)
    recs = trk.batch_records(len(specs))
    idx = trk.d_found_index[: len(specs) * n_hyp * T].cpu().numpy()
    flags = trk.d_found_batch[: len(specs)].cpu().numpy()
    return trk, ref, got, recs, idx, flags


def _check_problem(oracle, k, n_hyp, ref, got, rec, idx, flag, loc, K):
    """The invariants of the single-problem abort tests, on problem k's slice.  Returns the local ids of the flagged paths."""
    L = n_hyp * T
    s = slice(k * L, (k + 1) * L)
    tr0, cv0, inf0, st0 = (a[s] for a in ref)
    tr, cv, inf, st = (a[s] for a in got)
    reason = st[:, 3] >> 16
    done = reason < 4
    # paths that finished before the flag are the no-abort paths, bit for bit
    assert np.array_equal(cv[done], cv0[done]) and np.array_equal(inf[done], inf0[done]) and np.array_equal(st[done], st0[done])
    assert _bit_equal(tr[done][:, :30], tr0[done][:, :30])
    assert not cv[~done].any() and not inf[~done].any()
    # every flagged path passes the oracle's test with this problem's edgels and K; every finished, converged, passing path is flagged
    hits = np.nonzero(idx[s] >= 0)[0]
    assert np.array_equal(idx[s][hits], hits + k * L)
    im = np.abs(tr[:, 18:30].imag).astype(np.float64)
    gated = np.nonzero(done & (cv == 1) & np.all(im < 1e-5, axis=1))[0]
    passing = {int(b) for b in gated if oracle.score(tr[b], loc, K)[0]}
    assert set(hits.tolist()) == passing, (k, sorted(passing)[:5], hits[:5])
    assert flag == (1 if len(hits) else 0)
    if len(hits):
        ok, n21, n31, _ = oracle.score(tr[hits.min()], loc, K)
        assert rec == dict(found=1, path_id=int(hits.min()), inliers21=n21, inliers31=n31, n_passed=len(hits)), (k, rec)
    else:
        assert rec == dict(found=0, path_id=-1, inliers21=0, inliers31=0, n_passed=0), (k, rec)
    return hits


@pytest.mark.gpu
def test_a_pass_in_one_problem_does_not_stop_another(problem, oracle, ransac0):
    """Problem A (seed 0) passes on hypothesis 0 / track 104; problem B (seed 13) has no passing path in its first 30 hypotheses, so with 8 it
    must track everything: no end reason 4, and the no-abort results bit for bit."""
    import torch
    H = 8
    loc, tan, K = ransac0["locations"], ransac0["tangents"], ransac0["K"]
    trk, ref, got, recs, idx, flags = _run(problem, [(loc, tan, 0), (loc, tan, 13)], [loc, loc], [K, K], H)
    hits_a = _check_problem(oracle, 0, H, ref, got, recs[0], idx, flags[0], loc, K)
    _check_problem(oracle, 1, H, ref, got, recs[1], idx, flags[1], loc, K)
    assert 104 in hits_a and recs[0]["found"] == 1 and flags[0] == 1
    assert recs[1]["found"] == 0 and flags[1] == 0
    s = slice(H * T, 2 * H * T)
    assert ((got[3][s, 3] >> 16) < 4).all()
    assert np.array_equal(got[1][s], ref[1][s]) and np.array_equal(got[2][s], ref[2][s]) and np.array_equal(got[3][s], ref[3][s])
    assert _bit_equal(got[0][s], ref[0][s])
    # the record of a problem is the single-problem layout: hcb200_make_pose_record works on the problem's slice
    out = torch.zeros(32, dtype=torch.float32, device=trk.device)
    rc = trk.lib.hcb200_make_pose_record(trk._stream(), ctypes.c_void_p(trk.d_tracks[:H * T].data_ptr()), ctypes.c_void_p(trk.d_best_batch[0].data_ptr()),
                                         ctypes.c_void_p(trk.d_found_batch[0:].data_ptr()), 5000, 3, ctypes.c_void_p(out.data_ptr()))
    assert rc == 0
    r = hc.decode_pose_record(out.cpu().numpy())
    assert r["found"] == 1 and r["path_id"] == 5000 + recs[0]["path_id"] and r["abort_flag"] == 1 and r["rank"] == 3


@pytest.mark.gpu
def test_many_problems_each_keep_the_abort_invariants(problem, oracle, ransac0):
    """16 problems (dataset 0, sampler seeds 0-15, 40 hypotheses each; every seed has a passing path within its first 32 hypotheses)."""
    H = 40
    loc, tan, K = ransac0["locations"], ransac0["tangents"], ransac0["K"]
    specs = [(loc, tan, seed) for seed in range(16)]
    trk, ref, got, recs, idx, flags = _run(problem, specs, [loc] * 16, [K] * 16, H)
    for k in range(16):
        hits = _check_problem(oracle, k, H, ref, got, recs[k], idx, flags[k], loc, K)
        assert len(hits) >= 1, k
    assert ((got[3][:, 3] >> 16) == 4).sum() > 0                 # work behind the flags was skipped


@pytest.mark.gpu
def test_each_problem_is_scored_with_its_own_edgels_and_K(problem, oracle):
    """Problem 0 scores against the first 3 000 edgels of dataset 1 only; problem 1 against dataset 0 with K scaled by 1e-6, which makes every
    reprojection error tiny, so nearly every converged real path passes.  The flags and counts follow each problem's own inputs."""
    r1, r0 = fixtures.load_ransac(1), fixtures.load_ransac(0)
    loc1, tan1 = r1["locations"][:3000], r1["tangents"][:3000]
    K_small = (np.asarray(r0["K"], np.float32) * np.float32(1e-6)).astype(np.float32)
    H = 12
    specs = [(loc1, tan1, 0), (r0["locations"], r0["tangents"], 2)]
    trk, ref, got, recs, idx, flags = _run(problem, specs, [loc1, r0["locations"]], [r1["K"], K_small], H)
    _check_problem(oracle, 0, H, ref, got, recs[0], idx, flags[0], loc1, r1["K"])
    hits1 = _check_problem(oracle, 1, H, ref, got, recs[1], idx, flags[1], r0["locations"], K_small)
    if recs[0]["found"]:
        assert recs[0]["inliers21"] <= 3000 and recs[0]["inliers31"] <= 3000
    # with the true K the first passing path of seed 2 is path 2230 (hypothesis 7); the scaled K lets earlier converged real paths pass
    assert recs[1]["found"] == 1 and len(hits1) >= 1 and recs[1]["path_id"] < 2230


@pytest.mark.gpu
def test_one_problem_behaves_like_track_abort(problem, oracle, ransac0):
    """The assertions of test_abort_finds_gt_pose and test_abort_late_hit, for the batched launch with one problem."""
    loc, tan, K = ransac0["locations"], ransac0["tangents"], ransac0["K"]
    trk = hc.Tracker(problem=problem, stats=True)
    trk.set_edgel_batch([loc], [K])
    # seed 0: hypothesis 0 / track 104 is the ground-truth pose
    target, diff, _ = oracle.prepare_target_params(0, 4, loc, tan)
    trk.upload_params(target, diff)
    trk.track_abort_batched(1, 4, prune=True)
    tr_g, cv_g, _, _ = trk.results(4)
    rec = trk.batch_records(1)[0]
    idx = trk.d_found_index[: 4 * T].cpu().numpy()
    hits = np.nonzero(idx >= 0)[0]
    assert int(trk.d_found_batch.cpu()[0]) == 1 and len(hits) >= 1 and np.array_equal(idx[hits], hits)
    for b in hits:
        ok, n21, n31, gate = oracle.score(tr_g[b], loc, K)
        assert ok and gate and cv_g[b] == 1
    ok, n21, n31, _ = oracle.score(tr_g[rec["path_id"]], loc, K)
    assert rec == dict(found=1, path_id=int(hits.min()), inliers21=n21, inliers31=n31, n_passed=len(hits))
    assert 104 in hits and ((n21, n31) == (5117, 5117) or rec["path_id"] != 104)
    # seed 13: the first passing path is 9606 (hypothesis 30)
    H = 40
    target, diff, _ = oracle.prepare_target_params(13, H, loc, tan)
    tr_o, cv_o, inf_o, st_o = oracle.track(target, diff, True)
    passing = [int(b) for b in np.nonzero(cv_o)[0] if oracle.score(tr_o[b], loc, K)[0]]
    assert passing and min(passing) == 9606
    trk.upload_params(target, diff)
    trk.track_abort_batched(1, H, prune=True)
    tr_g, cv_g, inf_g, st_g = trk.results(H)
    rec = trk.batch_records(1)[0]
    idx = trk.d_found_index[: H * T].cpu().numpy()
    hits = np.nonzero(idx >= 0)[0]
    assert int(trk.d_found_batch.cpu()[0]) == 1 and len(hits) >= 1
    assert set(hits.tolist()) <= set(passing)
    assert rec["found"] == 1 and rec["path_id"] == hits.min() and rec["n_passed"] == len(hits)
    for b in hits:
        assert _bit_equal(tr_g[b, :30], tr_o[b, :30])
    reason = st_g[:, 3] >> 16
    assert (reason == 4).sum() > 0
    done = reason < 4
    assert np.array_equal(cv_g[done], cv_o[done]) and _bit_equal(tr_g[done][:, :30], tr_o[done][:, :30])


@pytest.mark.gpu
def test_empty_round_clears_every_record(problem, ransac0):
    loc, tan, K = ransac0["locations"], ransac0["tangents"], ransac0["K"]
    trk = hc.Tracker(problem=problem, stats=True)
    target, diff = _targets(problem, [(loc, tan, 0)] * 5, 1)
    trk.upload_params(target, diff)
    trk.set_edgel_batch([loc] * 5, [K] * 5)
    trk.track_abort_batched(5, 1, prune=True)
    assert any(r["found"] for r in trk.batch_records(5))
    trk.d_best_batch.fill_(7)
    trk.track_abort_batched(5, 0, prune=True)
    assert trk.batch_records(5) == [dict(found=0, path_id=-1, inliers21=0, inliers31=0, n_passed=0)] * 5
    assert (trk.d_best_batch[:5, 5:].cpu().numpy() == 0).all()          # reserved words cleared too
