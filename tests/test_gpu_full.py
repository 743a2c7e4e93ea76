"""GPU tests at BASELINE.json's full sizes and through the reference-facing host API.

 * the full default RANSAC round (100 hypotheses x 312 paths) must reproduce the oracle's golden run bit for bit
   (tests/golden/oracle_seed0_h100_*.npz: flags, step counts, SHA-256 of every hypothesis' end points);
 * size-independent properties on a 1000-hypothesis batch (replication / batch-position invariance, determinism);
 * the C++ host class GPU_HC_Solver (through include/hcb200_host.h) and the hc-main executable;
 * the UNMODIFIED reference GPU-HC++ kernels as a second oracle, compared statistically: their committed flags
   (tests/golden/ref_gpuhc_seed0_h100.npz), and their end points where oracle/_ref/libref_gpuhc.so is built."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest

from trifocal_pose_estimation_using_improved_gpuhc_b200 import fixtures, hc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
LIBDIR = os.path.join(ROOT, "trifocal_pose_estimation_using_improved_gpuhc_b200", "lib")


def _digest(tracks_h):
    a = np.ascontiguousarray(tracks_h[:, :30]).view(np.float32).copy()
    a[np.isnan(a)] = np.float32(np.nan)
    return hashlib.sha256(a.view(np.uint32).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def default_round(problem, ransac0):
    picked = hc.sample_hypotheses(0, 100, ransac0["locations"].shape[0])
    target, diff = hc.target_params_from_picks(picked, ransac0["locations"], ransac0["tangents"], problem["start_params"])
    return picked, target, diff


@pytest.mark.parametrize("prune", [True, False])
def test_full_default_round_is_bit_identical_to_oracle_golden(problem, default_round, prune):
    picked, target, diff = default_round
    g = np.load(os.path.join(GOLD, "oracle_seed0_h100_%s.npz" % ("prune" if prune else "noprune")))
    assert np.array_equal(picked, g["picked"])
    trk = hc.Tracker(problem=problem, stats=True)
    trk.upload_params(target, diff)
    trk.track(100, prune=prune)
    tr, cv, inf, st = trk.results(100)
    assert np.array_equal(np.packbits(cv), g["converged_bits"])
    assert np.array_equal(np.packbits(inf), g["infinity_bits"])
    assert np.array_equal(st[:, 0].astype(np.uint8), g["steps"])
    assert np.array_equal((st[:, 3] >> 16).astype(np.uint8), g["end_reason"])
    assert [int(st[:, 0].sum()), int(st[:, 1].sum()), int(st[:, 2].sum()), int((st[:, 3] & 0xffff).sum())] == g["stats_sum"][:4].tolist()
    assert np.array_equal(hc.count_solutions(tr, cv, inf, 100), g["counts"])          # per-hypothesis converged / inf / real
    mismatched = [h for h in range(100) if _digest(tr[h * 312:(h + 1) * 312]) != str(g["digests"][h])]
    assert mismatched == []
    assert np.array_equal(tr[104].view(np.uint64), g["track104_h0"].view(np.uint64))


def test_batch_position_invariance_and_determinism_1000_hypotheses(problem, default_round):
    """Synthetic sweep size (1000 hypotheses = 312 000 paths): the first 100 hypotheses repeated ten times.  Every replica
    must reproduce the golden flags whatever its position in the batch, and a second launch must be bit-identical."""
    picked, target, diff = default_round
    g = np.load(os.path.join(GOLD, "oracle_seed0_h100_prune.npz"))
    T, D = np.tile(target, (10, 1)), np.tile(diff, (10, 1))
    trk = hc.Tracker(problem=problem)
    trk.upload_params(T, D)
    trk.track(1000, prune=True)
    tr1, cv1, inf1, _ = trk.results(1000)
    trk.track(1000, prune=True)
    tr2, cv2, inf2, _ = trk.results(1000)
    assert np.array_equal(cv1, cv2) and np.array_equal(inf1, inf2)
    assert np.array_equal(np.nan_to_num(tr1.view(np.float32)), np.nan_to_num(tr2.view(np.float32)))
    gold_cv = np.unpackbits(g["converged_bits"])[:31200]
    for rep in range(10):
        assert np.array_equal(cv1[rep * 31200:(rep + 1) * 31200], gold_cv)
    assert _digest(tr1[9 * 31200 + 312 * 57: 9 * 31200 + 312 * 58]) == str(g["digests"][57])


@pytest.mark.parametrize("dataset,seed,prune", [(1, 3, True), (2, 5, False), (3, 11, True)])
def test_other_datasets_and_sampler_seeds_bit_exact(problem, oracle, dataset, seed, prune):
    """Inputs the committed goldens do not cover (they are all dataset 000 / sampler seed 0): other dataset files, other rand() streams,
    both pruning modes — 40 hypotheses each, tracked by the oracle on the box's CPU and compared bit for bit (flags, counters, end points).
    The one-off run over 1 872 000 such paths is profiles/parity_extended_r1.txt (tests/parity_extended.py)."""
    rs = fixtures.load_ransac(dataset)
    H = 40
    picked = hc.sample_hypotheses(seed, H, rs["locations"].shape[0])
    target, diff = hc.target_params_from_picks(picked, rs["locations"], rs["tangents"], problem["start_params"])
    tr_o, cv_o, inf_o, st_o = oracle.track(target, diff, prune)
    trk = hc.Tracker(problem=problem, stats=True)
    trk.upload_params(target, diff)
    trk.track(H, prune=prune)
    tr, cv, inf, st = trk.results(H)
    assert np.array_equal(cv, cv_o) and np.array_equal(inf, inf_o)
    assert np.array_equal(st[:, :3], st_o[:, :3]) and np.array_equal(st[:, 3] & 0xffff, st_o[:, 3]) and np.array_equal(st[:, 3] >> 16, st_o[:, 4])
    a, b = np.ascontiguousarray(tr[:, :30]), np.ascontiguousarray(tr_o[:, :30])
    assert bool(np.all((a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))))


def test_edge_cases_empty_and_invalid(problem):
    import torch
    trk = hc.Tracker(problem=problem)
    trk.reserve(1)
    trk.track(0)                                      # empty batch: success, no launch
    torch.cuda.synchronize()
    lib = hc.load_library()
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    rc = lib.hcb200_track(None, 1, 80, 3, 4, 1, p(trk.d_start_sols), p(trk.d_start_params), None, p(trk.d_diff),
                          p(trk.d_tracks), p(trk.d_conv), p(trk.d_inf), None, p(trk.d_ws))
    assert rc != 0                                    # NULL target parameters -> cudaErrorInvalidValue, nothing launched
    rc = lib.hcb200_track(None, -1, 80, 3, 4, 1, p(trk.d_start_sols), p(trk.d_start_params), p(trk.d_target), p(trk.d_diff),
                          p(trk.d_tracks), p(trk.d_conv), p(trk.d_inf), None, p(trk.d_ws))
    assert rc != 0
    rc = lib.hcb200_track(None, 4_000_000, 80, 3, 4, 1, p(trk.d_start_sols), p(trk.d_start_params), p(trk.d_target), p(trk.d_diff),
                          p(trk.d_tracks), p(trk.d_conv), p(trk.d_inf), None, p(trk.d_ws))
    assert rc != 0                                    # more hypotheses than 31-bit path ids allow: refused, nothing launched
    assert lib.hcb200_error_string(rc)


# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tree(tmp_path_factory):
    root = str(tmp_path_factory.mktemp("tree"))
    fixtures.materialize_tree(root, files=[0])
    return root


from trifocal_pose_estimation_using_improved_gpuhc_b200.host_solver import HostSolver  # noqa: E402


def test_host_class_default_round_matches_golden(tree):
    """GPU_HC_Solver with the shipped gpuhc_settings.yaml (100 iterations, no abort): same totals as the oracle golden, file
    column order converged / real / infinity, and the selected pose is the ground truth within the reference tolerances
    (ROT_RESIDUAL_TOL = TRANSL_RESIDUAL_TOL = 0.1, definitions.hpp:14-15)."""
    g = np.load(os.path.join(GOLD, "oracle_seed0_h100_prune.npz"))
    s = HostSolver(tree, "Num_Of_GPUs=1")
    r = s.round()
    s.close()
    assert r["H"] == 100
    c = g["counts"].sum(0)                                   # conv, inf, real
    assert r["totals"].tolist() == [int(c[0]), int(c[2]), int(c[1])]
    assert np.array_equal(r["per"].astype(np.int32), g["counts"])
    assert np.array_equal(np.packbits(r["conv"]), g["converged_bits"])
    assert r["pose_found"] == 1 and np.all(r["residuals"] < 0.1) and np.all(r["residuals"][:2] < 1e-2)
    assert 0 < r["seconds"] < 5
    # pose with maximal support: selected on the device (hcb200_score_tracks); the host-only path must pick the same one
    assert r["selected_path"] == 104 and r["selected_support"] == [5117, 5117]
    s2 = HostSolver(tree, "Num_Of_GPUs=1;Device_Scoring=false")
    r2 = s2.round()
    s2.close()
    assert r2["selected_path"] == 104 and r2["selected_support"] == [5117, 5117]
    assert np.array_equal(r2["residuals"], r["residuals"])


def test_host_class_refinement_option(tree):
    """Refine_Iterations = 3 (optional YAML key): converged end points are polished on the GPU before they are copied back;
    flags and counts are untouched, the selected pose is the same, and duplicates of one root now agree far below the
    reference's DUPLICATE_SOL_DIFF_TOL (Evaluations.cpp:184-233)."""
    s = HostSolver(tree, "Num_Of_GPUs=1;Num_Of_RANSAC_Iterations=10")
    r0 = s.round()
    s.close()
    s = HostSolver(tree, "Num_Of_GPUs=1;Num_Of_RANSAC_Iterations=10;Refine_Iterations=3")
    r1 = s.round()
    s.close()
    assert np.array_equal(r0["conv"], r1["conv"]) and np.array_equal(r0["inf"], r1["inf"])
    assert r1["selected_path"] == r0["selected_path"] == 104 and r1["pose_found"] == 1
    conv = r0["conv"] == 1
    moved = np.abs(r1["tracks"][conv, :30] - r0["tracks"][conv, :30]).max(axis=1) / np.maximum(1.0, np.abs(r0["tracks"][conv, :30]).max(axis=1))
    assert np.median(moved) < 1e-3 and (moved > 0).mean() > 0.5           # a polish, not a different answer
    assert np.array_equal(r1["tracks"][~conv], r0["tracks"][~conv])       # paths that did not converge are left alone


def test_host_class_early_abort_finds_gt_pose(tree):
    s = HostSolver(tree, "Num_Of_GPUs=1;Abort_RANSAC_by_Good_Sol=true")
    r = s.round()
    s.close()
    best = r["best"]
    assert best[0] == 1 and best[1] == 104 and (best[2], best[3]) == (5117, 5117) and best[4] >= 1
    assert r["conv"][104] == 1
    assert r["pose_found"] == 1 and np.all(r["residuals"] < 0.1)
    assert int(r["conv"].sum()) < 2640                        # later paths were skipped or aborted


def test_hc_main_writes_reference_output_files(tree):
    exe = os.path.join(LIBDIR, "hc-main")
    out = subprocess.run([exe, "-p", "trifocal_2op1p_30x30", "-s", "Num_Of_RANSAC_Iterations=10"], cwd=os.path.join(tree, "build", "bin"),
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "Number of Converged Solutions" in out.stdout
    g = np.load(os.path.join(GOLD, "oracle_seed0_h100_prune.npz"))
    c = g["counts"][:10].sum(0)
    stats = open(os.path.join(tree, "Output_Write_Files", "GPU_Sols_Statistics.txt")).read()
    assert stats == "%d\t%d\t%d\n" % (c[0], c[2], c[1])       # converged <TAB> real <TAB> infinity (SURVEY.md App. A.4)
    timing = open(os.path.join(tree, "Output_Write_Files", "GPU_Timings.txt")).read().split()
    assert len(timing) == 1 and 0 < float(timing[0]) < 5000


DROPIN = os.path.join(ROOT, "oracle", "_ref", "ref_gpuhc_on_hcb200")


@pytest.mark.skipif(not os.path.exists(DROPIN), reason="oracle/_ref/ref_gpuhc_on_hcb200 not built (needs /root/reference at build time)")
@pytest.mark.parametrize("abort,n_gpus", [(False, 1), (True, 1), (False, 2)])
def test_unmodified_reference_host_layer_runs_on_this_library(tmp_path, abort, n_gpus):
    """The drop-in claim itself: the reference's OWN GPU_HC_Solver.cpp / Data_Reader.cpp / Evaluations.cpp (compiled unmodified
    from /root/reference in the build container) linked against integration/hcb200_shim.cpp + libhcb200.so instead of the
    reference kernels.  The statistics file the reference writes must carry the golden counts of the default round."""
    import torch
    if torch.cuda.device_count() < n_gpus:
        pytest.skip("needs %d GPUs" % n_gpus)
    root = str(tmp_path)
    ov = {"Num_Of_GPUs": str(n_gpus)}
    if abort:
        ov["Abort_RANSAC_by_Good_Sol"] = "true"
    fixtures.materialize_tree(root, files=[0], settings_overrides=ov)
    out = subprocess.run([DROPIN, "trifocal_2op1p_30x30", "100"], cwd=os.path.join(root, "build", "bin"),
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "Number of Converged Solutions" in out.stdout
    stats = [int(v) for v in open(os.path.join(root, "Output_Write_Files", "GPU_Sols_Statistics.txt")).read().split()]
    g = np.load(os.path.join(GOLD, "oracle_seed0_h100_prune.npz"))
    c = g["counts"].sum(0)                                    # conv, inf, real
    if not abort:
        assert stats == [int(c[0]), int(c[2]), int(c[1])], (stats, out.stdout[-1500:])     # converged, real, infinity (App. A.4)
    else:
        assert 1 <= stats[0] < int(c[0])                      # the flag stopped the round early
    ms = float(open(os.path.join(root, "Output_Write_Files", "GPU_Timings.txt")).read().split()[0])
    assert 0 < ms < 1000


def test_host_class_two_gpus_same_answer(tree):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    g = np.load(os.path.join(GOLD, "oracle_seed0_h100_prune.npz"))
    s = HostSolver(tree, "Num_Of_GPUs=2")
    r = s.round()
    s.close()
    assert np.array_equal(np.packbits(r["conv"]), g["converged_bits"])
    assert np.array_equal(r["per"].astype(np.int32), g["counts"])


def test_host_class_abort_across_gpus(tree):
    """Abort_Across_GPUs (hcb200_track_abort_peers): with the reference's per-GPU flag a 4 000-hypothesis abort round on two GPUs lasts until BOTH
    shards have met a good hypothesis of their own; with the flag shared over NVLink it lasts until the FIRST one has.  Same pose either way."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = {}
    for key, ov in (("per_gpu", ""), ("shared", ";Abort_Across_GPUs=true")):
        s = HostSolver(tree, "Num_Of_GPUs=2;Abort_RANSAC_by_Good_Sol=true;Num_Of_RANSAC_Iterations=4000" + ov)
        s.round(fetch=False)
        secs = [s.round(fetch=False)["seconds"] for _ in range(3)]
        r = s.round(fetch=False)
        s.close()
        assert r["pose_found"] == 1 and r["best"][0] == 1 and r["best"][2] >= 4600 and r["best"][3] >= 4600, (key, r["best"][:5])
        if key == "per_gpu":
            assert r["best"][1] == 104          # (with the shared flag whichever GPU is first wins: hypothesis 0 on GPU 0 or 2003 on GPU 1)
        assert np.all(r["residuals"] < 0.1)     # either way it is the ground-truth pose
        out[key] = (min(secs), int(r["totals"][0]))
    print("abort round, 4000 hypotheses on 2 GPUs: per-GPU flags %.2f ms (%d converged), shared flag %.2f ms (%d converged)"
          % (out["per_gpu"][0] * 1e3, out["per_gpu"][1], out["shared"][0] * 1e3, out["shared"][1]))
    assert out["shared"][0] <= out["per_gpu"][0] * 1.25          # not slower beyond timer noise (observed 3.28 against 4.19 ms); faster whenever the
                                                                 # second shard's first hit comes later
    assert out["shared"][1] <= out["per_gpu"][1]                 # and less work was done


# ---------------------------------------------------------------------------------------------------------------------
def _refined_agreement(orc, target, tr, cv, tr_r, cv_r):
    """north_star: converged solutions within 1e-4 relative after Newton refinement.  Both end points of every path converged on both
    sides are polished in double precision against the target system; REGULAR end points (the polish settles nearby with residual
    < 1e-9 in both) are counted, and those that agree.  Returns (regular, agreeing)."""
    n_reg = n_same = 0
    for b in np.nonzero((cv == 1) & (cv_r == 1))[0]:
        xa, ra = orc.newton_refine(target[b // 312], tr[b], iters=8)
        xb, rb = orc.newton_refine(target[b // 312], tr_r[b], iters=8)
        nrm = max(1.0, np.abs(xb).max())
        if not (np.isfinite(ra) and np.isfinite(rb) and ra < 1e-9 and rb < 1e-9):
            continue
        if np.abs(xa - tr[b, :30]).max() / nrm > 1e-2 or np.abs(xb - tr_r[b, :30]).max() / nrm > 1e-2:
            continue
        n_reg += 1
        n_same += np.abs(xa - xb).max() / nrm < 1e-4
    return n_reg, n_same


def test_against_reference_gpu_kernels(problem, oracle, default_round):
    """Second oracle: the reference's own GPU-HC++ kernels, compiled unmodified for sm_100a; their flags on the seed-0 round (from a
    B200) are committed in tests/golden/ref_gpuhc_seed0_h100.npz.  They use a different LU operation order (and a shuffle reduction that
    reads two lanes that do not exist, …TrunPaths.cu:236-239), so integer results are compared at the noise floor the reference shows
    against itself.  End points: the committed ones are the reference CPU-HC's (tests/golden/ref_cpuhc_seed0_first6.npz); the GPU
    kernels' own are compared in test_end_points_against_reference_gpu_kernels where oracle/_ref is built."""
    picked, target, diff = default_round
    H = 30
    P = H * 312
    g = np.load(os.path.join(GOLD, "ref_gpuhc_seed0_h100.npz"))
    assert np.array_equal(g["picked"], picked)
    cv_r, inf_r, real_r = (np.unpackbits(g[k])[:P] for k in ("converged_bits", "infinity_bits", "real_bits"))
    trk = hc.Tracker(problem=problem)
    trk.upload_params(target[:H], diff[:H])
    trk.track(H, prune=True)
    tr, cv, inf, _ = trk.results(H)
    mine = hc.count_solutions(tr, cv, inf, H)
    theirs = np.stack([f.reshape(H, 312).sum(1) for f in (cv_r, inf_r, real_r)], axis=1)
    # gates at 1.5x what is observed on these 30 hypotheses (|d converged| max 3, mean 0.6, totals 764 vs 770, real max 0, flags 99.70 %);
    # the per-path statement — every difference is an unstable path — is tests/test_parity_envelope.py
    assert np.abs(mine[:, 0] - theirs[:, 0]).max() <= 4 and np.abs(mine[:, 0] - theirs[:, 0]).mean() <= 0.9
    assert abs(int(mine[:, 0].sum()) - int(theirs[:, 0].sum())) <= 0.012 * theirs[:, 0].sum()
    assert np.abs(mine[:, 2] - theirs[:, 2]).max() <= 1
    assert (cv == cv_r).mean() > 0.9955
    assert cv[104] == 1 and cv_r[104] == 1
    # the reference CPU-HC's end points of hypotheses 0..5 (no pruning, like it): observed track 104 at 2.0e-5 relative, 414 of 416
    # regular end points within 1e-4 after refinement
    r = np.load(os.path.join(GOLD, "ref_cpuhc_seed0_first6.npz"))
    assert np.array_equal(r["target_params"], target[:6])
    trk.upload_params(target[:6], diff[:6])
    trk.track(6, prune=False)
    tr6, cv6, _, _ = trk.results(6)
    assert cv6[104] == 1 and r["converged"][104] == 1
    assert np.abs(tr6[104, :30] - r["tracks"][104, :30]).max() / np.abs(r["tracks"][104, :30]).max() < 1e-3
    n_reg, n_same = _refined_agreement(oracle, target, tr6, cv6, r["tracks"], r["converged"])
    assert n_reg > 300 and n_same >= 0.995 * n_reg


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_gpuhc.so")),
                    reason="oracle/_ref/libref_gpuhc.so not built (needs the reference sources at build time)")
def test_end_points_against_reference_gpu_kernels(problem, oracle, ransac0, default_round):
    """The reference GPU-HC++ kernels run live: end points agree after Newton refinement, and in early-abort mode both stop on the
    ground-truth path."""
    from oracle.pyoracle import ReferenceGPU
    picked, target, diff = default_round
    H = 30
    ref = ReferenceGPU(problem)
    ref.setup(target[:H], diff[:H], ransac0["locations"], ransac0["K"])
    ref.track()
    tr_r, cv_r, inf_r = ref.results()
    trk = hc.Tracker(problem=problem)
    trk.upload_params(target[:H], diff[:H])
    trk.track(H, prune=True)
    tr, cv, inf, _ = trk.results(H)
    assert cv[104] == 1 and cv_r[104] == 1
    rel = np.abs(tr[104, :30] - tr_r[104, :30]).max() / np.abs(tr_r[104, :30]).max()
    assert rel < 1e-3
    n_reg, n_same = _refined_agreement(oracle, target, tr, cv, tr_r, cv_r)
    assert n_reg > 300 and n_same >= 0.995 * n_reg
    # early abort: both find hypothesis 0 / track 104
    ref.reload()
    ref.track_abort()
    ref.results()
    idx = ref.d_found_index.cpu().numpy()
    assert bool(ref.d_found.cpu()[0]) and 104 in idx[idx >= 0]


def test_device_scoring_matches_host_evaluations(problem, ransac0, default_round):
    """hcb200_score_tracks vs the host class's arithmetic (hcb200_host_score_track = Evaluations/mvg.hpp): same candidate set,
    identical inlier counts (integers), same selected pose."""
    picked, target, diff = default_round
    H = 40
    trk = hc.Tracker(problem=problem)
    trk.set_edgels(ransac0["locations"], ransac0["K"])
    trk.upload_params(target[:H], diff[:H])
    trk.track(H, prune=True)
    tr, cv, inf, _ = trk.results(H)
    support, best = trk.score_tracks(H)
    host = ctypes.CDLL(os.path.join(LIBDIR, "libhcb200_host.so"))
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    loc = np.ascontiguousarray(ransac0["locations"], np.float32)
    K = np.ascontiguousarray(ransac0["K"], np.float32).reshape(-1)
    n_cand, best_key, best_path = 0, -1, -1
    for pth in range(H * 312):
        if not cv[pth]:
            assert support[pth].tolist() == [-1, -1]
            continue
        x = np.ascontiguousarray(np.stack([tr[pth].real, tr[pth].imag], -1).astype(np.float32))
        n21, n31 = ctypes.c_int(), ctypes.c_int()
        is_cand = host.hcb200_host_score_track(vp(x), vp(loc), loc.shape[0], vp(K), ctypes.byref(n21), ctypes.byref(n31))
        if not is_cand:
            assert support[pth].tolist() == [-1, -1]
            continue
        n_cand += 1
        assert support[pth].tolist() == [n21.value, n31.value], pth
        if min(n21.value, n31.value) > best_key:
            best_key, best_path = min(n21.value, n31.value), pth
    assert n_cand >= 5
    assert best[0] == 1 and best[1] == best_path == 104 and best[4] == n_cand
    assert (best[2], best[3]) == (5117, 5117)


def test_device_statistics_equal_host_statistics(tree, problem, default_round):
    """hcb200_count_solutions (per-hypothesis converged / infinity / real counts reduced on the GPU) against the host's walk over every end
    point (Evaluations::Evaluate_HC_Sols, reference Evaluations.cpp:145-167) and against hc.count_solutions, and the host class gives the
    same round statistics with Device_Statistics on and off."""
    picked, target, diff = default_round
    trk = hc.Tracker(problem=problem)
    trk.upload_params(target, diff)
    trk.track(100, prune=True)
    tr, cv, inf, _ = trk.results(100)
    assert np.array_equal(trk.count_solutions_device(100), hc.count_solutions(tr, cv, inf, 100))
    a = HostSolver(tree, "Num_Of_GPUs=1;Device_Statistics=true")
    ra = a.round()
    a.close()
    b = HostSolver(tree, "Num_Of_GPUs=1;Device_Statistics=false")
    rb = b.round()
    b.close()
    assert np.array_equal(ra["per"], rb["per"]) and np.array_equal(ra["totals"], rb["totals"])
    assert np.array_equal(ra["per"].astype(np.int64), hc.count_solutions(tr, cv, inf, 100))


def test_lazy_results_host_class(tree):
    """Lazy_Results=true: statistics, scoring and the selected pose come from the GPU; the stacked end points are copied back only when
    asked for, and are then the golden ones."""
    g = np.load(os.path.join(GOLD, "oracle_seed0_h100_prune.npz"))
    s = HostSolver(tree, "Num_Of_GPUs=1;Lazy_Results=true")
    r0 = s.round(fetch=False)
    assert np.array_equal(r0["per"].astype(np.int32), g["counts"]) and r0["selected_path"] == 104 and r0["selected_support"] == [5117, 5117]
    assert r0["pose_found"] == 1 and max(r0["residuals"][:2]) < 0.1
    r1 = s.round(fetch=True)
    s.close()
    assert np.array_equal(np.packbits(r1["conv"]), g["converged_bits"]) and np.array_equal(np.packbits(r1["inf"]), g["infinity_bits"])
    assert np.array_equal(r1["tracks"][104].view(np.uint64), g["track104_h0"].view(np.uint64))


def test_device_scoring_is_pinned_to_the_reference_util(problem, ransac0, default_round):
    """(f2) hcb200_score_tracks against the REFERENCE's MVG helpers (magmaHC/util.hpp:29-209 through oracle/_ref/libref_cpuhc.so; golden
    tests/golden/ref_util_support.npz): same candidates, same selected pose, inlier counts identical on >= 34 of the 36 candidates and
    within one edgel on the rest (the reference binary is FMA-contracted, the kernel is not: tests/test_host_cpu.py), and the pose in
    the 128-byte exchange record equals the reference's normalised (R21, t21, R31, t31) to float rounding."""
    picked, target, diff = default_round
    g = np.load(os.path.join(GOLD, "ref_util_support.npz"))
    trk = hc.Tracker(problem=problem)
    trk.set_edgels(ransac0["locations"], ransac0["K"])
    trk.upload_params(target, diff)
    trk.track(100, prune=True)
    support, best = trk.score_tracks(100)
    assert np.array_equal(support[:, 0] >= 0, g["support"][:, 0] >= 0)              # the same candidate set
    d = np.abs(support - g["support"]).max(1)
    assert d.max() <= 1 and (d[g["candidates"]] == 0).sum() >= 34 and d[104] == 0
    assert best[0] == 1 and best[1] == 104 and best[4] == len(g["candidates"])
    import torch
    rec = hc.decode_pose_record(trk.make_pose_record(0, 0).cpu().numpy())
    torch.cuda.synchronize()
    ref_pose = g["poses"][g["candidates"].tolist().index(104)]
    mine = np.concatenate([rec["R21"].reshape(-1), rec["t21"], rec["R31"].reshape(-1), rec["t31"]])
    assert rec["path_id"] == 104 and (rec["inliers21"], rec["inliers31"]) == (5117, 5117)
    assert np.abs(mine - ref_pose).max() < 2e-6


def test_launch_is_stream_ordered_and_graph_capturable(problem, default_round):
    """The C ABI only ENQUEUES (workspace reset + one kernel) on the caller's stream — no synchronisation, no allocation — so a round
    can be captured in a CUDA graph and replayed; the replay gives the same bits as a direct launch."""
    import torch
    picked, target, diff = default_round
    H = 8
    trk = hc.Tracker(problem=problem)
    trk.upload_params(target[:H], diff[:H])
    trk.track(H, prune=True)
    tr0, cv0, inf0, _ = trk.results(H)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        trk.track(H, prune=True)                       # warm-up on the capture stream (function attributes are set here)
        side.synchronize()
        with torch.cuda.graph(graph, stream=side):
            trk.track(H, prune=True)
    for _ in range(2):
        trk.d_tracks.zero_(); trk.d_conv.zero_(); trk.d_inf.zero_()
        torch.cuda.synchronize()
        graph.replay()
        torch.cuda.synchronize()
        tr1, cv1, inf1, _ = trk.results(H)
        assert np.array_equal(cv0, cv1) and np.array_equal(inf0, inf1)
        assert np.array_equal(np.ascontiguousarray(tr0).view(np.uint64), np.ascontiguousarray(tr1).view(np.uint64)) or \
            bool(np.all((np.ascontiguousarray(tr0).view(np.uint64) == np.ascontiguousarray(tr1).view(np.uint64)) | np.isnan(tr0) & np.isnan(tr1)))
