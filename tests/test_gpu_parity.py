"""GPU parity tests proper: the CUDA tracker, called through the C ABI (include/hcb200.h), against the CPU oracle
(oracle/hc_oracle.c) on the same seeded inputs.  Bar: bit-exact — converged / infinity flags, per-path counters and
every end-point component are identical (NaNs compare equal), because kernel and oracle follow one arithmetic spec."""
import numpy as np
import pytest

from trifocal_pose_estimation_using_improved_gpuhc_b200 import hc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def tracker(problem):
    return hc.Tracker(problem=problem, stats=True)


def _bit_equal(a, b):
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    av, bv = a.view(np.uint32), b.view(np.uint32)
    both_nan = np.isnan(a.view(np.float32)) & np.isnan(b.view(np.float32))
    return bool(np.all((av == bv) | both_nan))


@pytest.mark.parametrize("prune", [True, False])
def test_tracker_bit_exact_vs_oracle(tracker, oracle, ransac0, prune):
    n_hyp = 3
    target, diff, _ = oracle.prepare_target_params(0, n_hyp, ransac0["locations"], ransac0["tangents"])
    tr_o, cv_o, inf_o, st_o = oracle.track(target, diff, prune)
    tracker.upload_params(target, diff)
    tracker.track(n_hyp, prune=prune)
    tr_g, cv_g, inf_g, st_g = tracker.results(n_hyp)
    assert np.array_equal(cv_g, cv_o), "converged flags differ on %d paths" % int((cv_g != cv_o).sum())
    assert np.array_equal(inf_g, inf_o)
    assert np.array_equal(st_g[:, 0], st_o[:, 0])          # steps
    assert np.array_equal(st_g[:, 1], st_o[:, 1])          # predictor stages
    assert np.array_equal(st_g[:, 2], st_o[:, 2])          # corrector stages
    assert np.array_equal(st_g[:, 3] & 0xffff, st_o[:, 3])  # rejected steps
    assert np.array_equal(st_g[:, 3] >> 16, st_o[:, 4])     # end reason
    assert _bit_equal(tr_g[:, :30], tr_o[:, :30])
    assert np.all(tr_g[:, 30] == 1.0)
    counts = hc.count_solutions(tr_g, cv_g, inf_g, n_hyp)
    assert np.array_equal(counts, hc.count_solutions(tr_o, cv_o, inf_o, n_hyp))


def test_abort_finds_gt_pose(tracker, oracle, ransac0):
    """Abort_RANSAC_by_Good_Sol = true: seed 0, hypothesis 0 / track 104 is the GT pose (SURVEY.md App. C.1)."""
    n_hyp = 4
    target, diff, _ = oracle.prepare_target_params(0, n_hyp, ransac0["locations"], ransac0["tangents"])
    tracker.set_edgels(ransac0["locations"], ransac0["K"])
    tracker.upload_params(target, diff)
    tracker.track_abort(n_hyp, prune=True)
    tr_g, cv_g, inf_g, st_g = tracker.results(n_hyp)
    found = int(tracker.d_found.cpu()[0])
    idx = tracker.d_found_index[: n_hyp * 312].cpu().numpy()
    best = tracker.d_best.cpu().numpy()
    assert found == 1
    hits = np.nonzero(idx >= 0)[0]
    assert len(hits) >= 1 and np.array_equal(idx[hits], hits)
    # every flagged path must pass the oracle's scoring of the SAME end point, with the same inlier counts
    for b in hits:
        ok, n21, n31, gate = oracle.score(tr_g[b], ransac0["locations"], ransac0["K"])
        assert ok and gate and cv_g[b] == 1
    assert best[0] == 1 and best[1] == hits.min() and best[4] == len(hits)
    ok, n21, n31, _ = oracle.score(tr_g[best[1]], ransac0["locations"], ransac0["K"])
    assert (best[2], best[3]) == (n21, n31)
    assert 104 in hits          # hypothesis 0, track 104
    assert (n21, n31) == (5117, 5117) or best[1] != 104


def test_device_target_params_match_host(tracker, oracle, ransac0):
    import torch
    n_hyp = 64
    target, diff, picked = oracle.prepare_target_params(3, n_hyp, ransac0["locations"], ransac0["tangents"])
    tracker.set_edgels(ransac0["locations"], ransac0["K"])
    tracker.reserve(n_hyp)
    d_picked = torch.from_numpy(picked).to(tracker.device)
    d_tan = torch.from_numpy(np.ascontiguousarray(ransac0["tangents"])).to(tracker.device)
    tracker.build_target_params(d_picked, d_tan, n_hyp)
    torch.cuda.synchronize()
    t = tracker.d_target[:n_hyp].cpu().numpy()
    d = tracker.d_diff[:n_hyp].cpu().numpy()
    assert np.array_equal(t[..., 0] + 1j * t[..., 1], target)
    assert np.array_equal((d[..., 0] + 1j * d[..., 1]).astype(np.complex64), diff)
    # and the python host mirror of Prepare_Target_Params agrees with both
    p2 = hc.sample_hypotheses(3, n_hyp, ransac0["locations"].shape[0])
    assert np.array_equal(p2, picked)
    t2, d2 = hc.target_params_from_picks(p2, ransac0["locations"], ransac0["tangents"], oracle.start_params)
    assert np.array_equal(t2, target) and np.array_equal(d2, diff)


def _assert_same(tracker, oracle, target, diff, prune):
    n_hyp = target.shape[0]
    tr_o, cv_o, inf_o, st_o = oracle.track(target, diff, prune)
    tracker.upload_params(target, diff)
    tracker.track(n_hyp, prune=prune)
    tr_g, cv_g, inf_g, st_g = tracker.results(n_hyp)
    assert np.array_equal(cv_g, cv_o) and np.array_equal(inf_g, inf_o)
    assert np.array_equal(st_g[:, :3], st_o[:, :3])
    assert np.array_equal(st_g[:, 3] & 0xffff, st_o[:, 3]) and np.array_equal(st_g[:, 3] >> 16, st_o[:, 4])
    assert _bit_equal(tr_g[:, :30], tr_o[:, :30])
    return tr_g, cv_g, inf_g, st_g


@pytest.mark.parametrize("dataset", [1, 2, 3])
def test_other_datasets_bit_exact(tracker, oracle, dataset):
    """RANSAC_Data/Synthetic/001-003 (SURVEY.md §8d config 5 draws hypotheses from the other dataset files)."""
    from trifocal_pose_estimation_using_improved_gpuhc_b200 import fixtures
    rs = fixtures.load_ransac(dataset)
    target, diff, _ = oracle.prepare_target_params(dataset, 2, rs["locations"], rs["tangents"])
    _assert_same(tracker, oracle, target, diff, True)


@pytest.mark.parametrize("prune", [True, False])
def test_random_complex_targets_bit_exact(tracker, oracle, prune):
    """Second input distribution of SURVEY.md §8d config 5: target = U(0,1) + i U(0,1) (the reference's Julia start-system
    script draws its parameters this way).  Generic complex targets keep almost every path alive to the step cap or send it
    to infinity, so this exercises the long-path, overflow and NaN branches that edgel-derived (real) targets rarely reach."""
    rng = np.random.default_rng(20240607)
    n_hyp = 2
    target = np.zeros((n_hyp, 34), np.complex64)
    target[:, :33] = (rng.random((n_hyp, 33)) + 1j * rng.random((n_hyp, 33))).astype(np.complex64)
    target[:, 33] = 1.0
    diff = (target - oracle.start_params[None, :]).astype(np.complex64)
    diff[:, 33] = 0.0
    tr_g, cv_g, inf_g, st_g = _assert_same(tracker, oracle, target, diff, prune)
    assert st_g[:, 0].max() >= 40          # long paths were exercised


def test_degenerate_targets_bit_exact(tracker, oracle):
    """target == start (zero parameter velocity: every predictor stage solves A k = 0), an all-zero target (singular Jacobians,
    zero pivots), a huge target (overflow -> the infinity exit) and NaN / Inf parameters (NaN pivot keys and norms)."""
    start = oracle.start_params.astype(np.complex64)
    target = np.zeros((5, 34), np.complex64)
    target[0] = start
    target[2, :33] = np.complex64(3.0e18 + 1.0e18j)
    target[3] = start
    target[3, 5] = np.complex64(complex(np.nan, 0.0))          # NaN parameter: NaN pivots, NaN norms
    target[4] = start
    target[4, 7] = np.complex64(complex(np.inf, 0.0))          # Inf parameter
    target[:, 33] = 1.0
    diff = (target - start[None, :]).astype(np.complex64)
    diff[:, 33] = 0.0
    tr_g, cv_g, inf_g, st_g = _assert_same(tracker, oracle, target, diff, False)
    # target == start: the start solutions already solve the system; every path runs to t = 1 and converges where it began
    assert cv_g[:312].all()


def test_abort_late_hit(tracker, oracle, ransac0):
    """SURVEY.md §8d config 3, second half: a sampler seed whose first passing pose comes late in the round (seed 13: hypothesis
    30, path 9606 — found with tools/find_abort_seeds.py).  The oracle tracks and scores all 40 hypotheses; the abort launch must
    flag only paths the oracle also passes, none before the oracle's first, and must skip the work queued behind the flag."""
    n_hyp = 40
    loc, K = ransac0["locations"], ransac0["K"]
    target, diff, _ = oracle.prepare_target_params(13, n_hyp, loc, ransac0["tangents"])
    tr_o, cv_o, inf_o, st_o = oracle.track(target, diff, True)
    passing = [int(b) for b in np.nonzero(cv_o)[0] if oracle.score(tr_o[b], loc, K)[0]]
    assert passing and min(passing) == 9606
    tracker.set_edgels(loc, K)
    tracker.upload_params(target, diff)
    tracker.track_abort(n_hyp, prune=True)
    tr_g, cv_g, inf_g, st_g = tracker.results(n_hyp)
    idx = tracker.d_found_index[: n_hyp * 312].cpu().numpy()
    best = tracker.d_best.cpu().numpy()
    hits = np.nonzero(idx >= 0)[0]
    assert int(tracker.d_found.cpu()[0]) == 1 and len(hits) >= 1
    assert set(hits.tolist()) <= set(passing)
    assert best[0] == 1 and best[1] == hits.min() and best[4] == len(hits)
    for b in hits:                                   # a flagged path ran to completion: same end point as the oracle, bit for bit
        assert _bit_equal(tr_g[b, :30], tr_o[b, :30])
    reason = st_g[:, 3] >> 16
    assert (reason == 4).sum() > 0                   # work behind the flag was skipped
    done = reason < 4                                # paths that finished before the flag are the oracle's, bit for bit
    assert np.array_equal(cv_g[done], cv_o[done]) and _bit_equal(tr_g[done][:, :30], tr_o[done][:, :30])


def test_device_refinement_bit_exact_vs_oracle(tracker, oracle, ransac0):
    """hcb200_refine_tracks: Newton refinement of converged end points against their target systems, same arithmetic spec as the
    tracker's corrector -> bit-identical to the oracle's hco_refine_path; paths that did not converge are left alone."""
    n_hyp = 3
    target, diff, _ = oracle.prepare_target_params(0, n_hyp, ransac0["locations"], ransac0["tangents"])
    tracker.upload_params(target, diff)
    tracker.track(n_hyp, prune=True)
    tr0, cv, inf, _ = tracker.results(n_hyp)
    sums = tracker.refine_tracks(n_hyp, iters=3)
    tr1, cv1, _, _ = tracker.results(n_hyp)
    assert np.array_equal(cv, cv1)
    not_conv = cv == 0
    assert _bit_equal(tr1[not_conv], tr0[not_conv]) and np.all(sums[not_conv] == -1.0)
    conv = np.nonzero(cv)[0]
    assert len(conv) > 50
    for b in conv:
        x, sd, sx = oracle.refine(target[b // 312], tr0[b], iters=3)
        assert _bit_equal(tr1[b, :30], x[:30]), b
        assert _bit_equal(np.array([sd, sx], np.float32), sums[b]), b
    # the ground-truth pose (hypothesis 0 / track 104) is a regular solution: the polish settles at the float floor
    assert sums[104, 0] < 1e-8 * sums[104, 1]
    # iters = 0: nothing moves
    tracker.refine_tracks(n_hyp, iters=0)
    tr2, _, _, _ = tracker.results(n_hyp)
    assert _bit_equal(tr2, tr1)


@pytest.mark.parametrize("prune", [True, False])
def test_split_long_paths_gives_identical_results(problem, ransac0, prune):
    """HCB200_FLAG_SPLIT_LONG_PATHS parks a path at a step boundary and resumes it on another warp: flags, end points and every counter must
    be those of the unsplit kernel bit for bit, wherever the cut is made (step 1: every path is cut; 79: only step-capped ones; default 64)."""
    H = 60
    picked = hc.sample_hypotheses(3, H, ransac0["locations"].shape[0])
    target, diff = hc.target_params_from_picks(picked, ransac0["locations"], ransac0["tangents"], problem["start_params"])
    base = hc.Tracker(problem=problem, stats=True, split=False)
    base.upload_params(target, diff)
    base.track(H, prune=prune)
    tr0, cv0, inf0, st0 = base.results(H)
    assert (st0[:, 0] > 64).sum() > 1000                      # there ARE long paths to cut
    trk = hc.Tracker(problem=problem, stats=True, split=True)
    trk.upload_params(target, diff)
    for cut in (0, 1, 2, 17, 64, 79, 80, 81):
        trk.suspend_step = cut
        trk.d_tracks.zero_(); trk.d_conv.fill_(7); trk.d_inf.fill_(7)
        for rep in range(2):                                  # (twice: the launch must leave the workspace reusable)
            trk.track(H, prune=prune)
        tr, cv, inf, st = trk.results(H)
        assert np.array_equal(cv, cv0) and np.array_equal(inf, inf0), cut
        assert np.array_equal(st, st0), cut
        assert _bit_equal(tr, tr0), cut


def test_early_abort_flag_crosses_gpus(problem, oracle, ransac0):
    """hcb200_track_abort_peers: GPU 1 is given edgels no pose can match, so on its own it tracks its whole shard; with GPU 0 as a peer in the same
    round it stops as soon as GPU 0's first passing path raises its flag through the NVLink peer mapping.  What GPU 1 did finish is its no-abort
    result, bit for bit; its own record says it found nothing."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    H = 100
    picked = hc.sample_hypotheses(0, H, ransac0["locations"].shape[0])
    target, diff = hc.target_params_from_picks(picked, ransac0["locations"], ransac0["tangents"], problem["start_params"])
    a = hc.Tracker(device="cuda:0", problem=problem, stats=True)
    b = hc.Tracker(device="cuda:1", problem=problem, stats=True)
    a.set_edgels(ransac0["locations"], ransac0["K"])
    rng = np.random.RandomState(5)
    b.set_edgels((rng.rand(*ransac0["locations"].shape) * 0.4 - 0.2).astype(np.float32), ransac0["K"])      # nothing reprojects within 2 px
    a.upload_params(target, diff)
    b.upload_params(target, diff)
    b.track(H, prune=True)
    tr_full, cv_full, inf_full, st_full = b.results(H)
    # GPU 1 alone: no hit, the whole shard is tracked
    b.track_abort(H, prune=True)
    tr1, cv1, inf1, st1 = b.results(H)
    assert int(b.d_found.cpu()[0]) == 0 and np.array_equal(cv1, cv_full) and ((st1[:, 3] >> 16) != 4).all()
    # the same round with GPU 0 as a peer: both stop on GPU 0's hit
    a.reset_abort(H); b.reset_abort(H)
    torch.cuda.synchronize(0); torch.cuda.synchronize(1)
    b.track_abort(H, prune=True, peers=[a], reset=False)
    a.track_abort(H, prune=True, peers=[b], reset=False)
    tr_a, cv_a, inf_a, st_a = a.results(H)
    tr_b, cv_b, inf_b, st_b = b.results(H)
    assert int(a.d_found.cpu()[0]) == 1 and int(b.d_found.cpu()[0]) == 1
    best_a, best_b = a.d_best.cpu().numpy(), b.d_best.cpu().numpy()
    assert best_a[0] == 1 and best_a[1] == 104 and best_b[0] == 0          # GPU 0 found track 104 of hypothesis 0; GPU 1 found nothing itself
    assert (b.d_found_index[:H * 312].cpu().numpy() == -1).all()
    cut = (st_b[:, 3] >> 16) == 4                                           # skipped or stopped by the flag
    assert cut.sum() > 20000, int(cut.sum())                                # GPU 1 did NOT track its whole shard this time
    ran = ~cut
    assert np.array_equal(cv_b[ran], cv_full[ran]) and np.array_equal(inf_b[ran], inf_full[ran])
    assert _bit_equal(tr_b[ran][:, :30], tr_full[ran][:, :30])


def test_split_workspace_is_not_overrun(problem, ransac0):
    """The split kernel writes a list entry and 16 bytes of state per parked path behind the 256-byte header: with EVERY path parked (step 1) the
    bytes beyond hcb200_workspace_bytes_for(H) must stay untouched, and so must the tail of the result arrays."""
    import torch
    H = 40
    picked = hc.sample_hypotheses(9, H, ransac0["locations"].shape[0])
    target, diff = hc.target_params_from_picks(picked, ransac0["locations"], ransac0["tangents"], problem["start_params"])
    trk = hc.Tracker(problem=problem, stats=True, split=True)
    trk.upload_params(target, diff)
    need = int(trk.lib.hcb200_workspace_bytes_for(H))
    ws = torch.full((need + 4096,), 0xA5, dtype=torch.uint8, device=trk.device)
    trk.d_ws = ws
    pad = 64
    tracks = torch.full((H * 312 * 31 * 2 + pad,), 7.0, dtype=torch.float32, device=trk.device)
    trk.d_tracks = tracks[:H * 312 * 31 * 2].view(H * 312, 31, 2)
    for cut in (1, 64):
        trk.suspend_step = cut
        trk.track(H, prune=True)
        torch.cuda.synchronize()
        assert bool((ws[need:] == 0xA5).all()), cut
        assert bool((tracks[H * 312 * 31 * 2:] == 7.0).all()), cut
    parked = ws[256:256 + H * 312 * 4].view(torch.int32)
    assert int((parked != 0).sum()) > 1000          # the list was really used


def test_repeated_launches_are_identical(problem, ransac0):
    """No race: warps hand paths to each other through atomics, shared-memory rows and (split mode) parked state, in an order that differs from
    launch to launch — the results must not."""
    H = 100
    picked = hc.sample_hypotheses(0, H, ransac0["locations"].shape[0])
    target, diff = hc.target_params_from_picks(picked, ransac0["locations"], ransac0["tangents"], problem["start_params"])
    for split in (True, False):
        trk = hc.Tracker(problem=problem, stats=True, split=split)
        trk.upload_params(target, diff)
        first = None
        for rep in range(8):
            trk.d_tracks.zero_()
            trk.track(H, prune=True)
            out = trk.results(H)
            if first is None:
                first = out
            else:
                assert np.array_equal(out[1], first[1]) and np.array_equal(out[2], first[2]) and np.array_equal(out[3], first[3]), (split, rep)
                assert _bit_equal(out[0], first[0]), (split, rep)
