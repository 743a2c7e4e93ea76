"""The HC tracker's step control across its run-time settings, down to a zero step size, and the settings the path counters cannot hold.

`hcb200_track`, the early-abort entry points and the batched abort take GPUHC_Max_Steps, GPUHC_Max_Correction_Steps and
GPUHC_Num_Of_Steps_to_Increase_Delta_t at run time.  Each entry of SETTINGS is (max_steps, max_corr, dt_inc) and tests one edge:

  (-1, 3, 4)                      no step runs: the end point is the start solution
  (0, 3, 4) (40, 2, 2) (120, 5, 6) (80, 1, 1)   small caps, one and two corrector steps, doubling after every accepted step
  (9, 3, 4) / (10, 3, 4)          either side of the split kernel's step limit (it needs max_steps >= 10)
  (200, 3, 255) / (200, 3, 256)   either side of its dt_inc limit (the parked state holds the success counter in 8 bits)
  (300, 4, 4)                     paths that keep being rejected halve delta_t through the subnormal range to exactly 0
  (1022, 4, 4)                    the packed counters filled: 1 023 steps, 4 059 corrector stages, 1 004 rejections on input R
  (1022, 4, 0) (1022, 4, -3)      dt_inc <= 0: delta_t doubles after every accepted step
  (80, 50, 4)                     up to 81 * 50 = 4 050 corrector stages at the default cap
  (1023, 3, 4) (1100, 5, 4)       more steps than the counters hold: refused with stats, tracked without

Inputs (all seeded): R, the random complex targets of test_gpu_parity.py (seed 20240607, 2 hypotheses); E, dataset 0 with sampler seed 5
(1 hypothesis); E0, dataset 0 with sampler seed 0 (8 hypotheses; track 104 is the ground-truth pose).

CPU part: the oracle's per-step trace shows that the inputs reach the edges; a numpy float32 restatement of the step-size rules reproduces
every traced t0 and delta_t bit for bit, subnormals and zeros included; the counters keep their invariants for the whole table; the
launchers refuse what the packed counters cannot hold.  GPU part: every kernel against the oracle, bit for bit (flags, end points, counters).
"""
import ctypes
import os

import numpy as np
import pytest

from trifocal_pose_estimation_using_improved_gpuhc_b200 import fixtures, hc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROBLEMS = sorted(os.listdir(os.path.join(ROOT, "problems")))
T = hc.NUM_TRACKS
INT_MAX = 2 ** 31 - 1
INVALID_VALUE = 1
TINY = np.float32(2.0 ** -126)          # smallest normal float32

SETTINGS = [(-1, 3, 4), (0, 3, 4), (40, 2, 2), (120, 5, 6), (80, 1, 1), (9, 3, 4), (10, 3, 4), (200, 3, 255), (200, 3, 256),
            (300, 4, 4), (1022, 4, 4), (1022, 4, 0), (1022, 4, -3), (80, 50, 4)]
NO_STATS = [(1023, 3, 4), (1100, 5, 4)]
ZERO_STEP = [(300, 4, 4), (1022, 4, 4), (1022, 4, 0), (1022, 4, -3)]


def _split_eligible(setting):
    """The launcher's condition for the split kernel (hc_tracker.cu, launch_common)."""
    ms, _, di = setting
    return 10 <= ms < 1024 and di < 256


# ---------------------------------------------------------------------------------------------------------------------
# inputs and oracle runs (cached: the CPU and GPU parts share them)

_RUNS = {}


def _complex_targets(start_params, n_hyp, seed):
    """target = U(0,1) + i U(0,1) per parameter, pad 1; diff = target - start component-wise in float32 (pad 0)."""
    rng = np.random.default_rng(seed)
    n = start_params.shape[0] - 1
    target = np.zeros((n_hyp, n + 1), np.complex64)
    target[:, :n] = (rng.random((n_hyp, n)) + 1j * rng.random((n_hyp, n))).astype(np.complex64)
    target[:, n] = 1.0
    diff = np.empty_like(target)
    diff.real, diff.imag = target.real - start_params.real[None, :], target.imag - start_params.imag[None, :]
    diff[:, n] = 0.0
    return target, diff


def _inputs(oracle, name):
    if name == "R":
        return _complex_targets(oracle.start_params, 2, 20240607)
    rs = fixtures.load_ransac(0)
    seed, n_hyp = {"E": (5, 1), "E0": (0, 8)}[name]
    target, diff, _ = oracle.prepare_target_params(seed, n_hyp, rs["locations"], rs["tangents"])
    return target, diff


def _oracle(oracle, name, setting, prune):
    key = (name, setting, prune)
    if key not in _RUNS:
        target, diff = _inputs(oracle, name)
        ms, mc, di = setting
        _RUNS[key] = oracle.track(target, diff, prune, max_steps=ms, max_corr=mc, dt_inc=di)
    return _RUNS[key]


def _replay(accepted, dt_inc):
    """The step-size rules in numpy float32, driven by a traced accept / reject sequence.  Returns the t0 and delta_t of every step, which
    steps the end zone clamped, t0 after the last step, and the state a path carries into each step: (delta_t before the clamps, success
    counter, end-zone flag)."""
    f32 = np.float32
    t0, dt, end_zone, counter = f32(0.0), f32(0.01), False, 0
    n = len(accepted)
    t0s, dts, clamped = np.empty(n, np.float32), np.empty(n, np.float32), np.zeros(n, bool)
    carried = []
    for i, acc in enumerate(accepted):
        carried.append((dt, counter, end_zone))
        if not end_zone and float(abs(f32(1.0) - t0)) <= 0.0500001:
            end_zone = True
        if end_zone:                                         # the last 5 %: never step beyond t = 1
            r = abs(f32(1.0) - t0)
            if dt > r:
                dt, clamped[i] = r, True
        else:                                                # before it: never step beyond t = 0.95 (compared in double)
            r = abs(0.95 - float(t0))
            if float(dt) > r:
                dt = f32(r)
        t0s[i], dts[i] = t0, dt
        half = f32(0.5) * dt
        if acc:                                              # RK4 stages 0 and 2 each advance t0 by half a step
            t0 = (t0 + half) + half
            counter += 1
            if counter >= dt_inc:
                counter, dt = 0, dt * f32(2.0)
        else:                                                # rejected: same t0, half the step
            dt, counter = dt * f32(0.5), 0
    return t0s, dts, clamped, t0, carried


def _traced_paths(st):
    """Up to 12 paths that reached the step cap, evenly spread, plus every 39th path of the round (all end reasons)."""
    capped = np.nonzero(st[:, 4] == 3)[0]
    return sorted(set(capped[::max(1, len(capped) // 12)].tolist()) | set(range(0, st.shape[0], 39)))


# ---------------------------------------------------------------------------------------------------------------------
# CPU

def test_inputs_reach_the_step_control_edges(oracle):
    """The oracle's trace of input R shows the edges the table claims: delta_t becomes subnormal and then exactly 0 in the settings of
    ZERO_STEP, steps are clamped inside the end zone, paths reach the step cap, and (1022, 4, 4) fills the counter fields."""
    target, diff = _inputs(oracle, "R")
    for setting in ZERO_STEP:
        ms, mc, di = setting
        tr, cv, inf, st = _oracle(oracle, "R", setting, False)
        capped = np.nonzero(st[:, 4] == 3)[0]
        assert len(capped) >= 10, setting
        through_zero = 0
        for p in capped:
            t0, dt, acc, s = oracle.trace_path(target[p // T], diff[p // T], p % T, False, ms, mc, di)
            sub = np.nonzero((dt > 0) & (dt < TINY))[0]
            zero = np.nonzero(dt == 0)[0]
            if len(sub) and len(zero) and sub[0] < zero[0]:
                through_zero += 1
                assert (dt[zero[0]:] == 0).all()             # once 0, delta_t stays 0 (0 * 2 == 0): the path burns steps up to the cap
        assert through_zero >= 10, (setting, through_zero)
    tr, cv, inf, st = _oracle(oracle, "R", (1022, 4, 4), False)
    assert st[:, 0].max() == 1023 and st[:, 2].max() == 4059 and st[:, 3].max() == 1004
    assert (st[:, 0] == 1023).sum() == 18
    tr, cv, inf, st = _oracle(oracle, "R", (1100, 5, 4), False)
    assert st[:, 0].max() == 1101 and st[:, 2].max() > 4095          # what the refused settings would have wrapped
    for setting in [(40, 2, 2), (300, 4, 4), (1022, 4, 0)]:
        ms, mc, di = setting
        tr, cv, inf, st = _oracle(oracle, "R", setting, False)
        clamps = 0
        for p in np.nonzero(cv)[0][:20]:
            t0, dt, acc, s = oracle.trace_path(target[p // T], diff[p // T], p % T, False, ms, mc, di)
            clamps += int(_replay(acc, di)[2].sum())
        assert clamps > 0, setting
    for setting in SETTINGS + NO_STATS:
        if setting[0] >= 0:
            assert (_oracle(oracle, "R", setting, False)[3][:, 4] == 3).any(), setting


@pytest.mark.parametrize("name", ["R", "E"])
@pytest.mark.parametrize("setting", [s for s in SETTINGS + NO_STATS if s[0] >= 0], ids=str)
def test_step_size_rules_replayed_in_float32(oracle, name, setting):
    """Halving on a rejection, doubling after dt_inc accepted steps (every step for dt_inc <= 0), the clamps to 0.95 - t0 and 1 - t0 and
    the t0 advance by two halves, restated in numpy float32, give the oracle's t0 and delta_t at every step bit for bit; the number of steps,
    the end at the cap and the converged flag follow from them."""
    ms, mc, di = setting
    target, diff = _inputs(oracle, name)
    for prune in (False, True):
        tr, cv, inf, st = _oracle(oracle, name, setting, prune)
        for p in _traced_paths(st):
            t0, dt, acc, s = oracle.trace_path(target[p // T], diff[p // T], p % T, prune, ms, mc, di)
            assert np.array_equal(s, st[p]), p
            r_t0, r_dt, _, t_end, _ = _replay(acc, di)
            assert np.array_equal(r_t0.view(np.uint32), t0.view(np.uint32)), (p, np.nonzero(r_t0 != t0)[0][:3])
            assert np.array_equal(r_dt.view(np.uint32), dt.view(np.uint32)), (p, np.nonzero(r_dt != dt)[0][:3])
            assert len(acc) == s[0] and s[3] == (~acc).sum() - (s[4] == 1)          # the step that overflowed is neither
            if s[4] == 1:                           # the overflow ends the path inside its step, after the predictor's two half steps
                half = np.float32(0.5) * dt[-1]
                t_end = (t0[-1] + half) + half
            assert bool(cv[p]) == (float(t_end) >= 1.0 or 1.0 - float(t_end) <= 1e-7), p
            if s[4] == 3:
                assert len(acc) == ms + 1


@pytest.mark.parametrize("name", ["R", "E"])
def test_counter_invariants_on_the_oracle(oracle, name):
    """For the whole table, both pruning modes: 4 predictor stages per step; rejected <= steps; accepted steps <= corrector stages <=
    steps * max_corr; end reason 3 only at steps == max_steps + 1; reason 2 only with pruning; converged paths end with reason 0, or with
    reason 1 when the corrector overflows in a step whose predictor reached t = 1; max_steps < 0 tracks nothing."""
    start = np.tile(oracle.start_sols, (_inputs(oracle, name)[0].shape[0], 1))
    for setting in SETTINGS + NO_STATS:
        ms, mc, di = setting
        for prune in (False, True):
            tr, cv, inf, st = _oracle(oracle, name, setting, prune)
            steps, pred, corr, rej, reason = st.T
            accepted = steps - rej - (reason == 1)
            assert np.array_equal(pred, 4 * steps), setting
            assert (rej <= steps).all() and (accepted >= 0).all(), setting
            assert (accepted <= corr).all() and (corr <= steps * mc).all(), setting
            assert (steps <= max(ms + 1, 0)).all(), setting
            assert (steps[reason == 3] == max(ms + 1, 0)).all(), setting
            assert prune or not (reason == 2).any(), setting
            assert (cv[reason == 0] == 1).all() and (cv[reason > 1] == 0).all(), setting      # (an overflow in the last step can converge)
            if ms < 0:
                assert (steps == 0).all() and (reason == 3).all() and not cv.any() and not inf.any()
                assert np.array_equal(tr, start)


def _fake_pointers(n):
    return [ctypes.c_void_p(0x1000 * (i + 1)) for i in range(n)]


def _call_entry(lib, entry, max_steps, max_corr, stats):
    """One track entry point with fake (never dereferenced) device pointers.  Only for settings the launcher refuses: a call it accepted
    would launch on them."""
    if entry == "track":
        bufs = _fake_pointers(9)
        bufs[7] = bufs[7] if stats else None                 # d_stats
        return lib.hcb200_track(None, 1, max_steps, max_corr, 4, hc.FLAG_PRUNE_PATHS, *bufs)
    bufs = _fake_pointers(14)
    bufs[12] = bufs[12] if stats else None                   # d_stats
    if entry == "abort":
        return lib.hcb200_track_abort(None, 1, 10, max_steps, max_corr, 4, hc.FLAG_PRUNE_PATHS, *bufs)
    if entry == "peers":
        return lib.hcb200_track_abort_peers(None, 1, 10, max_steps, max_corr, 4, hc.FLAG_PRUNE_PATHS, *bufs, None, 0)
    offsets = np.array([0, 10, 25], np.int32)
    return lib.hcb200_track_abort_batched(None, 2, 1, offsets.ctypes.data_as(ctypes.c_void_p), max_steps, max_corr, 4, hc.FLAG_PRUNE_PATHS,
                                          *bufs)


REFUSED = [(1023, 3, True),            # 1 024 steps: the steps field holds 1 023
           (1022, 5, True),            # 1 023 * 5 = 5 115 corrector stages: the field holds 4 095
           (80, 51, True),             # 81 * 51 = 4 131
           (INT_MAX, 3, False),        # step <= max_steps never ends
           (80, INT_MAX - 3, False)]   # 4 + max_corr overflows int


@pytest.mark.parametrize("entry", ["track", "abort", "peers", "batched"])
@pytest.mark.parametrize("max_steps,max_corr,stats", REFUSED)
def test_launchers_refuse_what_the_counters_cannot_hold(entry, max_steps, max_corr, stats):
    """cudaErrorInvalidValue before any CUDA call, so the result is the same without a GPU."""
    assert _call_entry(hc.load_library(), entry, max_steps, max_corr, stats) == INVALID_VALUE


@pytest.mark.parametrize("max_steps,max_corr,stats", REFUSED)
def test_compiled_problem_libraries_refuse_the_same_caps(max_steps, max_corr, stats):
    from trifocal_pose_estimation_using_improved_gpuhc_b200 import problem as pm
    built = [name for name in PROBLEMS if os.path.exists(pm.library_path(name))]
    if not built:
        pytest.skip("no compiled-problem library built (make problem PROBLEM_DIR=problems/<name>)")
    for name in built:
        assert _call_entry(pm.load_problem_library(pm.library_path(name)), "track", max_steps, max_corr, stats) == INVALID_VALUE, name


@pytest.mark.parametrize("name", PROBLEMS)
def test_compiled_problem_inputs_stay_above_the_subnormal_range(name):
    """The compiled problems' random complex targets (seed 7, 4 hypotheses) converge within 52 steps at every ZERO_STEP setting: on these
    problems the GPU runs below test the settings, not the subnormal regime, which the trifocal input R covers."""
    from oracle.pyoracle import Oracle
    from trifocal_pose_estimation_using_improved_gpuhc_b200 import problem as pm
    pdir = os.path.join(ROOT, "problems", name)
    prob = pm.read_problem(pdir)
    orc = Oracle(prob, problem_dir=pdir)
    target, diff = _complex_targets(orc.start_params, 4, 7)
    n_t = prob["spec"]["n_tracks"]
    for ms, mc, di in ZERO_STEP[:3]:
        tr, cv, inf, st = orc.track(target, diff, False, max_steps=ms, max_corr=mc, dt_inc=di)
        assert cv.all() and st[:, 0].max() <= 52, (ms, mc, di)
        p = int(np.argmax(st[:, 3]))                          # the path with the most rejections
        t0, dt, acc, s = orc.trace_path(target[p // n_t], diff[p // n_t], p % n_t, False, ms, mc, di)
        assert dt.min() >= TINY


# ---------------------------------------------------------------------------------------------------------------------
# GPU

def _bit_equal(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    av, bv = a.view(np.uint32), b.view(np.uint32)
    both_nan = np.isnan(a.view(np.float32)) & np.isnan(b.view(np.float32))
    return bool(np.all((av == bv) | both_nan))


def _assert_matches_oracle(got, ref, what, n_vars=30, stats=True):
    tr, cv, inf, st = got
    tr_o, cv_o, inf_o, st_o = ref
    assert np.array_equal(cv, cv_o) and np.array_equal(inf, inf_o), (what, int((cv != cv_o).sum()), int((inf != inf_o).sum()))
    assert _bit_equal(tr[:, :n_vars], tr_o[:, :n_vars]), what
    if stats:
        assert np.array_equal(st[:, 0], st_o[:, 0]), (what, np.nonzero(st[:, 0] != st_o[:, 0])[0][:5])
        assert np.array_equal(st[:, 1], st_o[:, 1]) and np.array_equal(st[:, 2], st_o[:, 2]), what
        assert np.array_equal(st[:, 3] & 0xffff, st_o[:, 3]) and np.array_equal(st[:, 3] >> 16, st_o[:, 4]), what


def _tile(ref, k):
    return tuple(np.concatenate([a] * k) for a in ref)


@pytest.fixture(scope="module")
def gpu(problem):
    """Trackers with and without stats, plain and split, sized for the largest launch; `tiles` copies of input R put more paths in the queue
    than the device has resident warps, so a path that reaches the suspend step while fresh paths wait is parked."""
    import torch
    plain = hc.Tracker(problem=problem, stats=True, split=False)
    info = plain.kernel_info()
    warps = info["grid"] * info["block"] // 32
    tiles = -(-4 * warps // (2 * T))
    trk = {(split, stats): hc.Tracker(problem=problem, stats=stats, split=split) for split in (False, True) for stats in (False, True)}
    for t in trk.values():
        t.reserve(2 * tiles)
    return dict(trk=trk, tiles=tiles, torch=torch)


def _track(trk, target, diff, setting, prune, suspend=0):
    """hcb200_track through the Tracker; returns (tracks, converged, infinity, stats) and the number of paths the split kernel parked."""
    trk.max_steps, trk.max_corr, trk.dt_inc = setting
    trk.suspend_step = suspend
    H = trk.upload_params(target, diff)
    if trk.split:
        trk.d_ws.zero_()
    trk.track(H, prune=prune)
    out = trk.results(H)
    parked = int((trk.d_ws[256:256 + 4 * H * T].view(trk.torch.int32) != 0).sum().item()) if trk.split else 0
    return out, parked


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["R", "E"])
@pytest.mark.parametrize("setting", SETTINGS + NO_STATS, ids=str)
def test_plain_and_split_kernels_match_the_oracle(gpu, oracle, name, setting):
    """Both pruning modes: the plain kernel, the split kernel at its own suspend step, and the split kernel parking at step 1 on input R or E
    repeated until the queue outlasts the first wave of warps.  Where the launcher may use the split kernel it must have parked paths; where
    it may not ((9, 3, 4), (200, 3, 256), caps >= 1024), nothing is parked.  At (1022, 4, 4) most paths are parked at step 1 and resumed, so
    the paths whose delta_t is 0 carry that state through about 1 000 steps on another warp."""
    stats = setting not in NO_STATS
    target, diff = _inputs(oracle, name)
    reps = gpu["tiles"] * 2 // target.shape[0]
    for prune in (False, True):
        ref = _oracle(oracle, name, setting, prune)
        for split in (False, True):
            got, _ = _track(gpu["trk"][(split, stats)], target, diff, setting, prune)
            _assert_matches_oracle(got, ref, (setting, prune, split), stats=stats)
        got, parked = _track(gpu["trk"][(True, stats)], np.concatenate([target] * reps), np.concatenate([diff] * reps), setting, prune, 1)
        _assert_matches_oracle(got, _tile(ref, reps), (setting, prune, "parked at step 1"), stats=stats)
        n_paths = reps * target.shape[0] * T
        if _split_eligible(setting):
            assert parked > 0, (setting, prune)
            if setting == (1022, 4, 4):
                assert parked > n_paths // 2, (parked, n_paths)
        else:
            assert parked == 0, (setting, prune)


@pytest.mark.gpu
def test_counters_at_their_limits(gpu, oracle):
    """(1022, 4, 4) fills the packed counters: 1 023 steps and 4 059 corrector stages come back equal to the oracle's.  With stats,
    (1023, 3, 4) and (1100, 5, 4) are refused; without stats their flags and end points are the oracle's."""
    target, diff = _inputs(oracle, "R")
    ref = _oracle(oracle, "R", (1022, 4, 4), False)
    for split in (False, True):
        got, _ = _track(gpu["trk"][(split, True)], target, diff, (1022, 4, 4), False)
        _assert_matches_oracle(got, ref, ("limits", split))
        st = got[3]
        assert st[:, 0].max() == 1023 and st[:, 2].max() == 4059 and (st[:, 3] & 0xffff).max() == 1004
    for setting in NO_STATS:
        for split in (False, True):
            with pytest.raises(hc.HCB200Error):
                _track(gpu["trk"][(split, True)], target, diff, setting, False)
            got, _ = _track(gpu["trk"][(split, False)], target, diff, setting, False)
            _assert_matches_oracle(got, _oracle(oracle, "R", setting, False), (setting, split), stats=False)


@pytest.mark.gpu
def test_parked_step_state_is_the_oracles_below_the_normal_range(gpu, oracle):
    """A launch exposes delta_t in one place: the state the split kernel parks for a path (t0, delta_t, counts, success counter, end-zone
    flag, step).  Input R at (1022, 4, 4), 64 copies, so the queue still holds fresh paths when the first wave's long paths reach the suspend
    step: at step 170 most of the capped paths carry a subnormal delta_t, at step 250 all carry 0.  For every parked path the state equals
    the float32 replay of the oracle's trace at that step, bit for bit, and the results are the oracle's."""
    setting, reps, n_r = (1022, 4, 4), 64, 2 * T
    target, diff = _inputs(oracle, "R")
    ref = _oracle(oracle, "R", setting, False)
    trk = gpu["trk"][(True, True)]
    replays = {}
    for cut in (170, 250):
        got, parked = _track(trk, np.concatenate([target] * reps), np.concatenate([diff] * reps), setting, False, cut)
        _assert_matches_oracle(got, _tile(ref, reps), ("parked at", cut))
        n_paths = reps * n_r
        ws = trk.d_ws.cpu().numpy()
        entries = ws[256:256 + 4 * n_paths].view(np.uint32)
        state = ws[256 + ((4 * n_paths + 15) & ~15):][:16 * n_paths].view(np.uint32).reshape(n_paths, 4)
        kinds = []
        for b in (entries[entries != 0].astype(np.int64) - 1):
            p = int(b % n_r)
            assert ref[3][p, 0] > cut, (cut, b)
            if p not in replays:
                t0, dt, acc, _ = oracle.trace_path(target[p // T], diff[p // T], p % T, False, *setting)
                replays[p] = (t0, acc, _replay(acc, setting[2])[4])
            t0, acc, carried = replays[p]
            dt_in, counter, end_zone = carried[cut]
            st = state[b]
            assert st[0] == t0[cut].view(np.uint32) and st[1] == dt_in.view(np.uint32), (cut, b, st[:2].view(np.float32), t0[cut], dt_in)
            assert st[2] & 1023 == cut and st[2] >> 22 == (~acc[:cut]).sum(), (cut, b)
            assert (st[3] & 0xff, (st[3] >> 8) & 1, st[3] >> 16) == (counter, int(end_zone), cut), (cut, b)
            kinds.append("zero" if dt_in == 0 else "subnormal" if dt_in < TINY else "normal")
        assert parked == len(kinds) and kinds.count({170: "subnormal", 250: "zero"}[cut]) >= 5, (cut, kinds.count("subnormal"), kinds.count("zero"))


def _track_abort(trk, n_hyp, setting, prune, split_flag):
    """hcb200_track_abort as Tracker.track_abort calls it, optionally with the split flag and suspend step 1 in `flags` (both ignored)."""
    p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    trk.max_steps, trk.max_corr, trk.dt_inc = setting
    trk.reset_abort(n_hyp)
    flags = (hc.FLAG_PRUNE_PATHS if prune else 0) | ((hc.FLAG_SPLIT_LONG_PATHS | (1 << 16)) if split_flag else 0)
    with trk.torch.cuda.device(trk.device):
        rc = trk.lib.hcb200_track_abort(trk._stream(), n_hyp, trk.n_edgels, trk.max_steps, trk.max_corr, trk.dt_inc, flags,
                                        p(trk.d_start_sols), p(trk.d_start_params), p(trk.d_target), p(trk.d_diff), p(trk.d_edgels),
                                        p(trk.d_K), p(trk.d_tracks), p(trk.d_conv), p(trk.d_inf), p(trk.d_found), p(trk.d_found_index),
                                        p(trk.d_best), p(trk.d_stats), p(trk.d_ws))
    hc._check(rc, "hcb200_track_abort")
    out = trk.results(n_hyp)
    return out, int(trk.d_found.cpu()[0]), trk.d_found_index[:n_hyp * T].cpu().numpy(), trk.d_best.cpu().numpy()


def _assert_nothing_passes(oracle, ref, rs):
    tr, cv, _, _ = ref
    conv = np.nonzero(cv)[0]
    assert len(conv) > 100
    assert not any(oracle.score(tr[b], rs["locations"], rs["K"])[0] for b in conv)


def _assert_abort_invariants(oracle, ref, got, idx, rec, rs, offset=0):
    """test_abort_late_hit's invariants: flagged paths pass the oracle's scoring of their end points, paths that finished before the flag
    (end reason < 4) are the oracle's bit for bit, and the record names the smallest flagged path with its inlier counts."""
    tr, cv, inf, st = got
    hits = np.nonzero(idx >= 0)[0]
    assert len(hits) >= 1 and np.array_equal(idx[hits], hits + offset)
    passing = {int(b) for b in np.nonzero(ref[1])[0] if oracle.score(ref[0][b], rs["locations"], rs["K"])[0]}
    assert set(hits.tolist()) <= passing
    for b in hits:
        assert oracle.score(tr[b], rs["locations"], rs["K"])[0] and cv[b] == 1
    done = (st[:, 3] >> 16) < 4
    _assert_matches_oracle(tuple(a[done] for a in got), tuple(a[done] for a in ref), "finished before the flag")
    ok, n21, n31, _ = oracle.score(tr[hits.min()], rs["locations"], rs["K"])
    assert (rec[0], rec[1], rec[2], rec[3], rec[4]) == (1, hits.min(), n21, n31, len(hits))


@pytest.mark.gpu
@pytest.mark.parametrize("setting", [(300, 4, 4), (1022, 4, 4), (1022, 4, 0)], ids=str)
def test_abort_kernel_matches_the_oracle_when_nothing_passes(gpu, oracle, setting):
    """Input R against dataset 0's edgels: complex end points fail the imaginary-part gate, so no path passes and the abort kernel tracks
    every path, with the rejected step's t read back from shared memory; results and counters are the oracle's, the split flag changes
    nothing.  Input E0 at (1022, 4, 4), where track 104 still converges to the ground-truth pose, keeps the abort invariants."""
    rs = fixtures.load_ransac(0)
    trk = gpu["trk"][(False, True)]
    trk.set_edgels(rs["locations"], rs["K"])
    target, diff = _inputs(oracle, "R")
    for prune in (False, True):
        ref = _oracle(oracle, "R", setting, prune)
        _assert_nothing_passes(oracle, ref, rs)
        trk.upload_params(target, diff)
        for split_flag in (False, True):
            got, found, idx, best = _track_abort(trk, 2, setting, prune, split_flag)
            _assert_matches_oracle(got, ref, (setting, prune, split_flag))
            assert found == 0 and (idx == -1).all() and best[0] == 0 and best[1] == -1 and best[4] == 0
    if setting != (1022, 4, 4):
        return
    ref = _oracle(oracle, "E0", setting, True)
    assert ref[1][104] == 1 and oracle.score(ref[0][104], rs["locations"], rs["K"]) == (True, 5117, 5117, True)
    target, diff = _inputs(oracle, "E0")
    trk.upload_params(target, diff)
    for split_flag in (False, True):
        got, found, idx, best = _track_abort(trk, 8, setting, True, split_flag)
        assert found == 1
        _assert_abort_invariants(oracle, ref, got, idx, best, rs)


@pytest.mark.gpu
def test_batched_abort_at_the_filled_counters(gpu, oracle):
    """(1022, 4, 4), three problems of two hypotheses: input R against dataset 0's edgels, input R against dataset 1's (neither ever
    passes), and the first two hypotheses of E0 against dataset 0's.  The first two are the oracle's bit for bit with empty records; the
    third keeps the abort invariants."""
    setting = (1022, 4, 4)
    r0, r1 = fixtures.load_ransac(0), fixtures.load_ransac(1)
    ref_r = _oracle(oracle, "R", setting, True)
    _assert_nothing_passes(oracle, ref_r, r0)
    _assert_nothing_passes(oracle, ref_r, r1)
    ref_e0 = tuple(a[:2 * T] for a in _oracle(oracle, "E0", setting, True))
    (tR, dR), (tE, dE) = _inputs(oracle, "R"), _inputs(oracle, "E0")
    trk = gpu["trk"][(False, True)]
    trk.max_steps, trk.max_corr, trk.dt_inc = setting
    trk.upload_params(np.concatenate([tR, tR, tE[:2]]), np.concatenate([dR, dR, dE[:2]]))
    trk.set_edgel_batch([r0["locations"], r1["locations"], r0["locations"]], [r0["K"], r1["K"], r0["K"]])
    trk.track_abort_batched(3, 2, prune=True)
    got = trk.results(6)
    recs = trk.batch_records(3)
    idx = trk.d_found_index[:6 * T].cpu().numpy()
    flags = trk.d_found_batch[:3].cpu().numpy()
    L = 2 * T
    for k in (0, 1):
        s = slice(k * L, (k + 1) * L)
        _assert_matches_oracle(tuple(a[s] for a in got), ref_r, ("problem", k))
        assert flags[k] == 0 and (idx[s] == -1).all()
        assert recs[k] == dict(found=0, path_id=-1, inliers21=0, inliers31=0, n_passed=0)
    s = slice(2 * L, 3 * L)
    rec = recs[2]
    assert flags[2] == 1
    _assert_abort_invariants(oracle, ref_e0, tuple(a[s] for a in got), idx[s], [rec["found"], rec["path_id"], rec["inliers21"],
                                                                               rec["inliers31"], rec["n_passed"]], r0, offset=2 * L)


@pytest.mark.gpu
@pytest.mark.parametrize("name", PROBLEMS)
def test_compiled_problems_match_their_oracle_at_large_caps(name):
    """Random complex targets (seed 7, 4 hypotheses) at the ZERO_STEP caps, plain and split, both pruning modes, against the problem's
    oracle bit for bit.  (These inputs converge within 52 steps: test_compiled_problem_inputs_stay_above_the_subnormal_range.)"""
    from oracle.pyoracle import Oracle
    from trifocal_pose_estimation_using_improved_gpuhc_b200 import problem as pm
    pdir = os.path.join(ROOT, "problems", name)
    prob = pm.read_problem(pdir)
    n = prob["spec"]["n_vars"]
    orc = Oracle(prob, problem_dir=pdir)
    target, diff = _complex_targets(orc.start_params, 4, 7)
    for split in (False, True):
        trk = pm.ProblemTracker(pdir, problem=prob, stats=True, split=split)
        trk.upload_params(target)
        assert np.array_equal(trk.diff_params(target), diff)
        for setting in ZERO_STEP[:3]:
            trk.max_steps, trk.max_corr, trk.dt_inc = setting
            for prune in (False, True):
                trk.track(4, prune=prune)
                ref = orc.track(target, diff, prune, max_steps=setting[0], max_corr=setting[1], dt_inc=setting[2])
                _assert_matches_oracle(trk.results(4), ref, (name, setting, prune, split), n_vars=n)
