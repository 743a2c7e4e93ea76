"""SURVEY.md §8 row f4: a minimal problem is DATA (a folder in the reference's layout), compiled into the tracker.

Two synthetic problems (tools/make_synthetic_problem.py) exercise the compiler beyond the trifocal tables: `coupled_quadrics_8x8`
(block structure found by the compiler: two private pivot columns + six shared; one-, two- and three-factor terms, two-parameter
coefficients, depth pruning on 2 unknowns) and `dense_quadrics_6x6` (no block structure: the all-warp-wide fallback, NSP == 0).

Pinning: the UNMODIFIED reference CPU-HC (its generic solver + index-table evaluators take every size from gpuhc_settings.yaml) was run on
both folders in the build container (tools/make_golden.py problem -> tests/golden/problem_*_h16.npz); the oracle built for each problem's
sizes must reproduce the reference's flags exactly and its end points to 1e-4 (median < 1e-6); the GPU library built from the generated header must
reproduce the oracle bit for bit (-m gpu)."""
import ctypes
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_synthetic_problem as msp  # noqa: E402

PKG = os.path.join(ROOT, "trifocal_pose_estimation_using_improved_gpuhc_b200")
GOLD = os.path.join(ROOT, "tests", "golden")
PROBLEMS = list(msp.NAMES)


def _pdir(name):
    return os.path.join(ROOT, "problems", name)


def _digest(tracks, n):
    a = np.ascontiguousarray(tracks[:, :n]).view(np.float32).copy()
    a[np.isnan(a)] = np.float32(np.nan)
    return hashlib.sha256(a.view(np.uint32).tobytes()).hexdigest()


def _inputs(name, n_hyp=16):
    from trifocal_pose_estimation_using_improved_gpuhc_b200 import problem as pm
    msp.select(name)
    prob = pm.read_problem(_pdir(name))
    tgt = msp.target_params(n_hyp)
    sp1 = np.concatenate([prob["start_params"], [1.0]]).astype(np.complex64)
    dif = np.empty_like(tgt)
    dif.real, dif.imag = tgt.real - sp1.real, tgt.imag - sp1.imag
    return prob, tgt, dif


# ---------------------------------------------------------------------------------------------------------------------
# CPU

@pytest.mark.parametrize("name", PROBLEMS)
def test_problem_folder_is_what_the_generator_script_writes(name, tmp_path):
    msp.select(name)
    msp.write_folder(str(tmp_path / name))
    for f in sorted(os.listdir(_pdir(name))):
        assert open(os.path.join(_pdir(name), f)).read() == open(str(tmp_path / name / f)).read(), f


@pytest.mark.parametrize("name", PROBLEMS)
def test_jacobian_table_is_the_derivative_of_the_H_table(name):
    """Central differences of the H table (float64) against the dHdx table, through the oracle-independent term lists of the compiler."""
    from trifocal_pose_estimation_using_improved_gpuhc_b200.codegen import gen_eval
    spec, hx, ht = gen_eval.read_problem_dir(_pdir(name))
    gen_eval.configure(spec)
    gen_eval._TABLES = (hx, ht)
    try:
        hx_terms, h_terms = gen_eval.parse_terms(*gen_eval.load_tables())
    finally:
        gen_eval.configure(dict(name="trifocal_2op1p_30x30", n_vars=30, n_params=33, n_tracks=312, hx_terms=8, hx_parts=5, ht_terms=16, ht_parts=6, n_depths=8, trifocal=1))
        gen_eval._TABLES = None
    n, npar = spec["n_vars"], spec["n_params"]
    rng = np.random.RandomState(3)
    x = np.concatenate([rng.randn(n) + 1j * rng.randn(n), [1.0]])
    p = np.concatenate([rng.randn(npar) + 1j * rng.randn(npar), [1.0]])

    def H(xv):
        return np.array([sum(c * p[a] * p[b] * np.prod([xv[k] for k in xs]) for c, a, b, xs in h_terms[r]) for r in range(n)])
    for col in range(n):
        e = np.zeros(n + 1)
        e[col] = 1e-6
        fd = (H(x + e) - H(x - e)) / 2e-6
        an = np.array([sum(c * p[a] * p[b] * np.prod([x[k] for k in xs]) for c, a, b, xs in hx_terms.get((r, col), [])) for r in range(n)])
        assert np.allclose(fd, an, rtol=1e-6, atol=1e-7), (name, col)


@pytest.mark.parametrize("name", PROBLEMS)
def test_committed_header_is_what_the_compiler_emits(name, tmp_path):
    out = str(tmp_path / "gen.h")
    subprocess.check_call([sys.executable, os.path.join(PKG, "codegen", "gen_eval.py"), "--problem-dir", _pdir(name), "--out", out], stdout=subprocess.DEVNULL)
    committed = os.path.join(PKG, "csrc", "hc_problem_gen_%s.h" % name)
    assert open(out).read() == open(committed).read()
    text = open(out).read()
    assert '#define HCG_PROBLEM_NAME "%s"' % name in text and "#define HCG_TRIFOCAL 0" in text
    if name == "dense_quadrics_6x6":
        assert "#define HCG_K1 0 " in text and "#define HCG_NSP 0 " in text          # no block structure: every pivot step warp-wide
    else:
        assert "#define HCG_K1 2 " in text                                           # block structure found in a non-trifocal system


def _csrc_snapshot():
    csrc = os.path.join(PKG, "csrc")
    snap = {}
    for d, _, files in os.walk(csrc):
        for f in files:
            p = os.path.join(d, f)
            with open(p, "rb") as fh:
                snap[os.path.relpath(p, csrc)] = fh.read()
    return snap


def test_trifocal_header_is_byte_identical_and_the_generator_leaves_csrc_untouched(tmp_path):
    out = str(tmp_path / "gen.h")
    before = _csrc_snapshot()                                      # the generator writes --out and nothing else: committed sources stay as they are
    subprocess.check_call([sys.executable, os.path.join(PKG, "codegen", "gen_eval.py"), "--out", out], stdout=subprocess.DEVNULL)
    assert open(out).read() == open(os.path.join(PKG, "csrc", "hc_problem_gen.h")).read()
    assert _csrc_snapshot() == before


@pytest.mark.parametrize("name", PROBLEMS)
def test_oracle_matches_the_reference_generic_cpu_hc_on_the_problem(name):
    """Golden = UNMODIFIED reference CPU-HC (LAPACK cgesv) on the same folder and targets: identical flags, end points to 1e-4 (median 1e-6); and the
    oracle reproduces its own committed digest (so the GPU test, which compares with the live oracle, is anchored to these files)."""
    from oracle.pyoracle import Oracle
    prob, tgt, dif = _inputs(name)
    n, T = prob["spec"]["n_vars"], prob["spec"]["n_tracks"]
    g = np.load(os.path.join(GOLD, "problem_%s_h16.npz" % name))
    assert np.array_equal(g["target"], tgt)
    orc = Oracle(prob, problem_dir=_pdir(name))
    P = 16 * T
    for prune in (False, True):
        k = "prune" if prune else "noprune"
        tr, cv, inf, st = orc.track(tgt, dif, prune)
        assert np.array_equal(np.packbits(cv), g["oracle_converged_" + k]) and np.array_equal(np.packbits(inf), g["oracle_infinity_" + k])
        assert np.array_equal(st[:, 0].astype(np.uint8), g["oracle_steps_" + k])
        assert _digest(tr, n) == str(g["oracle_digest_" + k])
        if not prune:
            cv_r, inf_r = np.unpackbits(g["ref_converged"])[:P], np.unpackbits(g["ref_infinity"])[:P]
            assert np.array_equal(cv, cv_r) and np.array_equal(inf, inf_r)
            both = cv != 0
            assert both.sum() > 0.9 * P
            d = np.abs(tr[both][:, :n] - g["ref_tracks"][both]).max(1)
            assert d.max() < 1e-4 and np.median(d) < 1e-6, (d.max(), np.median(d))      # observed 2e-6 / 1.2e-5 max, 6e-8 median
            # and the end points solve the TARGET system (float64 residual of the polynomial written out by hand)
            msp.select(name)
            x = tr[both][:, :n].astype(np.complex128)
            p = np.repeat(tgt, T, axis=0)[both].astype(np.complex128)
            res = 0.0
            for r, terms in enumerate(msp.system()):
                v = sum(c * p[:, a] * p[:, b] * np.prod([x[:, j] for j in xs], axis=0) if xs else c * p[:, a] * p[:, b] for c, a, b, xs in terms)
                res = max(res, np.abs(v).max())
            assert res < 2e-5, res


def test_libraries_export_problem_info():
    from trifocal_pose_estimation_using_improved_gpuhc_b200 import hc, problem as pm
    info = pm.problem_info(pm.load_problem_library(hc.LIB_PATH))
    assert info == dict(n_vars=30, n_params=33, n_tracks=312, trifocal=1, name="trifocal_2op1p_30x30")
    for name in PROBLEMS:
        path = pm.library_path(name)
        if not os.path.exists(path):
            pytest.skip(path + " not built (make problem PROBLEM_DIR=problems/%s)" % name)
        spec = pm.read_problem(_pdir(name))["spec"]
        info = pm.problem_info(pm.load_problem_library(path))
        assert (info["name"], info["n_vars"], info["n_params"], info["n_tracks"], info["trifocal"]) == (name, spec["n_vars"], spec["n_params"], spec["n_tracks"], 0)
        lib = ctypes.CDLL(path)
        for sym in hc.ABI_SYMBOLS:
            getattr(lib, sym)


def test_hc_main_refuses_what_it_cannot_run(tmp_path):
    """Host logic of `hc-main -p <problem>` that needs no GPU: a folder nobody compiled is refused with the build command; a compiled problem
    without a CUDA device is a loud error, not a CPU fallback."""
    import shutil
    import torch
    exe = os.path.join(PKG, "lib", "hc-main")
    name = PROBLEMS[0]
    root = str(tmp_path)
    os.makedirs(os.path.join(root, "Output_Write_Files"))
    shutil.copytree(_pdir(name), os.path.join(root, "problems", name))
    shutil.copytree(_pdir(name), os.path.join(root, "problems", "uncompiled"))
    y = os.path.join(root, "problems", "uncompiled", "gpuhc_settings.yaml")
    text = open(y).read().replace("problem_name: " + name, "problem_name: uncompiled")
    open(y, "w").write(text)
    out = subprocess.run([exe, "-p", "uncompiled", "-d", root], capture_output=True, text=True, timeout=60)
    assert out.returncode == 1 and "make problem PROBLEM_DIR=problems/uncompiled" in out.stdout + out.stderr
    if not torch.cuda.is_available() and os.path.exists(os.path.join(PKG, "lib", "libhcb200_%s.so" % name)):
        out = subprocess.run([exe, "-p", name, "-d", root], capture_output=True, text=True, timeout=60)
        assert out.returncode != 0 and "no CUDA device" in out.stdout + out.stderr
        assert not os.path.exists(os.path.join(root, "Output_Write_Files", "GPU_Sols_Statistics.txt"))


# ---------------------------------------------------------------------------------------------------------------------
# GPU

@pytest.mark.gpu
@pytest.mark.parametrize("name", PROBLEMS)
def test_gpu_tracker_of_a_compiled_problem_is_bit_identical_to_the_oracle(name):
    import torch
    from oracle.pyoracle import Oracle
    from trifocal_pose_estimation_using_improved_gpuhc_b200 import problem as pm
    H = 48
    prob, tgt, dif = _inputs(name, H)
    n, T = prob["spec"]["n_vars"], prob["spec"]["n_tracks"]
    orc = Oracle(prob, problem_dir=_pdir(name))
    trk = pm.ProblemTracker(_pdir(name), problem=prob, stats=True)
    trk.upload_params(tgt)
    assert np.array_equal(trk.diff_params(tgt), dif)
    for prune in (False, True):
        trk.track(H, prune=prune)
        tr, cv, inf, st = trk.results(H)
        tr_o, cv_o, inf_o, st_o = orc.track(tgt, dif, prune)
        assert np.array_equal(cv, cv_o) and np.array_equal(inf, inf_o)
        a, b = np.ascontiguousarray(tr[:, :n]), np.ascontiguousarray(tr_o[:, :n])
        assert bool(np.all((a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))))
        assert np.array_equal(st[:, 0], st_o[:, 0]) and np.array_equal(st[:, 2], st_o[:, 2]) and np.array_equal(st[:, 3] & 0xffff, st_o[:, 3])
        assert np.array_equal(st[:, 3] >> 16, st_o[:, 4])
        assert cv.sum() > 0.2 * H * T
        # device statistics == numpy on the same arrays (Evaluations.cpp:145-167 semantics)
        counts = trk.count_solutions(H)
        real = (cv != 0) & np.all(np.abs(tr[:, :n].imag).astype(np.float64) <= 1e-4, axis=1)
        ref = np.stack([cv.reshape(H, T).sum(1), inf.reshape(H, T).sum(1), real.reshape(H, T).sum(1)], 1)
        assert np.array_equal(counts, ref)
    # Newton refinement on the device == the oracle's, bit for bit, on the first hypothesis
    trk.track(H, prune=False)
    tr, cv, inf, st = trk.results(H)
    sums = trk.refine_tracks(H, iters=2)
    tr2 = trk.results(H)[0]
    for path in np.nonzero(cv[:T])[0][:40]:
        x1 = np.concatenate([tr[path, :n], [1.0]]).astype(np.complex64)
        xo, sd, sx = orc.refine(tgt[0], x1, iters=2)
        assert np.array_equal(np.ascontiguousarray(xo[:n]).view(np.uint64), np.ascontiguousarray(tr2[path, :n]).view(np.uint64))
        assert np.float32(sd) == sums[path, 0] and np.float32(sx) == sums[path, 1]
    # nothing is written beyond the problem's (smaller) arrays: guard bytes behind tracks, flags and workspace survive a launch
    P = H * T
    g_tr = torch.full((P * (n + 1) * 2 + 64,), 7.0, dtype=torch.float32, device=trk.device)
    g_cv = torch.full((P + 64,), 0x5A, dtype=torch.uint8, device=trk.device)
    g_inf = torch.full((P + 64,), 0x5A, dtype=torch.uint8, device=trk.device)
    need = int(trk.lib.hcb200_workspace_bytes_for(H))
    g_ws = torch.full((need + 1024,), 0xA5, dtype=torch.uint8, device=trk.device)
    trk.d_tracks, trk.d_conv, trk.d_inf, trk.d_ws = g_tr[:P * (n + 1) * 2].view(P, n + 1, 2), g_cv[:P], g_inf[:P], g_ws
    trk.track(H, prune=False)
    torch.cuda.synchronize()
    assert bool((g_tr[P * (n + 1) * 2:] == 7.0).all()) and bool((g_cv[P:] == 0x5A).all()) and bool((g_inf[P:] == 0x5A).all()) and bool((g_ws[need:] == 0xA5).all())
    assert np.array_equal(trk.d_conv.cpu().numpy(), cv)
    # the entry points that know what trifocal unknowns MEAN refuse to run on another problem
    rc = trk.lib.hcb200_track_abort(None, 1, 10, 80, 3, 4, 0, *([None] * 14))
    assert rc != 0 and b"not supported" in trk.lib.hcb200_error_string(rc).lower()
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("name", PROBLEMS)
def test_hc_main_runs_a_compiled_problem(name, tmp_path):
    """`hc-main -p <name>` — the original GPU-HC usage (reference README.md:25): the folder's start system is tracked to target_params.txt with
    the library compiled from the folder; statistics file and converged end points equal the oracle's (bit for bit: %.9g round-trips float32)."""
    import shutil
    from oracle.pyoracle import Oracle
    exe = os.path.join(PKG, "lib", "hc-main")
    root = str(tmp_path)
    shutil.copytree(_pdir(name), os.path.join(root, "problems", name))
    os.makedirs(os.path.join(root, "Output_Write_Files"))
    prob, tgt, dif = _inputs(name, 1)
    n, T = prob["spec"]["n_vars"], prob["spec"]["n_tracks"]
    tr_o, cv_o, inf_o, st_o = Oracle(prob, problem_dir=_pdir(name)).track(tgt, dif, False)
    real_o = (cv_o != 0) & np.all(np.abs(tr_o[:, :n].imag).astype(np.float64) <= 1e-4, axis=1)
    for H in (1, 37):
        out = subprocess.run([exe, "-p", name, "-d", root, "-s", "Num_Of_RANSAC_Iterations=%d" % H], capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
        stats = [int(v) for v in open(os.path.join(root, "Output_Write_Files", "GPU_Sols_Statistics.txt")).read().split()]
        assert stats == [H * int(cv_o.sum()), H * int(real_o.sum()), H * int(inf_o.sum())]          # converged <TAB> real <TAB> infinity
        assert float(open(os.path.join(root, "Output_Write_Files", "GPU_Timings.txt")).read()) > 0.0
    got, cur = {}, None
    for line in open(os.path.join(root, "Output_Write_Files", "GPU_Converged_HC_Tracks.txt")):
        if line.startswith("track"):
            cur = int(line.split()[1]); got[cur] = []
        else:
            re_, im_ = line.split(); got[cur].append(np.float32(re_) + 1j * np.float32(im_))
    assert sorted(got) == np.nonzero(cv_o)[0].tolist()
    for t, x in got.items():
        assert np.array_equal(np.asarray(x, np.complex64).view(np.uint64), np.ascontiguousarray(tr_o[t, :n]).view(np.uint64)), t
    # a folder nobody compiled is refused with a message, not tracked by something else
    shutil.copytree(_pdir(name), os.path.join(root, "problems", "uncompiled"))
    y = os.path.join(root, "problems", "uncompiled", "gpuhc_settings.yaml")
    text = open(y).read().replace("problem_name: " + name, "problem_name: uncompiled")
    open(y, "w").write(text)
    out = subprocess.run([exe, "-p", "uncompiled", "-d", root], capture_output=True, text=True, timeout=60)
    assert out.returncode == 1 and "make problem" in out.stdout + out.stderr
