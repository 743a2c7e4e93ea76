"""ctypes front-end of the CPU oracles.  TEST INFRASTRUCTURE ONLY — imported by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs; the product package never imports this module.

  Oracle     oracle/liboracle_hc.so      plain-C restatement (hc_oracle.c), built on demand with gcc
  Reference  oracle/_ref/libref_cpuhc.so the UNMODIFIED reference CPU-HC (built in the build container from /root/reference
                                         by `make -C oracle ref`; travels to the GPU box as a prebuilt file)
"""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "liboracle_hc.so")
REF_CPU_SO = os.path.join(HERE, "_ref", "libref_cpuhc.so")
REF_CPU_PRUNED_SO = os.path.join(HERE, "_ref", "libref_cpuhc_pruned.so")   # reference CPU-HC + the GPU kernels' path pruning (generated copy)
REF_GPU_SO = os.path.join(HERE, "_ref", "libref_gpuhc.so")
REF_GPU_DEBUG_SO = os.path.join(HERE, "_ref", "libref_gpuhc_debug.so")     # same sources with the reference's GPU_DEBUG switch on

N, NP1, TRACKS = 30, 34, 312


def _vp(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


def c2f(z):
    """complex64 array -> float32 array with trailing (re, im)."""
    z = np.asarray(z, np.complex64)
    return np.ascontiguousarray(np.stack([z.real, z.imag], -1).astype(np.float32))


def f2c(a):
    return (a[..., 0] + 1j * a[..., 1]).astype(np.complex64)


class Settings(ctypes.Structure):
    _fields_ = [("max_steps", ctypes.c_int), ("max_corr_steps", ctypes.c_int), ("dt_inc_steps", ctypes.c_int),
                ("prune", ctypes.c_int)]


class Variant(ctypes.Structure):
    """hco_variant (hc_oracle.h): an equally valid floating-point evaluation of the same algorithm; all zeros == the spec."""
    _fields_ = [("solver", ctypes.c_int), ("term_order", ctypes.c_int), ("contract", ctypes.c_int), ("sum_order", ctypes.c_int),
                ("rk_final_mul", ctypes.c_int), ("perturb_seed", ctypes.c_uint)]


def build_oracle(force=False):
    src = os.path.join(HERE, "hc_oracle.c")
    if force or not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", HERE, "oracle"], stdout=subprocess.DEVNULL)
    return ORACLE_SO


def build_problem_oracle(problem_dir):
    name = os.path.basename(os.path.normpath(problem_dir))
    so = os.path.join(HERE, "liboracle_hc_%s.so" % name)
    src = os.path.join(HERE, "hc_oracle.c")
    if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", HERE, "problem_oracle", "PROBLEM_DIR=" + os.path.abspath(problem_dir)], stdout=subprocess.DEVNULL)
    return so


class Oracle:
    def __init__(self, problem, problem_dir=None):
        """problem: dict with start_sols, start_params, dHdx_indx, dHdt_indx.  problem_dir: a problem folder (reference layout) other than
        the trifocal one — the same C source is built for its sizes (`make -C oracle problem_oracle`), problem["spec"] gives them."""
        if problem_dir is None:
            build_oracle()
            self.lib = ctypes.CDLL(ORACLE_SO)
            self.N, self.NP1, self.TRACKS = N, NP1, TRACKS
        else:
            self.lib = ctypes.CDLL(build_problem_oracle(problem_dir))
            spec = problem["spec"]
            self.N, self.NP1, self.TRACKS = spec["n_vars"], spec["n_params"] + 1, spec["n_tracks"]
        self.lib.hco_newton_refine_f64.restype = ctypes.c_double
        self.hx = np.ascontiguousarray(problem["dHdx_indx"], np.int32)
        self.ht = np.ascontiguousarray(problem["dHdt_indx"], np.int32)
        ss = np.ones((self.TRACKS, self.N + 1), np.complex64)
        ss[:, :self.N] = problem["start_sols"]
        self.start_sols = ss
        self.start_params = np.concatenate([problem["start_params"], [1.0]]).astype(np.complex64)
        self._ss = c2f(ss)
        self._sp = c2f(self.start_params)

    # evaluators -------------------------------------------------------------------------------------------------
    def eval_Hx(self, x31, p34):
        A = np.zeros((self.N, self.N, 2), np.float32)
        self.lib.hco_eval_Hx(_vp(self.hx), _vp(c2f(x31)), _vp(c2f(p34)), _vp(A))
        return f2c(A)

    def eval_H(self, x31, p34):
        b = np.zeros((self.N, 2), np.float32)
        self.lib.hco_eval_H(_vp(self.ht), _vp(c2f(x31)), _vp(c2f(p34)), _vp(b))
        return f2c(b)

    def eval_Ht(self, x31, p34, dp34):
        b = np.zeros((self.N, 2), np.float32)
        self.lib.hco_eval_Ht(_vp(self.ht), _vp(c2f(x31)), _vp(c2f(p34)), _vp(c2f(dp34)), _vp(b))
        return f2c(b)

    def param_homotopy(self, t, target34):
        p = np.zeros((self.NP1, 2), np.float32)
        self.lib.hco_param_homotopy(ctypes.c_float(t), _vp(self._sp), _vp(c2f(target34)), _vp(p))
        return f2c(p)

    def solve(self, A, b, lu_ref=False):
        Af, bf = c2f(A), c2f(b)
        fn = self.lib.hco_solve_lu_ref if lu_ref else self.lib.hco_solve
        info = fn(_vp(Af), _vp(bf))
        return f2c(bf), info

    # tracker ----------------------------------------------------------------------------------------------------
    def prepare_target_params(self, seed, n_hyp, locations, tangents):
        tgt = np.zeros((n_hyp, self.NP1, 2), np.float32)
        dif = np.zeros((n_hyp, self.NP1, 2), np.float32)
        picked = np.zeros((n_hyp, 3), np.int32)
        loc = np.ascontiguousarray(locations, np.float32)
        tan = np.ascontiguousarray(tangents, np.float32)
        self.lib.hco_prepare_target_params(ctypes.c_uint(seed), n_hyp, loc.shape[0], _vp(loc), _vp(tan), _vp(self._sp),
                                           _vp(tgt), _vp(dif), _vp(picked))
        return f2c(tgt), f2c(dif), picked

    def track(self, target, diff, prune, max_steps=80, max_corr=3, dt_inc=4, n_threads=0, variant=None):
        """Returns tracks[P,31] c64, converged[P] u8, infinity[P] u8, stats[P,5] i32 (steps,pred,corr,rejected,reason).
        variant: dict of hco_variant fields (None == the arithmetic spec)."""
        n_hyp = target.shape[0]
        P = n_hyp * self.TRACKS
        tr = np.zeros((P, self.N + 1, 2), np.float32)
        cv = np.zeros(P, np.uint8)
        inf = np.zeros(P, np.uint8)
        st = np.zeros((P, 5), np.int32)
        cfg = Settings(max_steps, max_corr, dt_inc, 1 if prune else 0)
        var = ctypes.byref(Variant(**variant)) if variant else None
        self.lib.hco_track_batch_v(_vp(self.hx), _vp(self.ht), _vp(self._ss), _vp(self._sp), _vp(c2f(target)), _vp(c2f(diff)),
                                   n_hyp, ctypes.byref(cfg), var, n_threads or (os.cpu_count() or 1), _vp(tr), _vp(cv), _vp(inf), _vp(st))
        return f2c(tr), cv, inf, st

    def trace_path(self, target34, diff34, track, prune, max_steps=80, max_corr=3, dt_inc=4):
        """Path `track` (start-solution index) of one hypothesis, with its step control traced.  Returns t0 float32 [S] at the start of each
        step, delta_t float32 [S] used by the step (after the clamps), accepted bool [S], and the path's stats [5] (as track()), S = steps."""
        cap = max(max_steps + 1, 0)
        t0, dt, acc = np.zeros(cap, np.float32), np.zeros(cap, np.float32), np.zeros(cap, np.uint8)
        tr, cv, inf = np.zeros((self.N + 1, 2), np.float32), ctypes.c_uint8(), ctypes.c_uint8()
        st = np.zeros(5, np.int32)
        cfg = Settings(max_steps, max_corr, dt_inc, 1 if prune else 0)
        n = self.lib.hco_trace_path(_vp(self.hx), _vp(self.ht), _vp(self._ss[track]), _vp(self._sp), _vp(c2f(target34)), _vp(c2f(diff34)),
                                    ctypes.byref(cfg), cap, _vp(t0), _vp(dt), _vp(acc), _vp(tr), ctypes.byref(cv), ctypes.byref(inf), _vp(st))
        assert n == st[0]
        return t0[:n], dt[:n], acc[:n].astype(bool), st

    def score(self, x31, locations, K):
        n21, n31, gate = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        loc = np.ascontiguousarray(locations, np.float32)
        Kf = np.ascontiguousarray(K, np.float32).reshape(-1)
        ok = self.lib.hco_score_solution(_vp(c2f(x31)), _vp(loc), loc.shape[0], _vp(Kf), ctypes.byref(n21), ctypes.byref(n31),
                                         ctypes.byref(gate))
        return bool(ok), n21.value, n31.value, bool(gate.value)

    def refine(self, target34, x31, iters=3):
        """Float Newton refinement in the arithmetic spec (oracle of hcb200_refine_tracks): returns x31 (copy), sum_d, sum_x."""
        x = np.ascontiguousarray(c2f(np.asarray(x31, np.complex64).copy()))
        sd, sx = ctypes.c_float(), ctypes.c_float()
        self.lib.hco_refine_path(_vp(self.hx), _vp(self.ht), _vp(c2f(target34)), _vp(x), int(iters), ctypes.byref(sd), ctypes.byref(sx))
        return f2c(x), sd.value, sx.value

    def newton_refine(self, target34, x31, iters=6):
        out = np.zeros((self.N, 2), np.float64)
        res = self.lib.hco_newton_refine_f64(_vp(self.hx), _vp(self.ht), _vp(c2f(target34)), _vp(c2f(x31)), iters, _vp(out))
        return out[:, 0] + 1j * out[:, 1], res


class ReferenceCPU:
    """The real reference CPU-HC (oracle/_ref/libref_cpuhc.so)."""

    def __init__(self, pruned=False):
        so = REF_CPU_PRUNED_SO if pruned else REF_CPU_SO
        if not os.path.exists(so):
            raise FileNotFoundError(so + " (run `make -C oracle ref` in the build container)")
        os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
        self.lib = ctypes.CDLL(so)

    def run(self, bin_dir, n_hyp, seed=0, dataset_index=0, n_cores=None, target=None):
        P = n_hyp * TRACKS
        tr = np.zeros((P, N + 1, 2), np.float32)
        cv = np.zeros(P, np.uint8)
        inf = np.zeros(P, np.uint8)
        tp = np.zeros((n_hyp, NP1, 2), np.float32)
        sec = ctypes.c_double()
        tin = c2f(target) if target is not None else None
        rc = self.lib.ref_cpuhc_run(bin_dir.encode(), n_hyp, ctypes.c_uint(seed), dataset_index, n_cores or (os.cpu_count() or 1),
                                    _vp(tin), _vp(tr), _vp(cv), _vp(inf), _vp(tp), ctypes.byref(sec))
        if rc != 0:
            raise RuntimeError("ref_cpuhc_run failed with code %d" % rc)
        return f2c(tr), cv, inf, f2c(tp), sec.value

    def run_problem(self, problem_dir, target, n_cores=None):
        """The reference's generic CPU-HC on ANOTHER problem folder (reference layout); target: complex64 [H][Num_Of_Params + 1].
        Returns tracks [H*T][N+1] c64, converged, infinity, seconds."""
        import shutil
        import tempfile
        from trifocal_pose_estimation_using_improved_gpuhc_b200.codegen import gen_eval
        spec = gen_eval.read_problem_dir(problem_dir)[0]
        n_hyp, P = target.shape[0], target.shape[0] * spec["n_tracks"]
        tr = np.zeros((P, spec["n_vars"] + 1, 2), np.float32)
        cv, inf, sec = np.zeros(P, np.uint8), np.zeros(P, np.uint8), ctypes.c_double()
        with tempfile.TemporaryDirectory() as tmp:
            shutil.copytree(problem_dir, os.path.join(tmp, "problems", spec["name"]))
            os.makedirs(os.path.join(tmp, "Output_Write_Files"))
            os.makedirs(os.path.join(tmp, "build", "bin"))
            rc = self.lib.ref_cpuhc_run_problem(os.path.join(tmp, "build", "bin").encode(), spec["name"].encode(), n_hyp, n_cores or (os.cpu_count() or 1),
                                                _vp(c2f(target)), _vp(tr), _vp(cv), _vp(inf), ctypes.byref(sec))
        if rc != 0:
            raise RuntimeError("ref_cpuhc_run_problem failed with code %d" % rc)
        return f2c(tr), cv, inf, sec.value

    def eval_Hx(self, hx, x31, p34):
        A = np.zeros((N * N, 2), np.float32)
        self.lib.ref_eval_dHdX(_vp(np.ascontiguousarray(hx, np.int32)), _vp(c2f(x31)), _vp(c2f(p34)), _vp(A))
        return f2c(A).reshape(N, N).T      # column-major -> [row][col]

    def eval_H(self, ht, x31, p34):
        b = np.zeros((N, 2), np.float32)
        self.lib.ref_eval_H(_vp(np.ascontiguousarray(ht, np.int32)), _vp(c2f(x31)), _vp(c2f(p34)), _vp(b))
        return f2c(b)

    def eval_Ht(self, ht, x31, p34, dp34):
        b = np.zeros((N, 2), np.float32)
        self.lib.ref_eval_dHdt(_vp(np.ascontiguousarray(ht, np.int32)), _vp(c2f(x31)), _vp(c2f(p34)), _vp(c2f(dp34)), _vp(b))
        return f2c(b)

    def cgesv(self, A, b):
        Acm = c2f(np.asarray(A).T)          # row-major [row][col] -> column-major
        bf = c2f(b)
        info = self.lib.ref_cgesv(_vp(Acm), _vp(bf))
        return f2c(bf), info


class ReferenceGPU:
    """The UNMODIFIED reference GPU-HC++ kernels compiled for sm_100a (oracle/_ref/libref_gpuhc.so), driven the way
    GPU_HC_Solver drives them.  GPU box only; used as the GPU baseline in bench.py and as a second oracle in tests."""

    def __init__(self, problem, device="cuda:0", debug=False):
        import torch
        so = REF_GPU_DEBUG_SO if debug else REF_GPU_SO
        if not os.path.exists(so):
            raise FileNotFoundError(so + " (run `make -C oracle ref` in the build container)")
        self.torch = torch
        self.lib = ctypes.CDLL(so)
        self.device = torch.device(device)
        ss = np.ones((TRACKS, N + 1), np.complex64)
        ss[:, :N] = problem["start_sols"]
        sp = np.concatenate([problem["start_params"], [1.0]]).astype(np.complex64)
        idx = np.concatenate([problem["dHdx_indx"], problem["dHdt_indx"]]).astype(np.int32)
        self.d_ss = torch.from_numpy(c2f(ss)).to(self.device)
        self.d_sp = torch.from_numpy(c2f(sp)).to(self.device)
        self.d_idx = torch.from_numpy(idx).to(self.device)
        self.n_hyp = 0

    def _s(self):
        return ctypes.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def setup(self, target, diff, locations=None, K=None):
        torch = self.torch
        H = target.shape[0]
        P = H * TRACKS
        dev = self.device
        self.n_hyp = H
        self.d_target = torch.from_numpy(c2f(target)).to(dev)
        self.d_diff = torch.from_numpy(c2f(diff)).to(dev)
        self.d_tracks = torch.empty((P, N + 1, 2), dtype=torch.float32, device=dev)
        self.d_conv = torch.zeros(P, dtype=torch.bool, device=dev)
        self.d_inf = torch.zeros(P, dtype=torch.bool, device=dev)
        self.d_dbg = torch.zeros((P, 2), dtype=torch.float32, device=dev)
        if locations is not None:
            self.d_edgels = torch.from_numpy(np.ascontiguousarray(locations, np.float32)).to(dev)
            self.d_K = torch.from_numpy(np.ascontiguousarray(K, np.float32).reshape(-1)).to(dev)
            self.n_edgels = int(locations.shape[0])
            self.d_found = torch.zeros(1, dtype=torch.bool, device=dev)
            self.d_found_index = torch.full((P,), -1, dtype=torch.int32, device=dev)
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        rc = self.lib.ref_gpuhc_prepare(self._s(), H, p(self.d_ss), p(self.d_tracks), p(self.d_idx), int(self.d_idx.numel()))
        if rc:
            raise RuntimeError("ref_gpuhc_prepare -> %d" % rc)

    def reload(self):
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        self.lib.ref_gpuhc_reload_tracks(self._s(), self.n_hyp, p(self.d_ss), p(self.d_tracks))
        self.d_inf.zero_()

    def track(self, max_steps=80, max_corr=3, dt_inc=4):
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        rc = self.lib.ref_gpuhc_track(self._s(), self.n_hyp, max_steps, max_corr, dt_inc, p(self.d_sp), p(self.d_target),
                                      p(self.d_diff), p(self.d_idx), p(self.d_conv), p(self.d_inf), p(self.d_dbg))
        if rc:
            raise RuntimeError("ref_gpuhc_track -> cudaError %d" % rc)

    def track_abort(self, max_steps=80, max_corr=3, dt_inc=4):
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        self.d_found.zero_()
        self.d_found_index.fill_(-1)
        rc = self.lib.ref_gpuhc_track_abort(self._s(), self.n_hyp, self.n_edgels, max_steps, max_corr, dt_inc, p(self.d_sp),
                                            p(self.d_target), p(self.d_diff), p(self.d_idx), p(self.d_edgels), p(self.d_K),
                                            p(self.d_conv), p(self.d_inf), p(self.d_dbg), p(self.d_found), p(self.d_found_index))
        if rc:
            raise RuntimeError("ref_gpuhc_track_abort -> cudaError %d" % rc)

    def debug_t0_dt(self):
        """GPU_DEBUG build only: per path (1, 0) if converged else (t0, delta_t) at the end of the track (…TrunPaths.cu:287-289)."""
        self.torch.cuda.synchronize(self.device)
        return self.d_dbg.cpu().numpy()

    def results(self):
        self.torch.cuda.synchronize(self.device)
        tr = self.d_tracks.cpu().numpy()
        return f2c(tr), self.d_conv.cpu().numpy().astype(np.uint8), self.d_inf.cpu().numpy().astype(np.uint8)
