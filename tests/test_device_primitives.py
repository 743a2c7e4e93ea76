"""The tracker's device primitives one at a time, against the oracle bit for bit and against float64, at their arithmetic edges.

Every other GPU test checks the whole tracker.  Its inputs are natural RANSAC rounds, on which the solve's special rules (DESIGN.md §4: the
pivot key with its row bits, exact-zero multipliers, all-zero pivot columns, the reciprocal's clamp, the fast/exact two-pass scheme) almost
never fire.  `make unit` builds the tracker source with -DHC_UNIT and the product's NVFLAGS into lib/libhcb200_unit.so (and
`make unit_problem` once per compiled problem); its kernels run one warp per system with the tracker's shared-memory setup, call the same
__forceinline__ functions (param_homotopy, build_cq/dq/xp, eval_Hx, eval_rhs, solve, eval_and_solve, c_recip), and run several systems
in sequence on one warp without clearing shared memory, as the tracker does across stages and paths.

Bars: bit-exact with oracle/hc_oracle.c (NaNs compare equal), with a float64 statement beside it so that a bug the kernel shares with the
oracle is caught too:
* evaluators: |gpu - f64| <= 2 (terms + 4) 2^-24 sum|term| (+ 2^-130 per term for subnormal products) per entry;
* solve: the float64 normwise backward error <= 30 * 2^-24 * growth, where growth is the element growth of the same elimination (same pivot
  order) run in complex128, and the forward error <= cond_inf(A) times that bound; a regular finite system never takes the exact pass;
* reciprocal: recip_newton == __frcp_rn on every float in [2^-100, 2^100], __frcp_rn == numpy's float32 1/d on a sample.

One documented deviation (DESIGN.md §4): a row that the spec leaves untouched because its multiplier is exactly zero still gets the kernel's
zero-multiplier update, which maps an entry that is exactly -0 to +0 or -0 depending on the pivot row's signs.  Only a rank-1 update whose
product underflows makes a -0 (sums start from +0), and a zero's sign only ever reaches the sign of a zero; the underflow construction
therefore compares zeros sign-insensitively, and every other case is bit-exact."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle.pyoracle import Oracle, Settings, c2f
from trifocal_pose_estimation_using_improved_gpuhc_b200 import fixtures, hc
from trifocal_pose_estimation_using_improved_gpuhc_b200 import problem as pm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "trifocal_pose_estimation_using_improved_gpuhc_b200", "lib")
TRIFOCAL = "trifocal_2op1p_30x30"
PROBLEMS = [TRIFOCAL, "coupled_quadrics_8x8", "dense_quadrics_6x6", "mixed_12x12"]
F32 = np.float32
EPS = 2.0 ** -24
TINY = F32(2.0 ** -76)                       # TINY * TINY = 2^-152: below half the smallest subnormal, rounds to a signed zero
SUBN = np.nextafter(F32(0), F32(1))          # 2^-149
STEP0_COL = 0     # column 0 is pivoted by the first elimination step of every compiled problem (a level-0 group, or the first warp-wide step)




def _p(a):
    return ctypes.c_void_p(a.ctypes.data)


def f2c(a):
    """float32 [..., 2] -> complex64 [...] as a view: every bit kept (an arithmetic re + 1j * im would turn (x, Inf) into (NaN, Inf) and
    drop the sign of a zero imaginary part)."""
    return np.ascontiguousarray(a, F32).view(np.complex64)[..., 0]


# ---------------------------------------------------------------------------------------------------------------------
# one problem: oracle, tables, unit library and its slot map

class Prim:
    def __init__(self, name):
        self.name = name
        if name == TRIFOCAL:
            self.problem = fixtures.load_problem()
            self.oracle = Oracle(self.problem)
            self.so = os.path.join(LIBDIR, "libhcb200_unit.so")
            make = ["make", "-C", ROOT, "unit"]
        else:
            pdir = os.path.join(ROOT, "problems", name)
            self.problem = pm.read_problem(pdir)
            self.oracle = Oracle(self.problem, problem_dir=pdir)
            self.so = os.path.join(LIBDIR, "libhcb200_unit_%s.so" % name)
            make = ["make", "-C", ROOT, "unit_problem", "PROBLEM_DIR=problems/" + name]
        subprocess.check_call(make, stdout=subprocess.DEVNULL)       # a no-op when build() made it
        self.lib = ctypes.CDLL(self.so)
        vp, i32, u32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint
        for fn, args in (("hcb200_unit_layout", [vp] * 4), ("hcb200_unit_eval", [vp, i32, i32] + [vp] * 8),
                         ("hcb200_unit_solve", [vp, i32, i32] + [vp] * 6), ("hcb200_unit_eval_and_solve", [vp, i32, i32] + [vp] * 7),
                         ("hcb200_unit_recip", [vp, i32, vp, vp, vp]), ("hcb200_unit_recip_sweep", [vp, u32, u32, vp, vp])):
            getattr(self.lib, fn).restype = i32
            getattr(self.lib, fn).argtypes = args
        sizes = np.zeros(7, np.int32)
        rol = np.zeros(32, np.int32)
        idle = np.zeros(32, np.int32)
        self.N, self.NP1 = self.oracle.N, self.oracle.NP1
        N = self.N
        cols = np.zeros(32 * 32, np.int32)            # [32][NSLOT], NSLOT <= 32
        self.lib.hcb200_unit_layout(_p(sizes), _p(rol), _p(cols), _p(idle))
        assert (sizes[0], sizes[1]) == (self.N, self.NP1), "unit library and oracle disagree on the sizes"
        self.nslot, self.nsp, self.k1 = int(sizes[2]), int(sizes[3]), int(sizes[4])
        cols = cols[:32 * self.nslot].reshape(32, self.nslot)
        self.row_of_lane, self.slot_cols, self.idle_levels = rol, cols, idle
        self.mask = np.zeros((N, N), bool)             # structural pattern: (row, col) reachable through a register slot
        for lane in range(N):
            for c in cols[lane]:
                if c >= 0:
                    self.mask[rol[lane], c] = True
        self.sp = np.concatenate([self.problem["start_params"], [1.0]]).astype(np.complex64)
        self.hx = np.asarray(self.problem["dHdx_indx"], np.int64)
        self.ht = np.asarray(self.problem["dHdt_indx"], np.int64)
        self.hx_terms = self.hx.size // (5 * N * N)
        self.ht_terms = self.ht.size // (6 * N)

    # oracle ----------------------------------------------------------------------------------------------------------
    def param_homotopy(self, t, sp, tp):
        p, spf, tpf = np.zeros((self.NP1, 2), F32), c2f(sp), c2f(tp)          # (the inputs are named: a pointer does not keep its array)
        self.oracle.lib.hco_param_homotopy(ctypes.c_float(t), _p(spf), _p(tpf), _p(p))
        return f2c(p)

    def oracle_eval(self, pt):
        N, lib, o = self.N, self.oracle.lib, self.oracle
        p = self.param_homotopy(pt["t"], pt["sp"], pt["tp"])
        x, pf, dpf = c2f(pt["x"]), c2f(p), c2f(pt["dp"])
        A, h, ht = np.zeros((N, N, 2), F32), np.zeros((N, 2), F32), np.zeros((N, 2), F32)
        lib.hco_eval_Hx(_p(o.hx), _p(x), _p(pf), _p(A))
        lib.hco_eval_H(_p(o.ht), _p(x), _p(pf), _p(h))
        lib.hco_eval_Ht(_p(o.ht), _p(x), _p(pf), _p(dpf), _p(ht))
        return f2c(A), f2c(h), f2c(ht), p

    def oracle_solve(self, A, b):
        Af, bf = c2f(A), c2f(b)
        info = self.oracle.lib.hco_solve(_p(Af), _p(bf))
        return f2c(bf), info

    def oracle_track(self, orc, target, diff, max_steps):
        """Oracle.track without its re + 1j * im conversion of the end points."""
        n = target.shape[0] * orc.TRACKS
        tr = np.zeros((n, orc.N + 1, 2), F32)
        cv, inf, st = np.zeros(n, np.uint8), np.zeros(n, np.uint8), np.zeros((n, 5), np.int32)
        cfg = Settings(max_steps, 3, 4, 0)
        tf, df = c2f(target), c2f(diff)
        orc.lib.hco_track_batch_v(_p(orc.hx), _p(orc.ht), _p(orc._ss), _p(orc._sp), _p(tf),
                                  _p(df), target.shape[0], ctypes.byref(cfg), None, os.cpu_count() or 1, _p(tr),
                                  _p(cv), _p(inf), _p(st))
        return f2c(tr), cv, inf

    def oracle_recip(self, z):
        z = np.ascontiguousarray(z, np.complex64)
        out, zf = np.zeros(z.shape + (2,), F32), c2f(z)
        self.oracle.lib.hco_recip(_p(zf), _p(out), int(z.size))
        return f2c(out)

    # device ----------------------------------------------------------------------------------------------------------
    def _run(self, fn, n_warps, ins, out_shapes, out_dtypes=None):
        import torch
        dev = torch.device("cuda:0")
        d_in = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in ins]
        d_out = [torch.zeros(s, dtype=(out_dtypes[i] if out_dtypes else torch.float32), device=dev) for i, s in enumerate(out_shapes)]
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        n = ins[0].shape[0]
        args = [stream] + ([n, n_warps] if n_warps is not None else []) + [ctypes.c_void_p(t.data_ptr()) for t in d_in + d_out]
        rc = getattr(self.lib, fn)(*args)
        assert rc == 0, "%s -> cudaError %d" % (fn, rc)
        torch.cuda.synchronize(dev)
        return [t.cpu().numpy() for t in d_out]

    def _point_arrays(self, pts):
        return [np.array([p["t"] for p in pts], F32)] + [np.stack([c2f(p[k]) for p in pts]) for k in ("x", "sp", "tp", "dp")]

    def gpu_eval(self, pts, n_warps=1):
        N, n = self.N, len(pts)
        A, h, ht = self._run("hcb200_unit_eval", n_warps, self._point_arrays(pts), [(n, N, N, 2), (n, N, 2), (n, N, 2)])
        return f2c(A), f2c(h), f2c(ht)

    def gpu_eval_and_solve(self, pts, n_warps=1):
        N, n = self.N, len(pts)
        pred, corr = self._run("hcb200_unit_eval_and_solve", n_warps, self._point_arrays(pts), [(n, N, 2), (n, N, 2)])
        return f2c(pred), f2c(corr)

    def gpu_solve(self, systems, n_warps=1):
        import torch
        N, n = self.N, len(systems)
        A = np.stack([c2f(s["A"]) for s in systems])
        b = np.stack([c2f(s["b"]) for s in systems])
        fast, exact, sel, info = self._run("hcb200_unit_solve", n_warps, [A, b], [(n, N, 2)] * 3 + [(n, 2)],
                                           [torch.float32] * 3 + [torch.int32])
        return f2c(fast), f2c(exact), f2c(sel), info


_PRIMS = {}


def prim(name):
    if name not in _PRIMS:
        _PRIMS[name] = Prim(name)
    return _PRIMS[name]


# ---------------------------------------------------------------------------------------------------------------------
# comparisons and float64 references

def same_bits(a, b, zero_sign=True):
    """Element-wise bit equality of complex64 arrays; NaNs compare equal; zero_sign=False also equates +0 and -0."""
    a = np.asarray(a, np.complex64)
    b = np.asarray(b, np.complex64)
    a, b = np.stack([a.real, a.imag], -1), np.stack([b.real, b.imag], -1)
    eq = (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))
    if not zero_sign:
        eq |= (a == 0) & (b == 0)
    return eq.all(-1)


def assert_same(a, b, what, zero_sign=True):
    eq = same_bits(a, b, zero_sign)
    if not eq.all():
        i = np.argwhere(~eq)[0]
        raise AssertionError("%s: %d entries differ from the oracle, first at %s: %r vs %r"
                             % (what, int((~eq).sum()), tuple(i), np.asarray(a)[tuple(i)], np.asarray(b)[tuple(i)]))


def f64_eval(P, x, p, dp):
    """Float64 statement of the three evaluators from dHdx_indx / dHdt_indx: every entry is the sum of coef * p_a * p_b * x_d * x_e (* x_f)
    (x[N] == 1, p[NP] == 1).  Returns (A, sum|term| of A, #terms of A, H, sum|term|, #terms, -dH/dt, sum|term|, #terms)."""
    N = P.N
    X = np.append(np.asarray(x[:N], np.complex128), 1.0)
    Pp = np.asarray(p, np.complex128)
    D = np.asarray(dp, np.complex128)
    hx = P.hx.reshape(N, P.hx_terms, 5, N)                    # [col][term][part][row]
    c, a, b, d, e = (hx[:, :, k, :] for k in range(5))
    with np.errstate(all="ignore"):
        term = c * Pp[a] * Pp[b] * X[d] * X[e]
        aterm = np.abs(c) * np.abs(Pp[a]) * np.abs(Pp[b]) * np.abs(X[d]) * np.abs(X[e])
        A = np.where(c != 0, term, 0).sum(1).T                 # [row][col]
        SA = np.where(c != 0, aterm, 0).sum(1).T
        TA = (c != 0).sum(1).T
        ht = P.ht.reshape(P.ht_terms, 6, N)                    # [term][part][row]
        c, a, b, d, e, f = (ht[:, k, :] for k in range(6))
        xp = X[d] * X[e] * X[f]
        axp = np.abs(X[d]) * np.abs(X[e]) * np.abs(X[f])
        H = np.where(c != 0, c * Pp[a] * Pp[b] * xp, 0).sum(0)
        SH = np.where(c != 0, np.abs(c) * np.abs(Pp[a]) * np.abs(Pp[b]) * axp, 0).sum(0)
        Ht = -np.where(c != 0, c * (D[a] * Pp[b] + D[b] * Pp[a]) * xp, 0).sum(0)
        SHt = np.where(c != 0, np.abs(c) * (np.abs(D[a]) * np.abs(Pp[b]) + np.abs(D[b]) * np.abs(Pp[a])) * axp, 0).sum(0)
        TH = (c != 0).sum(0)
    return A, SA, TA, H, SH, TH, Ht, SHt, TH


def eval_bound(S, T):
    return 2.0 * (T + 4) * (EPS * S + 2.0 ** -130)


def gj_growth(A):
    """Element growth max|entry during the elimination| / max|A| of the spec's Gauss-Jordan elimination (pivot = largest |re|+|im|, lowest
    row among ties) in complex128."""
    A = np.array(A, np.complex128)
    N = A.shape[0]
    big0 = np.abs(A).max()
    big = big0
    done = np.zeros(N, bool)
    for k in range(N):
        key = np.where(done, -1.0, np.abs(A[:, k].real) + np.abs(A[:, k].imag))
        p = int(np.argmax(key))
        done[p] = True
        m = A[:, k] / A[p, k]
        m[p] = 0
        A -= np.outer(m, A[p])
        big = max(big, np.abs(A).max())
    return big / big0


# ---------------------------------------------------------------------------------------------------------------------
# inputs

def _cplx(rng, shape, scale=1.0):
    return ((rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) * scale).astype(np.complex64)


def _point(P, t, x, tp, sp=None):
    sp = P.sp if sp is None else np.asarray(sp, np.complex64)
    x31 = np.ones(P.N + 1, np.complex64)
    x31[:P.N] = x
    tp = np.asarray(tp, np.complex64).copy()
    tp[-1] = 1
    dp = np.empty_like(tp)
    with np.errstate(all="ignore"):
        dp.real, dp.imag = tp.real - sp.real, tp.imag - sp.imag       # target - start per part in float32
    dp[-1] = 0
    return dict(t=F32(t), x=x31, sp=sp, tp=tp, dp=dp)


def eval_points(P, seed=0):
    """(class, finite, point) for every edge class of the evaluators."""
    rng = np.random.default_rng(seed)
    N, NP1 = P.N, P.NP1
    out = []
    for _ in range(6):
        out.append(("random", True, _point(P, rng.uniform(0, 1), _cplx(rng, N), P.sp + _cplx(rng, NP1, 0.5))))
    for _ in range(3):                                       # small integers: exact cancellations, terms summing to +0
        ints = lambda n: (rng.integers(-2, 3, n) + 1j * rng.integers(-2, 3, n)).astype(np.complex64)
        out.append(("int_grid", True, _point(P, 0.5, ints(N), ints(NP1), sp=ints(NP1))))
    for _ in range(3):
        pw = lambda n: (np.where(rng.random(n) < 0.5, -1, 1) * 2.0 ** rng.integers(-3, 4, n)
                        * np.where(rng.random(n) < 0.5, 1, 1j)).astype(np.complex64)
        out.append(("pow2_grid", True, _point(P, 0.25, pw(N), pw(NP1), sp=pw(NP1))))
    for _ in range(3):                                       # components +0 and -0 (both parts, and mixed)
        x = _cplx(rng, N)
        f = c2f(x)
        sel = rng.integers(0, 4, N)
        f[sel == 1] = [0.0, 0.0]
        f[sel == 2] = [-0.0, -0.0]
        f[sel == 3] = [0.0, -0.0]
        out.append(("zeros", True, _point(P, rng.uniform(0, 1), f2c(f), P.sp + _cplx(rng, NP1, 0.5))))
    for _ in range(3):                                       # subnormal components
        f = c2f(_cplx(rng, N))
        sub = rng.random((N, 2)) < 0.4
        f[sub] = (rng.integers(1, 1 << 20, int(sub.sum())) * np.where(rng.random(int(sub.sum())) < 0.5, -1, 1)).astype(F32) * SUBN
        out.append(("subnormal", True, _point(P, rng.uniform(0, 1), f2c(f), P.sp + _cplx(rng, NP1, 0.5))))
    for e in (40, -40):                                      # near 2^+-40: products overflow to Inf / underflow
        f = c2f(_cplx(rng, N))
        big = rng.random((N, 2)) < 0.5
        f[big] = (f[big] * F32(2.0 ** e)).astype(F32)
        out.append(("pow40", e < 0, _point(P, 0.5, f2c(f), P.sp + _cplx(rng, NP1, 0.5))))
    for bad in (np.nan, np.inf, -np.inf):                   # one non-finite component of x, of the target and of the start parameters
        for part in (0, 1):
            f = c2f(_cplx(rng, N))
            f[rng.integers(N), part] = bad
            out.append(("nonfinite_x", False, _point(P, 0.5, f2c(f), P.sp + _cplx(rng, NP1, 0.5))))
        tp = c2f(P.sp + _cplx(rng, NP1, 0.5))
        tp[rng.integers(NP1 - 1), rng.integers(2)] = bad
        out.append(("nonfinite_p", False, _point(P, 0.5, _cplx(rng, N), f2c(tp))))
        sp = c2f(P.sp.copy())
        sp[rng.integers(NP1 - 1), rng.integers(2)] = bad
        out.append(("nonfinite_p", False, _point(P, 0.25, _cplx(rng, N), P.sp + _cplx(rng, NP1, 0.5), sp=f2c(sp))))
    for t in (0.0, 1.0, 0.5, np.nextafter(F32(1), F32(0))):
        out.append(("t_edges", True, _point(P, t, _cplx(rng, N), P.sp + _cplx(rng, NP1, 0.5))))
    return out


def _regular(P, A, b):
    return bool(np.isfinite(A).all() and np.isfinite(b).all() and np.linalg.cond(np.asarray(A, np.complex128)) < 1e6)


def _generic(P, rng, density=1.0):
    for _ in range(100):
        keep = P.mask & (rng.random(P.mask.shape) < density)
        A = np.where(keep, _cplx(rng, P.mask.shape), 0).astype(np.complex64)
        if np.linalg.cond(A.astype(np.complex128)) < 1e4:
            return A, _cplx(rng, P.N)
    raise AssertionError("no well-conditioned system on the pattern")


def _matching(P):
    """A perfect matching of the structural pattern: col -> row (the pattern of a square system that can be regular has one)."""
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import maximum_bipartite_matching
    m = maximum_bipartite_matching(csr_matrix(P.mask.T.astype(np.int8)), perm_type="column")
    assert (m >= 0).all(), "the structural pattern has no perfect matching"
    return m                                                 # m[col] = row


def underflow_system(P):
    """The -0 construction.  A = a permutation pattern (every pivot column has one non-zero, every other multiplier is exactly zero), plus
    A[i, k1] = 2^-76 for the row i that pivots column k2: at step k1 row i gets the multiplier (2^-76, +0) against the pivot row's
    right-hand side (2^-76, -0), and fma(-2^-76, 2^-76, +0) = -0 makes b_i = (-0, +0).  Every other step leaves row i untouched in the
    spec (zero multiplier); x_k2 = b_i * 1/(1 - i) keeps the sign: (-0, +0)."""
    N = P.N
    m = _matching(P)
    A = np.zeros((N, N), np.complex64)
    b = np.full(N, 1 + 1j, np.complex64)
    for col in range(N):
        A[m[col], col] = 1
    for k1 in range(N - 1):
        cands = [k2 for k2 in range(N) if k2 != k1 and P.mask[m[k2], k1]]
        if cands:
            k2 = cands[0]
            break
    else:
        return None
    i = m[k2]
    A[i, k1] = TINY
    A[i, k2] = 1 - 1j
    b[i] = 0
    bf = c2f(b)
    bf[m[k1]] = [TINY, -0.0]
    return dict(A=A, b=f2c(bf), k1=k1, k2=k2, row=i)


def solve_cases(P, seed=0):
    """(label, kind, A, b): kind 'generic' (float64 bars), 'regular' (finite, well conditioned), 'other' (singular / non-finite / extreme),
    'underflow' (the documented -0 deviation)."""
    rng = np.random.default_rng(seed)
    N = P.N
    out = []
    for _ in range(8):
        out.append(("generic", "generic") + _generic(P, rng))
    for _ in range(4):
        out.append(("sparse", "generic") + _generic(P, rng, density=0.6))
    m = _matching(P)
    # exactly-zero multipliers in every step position: column k keeps its matched entry and one other
    for k in range(N):
        A, b = _generic(P, rng)
        rows = np.flatnonzero(P.mask[:, k])
        keep = {m[k], int(rng.choice(rows))}
        for r in rows:
            if r not in keep:
                A[r, k] = 0
        out.append(("zero_mult_col%d" % k, "regular" if _regular(P, A, b) else "other", A, b))
    # exact and near ties in the first step's column (inside a pivot group) and in the first warp-wide column
    for col in sorted({STEP0_COL, P.k1}):
        rows = np.flatnonzero(P.mask[:, col])
        for near in (False, True):
            A, b = _generic(P, rng)
            if col == P.k1 and P.nsp > 0:                     # rows that pivot no sparse column reach step K1 untouched: the tie decides there
                rows = np.array([r for r in rows if r not in {m[c] for c in range(col)}])
                A[rows, :col] = 0
            j = rng.permutation(len(rows))
            mag = F32(8) * (1 + j * F32(2.0 ** -23)) if near else np.full(len(rows), F32(8))
            for r, v, rot in zip(rows, mag, rng.integers(0, 3, len(rows))):
                A[r, col] = [v, 1j * v, (v / 2) * (1 + 1j)][rot]
            out.append(("%stie_col%d" % ("near_" if near else "", col), "regular" if _regular(P, A, b) else "other", A, b))
    # an all-zero pivot column: the first step's column (segmented where the problem has levels) and a warp-wide one
    for col in sorted({STEP0_COL, P.k1, N - 1}):
        A, b = _generic(P, rng)
        A[:, col] = 0
        out.append(("zero_col%d" % col, "other", A, b))
    # pivots with |z|^2 at the clamp: column 0 holds one non-zero z, which is the first pivot
    r0 = int(np.flatnonzero(P.mask[:, 0])[0])
    lo, hi = F32(2.0 ** -50), F32(2.0 ** 50)
    for z in (lo, np.nextafter(lo, F32(0)), np.nextafter(lo, F32(1)), F32(2.0 ** -51), F32(2.0 ** -70), hi, np.nextafter(hi, F32(0)),
              np.nextafter(hi, F32(np.inf)), F32(2.0 ** 51), F32(2.0 ** 60)):
        for zz in (complex(z, 0), complex(z, -z)):
            A, b = _generic(P, rng)
            A[:, 0] = 0
            A[r0, 0] = zz
            out.append(("clamp_%g" % abs(zz), "other", A, b))
    # subnormal entries, and a first column of subnormals only
    A, b = _generic(P, rng)
    sub = P.mask & (rng.random(P.mask.shape) < 0.2)
    A[sub] = (rng.integers(1, 1 << 20, int(sub.sum())) * SUBN).astype(F32) * (1 - 1j)
    out.append(("subnormal_entries", "other", A, b))
    A, b = _generic(P, rng)
    A[P.mask[:, 0], 0] = (rng.integers(1, 1 << 10, int(P.mask[:, 0].sum())) * SUBN).astype(F32)
    out.append(("subnormal_col0", "other", A, b))
    # Inf / NaN in the pivot row, in a non-pivot row, in the right-hand side, and in a row of a lane idle on some level
    for bad in (np.nan, np.inf):
        A, b = _generic(P, rng)
        A[:, 0] = 0
        A[r0, 0] = 4
        A[r0, [c for c in np.flatnonzero(P.mask[r0]) if c != 0][0]] = bad
        out.append(("nonfinite_pivot_row", "other", A, b))
        A, b = _generic(P, rng)
        r = [r for r in range(N) if r != r0][0]
        A[r, np.flatnonzero(P.mask[r])[-1]] = complex(bad, 0)
        out.append(("nonfinite_row", "other", A, b))
        A, b = _generic(P, rng)
        b[rng.integers(N)] = complex(0, bad)
        out.append(("nonfinite_rhs", "other", A, b))
        idle = [P.row_of_lane[l] for l in range(N) if P.idle_levels[l]]
        if idle:
            A, b = _generic(P, rng)
            A[idle[0], np.flatnonzero(P.mask[idle[0]])[0]] = bad
            out.append(("nonfinite_idle_row", "other", A, b))
    u = underflow_system(P)
    if u is not None:
        out.append(("underflow", "underflow", u["A"], u["b"]))
    return out


def with_regular_after_each(P, cases, seed=1):
    """Interleave: every case is followed by a fresh regular system, so that a stale pivot-row buffer left by a singular or non-finite
    system would show as an exact pass on the regular one."""
    rng = np.random.default_rng(seed)
    out = []
    for c in cases:
        out.append(c)
        out.append(("regular_after_" + c[0], "regular") + _generic(P, rng))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# CPU part

def test_the_float32_facts_of_the_zero_multiplier_update():
    """fmaf(-2^-76, 2^-76, +0) is -0 (denormals kept, the product is below 2^-150), and the kernel's zero-multiplier update
    (c_msub_m with m = (0, 0)) is not the identity on (-0, -0).  Zero products and sums of zeros are exact in float64, so float64
    arithmetic states the float32 fma here."""
    def fma(a, b, c):
        return F32(np.float64(a) * np.float64(b) + np.float64(c))

    assert np.signbit(fma(-TINY, TINY, F32(0.0))) and fma(-TINY, TINY, F32(0.0)) == 0

    def msub_zero(acc, u):          # c_msub_m(acc, make_mult(m, false), u): (fma(-0, u.x, acc.x) -> fma(+0, u.y, .), fma(-0, u.y, acc.y) -> fma(-u.x, +0, .))
        re = fma(F32(-0.0), u[0], acc[0])
        re = fma(F32(0.0), u[1], re)
        im = fma(F32(-0.0), u[1], acc[1])
        im = fma(-u[0], F32(0.0), im)
        return np.signbit(re), np.signbit(im)

    acc = (F32(-0.0), F32(-0.0))
    assert msub_zero(acc, (F32(1), F32(1))) == (False, True)
    assert msub_zero(acc, (F32(-1), F32(1))) == (False, False)
    assert msub_zero(acc, (F32(1), F32(-1))) == (True, False)
    assert msub_zero(acc, (F32(0), F32(0))) == (False, True)         # exact mode's zero row
    for u in ((F32(1.5), F32(-2)), (F32(-3), F32(0.25))):          # on a non-zero entry the update IS the identity
        assert msub_zero((F32(0.75), F32(-1e-30)), u) == (False, True)


@pytest.mark.parametrize("name", PROBLEMS)
def test_oracle_solve_keeps_an_underflowed_minus_zero_untouched(name):
    """The -0 construction on oracle.solve: a tiny multiplier times a tiny pivot-row entry turns a zero right-hand side into -0, and the
    later steps, whose multipliers for that row are exactly zero, leave it alone: x_k2 = (-0, +0), where a +0 right-hand side gives +0."""
    P = prim(name)
    u = underflow_system(P)
    assert u is not None
    x, info = P.oracle_solve(u["A"], u["b"])
    assert info == 0
    assert x[u["k2"]] == 0 and np.signbit(x[u["k2"]].real) and not np.signbit(x[u["k2"]].imag)
    b0 = u["b"].copy()
    b0[np.argmax(np.abs(u["A"][:, u["k1"]]))] = 0            # no underflow: the pivot row's right-hand side is +0
    x0, _ = P.oracle_solve(u["A"], b0)
    assert x0[u["k2"]] == 0 and not np.signbit(x0[u["k2"]].real)
    # every other component is the permutation system's plain solution
    ref = np.linalg.solve(u["A"].astype(np.complex128), u["b"].astype(np.complex128))
    assert np.allclose(x, ref, rtol=1e-6, atol=1e-30)


@pytest.mark.parametrize("name", PROBLEMS)
def test_inputs_respect_the_structural_pattern(name):
    """Every solve input lies on the slot map (so nothing is dropped when it is loaded into the register slots), every evaluator output
    does too, and the pattern is what the oracle's Jacobian can reach."""
    P = prim(name)
    for label, kind, A, b in with_regular_after_each(P, solve_cases(P)):
        off = ~P.mask & ~((A.real == 0) & (A.imag == 0))
        assert not off.any(), "%s: non-zero off the slot map at %s" % (label, np.argwhere(off)[:3].tolist())
    for cls, finite, pt in eval_points(P):
        A, _, _, _ = P.oracle_eval(pt)
        off = ~P.mask & ~((A.real == 0) & (A.imag == 0))
        assert not off.any(), "%s: the oracle's Jacobian is non-zero off the slot map" % cls
    # and the map is the table's: every column the Hx table gives a row is a slot of that row
    hx = P.hx.reshape(P.N, P.hx_terms, 5, P.N)
    assert np.array_equal((hx[:, :, 0, :] != 0).any(1).T, P.mask)


@pytest.mark.parametrize("name", PROBLEMS)
def test_float64_evaluator_reference_bounds_the_oracle(name):
    """The float64 statement and its bound hold for the oracle on the finite classes (so the same bound on the device measures the kernel,
    not the reference), and the oracle's parameter homotopy is within 2 ulp-scaled terms of float64."""
    P = prim(name)
    for cls, finite, pt in eval_points(P):
        A, h, ht, p = P.oracle_eval(pt)
        t, omt = np.float64(pt["t"]), np.float64(F32(1) - pt["t"])     # the spec rounds 1 - t to float once
        tp, sp = pt["tp"].astype(np.complex128), pt["sp"].astype(np.complex128)
        if finite:
            for part in ("real", "imag"):
                ref = t * getattr(tp, part) + omt * getattr(sp, part)
                scale = np.abs(t * getattr(tp, part)) + np.abs(omt * getattr(sp, part))
                assert (np.abs(getattr(p, part)[:-1] - ref[:-1]) <= 2 * EPS * scale[:-1]).all(), cls
            _check_f64(P, cls, pt, p, A, h, ht)


def _check_f64(P, cls, pt, p, A, h, ht):
    A64, SA, TA, H64, SH, TH, Ht64, SHt, THt = f64_eval(P, pt["x"], p, pt["dp"])
    for got, ref, S, T, what in ((A, A64, SA, TA, "Hx"), (h, H64, SH, TH, "H"), (ht, Ht64, SHt, THt, "-dH/dt")):
        err = np.abs(got.astype(np.complex128) - ref)
        bound = eval_bound(S, T)
        assert np.isfinite(got).all(), "%s %s: non-finite on finite input" % (cls, what)
        assert (err <= bound).all(), "%s %s: |err| %.3g exceeds the bound %.3g" % (cls, what, err.max(), bound[np.unravel_index(np.argmax(err - bound), err.shape)])


# ---------------------------------------------------------------------------------------------------------------------
# GPU part

@pytest.mark.gpu
@pytest.mark.parametrize("name", PROBLEMS)
def test_evaluators_against_the_oracle_and_float64(name):
    P = prim(name)
    items = eval_points(P)
    pts = [pt for _, _, pt in items]
    A, h, ht = P.gpu_eval(pts, n_warps=1)            # one warp, every point in sequence
    A2, h2, ht2 = P.gpu_eval(pts, n_warps=7)
    assert same_bits(A, A2).all() and same_bits(h, h2).all() and same_bits(ht, ht2).all(), "result depends on the warp"
    for s, (cls, finite, pt) in enumerate(items):
        Ao, ho, hto, p = P.oracle_eval(pt)
        assert_same(A[s], Ao, "%s Hx (%s)" % (cls, name))
        assert_same(h[s], ho, "%s H (%s)" % (cls, name))
        assert_same(ht[s], hto, "%s -dH/dt (%s)" % (cls, name))
        off = ~P.mask & ~((A[s].real == 0) & (A[s].imag == 0))
        assert not off.any()
        if finite:
            _check_f64(P, cls, pt, p, A[s], h[s], ht[s])


def _check_solves(P, cases, n_warps):
    fast, exact, sel, info = P.gpu_solve([dict(A=A, b=b) for _, _, A, b in cases], n_warps=n_warps)
    for s, (label, kind, A, b) in enumerate(cases):
        what = "%s (%s, system %d)" % (label, P.name, s)
        assert info[s, 1] == 0, "%s: %d non-zeros off the slot map were dropped" % (what, info[s, 1])
        xo, _ = P.oracle_solve(A, b)
        assert_same(sel[s], xo, what, zero_sign=(kind != "underflow"))
        if np.isfinite(fast[s]).all():
            assert_same(fast[s], sel[s], what + ": fast pass")
            assert_same(exact[s], sel[s], what + ": exact pass", zero_sign=(kind != "underflow"))
            assert info[s, 0] == 0
        else:
            assert info[s, 0] == 1
            assert_same(exact[s], sel[s], what + ": exact pass")
        if kind in ("generic", "regular", "underflow"):
            assert np.isfinite(xo).all(), what
            assert info[s, 0] == 0, "%s: a regular finite system took the exact pass" % what
        if kind == "generic":
            A64, b64, x = A.astype(np.complex128), b.astype(np.complex128), sel[s].astype(np.complex128)
            growth = max(1.0, gj_growth(A64))
            nA = np.abs(A64).sum(1).max()
            berr = np.abs(A64 @ x - b64).max() / (nA * np.abs(x).max() + np.abs(b64).max())
            assert berr <= 30 * EPS * growth, "%s: backward error %.3g > 30 * 2^-24 * growth %.3g" % (what, berr, growth)
            xr = np.linalg.solve(A64, b64)
            cond = np.linalg.cond(A64, np.inf)
            ferr = np.abs(x - xr).max() / np.abs(xr).max()
            assert ferr <= cond * 30 * EPS * growth, "%s: forward error %.3g, cond %.3g" % (what, ferr, cond)


@pytest.mark.gpu
@pytest.mark.parametrize("name", PROBLEMS)
def test_solve_against_the_oracle_and_float64(name):
    """Every constructed case, each followed by a fresh regular system, on ONE warp in sequence (stale pivot-row buffers carry over), and
    the same list spread over several warps."""
    P = prim(name)
    cases = with_regular_after_each(P, solve_cases(P))
    _check_solves(P, cases, n_warps=1)
    _check_solves(P, cases[::-1], n_warps=5)


@pytest.mark.gpu
@pytest.mark.parametrize("name", PROBLEMS)
def test_eval_and_solve_equals_the_oracle(name):
    """The tracker's eval_and_solve at the evaluator's edge points: the predictor's solve(Hx, -dH/dt) and the corrector's solve(Hx, H)
    equal oracle.eval_* followed by oracle.solve."""
    P = prim(name)
    items = eval_points(P, seed=3)
    pts = [pt for _, _, pt in items]
    pred, corr = P.gpu_eval_and_solve(pts, n_warps=1)
    for s, (cls, finite, pt) in enumerate(items):
        Ao, ho, hto, _ = P.oracle_eval(pt)
        assert_same(pred[s], P.oracle_solve(Ao, hto)[0], "%s predictor (%s)" % (cls, name))
        assert_same(corr[s], P.oracle_solve(Ao, ho)[0], "%s corrector (%s)" % (cls, name))


@pytest.mark.gpu
def test_reciprocal_step_is_correctly_rounded_on_the_whole_clamp_range():
    """recip_newton (MUFU.RCP + one FMA-Newton step) == __frcp_rn on every float in [2^-100, 2^100] (1.68e9 values)."""
    import torch
    P = prim(TRIFOCAL)
    dev = torch.device("cuda:0")
    count = torch.zeros(1, dtype=torch.int64, device=dev)
    first = torch.zeros(16, dtype=torch.int32, device=dev)
    lo, hi = int(np.array(2.0 ** -100, F32).view(np.uint32)), int(np.array(2.0 ** 100, F32).view(np.uint32))
    assert hi - lo + 1 == 200 * (1 << 23) + 1
    rc = P.lib.hcb200_unit_recip_sweep(ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream), lo, hi,
                                       ctypes.c_void_p(count.data_ptr()), ctypes.c_void_p(first.data_ptr()))
    assert rc == 0
    n = int(count.cpu()[0])
    assert n == 0, "%d mismatches, first bit patterns %s" % (n, [hex(v) for v in first.cpu().numpy().view(np.uint32)[:min(n, 16)]])


@pytest.mark.gpu
@pytest.mark.parametrize("name", PROBLEMS)
def test_c_recip_at_its_edges_and_frcp_against_numpy(name):
    P = prim(name)
    rng = np.random.default_rng(5)
    # __frcp_rn == numpy's float32 1/d on a sample of the range and beyond it (subnormals, huge, 0, Inf, NaN)
    bits = np.concatenate([rng.integers(0x0D800000, 0x71800001, 200000), rng.integers(1, 0x7F800000, 50000),
                           [0, 1, 0x007FFFFF, 0x00800000, 0x7F7FFFFF, 0x7F800000, 0x7FC00000]]).astype(np.uint32)
    d = bits.view(F32)
    d = np.concatenate([d, -d])
    z = np.stack([d, np.zeros_like(d)], -1)
    # c_recip at 0, subnormal, the clamp's ends +- 1 ulp (|z|^2 = 2^+-100 for z = 2^+-50), beyond, Inf and NaN
    edge = []
    for v in (0.0, -0.0, float(SUBN), 2.0 ** -130, 2.0 ** -50, 2.0 ** 50, 2.0 ** -51, 2.0 ** 51, 2.0 ** 70, np.inf, -np.inf, np.nan):
        v = F32(v)
        for w in (v, np.nextafter(v, F32(0)), np.nextafter(v, F32(np.inf))):
            edge += [(w, 0), (0, w), (w, w), (w, -w), (w, 1), (1, w)]
    ze = np.array(edge, F32)
    zz = np.concatenate([z, ze]).astype(F32)
    out, frcp = _recip(P, zz)
    with np.errstate(all="ignore"):
        want = (F32(1) / zz[:, 0]).astype(F32)
    assert np.array_equal(frcp.view(np.uint32)[~np.isnan(want)], want.view(np.uint32)[~np.isnan(want)])
    assert np.isnan(frcp[np.isnan(want)]).all()
    assert_same(f2c(out[len(z):]), P.oracle_recip(f2c(ze)), "c_recip at its edges")
    assert_same(f2c(out[:len(z)]), P.oracle_recip(f2c(z)), "c_recip on the sample")


def _recip(P, z):
    import torch
    dev = torch.device("cuda:0")
    dz = torch.from_numpy(np.ascontiguousarray(z, F32)).to(dev)
    out = torch.zeros_like(dz)
    frcp = torch.zeros(len(z), dtype=torch.float32, device=dev)
    rc = P.lib.hcb200_unit_recip(ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream), len(z), ctypes.c_void_p(dz.data_ptr()),
                                 ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(frcp.data_ptr()))
    assert rc == 0
    torch.cuda.synchronize(dev)
    return out.cpu().numpy(), frcp.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("name", PROBLEMS)
def test_production_tracker_on_crafted_start_points_and_parameters(name):
    """The primitive-level edges through the public ABI: hcb200_track with crafted d_start_sols / d_start_params (start points with +0 and -0
    components, points scaled into the subnormal range, small-integer parameters with exact ties), 1-3 HC steps, one or two hypotheses,
    against an Oracle built on the same crafted problem dict, bit for bit."""
    P = prim(name)
    rng = np.random.default_rng(11)
    prob = dict(P.problem)
    ss = np.array(prob["start_sols"], np.complex64)
    T, N = ss.shape
    f = c2f(ss)
    q = T // 4
    sel = rng.integers(0, 3, (q, N))
    f[:q][sel == 1] = [0.0, 0.0]
    f[:q][sel == 2] = [-0.0, -0.0]
    f[q:2 * q] = (f[q:2 * q] * F32(2.0 ** -140)).astype(F32)            # subnormal-scaled start points
    f[2 * q:3 * q] = np.round(f[2 * q:3 * q])                           # small integers: exact ties in pivot columns
    prob["start_sols"] = f2c(f)
    NP = len(prob["start_params"])
    prob["start_params"] = (rng.integers(-2, 3, NP) + 1j * rng.integers(-1, 2, NP)).astype(np.complex64)
    sp1 = np.concatenate([prob["start_params"], [1.0]]).astype(np.complex64)
    if name == TRIFOCAL:
        orc = Oracle(prob)
    else:
        orc = Oracle(prob, problem_dir=os.path.join(ROOT, "problems", name))
    for n_hyp, max_steps in ((1, 1), (2, 3)):
        tgt = (rng.integers(-3, 4, (n_hyp, NP + 1)) + 1j * rng.integers(-3, 4, (n_hyp, NP + 1)) * 0.5).astype(np.complex64)
        tgt[:, -1] = 1
        dif = np.empty_like(tgt)
        dif.real, dif.imag = tgt.real - sp1.real, tgt.imag - sp1.imag
        if name == TRIFOCAL:
            trk = hc.Tracker(device="cuda:0", problem=prob, max_steps=max_steps)
            trk.upload_params(tgt, dif)
            trk.track(n_hyp, prune=False)
            _, cv_g, inf_g, _ = trk.results(n_hyp)
        else:
            trk = pm.ProblemTracker(os.path.join(ROOT, "problems", name), problem=prob, device="cuda:0", max_steps=max_steps)
            trk.upload_params(tgt)
            trk.track(n_hyp)
            _, cv_g, inf_g = trk.results(n_hyp)[:3]
        tr_g = f2c(trk.d_tracks[:n_hyp * T].cpu().numpy())
        tr_o, cv_o, inf_o = P.oracle_track(orc, tgt, dif, max_steps)
        assert np.array_equal(cv_g, cv_o) and np.array_equal(inf_g, inf_o)
        assert_same(tr_g[:, :N], tr_o[:, :N], "tracks after %d steps (%s)" % (max_steps, name))
