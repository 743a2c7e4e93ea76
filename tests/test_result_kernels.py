"""The round-result kernels against float64 and host references, at their thresholds and edges.

After the tracker, a round runs hcb200_score_tracks (candidate gate, inlier supports, best record), hcb200_make_pose_record (the 128-byte
exchange record), hcb200_reduce_pose_records (the arg-max over the gathered records) and, in the host class, hcb200_count_solutions and
hcb200_build_target_params.  Comparing float32 with float32 only proves that two implementations agree, so this file also states every decision
in plain float64 arithmetic:

* a synthetic scene (fixed seed, K of dataset 0) whose edgel triplets sit clearly inside or outside the 2 px inlier threshold, 2-30 mpx from
  it (the near tier), or within 1 mpx of it (the band); the float64 reprojection error of the host formula (host/mvg.hpp) gives each edgel
  a STABILITY INTERVAL: the edgel is unstable when its float64 decision changes under perturbations of 4 float32 ulp of every input (R, T,
  g1, g2, K; 8 seeded draws).  As in test_parity_envelope.py, float32 may differ from float64 on unstable edgels only.  With fx = 2585 px a
  few ulp of R move the error by several mpx, so the band is all unstable; the near tier is what makes the interval tight: it resolves
  the threshold to 10 mpx (a 1.99 or 2.01 px threshold falls outside it);
* numpy float32 restatements of the pose arithmetic (host/mvg.hpp operation order), pinned bit for bit to mvg.hpp on the CPU;
* plain Python arg-max, sum and OR for the record reductions, and a float64 numpy statement of Evaluations.cpp:145-167 for the counts.

The CPU part runs without a GPU; the GPU part writes synthetic end points straight into device buffers (no tracking) except the early-abort
threshold test, which tracks hypothesis 0 of dataset 0."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from trifocal_pose_estimation_using_improved_gpuhc_b200 import fixtures, hc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "trifocal_pose_estimation_using_improved_gpuhc_b200")
LIBDIR = os.path.join(PKG, "lib")
F32, F64 = np.float32, np.float64
INVALID_VALUE = 1
T = hc.NUM_TRACKS
IM_TOL = F32(1e-5)                                 # float32(1e-5) < 1e-5 in double: passes the Cayley gate
IM_ABOVE = np.nextafter(IM_TOL, F32(1))            # the next float32: fails it
SUBNORMAL = np.nextafter(F32(0), F32(1))           # 2^-149
SENTINEL = 0x5A5A5A5A


def _vp(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _host():
    return ctypes.CDLL(os.path.join(LIBDIR, "libhcb200_host.so"))


# ---------------------------------------------------------------------------------------------------------------------
# references

def rotation32(r):
    """host_style_rotation / mvg::cayley_to_rotation in float32, operation for operation: un-normalised Cayley matrix, columns scaled to 1."""
    r0, r1, r2 = (F32(v) for v in r)
    one, two = F32(1), F32(2)
    with np.errstate(all="ignore"):
        R = [one + r0 * r0 - (r1 * r1 + r2 * r2), two * (r0 * r1 - r2), two * (r0 * r2 + r1),
             two * (r0 * r1 + r2), one + r1 * r1 - (r0 * r0 + r2 * r2), two * (r1 * r2 - r0),
             two * (r0 * r2 - r1), two * (r1 * r2 + r0), one + r2 * r2 - (r0 * r0 + r1 * r1)]
        for c in range(3):
            n = np.sqrt(R[c] * R[c] + R[3 + c] * R[3 + c] + R[6 + c] * R[6 + c])
            R[c], R[3 + c], R[6 + c] = R[c] / n, R[3 + c] / n, R[6 + c] / n
    return np.array(R, F32)


def unit32(t):
    """mvg::normalized in float32."""
    t0, t1, t2 = (F32(v) for v in t)
    with np.errstate(all="ignore"):
        n = np.sqrt(t0 * t0 + t1 * t1 + t2 * t2)
        return np.array([t0 / n, t1 / n, t2 / n], F32)


def pose32(x31):
    """The 24 pose floats hcb200_make_pose_record writes for end point x31 (complex64 [31]): R21, t21, R31, t31."""
    x = np.asarray(x31, np.complex64).real
    return np.concatenate([rotation32(x[24:27]), unit32(x[18:21]), rotation32(x[27:30]), unit32(x[21:24])])


def rotation64(r):
    """Cayley rotation in float64 with unit columns (an exact rotation up to float64 rounding)."""
    r0, r1, r2 = (F64(v) for v in r)
    R = np.array([1 + r0 * r0 - (r1 * r1 + r2 * r2), 2 * (r0 * r1 - r2), 2 * (r0 * r2 + r1),
                  2 * (r0 * r1 + r2), 1 + r1 * r1 - (r0 * r0 + r2 * r2), 2 * (r1 * r2 - r0),
                  2 * (r0 * r2 - r1), 2 * (r1 * r2 + r0), 1 + r2 * r2 - (r0 * r0 + r1 * r1)]).reshape(3, 3)
    return (R / np.linalg.norm(R, axis=0)).reshape(9)


def pose64(x31):
    x = np.asarray(x31, np.complex64).real.astype(F64)
    u = lambda t: t / np.linalg.norm(t)
    return np.concatenate([rotation64(x[24:27]), u(x[18:21]), rotation64(x[27:30]), u(x[21:24])])


def pair_pose64(x31, pair):
    """(R [9], unit t [3]) in float64 of view pair 1-2 (pair 0) or 1-3 (pair 1) of end point x31."""
    x = np.asarray(x31, np.complex64).real.astype(F64)
    t = x[18 + 3 * pair:21 + 3 * pair]
    return rotation64(x[24 + 3 * pair:27 + 3 * pair]), t / np.linalg.norm(t)


def reproj_error(R, T_, g1, g2, K):
    """mvg::depth_rho + mvg::reprojection_error_pixels in the host's operation order, vectorised over edgels.  Every argument has the same
    dtype: float32 restates the host bit for bit, float64 is the plain-mathematics reference.  R [..., 9], T [..., 3], g [..., 2], K [..., 9]."""
    one = R.dtype.type(1)
    with np.errstate(all="ignore"):
        Rtg2 = R[..., 2] * g2[..., 0] + R[..., 5] * g2[..., 1] + R[..., 8] * one
        RtT = R[..., 2] * T_[..., 0] + R[..., 5] * T_[..., 1] + R[..., 8] * T_[..., 2]
        Rg1 = R[..., 6] * g1[..., 0] + R[..., 7] * g1[..., 1] + R[..., 8] * one
        rho = (T_[..., 2] * Rtg2 - RtT) / (one - Rg1 * Rtg2)
        q0 = (R[..., 0] * g1[..., 0] + R[..., 1] * g1[..., 1] + R[..., 2] * one) * rho + T_[..., 0]
        q1 = (R[..., 3] * g1[..., 0] + R[..., 4] * g1[..., 1] + R[..., 5] * one) * rho + T_[..., 1]
        q2 = Rg1 * rho + T_[..., 2]
        u = (q0 / q2) * K[..., 0] + K[..., 2]
        v = (q1 / q2) * K[..., 4] + K[..., 5]
        du = u - (g2[..., 0] * K[..., 0] + K[..., 2])
        dv = v - (g2[..., 1] * K[..., 4] + K[..., 5])
        return np.sqrt(du * du + dv * dv)


def stability(x31, loc, K, pair, draws=8, seed=7):
    """Float64 decision (error < 2 px) of every edgel for view pair 1-2 (pair 0) or 1-3 (pair 1) of the pose in x31, and whether that
    decision is unstable: it changes when every input is moved by up to 4 ulp of its float32 value, in `draws` seeded draws.  The
    draws start from the float64 pose and from the float32 pose the host computes (rotation32 / unit32), which lies a few correlated ulp
    away: independent random draws around the float64 pose alone miss that direction on a few edgels."""
    g1 = loc[:, 0:2].astype(F64)
    g2 = loc[:, 2 + 2 * pair:4 + 2 * pair].astype(F64)
    K64 = np.asarray(K, F64).reshape(9)
    R, t = pair_pose64(x31, pair)
    e0 = reproj_error(R, t, g1, g2, K64)
    lo, hi = e0.copy(), e0.copy()
    rng = np.random.default_rng(seed + pair)
    n = loc.shape[0]
    p = lambda a: a + rng.uniform(-4, 4, (n,) + a.shape[-1:]) * np.spacing(np.abs(a).astype(F32)).astype(F64)
    x = np.asarray(x31, np.complex64).real
    for R, t in ((R, t), (rotation32(x[24 + 3 * pair:27 + 3 * pair]).astype(F64), unit32(x[18 + 3 * pair:21 + 3 * pair]).astype(F64))):
        e = reproj_error(R, t, g1, g2, K64)
        lo, hi = np.minimum(lo, e), np.maximum(hi, e)
        for _ in range(draws):
            e = reproj_error(p(np.broadcast_to(R, (n, 9))), p(np.broadcast_to(t, (n, 3))), p(g1), p(g2), p(np.broadcast_to(K64, (n, 9))))
            lo, hi = np.minimum(lo, e), np.maximum(hi, e)
    return e0 < 2, (lo < 2) & (hi >= 2)


def host_score(x31, loc, K, lib=None):
    """hcb200_host_score_track: (is candidate, n21, n31)."""
    lib = lib or _host()
    x = np.ascontiguousarray(np.stack([x31.real, x31.imag], -1).astype(F32))
    loc = np.ascontiguousarray(loc, F32)
    Kf = np.ascontiguousarray(K, F32).reshape(9)
    n21, n31 = ctypes.c_int(), ctypes.c_int()
    ok = lib.hcb200_host_score_track(_vp(x), _vp(loc), loc.shape[0], _vp(Kf), ctypes.byref(n21), ctypes.byref(n31))
    return bool(ok), n21.value, n31.value


# ---------------------------------------------------------------------------------------------------------------------
# the synthetic scene

N_EDGELS = 5117
BAND = 1e-3                 # the band: float64 error within 1e-3 px of 2 px, finer than float32 resolves here (all unstable)
NEAR = (2e-3, 3e-2)         # the near tier: float64 error 2-30 mpx from 2 px, on either side; mostly stable


def end_point(r21, t21, r31, t31, rng):
    """An end point carrying the pose: depths in lanes 0-7, other variables in 8-17, t21 t31 in 18-23, r21 r31 in 24-29, small imaginary
    parts below every gate, lane 30 = 1+0i."""
    x = np.zeros(31, np.complex64)
    x.real[0:8] = rng.uniform(0.5, 9.0, 8)
    x.real[8:18] = rng.uniform(-1, 1, 10)
    x.imag[0:30] = rng.uniform(-2e-6, 2e-6, 30)
    x.real[18:21], x.real[21:24], x.real[24:27], x.real[27:30] = t21, t31, r21, r31
    x[30] = 1
    return x


def _build_scene(seed=20261020):
    rng = np.random.default_rng(seed)
    K = np.asarray(fixtures.load_ransac(0)["K"], F32).reshape(9)
    K64 = K.astype(F64)
    # pose 0 generates the edgels; its translations are stored un-normalised, so the kernels' normalisation is part of what is tested
    r21, t21 = np.array([0.05, -0.1, 0.07], F32), np.array([0.39, -0.26, 1.3], F32)
    r31, t31 = np.array([-0.08, 0.06, 0.03], F32), np.array([-0.3, 0.06, 0.54], F32)
    poses = [end_point(r21, t21, r31, t31, rng),
             end_point(r21 + F32(4e-4), t21, r31, t31 + F32(2e-3), rng),                    # near pose 0: other edgels near 2 px
             end_point(np.array([0.2, 0.1, -0.1], F32), np.array([1, 0.2, 0.1], F32), r31 - F32(3e-3), t31, rng)]
    M = 24000
    z = rng.uniform(3, 8, M)
    X = np.c_[rng.uniform(-0.07, 0.07, M) * z, rng.uniform(-0.07, 0.07, M) * z, z]
    g1 = X[:, :2] / X[:, 2:]
    views, keep = [g1], np.ones(M, bool)
    for pair in (0, 1):
        R, t = pair_pose64(poses[0], pair)
        Q = X @ R.reshape(3, 3).T + t
        g = Q[:, :2] / Q[:, 2:]
        # 0 clearly inside, 1 clearly outside, 2 the band around 2 px, 3 the near tier
        cat = rng.choice(4, M, p=[0.28, 0.22, 0.15, 0.35])
        th = rng.uniform(0, 2 * np.pi, M)
        d = np.c_[np.cos(th) / K64[0], np.sin(th) / K64[4]]
        s = np.where(cat == 0, rng.uniform(0, 1.6, M), np.where(cat == 1, rng.uniform(3, 40, M), rng.uniform(2, 4, M)))
        band, near = cat == 2, cat == 3
        side = rng.choice([-1.0, 1.0], M)
        target = np.where(band, 2 + rng.uniform(-0.8 * BAND, 0.8 * BAND, M), 2 + side * rng.uniform(NEAR[0] * 1.2, NEAR[1] * 0.9, M))
        for _ in range(5):                                            # rescale the offsets until their float64 error is ~target
            e = reproj_error(R, t, g1, g + d * s[:, None], K64)
            with np.errstate(all="ignore"):
                s = np.where((band | near) & np.isfinite(e) & (e > 0), s * target / e, s)
        gp = g + d * s[:, None]
        e = np.abs(reproj_error(R, t, g1.astype(F32).astype(F64), gp.astype(F32).astype(F64), K64) - 2)
        # the tiers are selected by the float64 error of the stored float32 edgel, not by the offset (the depth is re-estimated from g2)
        keep &= np.isfinite(e) & np.where(band, e <= BAND, np.where(near, (e >= NEAR[0]) & (e <= NEAR[1]), e > 0.05))
        views.append(gp)
    loc = np.concatenate(views, 1).astype(F32)[keep]
    assert loc.shape[0] >= N_EDGELS
    return {"loc": np.ascontiguousarray(loc[:N_EDGELS]), "K": K, "poses": poses}


@pytest.fixture(scope="module")
def scene():
    sc = _build_scene()
    sc["stab"] = [[stability(x, sc["loc"], sc["K"], pair) for pair in (0, 1)] for x in sc["poses"]]
    return sc


def support_bounds(sc, pose, n_edgels):
    """[stable inliers, stable inliers + unstable] of pose `pose` on the first n_edgels edgels, for both view pairs."""
    out = []
    for pair in (0, 1):
        d64, unstable = (a[:n_edgels] for a in sc["stab"][pose][pair])
        lo = int((d64 & ~unstable).sum())
        out.append((lo, lo + int(unstable.sum())))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# CPU

def test_the_stability_interval_resolves_the_threshold_to_10_mpx(scene):
    """For pose 0 and both view pairs: the band (|e - 2| <= 1e-3 px) is finer than float32 resolves with fx = 2585 px, so all of it is
    unstable; the near tier (2-30 mpx from 2 px) is mostly stable, with at least 100 stable edgels within 10 mpx on EACH side of 2 px.  So the
    interval is tight: the float32 restatement with a threshold of 1.99 or 2.01 px instead of 2 px gives a count outside it."""
    loc, K = scene["loc"], scene["K"]
    x = scene["poses"][0]
    for pair in (0, 1):
        R, t = pair_pose64(x, pair)
        e = reproj_error(R, t, loc[:, 0:2].astype(F64), loc[:, 2 + 2 * pair:4 + 2 * pair].astype(F64), K.astype(F64)) - 2
        d64, unstable = scene["stab"][0][pair]
        band, near = np.abs(e) <= BAND, (np.abs(e) >= NEAR[0]) & (np.abs(e) <= NEAR[1])
        assert band.sum() >= 600 and near.sum() >= 1500 and (e < -0.05).sum() >= 1000 and (e > 0.05).sum() >= 500
        assert not np.any(unstable & ~band & ~near)                    # clearly inside or outside: always stable
        assert (unstable & near).sum() <= 0.2 * near.sum()
        assert unstable.sum() <= 0.25 * loc.shape[0]
        assert (~unstable & (e < 0) & (e > -0.01)).sum() >= 100 and (~unstable & (e > 0) & (e < 0.01)).sum() >= 100
        lo = int((d64 & ~unstable).sum())
        hi = lo + int(unstable.sum())
        e32 = reproj_error(rotation32(x.real[24 + 3 * pair:27 + 3 * pair]), unit32(x.real[18 + 3 * pair:21 + 3 * pair]), loc[:, 0:2],
                           loc[:, 2 + 2 * pair:4 + 2 * pair], K)
        assert lo <= int((e32 < 2).sum()) <= hi
        assert int((e32 < F32(1.99)).sum()) < lo and int((e32 < F32(2.01)).sum()) > hi, (pair, lo, hi)


@pytest.mark.parametrize("pose", [0, 1, 2])
def test_host_score_track_lies_in_the_float64_stability_interval(scene, pose):
    """hcb200_host_score_track counts lie in [stable inliers, stable inliers + unstable] for both view pairs, on the whole edgel set and on
    prefixes; the numpy float32 restatement gives the same counts, and every edgel where float32 and float64 decide differently is unstable."""
    loc, K, x = scene["loc"], scene["K"], scene["poses"][pose]
    lib = _host()
    R = [rotation32(x.real[24:27]), rotation32(x.real[27:30])]
    t = [unit32(x.real[18:21]), unit32(x.real[21:24])]
    for n in (1, 31, 255, 257, N_EDGELS):
        ok, n21, n31 = host_score(x, loc[:n], K, lib)
        assert ok
        for pair, got in ((0, n21), (1, n31)):
            lo, hi = support_bounds(scene, pose, n)[pair]
            assert lo <= got <= hi, (pose, n, pair, lo, got, hi)
            d32 = reproj_error(R[pair], t[pair], loc[:n, 0:2], loc[:n, 2 + 2 * pair:4 + 2 * pair], K) < 2
            assert int(d32.sum()) == got
            d64, unstable = (a[:n] for a in scene["stab"][pose][pair])
            assert not np.any((d32 != d64) & ~unstable)


def test_float32_restatements_are_bit_identical_to_mvg(tmp_path):
    """rotation32 / unit32 (used by the GPU tests as the expected pose) against mvg::cayley_to_rotation / mvg::normalized compiled as the host
    library is compiled."""
    src = tmp_path / "mvg_shim.cpp"
    src.write_text('#include "mvg.hpp"\n'
                   'extern "C" void pose(const float* r, const float* t, float* out) {\n'
                   '  const auto R = hcb200::mvg::cayley_to_rotation({r[0], r[1], r[2]});\n'
                   '  const auto u = hcb200::mvg::normalized({t[0], t[1], t[2]});\n'
                   '  for (int i = 0; i < 9; i++) out[i] = R[i];\n'
                   '  for (int i = 0; i < 3; i++) out[9 + i] = u[i];\n}\n')
    so = tmp_path / "libmvg_shim.so"
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-I" + os.path.join(PKG, "host"), "-o", str(so), str(src)])
    lib = ctypes.CDLL(str(so))
    rng = np.random.default_rng(3)
    rs = [rng.uniform(-a, a, 3).astype(F32) for a in (1e-3, 0.1, 1.0, 30.0) for _ in range(500)]
    rs += [np.zeros(3, F32), np.array([SUBNORMAL, 0, -SUBNORMAL], F32), np.array([1e19, 0, 0], F32)]
    ts = [rng.uniform(-a, a, 3).astype(F32) for a in (1e-20, 1e-3, 1.0, 1e18) for _ in range(500)]
    ts += [np.zeros(3, F32), np.array([SUBNORMAL, 0, 0], F32), np.array([np.nan, 1, 1], F32)]
    out = np.zeros(12, F32)
    for r, t in zip(rs, ts):
        lib.pose(_vp(r), _vp(t), _vp(out))
        mine = np.concatenate([rotation32(r), unit32(t)])
        assert np.array_equal(mine.view(np.uint32), out.view(np.uint32)) or \
            np.all((mine.view(np.uint32) == out.view(np.uint32)) | (np.isnan(mine) & np.isnan(out))), (r, t, mine, out)


def _owned_pointers(n):
    """n pointers into the middle of zeroed 64 KB buffers the test owns (device memory where there is a GPU).  The refusals below happen
    before any CUDA call; should an argument check regress, the launch reads and writes only these buffers (at most a few KB either side of
    the pointer, with every count and index zero), instead of unmapped addresses."""
    import torch
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    bufs = [torch.zeros(1 << 16, dtype=torch.uint8, device=dev) for _ in range(n)]
    return bufs, [ctypes.c_void_p(b.data_ptr() + (1 << 15)) for b in bufs]


@pytest.mark.parametrize("n", [0, -1, 33])
def test_reduce_pose_records_refuses_bad_counts(n):
    lib = hc.load_library()
    bufs, p = _owned_pointers(2)
    assert lib.hcb200_reduce_pose_records(None, n, p[0], p[1]) == INVALID_VALUE


def test_make_pose_record_refuses_a_negative_offset():
    lib = hc.load_library()
    bufs, p = _owned_pointers(3)
    for off in (-1, -312, -(1 << 62)):
        assert lib.hcb200_make_pose_record(None, p[0], p[1], None, off, 0, p[2]) == INVALID_VALUE


@pytest.mark.parametrize("case", ["no_edgels", "negative_edgels", "negative_paths", "tracks", "converged", "edgels", "K", "support", "best",
                                  "workspace"])
def test_score_tracks_refuses_bad_arguments(case):
    """A NULL argument is refused with n_paths = 0, so that only the workspace and the record would be touched if the check regressed."""
    lib = hc.load_library()
    names = ["tracks", "converged", "edgels", "K", "support", "best", "workspace"]
    bufs, owned = _owned_pointers(len(names))
    p = [None if n == case else owned[i] for i, n in enumerate(names)]
    n_paths = {"negative_paths": -1, "no_edgels": 8, "negative_edgels": 8}.get(case, 0)
    n_edgels = {"no_edgels": 0, "negative_edgels": -3}.get(case, 10)
    assert lib.hcb200_score_tracks(None, n_paths, p[0], p[1], n_edgels, p[2], p[3], p[4], p[5], p[6]) == INVALID_VALUE


@pytest.mark.parametrize("n_edgels", [0, -1])
def test_build_target_params_refuses_no_edgels(n_edgels):
    lib = hc.load_library()
    bufs, p = _owned_pointers(6)
    assert lib.hcb200_build_target_params(None, 4, p[0], n_edgels, *p[1:]) == INVALID_VALUE


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers

def _torch():
    import torch
    return torch


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(_torch().cuda.current_stream().cuda_stream)


def _c2f(z):
    z = np.asarray(z, np.complex64)
    return np.ascontiguousarray(np.stack([z.real, z.imag], -1).astype(F32))


def _dev(a):
    return _torch().from_numpy(np.ascontiguousarray(a)).cuda()


def _grid():
    """Grid of hcb200_score_tracks / hcb200_count_solutions on the current device, as the launchers compute it: 8 CTAs of 8 warps per SM."""
    torch = _torch()
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count * 8


# variants of an end point that stay pose candidates; the others ("im_above_tol", "depth_-subnormal", "depth_nan", "not_converged") are
# rejected.  The first five keep the end point's pose, so they tie with its plain path.
CANDIDATE_VARIANTS = ("plain", "im_at_tol", "depth_+0", "depth_-0", "im_in_translation", "t21_nan", "t31_zero")


def variant(x0, kind, j):
    """End point x0 changed at one edge of the candidate gate; j picks the lane."""
    x = x0.copy()
    if kind == "im_at_tol":
        x.imag[24 + j % 6] = IM_TOL * (1 if j % 2 else -1)
    elif kind == "im_above_tol":
        x.imag[24 + j % 6] = IM_ABOVE * (1 if j % 2 else -1)
    elif kind == "depth_+0":
        x.real[j % 8] = F32(0.0)
    elif kind == "depth_-0":
        x.real[j % 8] = F32(-0.0)
    elif kind == "depth_-subnormal":
        x.real[j % 8] = -SUBNORMAL
    elif kind == "depth_nan":
        x.real[j % 8] = np.nan
    elif kind == "im_in_translation":             # the gate reads the Cayley lanes only
        x.imag[18 + j % 6] = F32(0.5)
    elif kind == "t21_nan":
        x.real[18 + j % 3] = np.nan
    elif kind == "t31_zero":
        x.real[21:24] = 0
    return x


def path_layout(n_paths):
    """(pose, kind, j) of every path.  Every group of eight paths (one CTA's share) holds candidates; every third group holds candidates only;
    path 0 is not pose 0, so the lowest-id rule among the many pose-0 ties is not the trivial one, and the first pose-0 path sits at the
    |Im| = float32(1e-5) edge of the gate."""
    mixed = [(1, "plain"), (0, "im_at_tol"), (0, "im_above_tol"), (0, "depth_-0"), (0, "not_converged"), (0, "t21_nan"), (2, "plain"),
             (0, "depth_-subnormal"), (2, "depth_+0"), (0, "depth_nan"), (1, "t31_zero"), (1, "im_at_tol"), (0, "plain"),
             (2, "im_in_translation"), (0, "depth_+0")]
    full = [(0, "plain"), (1, "plain"), (2, "plain"), (0, "im_at_tol"), (0, "depth_-0"), (0, "im_in_translation"), (1, "depth_+0"),
            (2, "t21_nan")]
    out = []
    for p in range(n_paths):
        g, w = divmod(p, 8)
        pose, kind = full[(w + g) % 8] if g % 3 == 2 else mixed[p % len(mixed)]
        out.append((pose, kind, p % 6))
    return out


def expected_scores(sc, layout, n_edgels, cache):
    """Host supports of every path ([-1, -1] for non-candidates) and the plain-rule best record."""
    lib = _host()
    sup = np.empty((len(layout), 2), np.int64)
    for p, (pose, kind, j) in enumerate(layout):
        key = (pose, kind, j, n_edgels)
        if key not in cache:
            x = variant(sc["poses"][pose], kind, j)
            ok, n21, n31 = host_score(x, sc["loc"][:n_edgels], sc["K"], lib)
            ok = ok and kind != "not_converged"
            assert ok == (kind in CANDIDATE_VARIANTS), (kind, j)
            assert (kind != "t21_nan" or n21 == 0) and (kind != "t31_zero" or n31 == 0)      # a NaN translation counts no inlier
            cache[key] = (n21, n31) if ok else (-1, -1)
        sup[p] = cache[key]
    rec = np.zeros(16, np.int64)
    cand = np.nonzero(sup[:, 0] >= 0)[0]
    if len(cand):
        best = max(cand, key=lambda q: (min(sup[q]), -q))         # largest min(support21, support31), lowest path id among equals
        rec[:7] = [1, best, sup[best, 0], sup[best, 1], len(cand), sup[cand, 0].max(), sup[cand, 1].max()]
    else:
        rec[1] = -1
    return sup, rec


class Scorer:
    """hcb200_score_tracks on buffers this test owns: d_support has guard words after 2 * n_paths; d_best starts as garbage."""

    def __init__(self, sc, n_edgels):
        torch = _torch()
        self.lib = hc.load_library()
        self.d_loc = _dev(sc["loc"][:n_edgels])
        self.d_K = _dev(sc["K"])
        self.n_edgels = n_edgels
        self.d_ws = torch.zeros(256, dtype=torch.uint8, device="cuda")
        self.d_best = torch.full((16,), 7, dtype=torch.int32, device="cuda")

    def run(self, tracks, conv, guard=64):
        torch = _torch()
        n = len(conv)
        d_tr = _dev(_c2f(tracks) if n else np.zeros((1, 31, 2), F32))
        d_cv = _dev(conv if n else np.zeros(1, np.uint8))
        d_sup = torch.full((2 * n + guard,), SENTINEL, dtype=torch.int32, device="cuda")
        rc = self.lib.hcb200_score_tracks(_stream(), n, _ptr(d_tr), _ptr(d_cv), self.n_edgels, _ptr(self.d_loc), _ptr(self.d_K), _ptr(d_sup),
                                          _ptr(self.d_best), _ptr(self.d_ws))
        assert rc == 0
        torch.cuda.synchronize()
        s = d_sup.cpu().numpy()
        assert (s[2 * n:] == SENTINEL).all(), "hcb200_score_tracks wrote past 2 * n_paths"
        return s[:2 * n].reshape(n, 2), self.d_best.cpu().numpy()


def _paths(sc, layout):
    xs = np.stack([variant(sc["poses"][pose], kind, j) for pose, kind, j in layout]) if layout else np.zeros((0, 31), np.complex64)
    conv = np.array([kind != "not_converged" for _, kind, _ in layout], np.uint8)
    return xs, conv


# ---------------------------------------------------------------------------------------------------------------------
# GPU: hcb200_score_tracks

@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["1", "7", "8", "9", "3_sweeps"])
def test_score_tracks_against_host_and_float64(scene, shape):
    """Supports equal hcb200_host_score_track on every path and lie in the float64 stability interval; the candidate gate follows the plain rule
    at its edges (|Im| = float32(1e-5) passes and the next float32 fails, depths +0 and -0 pass, a negative subnormal and NaN fail, NaN or zero
    translations give the host's NaN counts, an unconverged path gives -1, -1); the record is the plain arg-max with the lowest id among ties,
    n_passed, the per-pair maxima in reserved[0..1] and zeros after.  3_sweeps has 8 * grid * 3 + 5 paths, so the grid-stride loop reuses its
    shared slots with candidates present in every sweep."""
    n_paths = 8 * _grid() * 3 + 5 if shape == "3_sweeps" else int(shape)
    layout = path_layout(n_paths)
    xs, conv = _paths(scene, layout)
    cache = {}
    for n_edgels in (1, 31, 255, 257, N_EDGELS):
        sup, rec = Scorer(scene, n_edgels).run(xs, conv)
        exp_sup, exp_rec = expected_scores(scene, layout, n_edgels, cache)
        bad = np.nonzero((sup != exp_sup).any(1))[0]
        assert len(bad) == 0, (n_edgels, [(int(p), layout[p], sup[p].tolist(), exp_sup[p].tolist()) for p in bad[:5]])
        assert rec.tolist() == exp_rec.tolist(), (n_edgels, rec.tolist(), exp_rec.tolist())
        for pose in (0, 1, 2):
            (lo21, hi21), (lo31, hi31) = support_bounds(scene, pose, n_edgels)
            sp = sup[[p for p, (q, kind, _) in enumerate(layout) if q == pose and kind in ("plain", "im_at_tol", "depth_+0", "depth_-0")]]
            assert ((lo21 <= sp[:, 0]) & (sp[:, 0] <= hi21) & (lo31 <= sp[:, 1]) & (sp[:, 1] <= hi31)).all(), (pose, n_edgels)
    if shape == "3_sweeps":
        groups = (sup[:8 * (n_paths // 8), 0] >= 0).reshape(-1, 8)
        assert groups.all(1).sum() >= _grid() and groups.any(1).all()
        best = rec[1]
        ties = [p for p in range(n_paths) if sup[p].min() == sup[best].min()]
        assert len(ties) >= 2 and best == min(ties) and best > 0
        assert rec[5] != rec[6]                                            # the per-pair maxima differ, so a swap is visible


@pytest.mark.gpu
def test_score_tracks_without_candidates_and_back_to_back_launches(scene):
    """No candidate, or no path at all: found 0, path -1, every other word 0.  A launch does not inherit the previous launch's best key,
    maxima or candidate count (same workspace and record buffers)."""
    s = Scorer(scene, N_EDGELS)
    lay = [(0, k, j) for j, k in enumerate(["not_converged", "im_above_tol", "depth_nan", "depth_-subnormal"] * 5)]
    xs, conv = _paths(scene, lay)
    sup, rec = s.run(xs, conv)
    assert (sup == -1).all() and rec.tolist() == [0, -1] + [0] * 14
    s.d_best.fill_(7)
    sup, rec = s.run(xs[:0], conv[:0])
    assert sup.size == 0 and rec.tolist() == [0, -1] + [0] * 14
    # a rich launch, then one whose best is worse: the second record is the second launch's alone
    lay1 = path_layout(300)
    xs1, conv1 = _paths(scene, lay1)
    _, rec1 = s.run(xs1, conv1)
    lay2 = [(2, "plain", j) for j in range(20)] + [(0, "not_converged", 0)]
    xs2, conv2 = _paths(scene, lay2)
    sup2, rec2 = s.run(xs2, conv2)
    exp_sup2, exp_rec2 = expected_scores(scene, lay2, N_EDGELS, {})
    assert np.array_equal(sup2, exp_sup2) and rec2.tolist() == exp_rec2.tolist()
    assert rec1[4] > rec2[4] and min(rec1[2:4]) > min(rec2[2:4]) and rec2[1] == 0


# ---------------------------------------------------------------------------------------------------------------------
# GPU: hcb200_make_pose_record

def _make_record(lib, d_tracks, best, found_byte, offset, rank):
    torch = _torch()
    d_best = _dev(np.asarray(best, np.int32))
    d_out = torch.full((32,), float("nan"), dtype=torch.float32, device="cuda")
    d_found = None if found_byte is None else _dev(np.array([found_byte], np.uint8))
    rc = lib.hcb200_make_pose_record(_stream(), _ptr(d_tracks), _ptr(d_best), None if d_found is None else _ptr(d_found), offset, rank,
                                     _ptr(d_out))
    assert rc == 0
    torch.cuda.synchronize()
    return d_out.cpu().numpy()


@pytest.mark.gpu
def test_make_pose_record_against_float32_and_float64(scene):
    """The pose is bit-identical to the float32 restatement of host/mvg.hpp and within a few ulp of float64 Cayley -> column-normalised R and
    unit t; R is orthonormal to 1e-6.  path_id = local id + path_offset exactly up to 312 * (2^31 - 1); abort_flag is 0 without a flag byte and
    1 with a set one; a best record with found == 0 or path_id == -1 gives path -1 and a zero pose."""
    lib = hc.load_library()
    rng = np.random.default_rng(11)
    xs = [end_point(rng.uniform(-s, s, 3).astype(F32), rng.uniform(-3, 3, 3).astype(F32), rng.uniform(-s, s, 3).astype(F32),
                    rng.uniform(-3, 3, 3).astype(F32), rng) for s in (1e-3, 0.1, 0.5, 1.0, 2.0) for _ in range(64)]
    xs = np.stack(list(scene["poses"]) + xs)
    d_tracks = _dev(_c2f(xs))
    offsets = [0, 312 * 977, 312 * (2 ** 31 - 1)]
    for path in range(xs.shape[0]):
        off = offsets[path % 3]
        best = [1, path, 100 + path, 200 + path, 7 + path] + [0] * 11
        found = [None, 1, 0][path % 3]
        rec = hc.decode_pose_record(_make_record(lib, d_tracks, best, found, off, path % 8))
        assert rec["path_id"] == path + off and rec["found"] == 1 and rec["rank"] == path % 8
        assert (rec["inliers21"], rec["inliers31"], rec["n_candidates"]) == (100 + path, 200 + path, 7 + path)
        assert rec["abort_flag"] == (1 if found == 1 else 0)
        mine = np.concatenate([rec["R21"].reshape(-1), rec["t21"], rec["R31"].reshape(-1), rec["t31"]])
        assert np.array_equal(mine.view(np.uint32), pose32(xs[path]).view(np.uint32)), path
        ref = pose64(xs[path])
        assert np.abs(mine - ref).max() <= 8 * 2.0 ** -24, (path, np.abs(mine - ref).max())
        for R in (rec["R21"].astype(F64), rec["R31"].astype(F64)):
            assert np.abs(R.T @ R - np.eye(3)).max() < 1e-6 and abs(np.linalg.det(R) - 1) < 1e-6
        for t in (rec["t21"].astype(F64), rec["t31"].astype(F64)):
            assert abs(np.linalg.norm(t) - 1) < 1e-6
    for best in ([0, 3, 10, 10, 4] + [0] * 11, [1, -1, 10, 10, 4] + [0] * 11, [0, -1, 0, 0, 0] + [0] * 11):
        raw = _make_record(lib, d_tracks, best, 1, 312 * 5, 2)
        rec = hc.decode_pose_record(raw)
        assert rec["path_id"] == -1 and (raw[8:] == 0).all() and not np.signbit(raw[8:]).any()
        assert (rec["found"], rec["inliers21"], rec["inliers31"], rec["n_candidates"], rec["abort_flag"], rec["rank"]) == \
            (best[0], best[2], best[3], best[4], 1, 2)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: hcb200_reduce_pose_records

MAX_PATH_ID = 312 * (2 ** 31 - 1) + 311


def plain_reduce(recs):
    """Python arg-max over 128-byte records (float32 [n, 32]): the 128 bytes hcb200_reduce_pose_records must write."""
    dec = [hc.decode_pose_record(r) for r in recs]
    live = [i for i, r in enumerate(dec) if r["found"] and r["path_id"] >= 0]
    n_cand = int(np.array(sum(r["n_candidates"] for r in dec)).astype(np.int32))
    flag = 0
    for r in dec:
        flag |= r["abort_flag"]
    if live:
        w = max(live, key=lambda i: (min(dec[i]["inliers21"], dec[i]["inliers31"]), -dec[i]["path_id"]))
        out = recs[w].copy()
        out.view(np.int32)[3], out.view(np.int32)[4] = n_cand, flag
        return out
    return hc.encode_pose_record(0, 0, 0, n_cand, flag, -1, -1)


def mirror_reduce(recs):
    """hc.reduce_pose_records_host, encoded back to 128 bytes."""
    r = hc.reduce_pose_records_host(recs)
    pose = np.concatenate([r["R21"].reshape(-1), r["t21"], r["R31"].reshape(-1), r["t31"]])
    return hc.encode_pose_record(r["found"], r["inliers21"], r["inliers31"], r["n_candidates"], r["abort_flag"], r["rank"], r["path_id"], pose)


def random_records(rng, n, kind):
    recs = []
    if kind == "huge":                                             # unique global path ids up to the largest, the extremes included
        ids = np.concatenate([[MAX_PATH_ID, 0], MAX_PATH_ID - 1 - rng.choice(MAX_PATH_ID - 2, n, replace=False)])[rng.permutation(n + 2)[:n]]
    else:
        ids = rng.permutation(np.arange(0, 20 * n, dtype=np.int64) * 312 + rng.integers(0, 312, 20 * n))[:n]
    for i in range(n):
        pose = rng.standard_normal(24).astype(F32)
        found = int(rng.random() < 0.7)
        pid = int(ids[i])
        if rng.random() < 0.15:
            found, pid = 1, -1                                     # found with path_id == -1 never wins
        if kind == "ties":
            lo = int(rng.choice([3, 5]))
            a, b = (lo, lo + int(rng.integers(0, 4))) if rng.random() < 0.5 else (lo + int(rng.integers(0, 4)), lo)
        elif kind == "zeros":
            a, b = int(rng.integers(0, 2)), 0
        else:
            a, b = (int(v) for v in rng.integers(0, 65536, 2)) if kind == "huge" else (int(v) for v in rng.integers(0, 40, 2))
        recs.append(hc.encode_pose_record(found, a, b, int(rng.integers(0, 1000)), int(rng.random() < 0.2), i, pid, pose))
    return np.stack(recs)


@pytest.mark.gpu
def test_reduce_pose_records_against_plain_argmax_and_host_mirror():
    """n = 1..32 seeded random records (found and not found, found with path -1, min-support ties across lanes with different path ids, support 0
    against not found, path ids up to 312 * (2^31 - 1) + 311 and inlier counts up to 65 535): the 128 bytes written equal a plain Python arg-max
    and hc.reduce_pose_records_host byte for byte — the winner's record unchanged but for the summed n_candidates and the OR-ed abort_flag; with
    no winner, found 0, rank -1, path -1 and a zero pose."""
    torch = _torch()
    lib = hc.load_library()
    rng = np.random.default_rng(5)
    cases = []
    for n in range(1, 33):
        for kind in ("mixed", "ties", "zeros", "huge"):
            cases.append(random_records(rng, n, kind))
    # hand-made edges: the winner on the highest lane by the lowest path id among equal min-supports; support 0 beats not found; nobody found
    tie = np.stack([hc.encode_pose_record(1, 9, 50, 1, 0, r, 1000 - r, np.full(24, r)) for r in range(32)])
    tie[31].view(np.int64)[3] = 5
    cases.append(tie)
    cases.append(np.stack([hc.encode_pose_record(0, 65535, 65535, 2, 0, 0, 17), hc.encode_pose_record(1, 0, 65535, 3, 1, 1, MAX_PATH_ID,
                                                                                                           np.arange(24))]))
    cases.append(np.stack([hc.encode_pose_record(0, 9, 9, 4, 0, r, r, np.ones(24)) for r in range(5)]))
    cases.append(np.stack([hc.encode_pose_record(1, 65535, 65534, 0, 0, 0, MAX_PATH_ID, np.ones(24)),
                           hc.encode_pose_record(1, 65534, 65535, 0, 0, 1, 0, np.ones(24)),
                           hc.encode_pose_record(1, 65535, 65535, 0, 0, 2, MAX_PATH_ID - 1, np.ones(24))]))
    d_in = torch.from_numpy(np.zeros((len(cases), 32, 32), F32)).cuda()
    for c, recs in enumerate(cases):
        d_in[c, :len(recs)] = torch.from_numpy(recs)
    d_out = torch.full((len(cases), 32), float("nan"), dtype=torch.float32, device="cuda")
    for c, recs in enumerate(cases):
        assert lib.hcb200_reduce_pose_records(_stream(), len(recs), _ptr(d_in[c]), _ptr(d_out[c])) == 0
    torch.cuda.synchronize()
    out = d_out.cpu().numpy()
    for c, recs in enumerate(cases):
        want = plain_reduce(recs)
        assert np.array_equal(out[c].view(np.uint8), want.view(np.uint8)), (c, hc.decode_pose_record(out[c]), hc.decode_pose_record(want))
        assert np.array_equal(out[c].view(np.uint8), mirror_reduce(recs).view(np.uint8)), c
    assert hc.decode_pose_record(out[-4])["rank"] == 31 and hc.decode_pose_record(out[-3])["path_id"] == MAX_PATH_ID
    assert hc.decode_pose_record(out[-2])["rank"] == -1 and hc.decode_pose_record(out[-1])["rank"] == 2
    winners = {hc.decode_pose_record(out[c])["rank"] for c in range(len(cases))}
    assert len(winners) >= 16                                      # winners on many different lanes


# ---------------------------------------------------------------------------------------------------------------------
# GPU: hcb200_count_solutions

def count_solutions64(tracks, conv, inf, n_hyp):
    """Evaluations.cpp:145-167 in float64: per hypothesis converged, infinity, and converged with all 30 |imag| <= 1e-4."""
    im = np.abs(tracks[:, :30].imag.astype(F64))
    real = conv.astype(bool) & np.all(im <= 1e-4, axis=1)
    per = lambda a: a.reshape(n_hyp, T).sum(1)
    return np.stack([per(conv.astype(bool)), per(inf.astype(bool)), per(real)], 1)


@pytest.mark.gpu
def test_count_solutions_at_the_tolerance_edges():
    """|Im| = float32(1e-4) counts as real, the next float32 does not, NaN does not; the pad slot (lane 30) is never read; a path both
    converged and infinity counts in both columns; 100 hypotheses make several grid sweeps; n_hyp = 0 succeeds and writes nothing."""
    torch = _torch()
    lib = hc.load_library()
    rng = np.random.default_rng(9)
    H = 100
    P = H * T
    assert P > 3 * 8 * _grid()
    tr = (rng.uniform(-1, 1, (P, 31)) + 1j * rng.uniform(-5e-5, 5e-5, (P, 31))).astype(np.complex64)
    tol, above = F32(1e-4), np.nextafter(F32(1e-4), F32(1))
    kind = rng.integers(0, 6, P)
    lane = rng.integers(0, 30, P)
    rows = np.arange(P)
    tr.imag[rows[kind == 1], lane[kind == 1]] = tol
    tr.imag[rows[kind == 2], lane[kind == 2]] = -tol
    tr.imag[rows[kind == 3], lane[kind == 3]] = above
    tr.imag[rows[kind == 4], lane[kind == 4]] = np.nan
    tr[:, 30] = (rng.uniform(-1e6, 1e6, P) + 1j * rng.choice([1.0, np.nan, 3e-4], P)).astype(np.complex64)   # pad slot: garbage
    conv = (rng.random(P) < 0.6).astype(np.uint8)
    inf = (rng.random(P) < 0.3).astype(np.uint8)
    want = count_solutions64(tr, conv, inf, H)
    assert np.array_equal(want, hc.count_solutions(tr, conv, inf, H))
    assert (conv & inf).sum() > 1000 and want[:, 2].sum() > 1000 and (want[:, 0] > want[:, 2]).all()
    d_tr, d_cv, d_inf = _dev(_c2f(tr)), _dev(conv), _dev(inf)
    d_counts = torch.full((3 * H + 32,), SENTINEL, dtype=torch.int32, device="cuda")
    assert lib.hcb200_count_solutions(_stream(), H, _ptr(d_tr), _ptr(d_cv), _ptr(d_inf), _ptr(d_counts)) == 0
    torch.cuda.synchronize()
    got = d_counts.cpu().numpy()
    assert np.array_equal(got[:3 * H].reshape(H, 3), want) and (got[3 * H:] == SENTINEL).all()
    # one hypothesis whose every converged path sits exactly at the tolerance in one lane, or just above it
    for val, real in ((tol, True), (above, False)):
        t1 = np.zeros((T, 31), np.complex64)
        t1.imag[np.arange(T), np.arange(T) % 30] = val
        t1[:, 30] = 5 + 1j
        d_t1, d_c1, d_i1 = _dev(_c2f(t1)), _dev(np.ones(T, np.uint8)), _dev((np.arange(T) % 2).astype(np.uint8))
        d_counts.fill_(SENTINEL)
        assert lib.hcb200_count_solutions(_stream(), 1, _ptr(d_t1), _ptr(d_c1), _ptr(d_i1), _ptr(d_counts)) == 0
        torch.cuda.synchronize()
        assert d_counts[:3].cpu().tolist() == [T, T // 2, T if real else 0]
    d_counts.fill_(SENTINEL)
    assert lib.hcb200_count_solutions(_stream(), 0, _ptr(d_tr), _ptr(d_cv), _ptr(d_inf), _ptr(d_counts)) == 0
    torch.cuda.synchronize()
    assert (d_counts.cpu().numpy() == SENTINEL).all()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: hcb200_build_target_params

@pytest.mark.gpu
@pytest.mark.parametrize("n_hyp", [0, 1, 7, 1000])
def test_build_target_params_is_bit_identical_to_the_host_and_clamps_picks(problem, ransac0, n_hyp):
    """Targets and target - start are bit-identical to hc.target_params_from_picks (constants at 30-33 included); picks at 0 and n_edgels - 1
    are read, picks outside (-5, n_edgels + 3) are clamped to them.  The edgel arrays sit between NaN sentinel rows of a larger allocation,
    so a read outside them shows up as NaN and never leaves memory the test owns; nothing is written past n_hyp * 34."""
    torch = _torch()
    lib = hc.load_library()
    loc, tan = np.asarray(ransac0["locations"], F32), np.asarray(ransac0["tangents"], F32)
    E, pad = loc.shape[0], 8
    rng = np.random.default_rng(n_hyp)
    picked = rng.integers(0, E, (max(n_hyp, 1), 3)).astype(np.int32)[:n_hyp]
    edge = np.array([0, E - 1, -5, E + 3], np.int32)
    if n_hyp:
        flat = picked.reshape(-1)
        flat[: min(flat.size, 12)] = np.resize(np.concatenate([edge, edge[::-1], edge[[2, 0, 3, 1]]]), min(flat.size, 12))
    nan_rows = np.full((pad, 6), np.nan, F32)
    d_loc = _dev(np.concatenate([nan_rows, loc, nan_rows]))
    d_tan = _dev(np.concatenate([nan_rows, tan, nan_rows]))
    d_sp = _dev(_c2f(hc.padded_start_params(problem["start_params"])))
    d_picked = _dev(picked if n_hyp else np.zeros((1, 3), np.int32))
    guard = 16
    d_tgt = torch.full((max(n_hyp, 1) * 68 + guard,), float("inf"), dtype=torch.float32, device="cuda")
    d_dif = torch.full_like(d_tgt, float("inf"))
    rc = lib.hcb200_build_target_params(_stream(), n_hyp, _ptr(d_picked), E, _ptr(d_loc[pad:]), _ptr(d_tan[pad:]), _ptr(d_sp), _ptr(d_tgt),
                                        _ptr(d_dif))
    assert rc == 0
    torch.cuda.synchronize()
    tgt, dif = d_tgt.cpu().numpy(), d_dif.cpu().numpy()
    assert np.isposinf(tgt[n_hyp * 68:]).all() and np.isposinf(dif[n_hyp * 68:]).all()
    if n_hyp == 0:
        return
    want_t, want_d = hc.target_params_from_picks(np.clip(picked, 0, E - 1), loc, tan, problem["start_params"])
    assert np.array_equal(tgt[:n_hyp * 68].view(np.uint32), _c2f(want_t).reshape(-1).view(np.uint32))
    assert np.array_equal(dif[:n_hyp * 68].view(np.uint32), _c2f(want_d).reshape(-1).view(np.uint32))
    t = tgt[:n_hyp * 68].reshape(n_hyp, 34, 2)
    assert (t[:, 30:, 0] == [1, 0.5, 1, 1]).all() and (t[:, :, 1] == 0).all()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the early-abort pass threshold

@pytest.fixture(scope="module")
def abort_sets(ransac0, oracle):
    return make_abort_sets(ransac0, oracle)


def make_abort_sets(ransac0, oracle):
    """Edgel sets of m ground-truth inliers of dataset 0 plus n - m outliers (view-2 and view-3 points moved by 20-40 px, each checked to be
    an outlier of path 104 for both pairs), and the end points of a no-abort run of hypothesis 0."""
    loc, K = np.asarray(ransac0["locations"], F32), np.asarray(ransac0["K"], F32)
    target, diff, _ = oracle.prepare_target_params(0, 1, loc, ransac0["tangents"])
    tr, cv, _, _ = oracle.track(target, diff, prune=True)
    x104 = tr[104]
    assert oracle.score(x104, loc, K)[:3] == (True, loc.shape[0], loc.shape[0])
    rng = np.random.default_rng(2)
    pool = loc[rng.permutation(loc.shape[0])[:900]].copy()
    th = rng.uniform(0, 2 * np.pi, (900, 2))
    s = rng.uniform(20, 40, (900, 2))
    for v in (0, 1):
        pool[:, 2 + 2 * v] += (s[:, v] * np.cos(th[:, v]) / K[0, 0]).astype(F32)
        pool[:, 3 + 2 * v] += (s[:, v] * np.sin(th[:, v]) / K[1, 1]).astype(F32)
    outliers = np.stack([e for e in pool if oracle.score(x104, e[None, :], K)[1:3] == (0, 0)])
    assert outliers.shape[0] >= 501
    inliers = loc[rng.permutation(loc.shape[0])]
    sets = {}
    for n in (10, 5000):
        for m in (n * 9 // 10 - 1, n * 9 // 10, n * 9 // 10 + 1):
            sets[(n, m)] = np.ascontiguousarray(rng.permutation(np.concatenate([inliers[:m], outliers[:n - m]])))
    return {"target": target, "diff": diff, "tracks": tr, "conv": cv, "sets": sets, "K": K}


@pytest.mark.gpu
def test_early_abort_pass_threshold_is_the_references(problem, oracle, abort_sets):
    """A path passes the early-abort test when (double)(float(n21) / float(n_edgels)) >= 0.90 and the same for n31: the reference's
    PASS_RANSAC_INLIER_SUPPORT_RATIO test (TrunRANSAC.cu:241-242), kept as it is.  The float quotient of exactly 90 % is 0.9f < 0.9, so
    exactly 90 % does NOT pass; one inlier more does.  Hypothesis 0 of dataset 0 (its target parameters from the original edgels) is tracked
    with early abort against edgel sets of m inliers of the ground-truth path 104 and n - m outliers, for m/n = 90 % - 1, 90 %, 90 % + 1 at
    n = 10 and 5000.  On each set path 104 is the only converged end point of the no-abort run that the rule can pass (asserted first), so the
    flag and the best record follow the rule and the oracle's score for path 104 alone."""
    K = abort_sets["K"]
    tr, cv = abort_sets["tracks"], abort_sets["conv"]
    trk = hc.Tracker(problem=problem)
    trk.upload_params(abort_sets["target"], abort_sets["diff"])
    for (n, m), edgels in sorted(abort_sets["sets"].items()):
        passes = float(F32(m) / F32(n)) >= 0.90
        assert passes == (m > n * 9 // 10)
        ok, n21, n31, gate = oracle.score(tr[104], edgels, K)
        assert (ok, n21, n31, gate) == (passes, m, m, True), (n, m)
        passing = [int(b) for b in np.nonzero(cv)[0] if oracle.score(tr[b], edgels, K)[0]]
        assert passing == ([104] if passes else []), (n, m, passing)
        trk.set_edgels(edgels, K)
        trk.track_abort(1, prune=True)
        _torch().cuda.synchronize()
        found = int(trk.d_found.cpu()[0])
        best = trk.d_best.cpu().numpy()
        assert found == int(passes), (n, m)
        want = [1, 104, m, m, 1] if passes else [0, -1, 0, 0, 0]
        assert best[:5].tolist() == want and (best[5:] == 0).all(), (n, m, best.tolist())
