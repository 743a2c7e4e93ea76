"""ctypes binding of the C ABI (`include/hcb200.h`) plus the thin host logic the benchmarks and tests need.

PyTorch is used for device memory, streams and `torch.distributed` only; every kernel launched here lives in
`lib/libhcb200.so` (built by `make` / `__graft_entry__.build()`).  There is NO CPU fallback: if the library is missing
or a launch fails this module raises.
"""
import ctypes
import os

import numpy as np

from . import fixtures

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libhcb200.so")

NUM_VARS = 30
NUM_PARAMS = 33
NUM_TRACKS = 312
FLAG_PRUNE_PATHS = 1
FLAG_SPLIT_LONG_PATHS = 2      # needs a workspace of hcb200_workspace_bytes_for(n_hyp) bytes
SPLIT_MAX_HYPOTHESES = 2048    # HCB200_SPLIT_MAX_HYPOTHESES: larger rounds never use the split kernel, so they are not given its workspace

_lib = None

# every symbol include/hcb200.h declares
ABI_SYMBOLS = ("hcb200_workspace_bytes", "hcb200_abi_version", "hcb200_track", "hcb200_track_abort",
               "hcb200_build_target_params", "hcb200_score_tracks", "hcb200_refine_tracks", "hcb200_kernel_info", "hcb200_ffma_probe",
               "hcb200_error_string", "hcb200_make_pose_record", "hcb200_reduce_pose_records", "hcb200_count_solutions", "hcb200_problem_info",
               "hcb200_workspace_bytes_for", "hcb200_track_abort_peers", "hcb200_enable_peer_access", "hcb200_batch_workspace_bytes",
               "hcb200_track_abort_batched")
BATCH_MAX_PROBLEMS = 4095      # HCB200_BATCH_MAX_PROBLEMS


class HCB200Error(RuntimeError):
    pass


def load_library(path=None):
    """Load libhcb200.so (once).  Raises HCB200Error when it has not been built — never falls back to the CPU."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise HCB200Error("CUDA extension %s is missing: run `make` (or __graft_entry__.build()) first" % path)
    lib = ctypes.CDLL(path)
    vp, i32, u32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint
    lib.hcb200_workspace_bytes.restype = ctypes.c_size_t
    lib.hcb200_workspace_bytes.argtypes = []
    lib.hcb200_workspace_bytes_for.restype = ctypes.c_size_t
    lib.hcb200_workspace_bytes_for.argtypes = [i32]
    lib.hcb200_abi_version.restype = i32
    lib.hcb200_error_string.restype = ctypes.c_char_p
    lib.hcb200_error_string.argtypes = [i32]
    lib.hcb200_track.restype = i32
    lib.hcb200_track.argtypes = [vp, i32, i32, i32, i32, u32] + [vp] * 9
    lib.hcb200_track_abort.restype = i32
    lib.hcb200_track_abort.argtypes = [vp, i32, i32, i32, i32, i32, u32] + [vp] * 14
    lib.hcb200_track_abort_peers.restype = i32
    lib.hcb200_track_abort_peers.argtypes = [vp, i32, i32, i32, i32, i32, u32] + [vp] * 14 + [ctypes.POINTER(vp), i32]
    lib.hcb200_batch_workspace_bytes.restype = ctypes.c_size_t
    lib.hcb200_batch_workspace_bytes.argtypes = [i32]
    lib.hcb200_track_abort_batched.restype = i32
    lib.hcb200_track_abort_batched.argtypes = [vp, i32, i32, vp, i32, i32, i32, u32] + [vp] * 14
    lib.hcb200_enable_peer_access.restype = i32
    lib.hcb200_enable_peer_access.argtypes = [i32, i32]
    lib.hcb200_build_target_params.restype = i32
    lib.hcb200_build_target_params.argtypes = [vp, i32, vp, i32, vp, vp, vp, vp, vp]
    lib.hcb200_kernel_info.restype = i32
    lib.hcb200_kernel_info.argtypes = [i32] + [ctypes.POINTER(i32)] * 5
    lib.hcb200_score_tracks.restype = i32
    lib.hcb200_score_tracks.argtypes = [vp, i32, vp, vp, i32, vp, vp, vp, vp, vp]
    lib.hcb200_refine_tracks.restype = i32
    lib.hcb200_refine_tracks.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp]
    lib.hcb200_count_solutions.restype = i32
    lib.hcb200_count_solutions.argtypes = [vp, i32, vp, vp, vp, vp]
    lib.hcb200_make_pose_record.restype = i32
    lib.hcb200_make_pose_record.argtypes = [vp, vp, vp, vp, ctypes.c_longlong, i32, vp]
    lib.hcb200_reduce_pose_records.restype = i32
    lib.hcb200_reduce_pose_records.argtypes = [vp, i32, vp, vp]
    lib.hcb200_ffma_probe.restype = i32
    lib.hcb200_ffma_probe.argtypes = [vp, i32, vp, ctypes.POINTER(ctypes.c_double)]
    _lib = lib
    return lib


def _check(code, what):
    if code != 0:
        msg = load_library().hcb200_error_string(code)
        raise HCB200Error("%s failed: cudaError %d (%s)" % (what, code, msg.decode() if msg else "?"))


# ------------------------------------------------------------------------------------------------------------------
# host logic mirrored from the reference (no device work)

def shard_sizes(n_hyp, n_gpus):
    """GPU_HC_Solver.cpp:85-88: sub_RANSAC_iters[g] = H / N + (g < H % N)."""
    return [n_hyp // n_gpus + (1 if g < n_hyp % n_gpus else 0) for g in range(n_gpus)]


def shard_offsets(n_hyp, n_gpus):
    sizes = shard_sizes(n_hyp, n_gpus)
    offs = [0]
    for s in sizes:
        offs.append(offs[-1] + s)
    return offs


_libc = None


def sample_hypotheses(seed, n_hyp, n_edgels):
    """GPU_HC_Solver.cpp:263-271: srand(seed); three rand() % E per attempt, accept when e0 != e1 and e1 != e2
    (the reference never checks e0 != e2, SURVEY.md App. E-1).  Uses the C library's rand() stream."""
    global _libc
    if _libc is None:
        _libc = ctypes.CDLL(None)
        _libc.rand.restype = ctypes.c_int
        _libc.srand.argtypes = [ctypes.c_uint]
    _libc.srand(seed)
    out = np.empty((n_hyp, 3), np.int32)
    for h in range(n_hyp):
        while True:
            e = [_libc.rand() % n_edgels for _ in range(3)]
            if e[0] != e[1] and e[1] != e[2]:
                break
        out[h] = e
    return out


def target_params_from_picks(picked, locations, tangents, start_params):
    """GPU_HC_Solver.cpp:276-296 on the host, vectorised.  Returns (target[H,34], diff[H,34]) complex64."""
    picked = np.asarray(picked)
    H = picked.shape[0]
    tgt = np.zeros((H, NUM_PARAMS + 1), np.complex64)
    tgt[:, 0:18] = locations[picked].reshape(H, 18)
    tgt[:, 18:30] = tangents[picked[:, :2]].reshape(H, 12)
    tgt[:, 30] = 1.0
    tgt[:, 31] = 0.5
    tgt[:, 32] = 1.0
    tgt[:, 33] = 1.0
    sp = np.concatenate([np.asarray(start_params, np.complex64)[:NUM_PARAMS], [1.0]]).astype(np.complex64)
    diff = np.empty_like(tgt)
    diff.real = tgt.real - sp.real[None, :]
    diff.imag = tgt.imag - sp.imag[None, :]
    return tgt, diff


def padded_start_sols(start_sols):
    """[312,30] -> [312,31] with the constant-one pad (Data_Reader.cpp:55-57)."""
    ss = np.ones((NUM_TRACKS, NUM_VARS + 1), np.complex64)
    ss[:, :NUM_VARS] = start_sols
    return ss


def padded_start_params(start_params):
    return np.concatenate([np.asarray(start_params, np.complex64)[:NUM_PARAMS], [1.0]]).astype(np.complex64)


# ------------------------------------------------------------------------------------------------------------------

class Tracker:
    """Device-side state of one GPU's share of a RANSAC round (mirrors the per-GPU arrays of GPU_HC_Solver,
    GPU_HC_Solver.cpp:137-184) and the two launches.  All tensors are torch CUDA tensors owned by this object."""

    def __init__(self, device=None, problem=None, max_steps=80, max_corr=3, dt_inc=4, stats=False, split=True):
        import torch
        self.torch = torch
        self.lib = load_library()
        if not torch.cuda.is_available():
            raise HCB200Error("no CUDA device: the tracker has no CPU path")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        problem = problem or fixtures.load_problem()
        self.max_steps, self.max_corr, self.dt_inc = max_steps, max_corr, dt_inc
        self.start_sols_h = padded_start_sols(problem["start_sols"])
        self.start_params_h = padded_start_params(problem["start_params"])
        with torch.cuda.device(self.device):
            self.d_start_sols = torch.view_as_real(torch.from_numpy(self.start_sols_h)).contiguous().to(self.device)
            self.d_start_params = torch.view_as_real(torch.from_numpy(self.start_params_h)).contiguous().to(self.device)
            self.d_ws = torch.zeros(int(self.lib.hcb200_workspace_bytes()), dtype=torch.uint8, device=self.device)
        self.capacity = 0
        self.launches = 0
        self.want_stats = stats
        self.d_stats = None
        self.split = bool(split)       # HCB200_FLAG_SPLIT_LONG_PATHS: long paths are parked and finished by idle warps (same results, shorter tail)

    def kernel_info(self, abort=False):
        v = [ctypes.c_int() for _ in range(5)]
        with self.torch.cuda.device(self.device):
            _check(self.lib.hcb200_kernel_info(1 if abort else 0, *[ctypes.byref(x) for x in v]), "hcb200_kernel_info")
        return dict(zip(("regs", "smem_bytes", "ctas_per_sm", "grid", "block"), [x.value for x in v]))

    def reserve(self, n_hyp):
        torch = self.torch
        stats = self.want_stats
        if n_hyp <= self.capacity:
            return
        n_paths = n_hyp * NUM_TRACKS
        dev = self.device
        self.d_target = torch.empty((n_hyp, NUM_PARAMS + 1, 2), dtype=torch.float32, device=dev)
        self.d_diff = torch.empty_like(self.d_target)
        self.d_tracks = torch.empty((n_paths, NUM_VARS + 1, 2), dtype=torch.float32, device=dev)
        self.d_conv = torch.empty(n_paths, dtype=torch.uint8, device=dev)
        self.d_inf = torch.empty(n_paths, dtype=torch.uint8, device=dev)
        self.d_stats = torch.empty((n_paths, 4), dtype=torch.int32, device=dev) if stats else None
        self.d_found = torch.zeros(1, dtype=torch.uint8, device=dev)
        self.d_found_index = torch.empty(n_paths, dtype=torch.int32, device=dev)
        self.d_best = torch.zeros(16, dtype=torch.int32, device=dev)
        if self.split:
            self.d_ws = torch.zeros(int(self.lib.hcb200_workspace_bytes_for(min(n_hyp, SPLIT_MAX_HYPOTHESES))), dtype=torch.uint8, device=dev)
        self.capacity = n_hyp

    def set_edgels(self, locations, K):
        torch = self.torch
        self.d_edgels = torch.from_numpy(np.ascontiguousarray(locations, np.float32)).to(self.device)
        self.d_K = torch.from_numpy(np.ascontiguousarray(K, np.float32).reshape(-1)).to(self.device)
        self.n_edgels = int(locations.shape[0])

    def upload_params(self, target, diff, non_blocking=False):
        """target/diff: complex64 numpy [H,34] or pinned float32 torch tensors [H,34,2]."""
        torch = self.torch
        if isinstance(target, np.ndarray):
            target = torch.view_as_real(torch.from_numpy(np.ascontiguousarray(target, np.complex64)))
            diff = torch.view_as_real(torch.from_numpy(np.ascontiguousarray(diff, np.complex64)))
        H = target.shape[0]
        self.reserve(H)
        self.d_target[:H].copy_(target, non_blocking=non_blocking)
        self.d_diff[:H].copy_(diff, non_blocking=non_blocking)
        return H

    def _stream(self):
        return ctypes.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def track(self, n_hyp, prune=True):
        """Enqueue hcb200_track on torch's current stream (asynchronous, like the reference wrapper)."""
        p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        with self.torch.cuda.device(self.device):
            rc = self.lib.hcb200_track(self._stream(), n_hyp, self.max_steps, self.max_corr, self.dt_inc,
                                       (FLAG_PRUNE_PATHS if prune else 0) | (FLAG_SPLIT_LONG_PATHS if (self.split and n_hyp <= SPLIT_MAX_HYPOTHESES) else 0) |
                                       (int(getattr(self, "suspend_step", 0)) << 16),
                                       p(self.d_start_sols), p(self.d_start_params), p(self.d_target), p(self.d_diff),
                                       p(self.d_tracks), p(self.d_conv), p(self.d_inf), p(self.d_stats), p(self.d_ws))
        _check(rc, "hcb200_track")
        self.launches += 1

    def reset_abort(self, n_hyp):
        """Clear the early-abort flag and the found indices (the caller's job in the reference too, GPU_HC_Solver.cpp:321-324)."""
        self.d_found.zero_()
        self.d_found_index[:n_hyp * NUM_TRACKS].fill_(-1)

    def track_abort(self, n_hyp, prune=True, peers=None, reset=True):
        """Early-abort launch.  peers: Trackers on OTHER GPUs of this process taking part in the same round — the first passing path raises their
        flags too (hcb200_track_abort_peers, NVLink peer stores); every participant must then be reset (reset_abort) before the first launch of
        the round, so pass reset=False here."""
        p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        if reset:
            self.reset_abort(n_hyp)
        args = [self._stream(), n_hyp, self.n_edgels, self.max_steps, self.max_corr, self.dt_inc, FLAG_PRUNE_PATHS if prune else 0,
                p(self.d_start_sols), p(self.d_start_params), p(self.d_target), p(self.d_diff), p(self.d_edgels), p(self.d_K),
                p(self.d_tracks), p(self.d_conv), p(self.d_inf), p(self.d_found), p(self.d_found_index), p(self.d_best), p(self.d_stats), p(self.d_ws)]
        with self.torch.cuda.device(self.device):
            if peers:
                for q in peers:
                    _check(self.lib.hcb200_enable_peer_access(self.device.index, q.device.index), "hcb200_enable_peer_access")
                arr = (ctypes.c_void_p * len(peers))(*[q.d_found.data_ptr() for q in peers])
                rc = self.lib.hcb200_track_abort_peers(*args, arr, len(peers))
            else:
                rc = self.lib.hcb200_track_abort(*args)
        _check(rc, "hcb200_track_abort")
        self.launches += 2

    # ---- early-abort rounds of many image triplets ("problems") in one launch (hcb200_track_abort_batched).  The parameters are uploaded
    # stacked problem-major (upload_params of [n_problems * n_hyp, 34]); tracks, flags, stats and found indices come back in the same order.

    def set_edgel_batch(self, locations_list, K_list):
        """Problem k's edgel locations [E_k, 6] and 3x3 intrinsics: concatenated and uploaded; the host keeps the edgel offsets."""
        torch = self.torch
        locs = [np.ascontiguousarray(loc, np.float32).reshape(-1, 6) for loc in locations_list]
        if len(locs) != len(K_list) or not locs:
            raise ValueError("one K per edgel set, at least one problem")
        self.batch_offsets = np.concatenate([[0], np.cumsum([loc.shape[0] for loc in locs])]).astype(np.int32)
        self.d_edgels_batch = torch.from_numpy(np.concatenate(locs)).to(self.device)
        self.d_K_batch = torch.from_numpy(np.stack([np.asarray(K, np.float32).reshape(9) for K in K_list])).to(self.device)

    def _reserve_batch(self, n_problems):
        torch = self.torch
        if getattr(self, "d_found_batch", None) is not None and self.d_found_batch.shape[0] >= n_problems:
            return
        self.d_found_batch = torch.zeros(n_problems, dtype=torch.uint8, device=self.device)
        self.d_best_batch = torch.zeros((n_problems, 16), dtype=torch.int32, device=self.device)
        self.d_ws_batch = torch.zeros(int(self.lib.hcb200_batch_workspace_bytes(n_problems)), dtype=torch.uint8, device=self.device)

    def reset_abort_batched(self, n_problems, n_hyp):
        """Clear the problems' early-abort flags and the found indices of their paths."""
        self._reserve_batch(n_problems)
        self.d_found_batch[:n_problems].zero_()
        self.d_found_index[:n_problems * n_hyp * NUM_TRACKS].fill_(-1)

    def track_abort_batched(self, n_problems, n_hyp, prune=True):
        """Early-abort rounds of the first n_problems problems of set_edgel_batch, n_hyp hypotheses each, in one launch; every problem stops on
        its own first passing path.  Resets the flags and the found indices, then enqueues the launch; batch_records reads the results."""
        if n_problems > len(self.batch_offsets) - 1:
            raise ValueError("%d problems, but set_edgel_batch gave %d" % (n_problems, len(self.batch_offsets) - 1))
        p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        self.reset_abort_batched(n_problems, n_hyp)
        offsets = np.ascontiguousarray(self.batch_offsets[:n_problems + 1])
        with self.torch.cuda.device(self.device):
            rc = self.lib.hcb200_track_abort_batched(
                self._stream(), n_problems, n_hyp, offsets.ctypes.data_as(ctypes.c_void_p), self.max_steps, self.max_corr, self.dt_inc,
                FLAG_PRUNE_PATHS if prune else 0, p(self.d_start_sols), p(self.d_start_params), p(self.d_target), p(self.d_diff),
                p(self.d_edgels_batch), p(self.d_K_batch), p(self.d_tracks), p(self.d_conv), p(self.d_inf), p(self.d_found_batch),
                p(self.d_found_index), p(self.d_best_batch), p(self.d_stats), p(self.d_ws_batch))
        _check(rc, "hcb200_track_abort_batched")
        self.launches += 2

    def batch_records(self, n_problems):
        """Synchronise and return the problems' best records: found, path_id (local to the problem: hypothesis * 312 + track, -1 when none),
        inliers21, inliers31, n_passed."""
        self.torch.cuda.synchronize(self.device)
        best = self.d_best_batch[:n_problems].cpu().numpy()
        return [dict(found=int(b[0]), path_id=int(b[1]), inliers21=int(b[2]), inliers31=int(b[3]), n_passed=int(b[4])) for b in best]

    def score_tracks_batched(self, n_problems, n_hyp):
        """No-abort counterpart of track_abort_batched: hcb200_score_tracks on each problem's slice of the last round, with the problem's edgels
        and K.  Returns (support int32 [n_problems * n_hyp * 312, 2], best records int32 [n_problems, 16], path ids local to each problem)."""
        torch = self.torch
        L = n_hyp * NUM_TRACKS
        if getattr(self, "d_support", None) is None or self.d_support.shape[0] < n_problems * L:
            self.d_support = torch.empty((n_problems * L, 2), dtype=torch.int32, device=self.device)
        self._reserve_batch(n_problems)
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        off = self.batch_offsets
        with torch.cuda.device(self.device):
            for k in range(n_problems):
                s = slice(k * L, (k + 1) * L)
                rc = self.lib.hcb200_score_tracks(self._stream(), L, p(self.d_tracks[s]), p(self.d_conv[s]), int(off[k + 1] - off[k]),
                                                  p(self.d_edgels_batch[int(off[k]):]), p(self.d_K_batch[k]), p(self.d_support[s]),
                                                  p(self.d_best_batch[k]), p(self.d_ws))
                _check(rc, "hcb200_score_tracks")
                self.launches += 2
        torch.cuda.synchronize(self.device)
        return self.d_support[:n_problems * L].cpu().numpy(), self.d_best_batch[:n_problems].cpu().numpy()

    def refine_tracks(self, n_hyp, iters=3):
        """Device-side Newton refinement of the converged end points of the last round against their target systems (in place).
        Returns sums float32 [P,2] = (sum|dx|^2, sum|x|^2) of the last iteration, (-1,-1) for paths that were not refined."""
        torch = self.torch
        n_paths = n_hyp * NUM_TRACKS
        if getattr(self, "d_sums", None) is None or self.d_sums.shape[0] < n_paths:
            self.d_sums = torch.empty((n_paths, 2), dtype=torch.float32, device=self.device)
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        with torch.cuda.device(self.device):
            rc = self.lib.hcb200_refine_tracks(self._stream(), n_paths, int(iters), p(self.d_target), p(self.d_conv), p(self.d_tracks),
                                               p(self.d_sums), p(self.d_ws))
        _check(rc, "hcb200_refine_tracks")
        self.launches += 1
        torch.cuda.synchronize(self.device)
        return self.d_sums[:n_paths].cpu().numpy()

    def score_tracks(self, n_hyp):
        """Device-side final scoring of the last round: returns (support int32 [P,2], best record int32 [16]) after a sync."""
        torch = self.torch
        n_paths = n_hyp * NUM_TRACKS
        if getattr(self, "d_support", None) is None or self.d_support.shape[0] < n_paths:
            self.d_support = torch.empty((n_paths, 2), dtype=torch.int32, device=self.device)
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        with torch.cuda.device(self.device):
            rc = self.lib.hcb200_score_tracks(self._stream(), n_paths, p(self.d_tracks), p(self.d_conv), self.n_edgels, p(self.d_edgels),
                                              p(self.d_K), p(self.d_support), p(self.d_best), p(self.d_ws))
        _check(rc, "hcb200_score_tracks")
        self.launches += 2
        torch.cuda.synchronize(self.device)
        return self.d_support[:n_paths].cpu().numpy(), self.d_best.cpu().numpy()

    def score_tracks_async(self, n_hyp):
        """Enqueue the device-side final scoring of the last round (no synchronisation); the best record lands in self.d_best."""
        torch = self.torch
        n_paths = n_hyp * NUM_TRACKS
        if getattr(self, "d_support", None) is None or self.d_support.shape[0] < n_paths:
            self.d_support = torch.empty((n_paths, 2), dtype=torch.int32, device=self.device)
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        with torch.cuda.device(self.device):
            rc = self.lib.hcb200_score_tracks(self._stream(), n_paths, p(self.d_tracks), p(self.d_conv), self.n_edgels, p(self.d_edgels),
                                              p(self.d_K), p(self.d_support), p(self.d_best), p(self.d_ws))
        _check(rc, "hcb200_score_tracks")
        self.launches += 2

    def count_solutions_device(self, n_hyp):
        """Per-hypothesis (converged, infinity, real) counts of the last round, computed on the device; returns int array [H,3]."""
        torch = self.torch
        d_counts = torch.zeros((n_hyp, 3), dtype=torch.int32, device=self.device)
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        with torch.cuda.device(self.device):
            rc = self.lib.hcb200_count_solutions(self._stream(), n_hyp, p(self.d_tracks), p(self.d_conv), p(self.d_inf), p(d_counts))
        _check(rc, "hcb200_count_solutions")
        self.launches += 1
        torch.cuda.synchronize(self.device)
        return d_counts.cpu().numpy()

    def make_pose_record(self, path_offset, rank, abort=False):
        """Enqueue: best record of the last score / abort launch -> the 128-byte exchange record self.d_pose_record (float32 [32])."""
        torch = self.torch
        if getattr(self, "d_pose_record", None) is None:
            self.d_pose_record = torch.zeros(32, dtype=torch.float32, device=self.device)
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        with torch.cuda.device(self.device):
            rc = self.lib.hcb200_make_pose_record(self._stream(), p(self.d_tracks), p(self.d_best), p(self.d_found) if abort else None,
                                                  int(path_offset), int(rank), p(self.d_pose_record))
        _check(rc, "hcb200_make_pose_record")
        self.launches += 1
        return self.d_pose_record

    def reduce_pose_records(self, d_records, n):
        """Enqueue the arg-max over n gathered 128-byte records ([n,32] float32 device tensor) -> self.d_round_record."""
        torch = self.torch
        if getattr(self, "d_round_record", None) is None:
            self.d_round_record = torch.zeros(32, dtype=torch.float32, device=self.device)
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        with torch.cuda.device(self.device):
            rc = self.lib.hcb200_reduce_pose_records(self._stream(), int(n), p(d_records), p(self.d_round_record))
        _check(rc, "hcb200_reduce_pose_records")
        self.launches += 1
        return self.d_round_record

    def build_target_params(self, d_picked, d_tangents, n_hyp):
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        with self.torch.cuda.device(self.device):
            rc = self.lib.hcb200_build_target_params(self._stream(), n_hyp, p(d_picked), self.n_edgels, p(self.d_edgels),
                                                     p(d_tangents), p(self.d_start_params), p(self.d_target), p(self.d_diff))
        _check(rc, "hcb200_build_target_params")
        self.launches += 1

    def ffma_probe(self, iters=20000, reps=5):
        """Measured FP32 FMA throughput of this GPU in TFLOP/s (best of `reps`, CUDA events)."""
        torch = self.torch
        scratch = torch.zeros(4, dtype=torch.float32, device=self.device)
        flops = ctypes.c_double()
        best = 0.0
        for _ in range(reps + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _check(self.lib.hcb200_ffma_probe(self._stream(), iters, ctypes.c_void_p(scratch.data_ptr()), ctypes.byref(flops)),
                   "hcb200_ffma_probe")
            e1.record()
            e1.synchronize()
            best = max(best, flops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        return best

    def results(self, n_hyp):
        """Synchronise and fetch (tracks complex64 [P,31], converged uint8 [P], infinity uint8 [P], stats or None)."""
        self.torch.cuda.synchronize(self.device)
        n = n_hyp * NUM_TRACKS
        tr = self.d_tracks[:n].cpu().numpy()
        tracks = (tr[..., 0] + 1j * tr[..., 1]).astype(np.complex64)
        stats = self.d_stats[:n].cpu().numpy() if self.d_stats is not None else None
        return tracks, self.d_conv[:n].cpu().numpy(), self.d_inf[:n].cpu().numpy(), stats


def decode_pose_record(rec):
    """128-byte exchange record (float32 [32] host array, hcb200_pose_record) -> dict."""
    b = np.ascontiguousarray(rec, np.float32).view(np.uint8)
    i = b[:24].view(np.int32)
    return {"found": int(i[0]), "inliers21": int(i[1]), "inliers31": int(i[2]), "n_candidates": int(i[3]), "abort_flag": int(i[4]),
            "rank": int(i[5]), "path_id": int(b[24:32].view(np.int64)[0]), "R21": b[32:68].view(np.float32).reshape(3, 3).copy(),
            "t21": b[68:80].view(np.float32).copy(), "R31": b[80:116].view(np.float32).reshape(3, 3).copy(), "t31": b[116:128].view(np.float32).copy()}


def encode_pose_record(found, inliers21, inliers31, n_candidates, abort_flag, rank, path_id, pose24=None):
    """Build a 128-byte exchange record (hcb200_pose_record) on the host; returns float32 [32]."""
    b = np.zeros(128, np.uint8)
    b[:24].view(np.int32)[:] = [found, inliers21, inliers31, n_candidates, abort_flag, rank]
    b[24:32].view(np.int64)[0] = path_id
    if pose24 is not None:
        b[32:128].view(np.float32)[:] = np.asarray(pose24, np.float32).reshape(24)
    return b.view(np.float32).copy()


def reduce_pose_records_host(records):
    """Host mirror of hcb200_reduce_pose_records (csrc/hc_tracker.cu): arg-max over the gathered records — largest
    min(inliers21, inliers31), lowest global path id among equals; abort flags OR-ed, candidate counts summed.
    records: float32 [n, 32].  Returns the winning record as a dict (decode_pose_record layout)."""
    recs = [decode_pose_record(r) for r in np.asarray(records, np.float32).reshape(-1, 32)]
    best = None
    for r in recs:
        if not (r["found"] and r["path_id"] >= 0):
            continue
        key = (min(r["inliers21"], r["inliers31"]), -r["path_id"])
        if best is None or key > best[0]:
            best = (key, r)
    out = dict(best[1]) if best else {"found": 0, "inliers21": 0, "inliers31": 0, "rank": -1, "path_id": -1,
                                     "R21": np.zeros((3, 3), np.float32), "t21": np.zeros(3, np.float32),
                                     "R31": np.zeros((3, 3), np.float32), "t31": np.zeros(3, np.float32)}
    out["n_candidates"] = sum(r["n_candidates"] for r in recs)
    out["abort_flag"] = int(any(r["abort_flag"] for r in recs))
    return out


def count_solutions(tracks, converged, infinity, n_hyp):
    """Evaluations::Evaluate_HC_Sols (Evaluations.cpp:145-167): per hypothesis (#converged, #infinity, #real) with
    real == converged and all 30 |imag| <= 1e-4 (ZERO_IMAG_PART_TOL_FOR_SP)."""
    conv = converged.reshape(n_hyp, NUM_TRACKS).astype(bool)
    inf = infinity.reshape(n_hyp, NUM_TRACKS).astype(bool)
    im = np.abs(tracks.reshape(n_hyp, NUM_TRACKS, NUM_VARS + 1)[:, :, :NUM_VARS].imag)
    real = conv & np.all(im.astype(np.float64) <= 1e-4, axis=2)
    return np.stack([conv.sum(1), inf.sum(1), real.sum(1)], axis=1)
