/* hcb200.h — C ABI of the B200-native homotopy-continuation path tracker for trifocal_2op1p_30x30.
 *
 * This is the drop-in boundary: the entry points below replace the reference's kernel launch wrappers
 *
 *   kernel_GPUHC_trifocal_2op1p_30x30_PH_CodeOpt_TrunPaths            magmaHC/gpu-kernels/magmaHC-kernels.hpp:24-39
 *   kernel_GPUHC_trifocal_2op1p_30x30_PH_CodeOpt_TrunPaths_TrunRANSAC magmaHC/gpu-kernels/magmaHC-kernels.hpp:61-81
 *
 * (called from GPU_HC_Solver::Solve_by_GPU_HC, magmaHC/GPU_HC_Solver.cpp:395-433).  Conventions kept from the
 * reference: the CALLER owns every buffer; the current CUDA device is the caller's; work is ENQUEUED on `stream`
 * and the call returns immediately (the caller synchronises, GPU_HC_Solver.cpp:440-444).  Differences: plain C
 * types (cudaStream_t as void*, float2 as float[2]), an int (cudaError_t) status instead of a dummy time, and no
 * MAGMA queue / pointer arrays / index table (the polynomial system is compiled into the library).
 * INTEGRATION.md shows the ten-line shim that gives the reference's exact C++ signatures on top of this ABI.
 *
 * Layouts (reference: SURVEY.md App. A.5)
 *   start_sols    [312][31] complex64   start solutions, entry 30 == 1+0i        (d_Start_Sols,  Data_Reader.cpp:37-60)
 *   start_params  [34]      complex64   entry 33 == 1+0i                          (d_Start_Params)
 *   target_params [n_hyp][34] complex64 per RANSAC hypothesis                     (d_Target_Params, GPU_HC_Solver.cpp:276-292)
 *   diff_params   [n_hyp][34] complex64 target - start                            (d_diffParams,  GPU_HC_Solver.cpp:295-296)
 *   tracks        [n_hyp*312][31] complex64  OUT: end point of every path (need not be pre-loaded with the start
 *                                        solutions — the reference requires that, GPU_HC_Solver.cpp:208,342)
 *   converged / infinity [n_hyp*312] uint8 (C++ bool)  OUT                        (d_is_GPU_HC_Sol_Converge / _Infinity)
 *   path id = hypothesis*312 + start-solution index                              (…TrunPaths.cu:67-69)
 */
#ifndef HCB200_H
#define HCB200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HCB200_NUM_VARS 30
#define HCB200_NUM_PARAMS 33
#define HCB200_NUM_TRACKS 312
#define HCB200_ABI_VERSION 3

/* flags */
#define HCB200_FLAG_PRUNE_PATHS 1u   /* positive-depth path pruning (always on in the reference GPU kernels, …TrunPaths.cu:148-154) */
/* Split long paths (ABI 3): a path that reaches 4/5 of the step cap while fresh paths are still queued is parked and finished by the first
 * warp that runs out of fresh paths, so a round ends on many short remainders instead of a few long paths (default round: -5 % time).
 * Results are bit-identical with and without the flag.  The caller promises that d_workspace holds hcb200_workspace_bytes_for(n_hyp) bytes
 * (256 + 20 bytes per path) instead of hcb200_workspace_bytes().  Ignored by hcb200_track_abort.  Bits 16..31 of `flags`, when non-zero,
 * replace the step at which a path is parked (tuning; default 4/5 of hc_max_steps).  The launcher uses the split kernel only while the round
 * is small (fewer than 48 paths per resident warp: about 450 hypotheses on a B200), so callers need not pay for the large workspace of big
 * rounds: pass the flag only when n_hyp <= HCB200_SPLIT_MAX_HYPOTHESES. */
#define HCB200_SPLIT_MAX_HYPOTHESES 2048
#define HCB200_FLAG_SPLIT_LONG_PATHS 2u

/* Optional per-path counters (all int32): HC steps attempted, predictor stages, corrector stages,
 * rejected steps | end reason << 16 (0 converged, 1 infinity, 2 pruned, 3 step cap, 4 skipped after abort). */
typedef struct { int32_t steps, pred_stages, corr_stages, rejected_reason; } hcb200_path_stats;

/* Best candidate of an early-abort launch, reduced on the device (64 bytes). */
typedef struct {
  int32_t found;            /* 0/1: some path passed the inlier test                                   */
  int32_t path_id;          /* smallest passing path id of this launch (hypothesis*312 + track), or -1 */
  int32_t inliers21, inliers31;   /* its reprojection inlier counts (views 1-2, 1-3)                   */
  int32_t n_passed;         /* number of paths that passed before the launch drained                   */
  int32_t reserved[11];
} hcb200_best_record;

/* What one GPU contributes to the multi-GPU result exchange (128 bytes): its best candidate with the pose, and its early-abort
 * flag.  Replaces the host-side stacking of every GPU's tracks (GPU_HC_Solver.cpp:449-506) when only the selected pose is needed
 * (BASELINE.json north_star (4): "only a tiny gather of each GPU's best pose and early-abort flag"). */
typedef struct {
  int32_t found;            /* this GPU has a pose candidate (score launch) / a passing path (abort launch)      */
  int32_t inliers21, inliers31;
  int32_t n_candidates;     /* candidates (score) or passing paths (abort) on this GPU; summed by the reduction   */
  int32_t abort_flag;       /* the GPU's early-abort flag; OR-ed by the reduction                                 */
  int32_t rank;             /* GPU / rank that owns the winning record                                            */
  long long path_id;        /* GLOBAL path id (hypothesis * 312 + track over the whole round), -1 when none       */
  float pose[24];           /* R21 row-major [9], t21 [3] (unit length), R31 [9], t31 [3] of that path            */
} hcb200_pose_record;

/* Device workspace the launches need (work counter + reduction scratch); zeroing is done by the launch itself. */
size_t hcb200_workspace_bytes(void);
size_t hcb200_workspace_bytes_for(int n_hyp);      /* workspace size that HCB200_FLAG_SPLIT_LONG_PATHS needs for rounds of up to n_hyp hypotheses */
int hcb200_abi_version(void);

/* The minimal problem compiled into this library (the reference reads these from problems/<name>/gpuhc_settings.yaml:
 * Num_Of_Vars, Num_Of_Params, Num_Of_Tracks, problem_name).  libhcb200.so is trifocal_2op1p_30x30 (30, 33, 312, 1); a library built by
 * `make problem PROBLEM_DIR=…` for another problem folder reports that problem's sizes, takes arrays of those sizes in hcb200_track /
 * hcb200_refine_tracks / hcb200_count_solutions, and answers cudaErrorNotSupported in the trifocal-only entry points (abort, scoring,
 * pose records, target parameters from edgels).  Any pointer may be NULL.  Returns 0. */
int hcb200_problem_info(int* n_vars, int* n_params, int* n_tracks, int* is_trifocal, const char** name);

/* Replaces kernel_GPUHC_trifocal_2op1p_30x30_PH_CodeOpt_TrunPaths (…TrunPaths.cu:292-386).
 * Tracks all 312*n_hyp paths in one launch (0 <= n_hyp <= 3 441 480: path ids are 31-bit).  `stats` may be NULL.
 * Returns a cudaError_t value (0 == success; cudaErrorInvalidValue for NULL buffers or out-of-range counts, nothing launched). */
int hcb200_track(void* stream, int n_hyp,
                 int hc_max_steps, int hc_max_correction_steps, int hc_delta_t_incremental_steps, unsigned flags,
                 const float* d_start_sols, const float* d_start_params,
                 const float* d_target_params, const float* d_diff_params,
                 float* d_tracks, uint8_t* d_converged, uint8_t* d_infinity,
                 hcb200_path_stats* d_stats, void* d_workspace);

/* Replaces kernel_GPUHC_trifocal_2op1p_30x30_PH_CodeOpt_TrunPaths_TrunRANSAC (…TrunRANSAC.cu:329-453): as above plus
 * in-kernel scoring of every converged path against all edgel triplets and a device-side abort flag.
 *   d_edgel_locations [n_edgels][6] float32  (x1 y1 x2 y2 x3 y3, normalised coordinates)   (d_Triplet_Edge_Locations)
 *   d_intrinsic       [9] float32 row-major K                                             (d_Intrinsic_Matrix)
 *   d_found           [1] uint8 in/out: must be 0 on entry; set to 1 by the first passing path (d_Found_Trifocal_Sols)
 *   d_found_index     [n_hyp*312] int32 in/out: pre-set to -1 by the caller, entry b becomes b if path b passed
 *                                                                                          (d_Trifocal_Sols_Batch_Index)
 *   d_best            optional (may be NULL) hcb200_best_record, written when the launch drains.
 * Paths that start after the flag is up are skipped (converged = 0, end point = start solution) like the reference;
 * unlike the reference the flag is also polled at every HC step, and the infinity flag of skipped paths is 0. */
int hcb200_track_abort(void* stream, int n_hyp, int n_edgels,
                       int hc_max_steps, int hc_max_correction_steps, int hc_delta_t_incremental_steps, unsigned flags,
                       const float* d_start_sols, const float* d_start_params,
                       const float* d_target_params, const float* d_diff_params,
                       const float* d_edgel_locations, const float* d_intrinsic,
                       float* d_tracks, uint8_t* d_converged, uint8_t* d_infinity,
                       uint8_t* d_found, int32_t* d_found_index, hcb200_best_record* d_best,
                       hcb200_path_stats* d_stats, void* d_workspace);

/* Early abort ACROSS the GPUs of one process (ABI 3).  The reference keeps the flag per GPU (GPU_HC_Solver.cpp:329,402): a GPU whose shard holds
 * no good hypothesis tracks all of it while another GPU has long found the pose.  Here the first passing path also raises the flags of the
 * peer GPUs: d_peer_found[i] (host array of n_peers <= 7 device pointers) are the d_found bytes of the other GPUs' launches of the same round,
 * written through NVLink peer mappings — the caller enables peer access (cudaDeviceEnablePeerAccess) and resets every flag before the first
 * launch of the round.  Each GPU still polls only its own flag.  A GPU stopped by a peer reports found == 0 in its own best record and leaves
 * d_found_index at -1; its d_found byte reads 1. */
int hcb200_track_abort_peers(void* stream, int n_hyp, int n_edgels,
                       int hc_max_steps, int hc_max_correction_steps, int hc_delta_t_incremental_steps, unsigned flags,
                       const float* d_start_sols, const float* d_start_params,
                       const float* d_target_params, const float* d_diff_params,
                       const float* d_edgel_locations, const float* d_intrinsic,
                       float* d_tracks, uint8_t* d_converged, uint8_t* d_infinity,
                       uint8_t* d_found, int32_t* d_found_index, hcb200_best_record* d_best,
                       hcb200_path_stats* d_stats, void* d_workspace,
                             uint8_t* const* d_peer_found, int n_peers);

/* Early-abort rounds of MANY image triplets ("problems": dataset, edgel set, K) in one launch.  An abort round is bound by the latency of
 * one long path (~80 HC steps) while most resident warps track hypotheses whose work the flag then throws away; here the queue interleaves
 * the problems, so the first wave of warps holds the first hypotheses of every problem and K early-hit problems end in about the time of one.
 * Every problem has n_hyp_per_problem hypotheses.
 *   Storage is problem-major: path id b = problem * n_hyp_per_problem * 312 + hypothesis * 312 + track, so each problem's target / diff
 *     parameters ([n_problems * n_hyp_per_problem][34]), tracks, flags, stats and found indices form one contiguous slice.  d_found_index
 *     [all paths] is pre-set to -1 by the caller; entry b becomes b (the storage id) when path b passes.
 *   The queue is interleaved: queue position q tracks problem q % n_problems, local path q / n_problems.  Within a problem, paths start in
 *     the order of a single-problem launch.  The order is fixed.
 *   Each problem has its own early abort: d_found [n_problems] uint8, 0 on entry.  A passing path of problem k raises only d_found[k]; the
 *     paths of problem k poll only that byte, at path start and at every HC step, like hcb200_track_abort.  Skipped paths of a problem are
 *     as there: converged = 0, infinity = 0, end reason 4.  The pass test is hcb200_track_abort's, against problem k's edgels
 *     [off[k], off[k+1]) of d_edgel_locations ([off[n_problems]][6]) and its K, d_intrinsics + 9 k ([n_problems][9] row-major).
 *   Each problem has its own result: d_best [n_problems] (may be NULL) receives problem k's record: found, smallest passing path id LOCAL to
 *     the problem (hypothesis * 312 + track), its inlier counts, n_passed.  The layout is hcb200_track_abort's, so
 *     hcb200_make_pose_record(d_tracks + 62 * 312 * n_hyp_per_problem * k, d_best + k, d_found + k, path_offset, rank, ...) works on the slice.
 *     An empty round (n_hyp_per_problem == 0) clears every record.
 *   h_edgel_offsets is a HOST array [n_problems + 1]: off[0] == 0, problem k owns edgels [off[k], off[k+1]).  The launcher copies it into the
 *     workspace (cudaMemcpyAsync from pageable memory: the array may be reused when the call returns).  d_workspace holds
 *     hcb200_batch_workspace_bytes(n_problems) = 256 + 16 * (n_problems + 1) bytes: per-problem best keys, pass counters and edgel offsets.
 *   flags: HCB200_FLAG_PRUNE_PATHS; the split flag is ignored, as in hcb200_track_abort.
 * Returns cudaErrorInvalidValue, before any CUDA call and with nothing launched, for NULL buffers (d_best and d_stats may be NULL),
 * n_problems outside [1, HCB200_BATCH_MAX_PROBLEMS], n_hyp_per_problem < 0, n_problems * n_hyp_per_problem > 3 441 480 (31-bit path ids),
 * hc_max_correction_steps < 1, off[0] != 0, or a problem with 0 or more than 65 535 edgels.  cudaErrorNotSupported in a compiled-problem
 * library.  The limit on n_problems keeps the staged offsets (16 bytes per problem) in one 64 KB copy. */
#define HCB200_BATCH_MAX_PROBLEMS 4095
size_t hcb200_batch_workspace_bytes(int n_problems);
int hcb200_track_abort_batched(void* stream, int n_problems, int n_hyp_per_problem, const int32_t* h_edgel_offsets,
                               int hc_max_steps, int hc_max_correction_steps, int hc_delta_t_incremental_steps, unsigned flags,
                               const float* d_start_sols, const float* d_start_params,
                               const float* d_target_params, const float* d_diff_params,
                               const float* d_edgel_locations, const float* d_intrinsics,
                               float* d_tracks, uint8_t* d_converged, uint8_t* d_infinity,
                               uint8_t* d_found, int32_t* d_found_index, hcb200_best_record* d_best,
                               hcb200_path_stats* d_stats, void* d_workspace);

/* Lets kernels running on `device` store into memory of `peer_device` (cudaDeviceEnablePeerAccess in `device`'s context; "already enabled" is
 * success; cudaErrorPeerAccessUnsupported when the two GPUs have no peer path).  Needed once per ordered pair before hcb200_track_abort_peers. */
int hcb200_enable_peer_access(int device, int peer_device);

/* Device-side hypothesis generation (Prepare_Target_Params at scale, GPU_HC_Solver.cpp:252-306): given the picked
 * edgel indices [n_hyp][3] it gathers the 34 target parameters and target - start for every hypothesis. */
int hcb200_build_target_params(void* stream, int n_hyp, const int32_t* d_picked, int n_edgels,
                               const float* d_edgel_locations, const float* d_edgel_tangents,
                               const float* d_start_params, float* d_target_params, float* d_diff_params);

/* Final scoring of a round on the device (Evaluations::Transform_GPUHC_Sols_to_Trifocal_Relative_Pose +
 * ::get_Solution_with_Maximal_Support, reference Evaluations.cpp:298-504, with the intended per-solution indexing).
 * For every path: d_support[2*path + {0,1}] = number of edgel triplets whose reprojection error is < 2 px for view pairs
 * (1,2) / (1,3), or -1 when the path is not a pose candidate (not converged, |Im| of a Cayley parameter >= 1e-5, or a negative
 * depth).  d_best: found, path_id = candidate maximising min(support21, support31) (lowest path id on ties), its two supports,
 * n_passed = number of candidates, reserved[0..1] = the per-pair maxima over all candidates.  Uses bytes [128, 160) of the
 * workspace.  The float arithmetic is the host class's (host/mvg.hpp) operation for operation, so counts are identical. */
int hcb200_score_tracks(void* stream, int n_paths, const float* d_tracks, const uint8_t* d_converged, int n_edgels,
                        const float* d_edgel_locations, const float* d_intrinsic, int32_t* d_support,
                        hcb200_best_record* d_best, void* d_workspace);

/* Evaluations::Evaluate_HC_Sols on the device (reference Evaluations.cpp:145-167): d_counts[3*h + {0,1,2}] = number of converged,
 * infinity-failed and real (converged, all 30 |imag| <= 1e-4) paths of hypothesis h.  Lets a host driver report the round's
 * statistics without walking 248 bytes per path on the CPU. */
int hcb200_count_solutions(void* stream, int n_hyp, const float* d_tracks, const uint8_t* d_converged, const uint8_t* d_infinity,
                           unsigned int* d_counts);

/* Multi-GPU result exchange, device side.  hcb200_make_pose_record turns the best record of the last score / abort launch on
 * this GPU into the 128-byte exchange record (pose from the track's Cayley parameters, host/mvg.hpp arithmetic; path_offset =
 * 312 * first hypothesis of this GPU's shard; d_found may be NULL).  hcb200_reduce_pose_records reduces n <= 32 gathered records
 * to the round's result: largest min(inliers21, inliers31), lowest global path id among equals. */
int hcb200_make_pose_record(void* stream, const float* d_tracks, const hcb200_best_record* d_best, const uint8_t* d_found,
                            long long path_offset, int rank, hcb200_pose_record* d_out);
int hcb200_reduce_pose_records(void* stream, int n_records, const hcb200_pose_record* d_records, hcb200_pose_record* d_out);

/* Newton refinement of converged end points on the device (next row of SURVEY.md §8f-3; the reference has no such kernel — it is
 * what Evaluations::Find_Unique_Sols, reference Evaluations.cpp:184-233, needs before end points can be compared at
 * DUPLICATE_SOL_DIFF_TOL = 1e-4).  For every path with d_converged[path] != 0: n_iters Newton corrector iterations
 * x -= Hx(x, target)^-1 H(x, target) against the path's TARGET system (hypothesis = path / 312), evaluators and 30x30 solve of the
 * tracker (same arithmetic spec).  d_tracks is updated in place; d_sums[2*path + {0,1}] = sum |dx|^2 and sum |x|^2 of the last
 * iteration (the tracker's convergence test is sum|dx|^2 < 1e-6 sum|x|^2), or -1, -1 for paths that were not refined. */
int hcb200_refine_tracks(void* stream, int n_paths, int n_iters, const float* d_target_params, const uint8_t* d_converged,
                         float* d_tracks, float* d_sums, void* d_workspace);

/* Introspection for benchmarks/tests: registers per thread, static+dynamic shared bytes per CTA, resident CTAs per SM,
 * grid size a launch would use on the current device.  Any pointer may be NULL. */
int hcb200_kernel_info(int abort_variant, int* regs, int* smem_bytes, int* ctas_per_sm, int* grid, int* block);

/* Benchmark helper: enqueue an FP32 FFMA issue-rate probe (16 independent chains per thread, 8 CTAs of 256 threads per
 * SM); *flops_out = floating-point operations performed.  bench.py times it to obtain the measured FP32 peak that the
 * tracker's roofline fraction is quoted against (MEASURED_PEAKS.json has no FP32 entry). */
int hcb200_ffma_probe(void* stream, int iters, float* d_scratch, double* flops_out);

const char* hcb200_error_string(int code);

#ifdef __cplusplus
}
#endif
#endif
