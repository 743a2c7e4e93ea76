/* hc_oracle.h — CPU oracle for the trifocal_2op1p_30x30 homotopy-continuation path tracker.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product library links, loads or calls this.  It may be used by
 * tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs (when oracle/_ref is absent).
 *
 * It is a plain-C restatement of the reference's algorithm for the hot path:
 *   tracker loop .......... magmaHC/gpu-kernels/kernel_GPUHC_trifocal_2op1p_30x30_PH_CodeOpt_TrunPaths.cu:137-286
 *                           (== magmaHC/cpuhc-solvers/CPUHC_Generic_Solver_Eval_by_Indx.cpp:67-172 plus path pruning)
 *   evaluators ............ magmaHC/cpu-jacobian-evals/cpu-eval-indx_trifocal_2op1p_30x30.hpp:22-89
 *                           (== gpu-idx-evals/dev-eval-indxing-trifocal_2op1p_30x30_LimUnroll_L2Cache.cuh:40-148)
 *   linear solve .......... magmaHC/dev-cgesv-batched-small.cuh:38-107 (pivot rule, zero pivot) — see hc_oracle.c
 *   early-abort scoring ... magmaHC/dev-trifocal_2op1p-eval.cuh:28-250
 *   hypothesis sampling ... magmaHC/GPU_HC_Solver.cpp:252-306
 * with ONE fixed floating-point evaluation order ("the arithmetic spec", DESIGN.md §4) that the CUDA kernels follow
 * operation for operation, so kernel and oracle agree bit for bit.  PINNING: the oracle is checked against outputs of the
 * real reference run in the build container (oracle/_ref/libref_cpuhc.so, built from /root/reference; goldens in tests/golden/
 * made by tools/make_golden.py) and against the known answers of SURVEY.md App. C — tests/test_oracle.py.  Unpinned: the
 * arithmetic of MAGMA's complex operators and of OpenBLAS cgesv, whose sources are not part of the reference tree (DESIGN.md §4).
 */
#ifndef HC_ORACLE_H
#define HC_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Problem sizes (gpuhc_settings.yaml: Num_Of_Vars, Num_Of_Params, Num_Of_Tracks, dHdx_Max_Terms, dHdt_Max_Terms).  Defaults: the
 * trifocal problem; `make -C oracle problem_oracle PROBLEM_DIR=…` builds the same source for another problem folder with -D overrides. */
#ifndef HCO_N
#define HCO_N 30          /* variables == equations */
#endif
#ifndef HCO_NP
#define HCO_NP 33         /* parameters (index 33 is the constant-one pad) */
#endif
#ifndef HCO_TRACKS
#define HCO_TRACKS 312
#endif
#ifndef HCO_HX_TERMS
#define HCO_HX_TERMS 8
#endif
#define HCO_HX_PARTS 5
#ifndef HCO_HT_TERMS
#define HCO_HT_TERMS 16
#endif
#define HCO_HT_PARTS 6
#ifndef HCO_NUM_DEPTHS
#define HCO_NUM_DEPTHS 8  /* leading unknowns tested by the positive-depth pruning (…TrunPaths.cu:148-154) */
#endif
#define HCO_TRIFOCAL (HCO_N == 30 && HCO_NP == 33)     /* pose scoring / target parameters from edgels exist for this problem only */

typedef struct { float re, im; } hco_c32;

typedef struct {
  int max_steps;        /* GPUHC_Max_Steps (80) */
  int max_corr_steps;   /* GPUHC_Max_Correction_Steps (3) */
  int dt_inc_steps;     /* GPUHC_Num_Of_Steps_to_Increase_Delta_t (4) */
  int prune;            /* 1: positive-depth path pruning (GPU kernels), 0: none (reference CPU-HC) */
} hco_settings;

typedef struct {          /* per-path counters (for the flop model of SURVEY.md §8d) */
  int32_t steps, pred_stages, corr_stages, rejected, end_reason; /* end_reason: 0 conv, 1 inf, 2 pruned, 3 step cap */
} hco_path_stats;

/* Arithmetic variant of the tracker (all zeros == the spec).  Every variant is the same algorithm with a different, equally
 * valid floating-point evaluation at one point — what the reference's own CPU and GPU implementations do there.  Used only by
 * the per-path parity analysis (tools/parity_envelope.py): a path whose flags differ between any two variants is UNSTABLE. */
typedef struct {
  int solver;         /* 0 spec; 1 literal reference LU + back substitution (dev-cgesv-batched-small.cuh:38-107), no contraction;
                         2 the same with nvcc-style FMA contraction; 3 spec with the reference's exact-maximum pivot rule;
                         4 spec with cuCdivf reciprocal; 5 spec with both */
  int term_order;     /* 0 spec: (coef*p*p) * (x*x*x); 1 left to right as the reference evaluators multiply */
  int contract;       /* with term_order 1: complex products with (1) / without (0) FMA contraction */
  int sum_order;      /* 0 xor butterfly; 1 sequential (reference CPU); 2 reference GPU shuffle-down tree with own-value reads */
  int rk_final_mul;   /* 1: last RK stage multiplies by (float)(1/6) (round-1 spec) instead of dividing by 6.0f (reference) */
  unsigned perturb_seed; /* != 0: every solve result moved by -1/0/+1 ulp pseudo-randomly (stochastic arithmetic) */
} hco_variant;

/* evaluators: x31[30] and p34[33] must hold 1+0i; dHdx has 36000 ints, dHdt 2880 (reference token order) */
void hco_eval_Hx(const int* dHdx, const hco_c32* x31, const hco_c32* p34, hco_c32* A_rowmajor);
void hco_eval_Ht(const int* dHdt, const hco_c32* x31, const hco_c32* p34, const hco_c32* dp34, hco_c32* b30);
void hco_eval_H(const int* dHdt, const hco_c32* x31, const hco_c32* p34, hco_c32* b30);
void hco_param_homotopy(float t, const hco_c32* start34, const hco_c32* target34, hco_c32* p34);

/* linear solves: A row-major 30x30 (destroyed), b in / x out.  Return 0, or k+1 if the k-th pivot was exactly zero. */
void hco_recip(const hco_c32* z, hco_c32* out, int n);   /* the spec's 1/z (conj(z) / clamp(|z|^2, 2^-100, 2^100)), element-wise */
int hco_solve(hco_c32* A, hco_c32* b);          /* the spec: partial-pivot elimination, U-solve folded into the sweep */
int hco_solve_lu_ref(hco_c32* A, hco_c32* b);   /* literal dev-cgesv-batched-small.cuh order (LU + back substitution) */

/* one path */
void hco_track_path(const int* dHdx, const int* dHdt, const hco_c32* start_sol31, const hco_c32* start_params34,
                    const hco_c32* target34, const hco_c32* diff34, const hco_settings* cfg,
                    hco_c32* out_track31, uint8_t* out_converged, uint8_t* out_infinity, hco_path_stats* out_stats);

/* n_hyp * 312 paths, OpenMP over paths; tracks[n_hyp*312][31] out; stats may be NULL */
void hco_track_batch(const int* dHdx, const int* dHdt, const hco_c32* start_sols /*[312][31]*/,
                     const hco_c32* start_params34, const hco_c32* target /*[n_hyp][34]*/, const hco_c32* diff,
                     int n_hyp, const hco_settings* cfg, int n_threads,
                     hco_c32* tracks, uint8_t* converged, uint8_t* infinity, hco_path_stats* stats);

/* the same under an arithmetic variant (NULL == spec); path_key seeds the perturbation stream of this path */
void hco_track_path_v(const int* dHdx, const int* dHdt, const hco_c32* start_sol31, const hco_c32* start_params34,
                      const hco_c32* target34, const hco_c32* diff34, const hco_settings* cfg, const hco_variant* v, uint32_t path_key,
                      hco_c32* out_track31, uint8_t* out_converged, uint8_t* out_infinity, hco_path_stats* out_stats);
void hco_track_batch_v(const int* dHdx, const int* dHdt, const hco_c32* start_sols, const hco_c32* start_params34,
                       const hco_c32* target, const hco_c32* diff, int n_hyp, const hco_settings* cfg, const hco_variant* v, int n_threads,
                       hco_c32* tracks, uint8_t* converged, uint8_t* infinity, hco_path_stats* stats);

/* one path as hco_track_path, with a per-step trace (test helper): for each of the first `cap` steps the path attempts, t0 at the start of
 * the step, the delta_t the step uses after the end-zone / 0.95 clamps, and 1 if the step was accepted (0 if rejected or if the step
 * ended the path at infinity).  Returns the number of steps recorded (min(steps, cap)). */
int hco_trace_path(const int* dHdx, const int* dHdt, const hco_c32* start_sol31, const hco_c32* start_params34,
                   const hco_c32* target34, const hco_c32* diff34, const hco_settings* cfg, int cap, float* t0, float* delta_t,
                   uint8_t* accepted, hco_c32* out_track31, uint8_t* out_converged, uint8_t* out_infinity, hco_path_stats* out_stats);

/* early-abort scoring of one end point: returns 1 if the solution passes (>= 90 % inliers in both view pairs);
 * n21/n31 receive the inlier counts (0 when the imaginary-part gate fails, gate_out tells). */
int hco_score_solution(const hco_c32* x31, const float* edgel_locations /*[E][6]*/, int n_edgels, const float* K9,
                       int* n21, int* n31, int* gate_out);

/* hypothesis sampler + target parameters (glibc srand/rand stream, GPU-major order == plain order) */
void hco_prepare_target_params(unsigned seed, int n_hyp, int n_edgels, const float* locations, const float* tangents,
                               const hco_c32* start_params34, hco_c32* target, hco_c32* diff, int* picked /*[n_hyp][3]*/);

/* Newton refinement in double precision of an end point against the TARGET system (t = 1); used by tests to compare
 * end points "within 1e-4 relative after Newton refinement".  Returns the final residual norm. */
double hco_newton_refine_f64(const int* dHdx, const int* dHdt, const hco_c32* target34, const hco_c32* x31_in,
                             int iters, double* x_out_re_im /*[30][2]*/);

/* Newton refinement in float, in the arithmetic spec (the oracle of hcb200_refine_tracks): `iters` corrector iterations against the
 * target system; x31 in/out; sums = sum|dx|^2, sum|x|^2 of the last iteration (-1 when iters == 0). */
void hco_refine_path(const int* dHdx, const int* dHdt, const hco_c32* target34, hco_c32* x31, int iters, float* out_sum_d, float* out_sum_x);

#ifdef __cplusplus
}
#endif
#endif
