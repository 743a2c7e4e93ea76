/* hc_oracle.c — see hc_oracle.h.  TEST INFRASTRUCTURE ONLY (never linked into the product).
 *
 * Build: gcc -std=c11 -O2 -march=x86-64-v3 -ffp-contract=off -fno-fast-math -fopenmp -fPIC -shared hc_oracle.c -lm
 * -ffp-contract=off matters: every fused multiply-add below is an explicit fmaf(), every other operation is
 * individually rounded (IEEE-754 binary32, round to nearest even, denormals kept) — the same contract the CUDA
 * kernels are compiled under (-fmad=false + explicit fmaf, -prec-div=true, -prec-sqrt=true, -ftz=false).
 */
#include "hc_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* ------------------------------------------------------------------------------------------------------------
 * complex helpers (the arithmetic spec)
 * MAGMA's operator* is (ar*br - ai*bi, ai*br + ar*bi) (SURVEY.md §8c-4); the spec fixes where the single FMA sits. */
static inline hco_c32 c_make(float re, float im) { hco_c32 z; z.re = re; z.im = im; return z; }
static inline hco_c32 c_mul(hco_c32 a, hco_c32 b)
{ return c_make(fmaf(a.re, b.re, -(a.im * b.im)), fmaf(a.re, b.im, a.im * b.re)); }
static inline hco_c32 c_add(hco_c32 a, hco_c32 b) { return c_make(a.re + b.re, a.im + b.im); }
static inline hco_c32 c_sub(hco_c32 a, hco_c32 b) { return c_make(a.re - b.re, a.im - b.im); }
static inline hco_c32 c_scale(float s, hco_c32 a) { return c_make(s * a.re, s * a.im); }
/* acc - m*u, four dependent FMAs */
static inline hco_c32 c_msub(hco_c32 acc, hco_c32 m, hco_c32 u)
{
  float re = fmaf(-m.re, u.re, acc.re); re = fmaf(m.im, u.im, re);
  float im = fmaf(-m.re, u.im, acc.im); im = fmaf(-m.im, u.re, im);
  return c_make(re, im);
}
/* 1/z = conj(z) / |z|^2 with ONE IEEE reciprocal.  The reference divides with cuCdivf (MAGMA_C_DIV,
 * dev-cgesv-batched-small.cuh:84), which pre-scales by |re|+|im|; here |z|^2 is clamped to [2^-100, 2^100] instead
 * (|pivot| in [9e-16, 1e15] — a pivot outside that range means a numerically singular or overflowed system), which keeps the
 * reciprocal's argument in the range where the device's MUFU.RCP + one FMA-Newton step is the correctly rounded 1/d. */
static inline hco_c32 c_recip(hco_c32 z)
{
  float d = fmaf(z.re, z.re, z.im * z.im);
  d = fminf(fmaxf(d, 0x1p-100f), 0x1p100f);
  float q = 1.0f / d;
  return c_make(z.re * q, -(z.im * q));
}
void hco_recip(const hco_c32* z, hco_c32* out, int n) { for (int i = 0; i < n; i++) out[i] = c_recip(z[i]); }
static inline uint32_t f_bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
/* pivot key as the device sees it: NaN is the canonical 0x7fffffff */
static inline uint32_t key_bits(float f) { return (f != f) ? 0x7fffffffu : f_bits(f); }

/* ------------------------------------------------------------------------------------------------------------
 * evaluators — restatement of cpu-eval-indx_trifocal_2op1p_30x30.hpp:22-89: every entry is the sum, in table order, of
 *     coef * p[a] * p[b] * x[d] * x[e] (* x[f])
 * The reference multiplies left to right; the spec groups each term as  (coef * p[a]*p[b]) * (x[d]*x[e]*x[f])  — the
 * parameter part and the variable part are formed separately (each left to right) and multiplied once, so that an
 * implementation can share both parts between rows.  Padded factors: p[33] == 1 is multiplied like any parameter (p is
 * always finite, so that is exact); trailing padded x factors (index 30) are skipped, an all-padded variable part is 1.
 * Table index: Hx (col*40 + term*5 + part)*30 + row ; Ht/H (term*6 + part)*30 + row  (SURVEY.md App. A.3). */
void hco_param_homotopy(float t, const hco_c32* start34, const hco_c32* target34, hco_c32* p34)
{
  /* CPU_HC_Solver.hpp:102-106 / …L2Cache.cuh:40-54: target*t + start*(1.0-t); (1.0-t) rounds once to float */
  float omt = 1.0f - t;
  for (int i = 0; i < HCO_NP; i++) {
    p34[i].re = fmaf(target34[i].re, t, start34[i].re * omt);
    p34[i].im = fmaf(target34[i].im, t, start34[i].im * omt);
  }
  p34[HCO_NP] = c_make(1.0f, 0.0f);
}

static inline hco_c32 coef_pp(int coef, hco_c32 pa, hco_c32 pb)   /* coef * p[a] * p[b] */
{ return c_scale((float)coef, c_mul(pa, pb)); }

static inline hco_c32 x_product(const hco_c32* x, int d, int e, int f)   /* x[d]*x[e]*x[f], padded factors (30) are trailing */
{
  if (d == HCO_N) return c_make(1.0f, 0.0f);
  if (e == HCO_N) return x[d];
  hco_c32 v = c_mul(x[d], x[e]);
  if (f == HCO_N) return v;
  return c_mul(v, x[f]);
}

void hco_eval_Hx(const int* dHdx, const hco_c32* x, const hco_c32* p, hco_c32* A)
{
  for (int row = 0; row < HCO_N; row++)
    for (int col = 0; col < HCO_N; col++) {
      hco_c32 acc = c_make(0.0f, 0.0f);
      for (int j = 0; j < HCO_HX_TERMS; j++) {
        const int base = (col * HCO_HX_TERMS * HCO_HX_PARTS + j * HCO_HX_PARTS) * HCO_N + row;
        int coef = dHdx[base];
        if (coef == 0) continue;                               /* adds an exact +0 in the reference */
        hco_c32 cq = coef_pp(coef, p[dHdx[base + 1 * HCO_N]], p[dHdx[base + 2 * HCO_N]]);
        hco_c32 xp = x_product(x, dHdx[base + 3 * HCO_N], dHdx[base + 4 * HCO_N], HCO_N);
        acc = c_add(acc, c_mul(cq, xp));
      }
      A[row * HCO_N + col] = acc;
    }
}

void hco_eval_H(const int* dHdt, const hco_c32* x, const hco_c32* p, hco_c32* b)
{
  for (int row = 0; row < HCO_N; row++) {
    hco_c32 acc = c_make(0.0f, 0.0f);
    for (int j = 0; j < HCO_HT_TERMS; j++) {
      const int base = (j * HCO_HT_PARTS) * HCO_N + row;
      int coef = dHdt[base];
      if (coef == 0) continue;
      hco_c32 cq = coef_pp(coef, p[dHdt[base + 1 * HCO_N]], p[dHdt[base + 2 * HCO_N]]);
      hco_c32 xp = x_product(x, dHdt[base + 3 * HCO_N], dHdt[base + 4 * HCO_N], dHdt[base + 5 * HCO_N]);
      acc = c_add(acc, c_mul(cq, xp));
    }
    b[row] = acc;
  }
}

void hco_eval_Ht(const int* dHdt, const hco_c32* x, const hco_c32* p, const hco_c32* dp, hco_c32* b)
{
  for (int row = 0; row < HCO_N; row++) {
    hco_c32 acc = c_make(0.0f, 0.0f);
    for (int j = 0; j < HCO_HT_TERMS; j++) {
      const int base = (j * HCO_HT_PARTS) * HCO_N + row;
      int coef = dHdt[base];
      int ia = dHdt[base + 1 * HCO_N], ib = dHdt[base + 2 * HCO_N];
      if (coef == 0) continue;
      if (ia == HCO_NP && ib == HCO_NP) continue;              /* dp[33] == 0: the term is an exact 0 */
      hco_c32 s = c_add(c_mul(dp[ia], p[ib]), c_mul(dp[ib], p[ia]));
      hco_c32 dq = c_scale((float)coef, s);
      hco_c32 xp = x_product(x, dHdt[base + 3 * HCO_N], dHdt[base + 4 * HCO_N], dHdt[base + 5 * HCO_N]);
      acc = c_sub(acc, c_mul(dq, xp));                         /* r_cgesvB -= … (…L2Cache.cuh:110) */
    }
    b[row] = acc;
  }
}

/* ------------------------------------------------------------------------------------------------------------
 * linear solve — the spec.
 * Partial-pivot elimination in natural column order with the pivot key of dev-cgesv-batched-small.cuh:55-65 (|re|+|im|),
 * multipliers = row entry times the pivot's reciprocal (:84-86) and the same rank-1 updates (:87-93), re-organised as
 * Gauss-Jordan: rows that were already pivoted are swept too, which performs the U-solve (:97-106) inside the same 30
 * steps; x_k = b_pivot(k) * (1/pivot_k).  Three rules make the result independent of HOW a (block-parallel) implementation
 * schedules the steps:
 *   - the pivot is the row with the largest key after the key's five lowest mantissa bits are replaced by (31 - row index):
 *     i.e. the largest |re|+|im| to within 2^-18 relative, lowest row index among (near-)ties — one integer maximum finds
 *     the row.  (The reference takes the first exact maximum in its current, virtually permuted row order, :57-65.);
 *   - a row whose entry in the pivot column is exactly zero is not touched (its multiplier would be 0);
 *   - a pivot column whose candidates are all exactly zero makes the system singular: every component of the result is NaN
 *     (the reference continues with a multiplier of 1 and later divides by the zero diagonal, :66-68,100). */
int hco_solve(hco_c32* A, hco_c32* b)
{
  int done[HCO_N], piv[HCO_N];
  hco_c32 rsave[HCO_N];
  for (int i = 0; i < HCO_N; i++) done[i] = 0;
  for (int k = 0; k < HCO_N; k++) {
    uint32_t maxkey = 0;
    int p = -1;
    for (int i = 0; i < HCO_N; i++) {
      if (done[i]) continue;
      const uint32_t key = (key_bits(fabsf(A[i * HCO_N + k].re) + fabsf(A[i * HCO_N + k].im)) & ~31u) | (uint32_t)(31 - i);
      if (key > maxkey) { maxkey = key; p = i; }
    }
    if (maxkey < 32u) {                                  /* every candidate is (within 2^-144 of) zero */
      for (int i = 0; i < HCO_N; i++) b[i] = c_make(NAN, NAN);
      return k + 1;
    }
    done[p] = 1; piv[k] = p;
    const hco_c32 r = c_recip(A[p * HCO_N + k]);
    rsave[p] = r;
    for (int i = 0; i < HCO_N; i++) {
      if (i == p) continue;
      if (A[i * HCO_N + k].re == 0.0f && A[i * HCO_N + k].im == 0.0f) continue;
      const hco_c32 m = c_mul(A[i * HCO_N + k], r);
      for (int j = k + 1; j < HCO_N; j++)
        A[i * HCO_N + j] = c_msub(A[i * HCO_N + j], m, A[p * HCO_N + j]);
      b[i] = c_msub(b[i], m, b[p]);
    }
  }
  hco_c32 x[HCO_N];
  for (int k = 0; k < HCO_N; k++) x[k] = c_mul(b[piv[k]], rsave[piv[k]]);
  memcpy(b, x, sizeof x);
  return 0;
}

/* Literal operation order of cgesv_batched_small_device<30> (dev-cgesv-batched-small.cuh:38-107), kept to show that
 * the spec above solves the same systems to rounding (tests/test_oracle.py).  cuCdivf is restated from cuComplex.h. */
static inline hco_c32 c_div_cu(hco_c32 x, hco_c32 y)
{
  float s = fabsf(y.re) + fabsf(y.im);
  float oos = 1.0f / s;
  float ars = x.re * oos, ais = x.im * oos, brs = y.re * oos, bis = y.im * oos;
  s = (brs * brs) + (bis * bis);
  oos = 1.0f / s;
  return c_make(((ars * brs) + (ais * bis)) * oos, ((ais * brs) - (ars * bis)) * oos);
}
static inline hco_c32 c_mul_plain(hco_c32 a, hco_c32 b)
{ return c_make(a.re * b.re - a.im * b.im, a.im * b.re + a.re * b.im); }

int hco_solve_lu_ref(hco_c32* A, hco_c32* b)
{
  int rowid[HCO_N], info = 0;
  hco_c32 sx[HCO_N], sB[HCO_N];
  float dsx[HCO_N];
  for (int i = 0; i < HCO_N; i++) rowid[i] = i;
  for (int i = 0; i < HCO_N; i++) {
    for (int t = 0; t < HCO_N; t++) dsx[rowid[t]] = fabsf(A[t * HCO_N + i].re) + fabsf(A[t * HCO_N + i].im);
    float mx = dsx[i]; int max_id = i;
    for (int j = i + 1; j < HCO_N; j++) if (dsx[j] > mx) { max_id = j; mx = dsx[j]; }
    int zero = (mx == 0.0f);
    if (zero && !info) info = i + 1;
    float update = zero ? 0.0f : 1.0f;
    hco_c32 sB0 = c_make(0, 0);
    for (int t = 0; t < HCO_N; t++) {
      if (rowid[t] == max_id) {
        rowid[t] = i;
        for (int j = i; j < HCO_N; j++) sx[j] = c_scale(update, A[t * HCO_N + j]);
        sB0 = b[t];
      } else if (rowid[t] == i) rowid[t] = max_id;
    }
    hco_c32 reg = zero ? c_make(1, 0) : c_div_cu(c_make(1, 0), sx[i]);
    for (int t = 0; t < HCO_N; t++) {
      if (rowid[t] > i) {
        A[t * HCO_N + i] = c_mul_plain(A[t * HCO_N + i], reg);
        for (int j = i + 1; j < HCO_N; j++)
          A[t * HCO_N + j] = c_sub(A[t * HCO_N + j], c_mul_plain(A[t * HCO_N + i], sx[j]));
        b[t] = c_sub(b[t], c_mul_plain(A[t * HCO_N + i], sB0));
      }
    }
  }
  for (int t = 0; t < HCO_N; t++) sB[rowid[t]] = b[t];
  for (int i = HCO_N - 1; i >= 0; i--) {
    for (int t = 0; t < HCO_N; t++) sx[rowid[t]] = A[t * HCO_N + i];
    hco_c32 reg = c_div_cu(sB[i], sx[i]);
    for (int t = 0; t < i; t++) sB[t] = c_sub(sB[t], c_mul_plain(reg, sx[t]));
    sB[i] = reg;
  }
  memcpy(b, sB, sizeof sB);
  return info;
}

/* ------------------------------------------------------------------------------------------------------------
 * warp-order sum of 30 per-row values (the kernel adds lanes 30,31 as zeros in an xor butterfly 16,8,4,2,1;
 * the reference's shuffle-down tree is …TrunPaths.cu:236-239) */
static float butterfly_sum(const float* v30)
{
  float v[32];
  for (int i = 0; i < 32; i++) v[i] = i < HCO_N ? v30[i] : 0.0f;
  for (int off = 16; off > 0; off >>= 1) {
    float w[32];
    for (int i = 0; i < 32; i++) w[i] = v[i] + v[i ^ off];
    memcpy(v, w, sizeof v);
  }
  return v[0];
}

/* ------------------------------------------------------------------------------------------------------------
 * ARITHMETIC VARIANTS (hco_variant, hc_oracle.h) — equally valid floating-point evaluations of the SAME algorithm, used only to
 * measure how far rounding alone moves the integer results (tools/parity_envelope.py, tests/test_parity_envelope.py).  Variant 0
 * everywhere is the spec above; the others restate what the reference's own two implementations do at that point. */
static inline hco_c32 c_mul_v(hco_c32 a, hco_c32 b, int contract)      /* MAGMA operator*: (ar*br - ai*bi, ai*br + ar*bi) */
{
  if (contract) return c_make(fmaf(a.re, b.re, -(a.im * b.im)), fmaf(a.im, b.re, a.re * b.im));   /* nvcc / gcc -ffp-contract=fast */
  return c_make(a.re * b.re - a.im * b.im, a.im * b.re + a.re * b.im);
}
/* term = coef * p[a] * p[b] * x[d] * x[e] (* x[f]) multiplied LEFT TO RIGHT, padded factors (== 1+0i) included, exactly as
 * cpu-eval-indx_trifocal_2op1p_30x30.hpp:22-89 / …L2Cache.cuh:57-148 do (the integer coefficient enters as a real scale) */
static void eval_Hx_ltr(const int* dHdx, const hco_c32* x, const hco_c32* p, hco_c32* A, int contract)
{
  for (int row = 0; row < HCO_N; row++)
    for (int col = 0; col < HCO_N; col++) {
      hco_c32 acc = c_make(0.0f, 0.0f);
      for (int j = 0; j < HCO_HX_TERMS; j++) {
        const int base = (col * HCO_HX_TERMS * HCO_HX_PARTS + j * HCO_HX_PARTS) * HCO_N + row;
        hco_c32 t = c_scale((float)dHdx[base], p[dHdx[base + 1 * HCO_N]]);
        t = c_mul_v(t, p[dHdx[base + 2 * HCO_N]], contract);
        t = c_mul_v(t, x[dHdx[base + 3 * HCO_N]], contract);
        t = c_mul_v(t, x[dHdx[base + 4 * HCO_N]], contract);
        acc = c_add(acc, t);
      }
      A[row * HCO_N + col] = acc;
    }
}
static void eval_H_ltr(const int* dHdt, const hco_c32* x, const hco_c32* p, hco_c32* b, int contract)
{
  for (int row = 0; row < HCO_N; row++) {
    hco_c32 acc = c_make(0.0f, 0.0f);
    for (int j = 0; j < HCO_HT_TERMS; j++) {
      const int base = (j * HCO_HT_PARTS) * HCO_N + row;
      hco_c32 t = c_scale((float)dHdt[base], p[dHdt[base + 1 * HCO_N]]);
      t = c_mul_v(t, p[dHdt[base + 2 * HCO_N]], contract);
      t = c_mul_v(t, x[dHdt[base + 3 * HCO_N]], contract);
      t = c_mul_v(t, x[dHdt[base + 4 * HCO_N]], contract);
      t = c_mul_v(t, x[dHdt[base + 5 * HCO_N]], contract);
      acc = c_add(acc, t);
    }
    b[row] = acc;
  }
}
static void eval_Ht_ltr(const int* dHdt, const hco_c32* x, const hco_c32* p, const hco_c32* dp, hco_c32* b, int contract)
{
  for (int row = 0; row < HCO_N; row++) {
    hco_c32 acc = c_make(0.0f, 0.0f);
    for (int j = 0; j < HCO_HT_TERMS; j++) {
      const int base = (j * HCO_HT_PARTS) * HCO_N + row;
      const int ia = dHdt[base + 1 * HCO_N], ib = dHdt[base + 2 * HCO_N];
      /* …L2Cache.cuh:110-116: coef * (dp[a]*p[b] + dp[b]*p[a]) * x * x * x */
      hco_c32 t = c_scale((float)dHdt[base], c_add(c_mul_v(dp[ia], p[ib], contract), c_mul_v(dp[ib], p[ia], contract)));
      t = c_mul_v(t, x[dHdt[base + 3 * HCO_N]], contract);
      t = c_mul_v(t, x[dHdt[base + 4 * HCO_N]], contract);
      t = c_mul_v(t, x[dHdt[base + 5 * HCO_N]], contract);
      acc = c_sub(acc, t);
    }
    b[row] = acc;
  }
}

/* the spec's elimination with the reference's pivot rule (exact |re|+|im| maximum, first one in row order wins) and/or the
 * reference's division (cuCdivf scaling) for 1/pivot */
static int solve_gj_variant(hco_c32* A, hco_c32* b, int exact_key, int cudiv_recip)
{
  int done[HCO_N], piv[HCO_N];
  hco_c32 rsave[HCO_N];
  for (int i = 0; i < HCO_N; i++) done[i] = 0;
  for (int k = 0; k < HCO_N; k++) {
    int p = -1;
    if (exact_key) {
      float best = -1.0f;
      for (int i = 0; i < HCO_N; i++) {
        if (done[i]) continue;
        float v = fabsf(A[i * HCO_N + k].re) + fabsf(A[i * HCO_N + k].im);
        if (v != v) v = INFINITY;
        if (v > best) { best = v; p = i; }
      }
      if (!(best > 0.0f)) { for (int i = 0; i < HCO_N; i++) b[i] = c_make(NAN, NAN); return k + 1; }
    } else {
      uint32_t maxkey = 0;
      for (int i = 0; i < HCO_N; i++) {
        if (done[i]) continue;
        const uint32_t key = (key_bits(fabsf(A[i * HCO_N + k].re) + fabsf(A[i * HCO_N + k].im)) & ~31u) | (uint32_t)(31 - i);
        if (key > maxkey) { maxkey = key; p = i; }
      }
      if (maxkey < 32u) { for (int i = 0; i < HCO_N; i++) b[i] = c_make(NAN, NAN); return k + 1; }
    }
    done[p] = 1; piv[k] = p;
    const hco_c32 r = cudiv_recip ? c_div_cu(c_make(1.0f, 0.0f), A[p * HCO_N + k]) : c_recip(A[p * HCO_N + k]);
    rsave[p] = r;
    for (int i = 0; i < HCO_N; i++) {
      if (i == p) continue;
      if (A[i * HCO_N + k].re == 0.0f && A[i * HCO_N + k].im == 0.0f) continue;
      const hco_c32 m = c_mul(A[i * HCO_N + k], r);
      for (int j = k + 1; j < HCO_N; j++) A[i * HCO_N + j] = c_msub(A[i * HCO_N + j], m, A[p * HCO_N + j]);
      b[i] = c_msub(b[i], m, b[p]);
    }
  }
  hco_c32 x[HCO_N];
  for (int k = 0; k < HCO_N; k++) x[k] = c_mul(b[piv[k]], rsave[piv[k]]);
  memcpy(b, x, sizeof x);
  return 0;
}

/* literal reference LU (hco_solve_lu_ref) with the multiply-adds contracted the way nvcc -O3 (fmad on) compiles
 * dev-cgesv-batched-small.cuh:84-106: a - m*u  ->  re = fma(-m.re,u.re, fma(m.im,u.im,a.re)) … */
static inline hco_c32 c_msub_contract(hco_c32 a, hco_c32 m, hco_c32 u)
{
  const hco_c32 t = c_make(fmaf(m.re, u.re, -(m.im * u.im)), fmaf(m.im, u.re, m.re * u.im));
  return c_make(a.re - t.re, a.im - t.im);
}
static int solve_lu_ref_contract(hco_c32* A, hco_c32* b)
{
  int rowid[HCO_N], info = 0;
  hco_c32 sx[HCO_N], sB[HCO_N];
  float dsx[HCO_N];
  for (int i = 0; i < HCO_N; i++) rowid[i] = i;
  for (int i = 0; i < HCO_N; i++) {
    for (int t = 0; t < HCO_N; t++) dsx[rowid[t]] = fabsf(A[t * HCO_N + i].re) + fabsf(A[t * HCO_N + i].im);
    float mx = dsx[i]; int max_id = i;
    for (int j = i + 1; j < HCO_N; j++) if (dsx[j] > mx) { max_id = j; mx = dsx[j]; }
    int zero = (mx == 0.0f);
    if (zero && !info) info = i + 1;
    float update = zero ? 0.0f : 1.0f;
    hco_c32 sB0 = c_make(0, 0);
    for (int t = 0; t < HCO_N; t++) {
      if (rowid[t] == max_id) {
        rowid[t] = i;
        for (int j = i; j < HCO_N; j++) sx[j] = c_scale(update, A[t * HCO_N + j]);
        sB0 = b[t];
      } else if (rowid[t] == i) rowid[t] = max_id;
    }
    hco_c32 reg = zero ? c_make(1, 0) : c_div_cu(c_make(1, 0), sx[i]);
    for (int t = 0; t < HCO_N; t++) {
      if (rowid[t] > i) {
        A[t * HCO_N + i] = c_mul_v(A[t * HCO_N + i], reg, 1);
        for (int j = i + 1; j < HCO_N; j++) A[t * HCO_N + j] = c_msub_contract(A[t * HCO_N + j], A[t * HCO_N + i], sx[j]);
        b[t] = c_msub_contract(b[t], A[t * HCO_N + i], sB0);
      }
    }
  }
  for (int t = 0; t < HCO_N; t++) sB[rowid[t]] = b[t];
  for (int i = HCO_N - 1; i >= 0; i--) {
    for (int t = 0; t < HCO_N; t++) sx[rowid[t]] = A[t * HCO_N + i];
    hco_c32 reg = c_div_cu(sB[i], sx[i]);
    for (int t = 0; t < i; t++) sB[t] = c_msub_contract(sB[t], reg, sx[t]);
    sB[i] = reg;
  }
  memcpy(b, sB, sizeof sB);
  return info;
}

static void solve_variant(const hco_variant* v, hco_c32* A, hco_c32* b)
{
  switch (v ? v->solver : 0) {
    case 1: hco_solve_lu_ref(A, b); break;
    case 2: solve_lu_ref_contract(A, b); break;
    case 3: solve_gj_variant(A, b, 1, 0); break;
    case 4: solve_gj_variant(A, b, 0, 1); break;
    case 5: solve_gj_variant(A, b, 1, 1); break;
    default: hco_solve(A, b);
  }
}

/* norm sums.  0: the spec's xor butterfly (== the reference GPU's shuffle-down tree as lane 0 sees it when the two lanes that
 * do not exist contribute 0); 1: sequential i = 0..29 (reference CPU-HC, CPUHC_make_correction); 2: the reference GPU's
 * shuffle-down tree when a shuffle from a lane that does not exist returns the CALLER's own value (lanes 14 and 15 count twice
 * at offset 16, …TrunPaths.cu:236-239; which of 0 / 2 the hardware does is measured by tools/probes.cu) */
static float sum_variant(const hco_variant* v, const float* v30)
{
  const int mode = v ? v->sum_order : 0;
  if (mode == 1) { float s = 0.0f; for (int i = 0; i < HCO_N; i++) s += v30[i]; return s; }
  if (mode == 2) {
    float a[32];
    for (int i = 0; i < 32; i++) a[i] = i < HCO_N ? v30[i] : 0.0f;
    for (int off = 16; off > 0; off >>= 1) {
      float w[32];
      for (int i = 0; i < HCO_N; i++) { const int src = i + off; w[i] = a[i] + ((src < HCO_N) ? a[src] : a[i]); }
      for (int i = 0; i < HCO_N; i++) a[i] = w[i];
    }
    return a[0];
  }
  return butterfly_sum(v30);
}

/* stochastic-arithmetic variants: every component of every solve result is moved by -1 / 0 / +1 ulp, pseudo-randomly but
 * reproducibly (counter-based hash of seed, path, solve number, component).  A perturbation of one unit in the last place of
 * the linear-solve result is far below the solve's own backward error, so each seed is another legitimate rounding of the path. */
static inline uint32_t mix32(uint32_t x) { x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16; return x; }
static inline float ulp_nudge(float f, uint32_t r)
{
  if (!(f == f) || isinf(f) || f == 0.0f) return f;
  const uint32_t k = r % 3u;           /* 0: keep, 1: up, 2: down */
  if (k == 0) return f;
  return nextafterf(f, k == 1 ? INFINITY : -INFINITY);
}
static void perturb_solution(const hco_variant* v, uint32_t path_key, uint32_t solve_no, hco_c32* b)
{
  if (!v || !v->perturb_seed) return;
  for (int i = 0; i < HCO_N; i++) {
    const uint32_t r = mix32(v->perturb_seed * 0x9e3779b9u ^ mix32(path_key * 0x85ebca6bu ^ mix32(solve_no * 64u + (uint32_t)i)));
    b[i].re = ulp_nudge(b[i].re, r);
    b[i].im = ulp_nudge(b[i].im, r >> 8);
  }
}

typedef struct { float* t0; float* delta_t; uint8_t* accepted; int cap, n; } step_trace;   /* hco_trace_path */

/* ------------------------------------------------------------------------------------------------------------
 * one path: …TrunPaths.cu:80-286 (SURVEY.md App. B), cfg->prune == 0 gives CPUHC_Generic_Solver_Eval_by_Indx.cpp:67-172 */
static void track_path(const int* dHdx, const int* dHdt, const hco_c32* start_sol31, const hco_c32* sp,
                       const hco_c32* tp, const hco_c32* dp, const hco_settings* cfg, const hco_variant* v, uint32_t path_key,
                       hco_c32* out_track31, uint8_t* out_conv, uint8_t* out_inf, hco_path_stats* st, step_trace* trace)
{
  const int ltr = v ? v->term_order : 0, contract = v ? v->contract : 0;
  uint32_t solve_no = 0;
  hco_c32 x[HCO_N + 1], last[HCO_N], sols[HCO_N], p[HCO_NP + 1], A[HCO_N * HCO_N], b[HCO_N];
  for (int i = 0; i < HCO_N; i++) x[i] = last[i] = sols[i] = start_sol31[i];
  x[HCO_N] = c_make(1.0f, 0.0f);
  float t0 = 0.0f, t_step = 0.0f, delta_t = 0.01f;
  int end_zone = 0, counter = 0, ok = 0, inf_fail = 0, check_depths = 1;
  hco_path_stats s = {0, 0, 0, 0, 3};
  static const float c6[3] = {(float)(1.0 / 6.0), (float)(2.0 / 6.0), (float)(2.0 / 6.0)};   /* …TrunPaths.cu:193 */

  for (int step = 0; step <= cfg->max_steps; step++) {
    if (!((double)t0 < 1.0 && (1.0 - (double)t0 > 0.0000001))) { s.end_reason = 0; break; }        /* :139 */
    if (!end_zone && (double)fabsf(1.0f - t0) <= 0.0500001) end_zone = 1;                            /* :144-146 */
    if (cfg->prune) {                                                                               /* :148-154 */
      if (check_depths) {
        int all_pos = 1;
        for (int i = 0; i < HCO_NUM_DEPTHS; i++) all_pos &= (x[i].re > 0.0f);
        if (t0 > 0.0f) check_depths = all_pos ? 0 : 1;
      }
      if ((double)t0 > 0.95 && check_depths) { s.end_reason = 2; break; }
    }
    if (end_zone) { float r = fabsf(1.0f - t0); if (delta_t > r) delta_t = r; }                      /* :156-162 */
    else { double r = fabs(0.95 - (double)t0); if ((double)delta_t > r) delta_t = (float)r; }
    t_step = t0;
    const float half = 0.5f * delta_t;
    s.steps++;
    if (trace && trace->n < trace->cap) { trace->t0[trace->n] = t0; trace->delta_t[trace->n] = delta_t; trace->accepted[trace->n++] = 0; }

    /* RK4 predictor, "loopy" form (:170-211) */
    for (int r = 0; r < 4; r++) {
      hco_param_homotopy(t0, sp, tp, p);
      if (ltr) { eval_Hx_ltr(dHdx, x, p, A, contract); eval_Ht_ltr(dHdt, x, p, dp, b, contract); }
      else { hco_eval_Hx(dHdx, x, p, A); hco_eval_Ht(dHdt, x, p, dp, b); }
      solve_variant(v, A, b);
      perturb_solution(v, path_key, solve_no++, b);
      s.pred_stages++;
      if (r < 3) {
        const float sc = (r < 2) ? half : delta_t;
        for (int i = 0; i < HCO_N; i++) {
          sols[i].re = fmaf(b[i].re * delta_t, c6[r], sols[i].re);
          sols[i].im = fmaf(b[i].im * delta_t, c6[r], sols[i].im);
          x[i].re = fmaf(b[i].re, sc, last[i].re);
          x[i].im = fmaf(b[i].im, sc, last[i].im);
        }
        if (r != 1) t0 += half;
      } else if (v && v->rk_final_mul) {                  /* variant: multiply by (float)(1/6) like the first three stages */
        for (int i = 0; i < HCO_N; i++) {
          sols[i].re = fmaf(b[i].re * delta_t, c6[0], sols[i].re);
          sols[i].im = fmaf(b[i].im * delta_t, c6[0], sols[i].im);
          x[i] = sols[i];
        }
      } else {                                            /* :209  s_sols += sB * delta_t * 1.0/6.0  ==  (sB*delta_t) / 6.0f, IEEE division */
        for (int i = 0; i < HCO_N; i++) {
          sols[i].re = sols[i].re + (b[i].re * delta_t) / 6.0f;
          sols[i].im = sols[i].im + (b[i].im * delta_t) / 6.0f;
          x[i] = sols[i];
        }
      }
    }

    /* Newton corrector (:216-250); the parameter homotopy is NOT re-evaluated */
    for (int c = 0; c < cfg->max_corr_steps; c++) {
      if (ltr) { eval_Hx_ltr(dHdx, x, p, A, contract); eval_H_ltr(dHdt, x, p, b, contract); }
      else { hco_eval_Hx(dHdx, x, p, A); hco_eval_H(dHdt, x, p, b); }
      solve_variant(v, A, b);
      perturb_solution(v, path_key, solve_no++, b);
      s.corr_stages++;
      float vd[HCO_N], vx[HCO_N];
      for (int i = 0; i < HCO_N; i++) {
        x[i] = c_sub(x[i], b[i]);
        vd[i] = fmaf(b[i].re, b[i].re, b[i].im * b[i].im);
        vx[i] = fmaf(x[i].re, x[i].re, x[i].im * x[i].im);
      }
      const float sum_d = sum_variant(v, vd), sum_x = sum_variant(v, vx);
      ok = (double)sum_d < 0.000001 * (double)sum_x;
      inf_fail = (double)sum_x > 1e14;
      if (inf_fail) break;
      if (ok) break;
    }
    if (inf_fail) { s.end_reason = 1; break; }                                                       /* :252 */

    if (!ok) {                                                                                      /* :257-275 */
      delta_t *= 0.5f;
      for (int i = 0; i < HCO_N; i++) x[i] = sols[i] = last[i];
      counter = 0;
      t0 = t_step;
      s.rejected++;
    } else {
      counter++;
      for (int i = 0; i < HCO_N; i++) last[i] = sols[i] = x[i];
      if (counter >= cfg->dt_inc_steps) { counter = 0; delta_t *= 2.0f; }
      if (trace && trace->n == s.steps) trace->accepted[trace->n - 1] = 1;
    }
  }
  const int conv = ((double)t0 >= 1.0 || (1.0 - (double)t0 <= 0.0000001));                           /* :284 */
  if (conv && s.end_reason == 3) s.end_reason = 0;
  memcpy(out_track31, x, sizeof(hco_c32) * (HCO_N + 1));
  *out_conv = (uint8_t)conv;
  *out_inf = (uint8_t)inf_fail;
  if (st) *st = s;
}

void hco_track_path_v(const int* dHdx, const int* dHdt, const hco_c32* start_sol31, const hco_c32* sp,
                      const hco_c32* tp, const hco_c32* dp, const hco_settings* cfg, const hco_variant* v, uint32_t path_key,
                      hco_c32* out_track31, uint8_t* out_conv, uint8_t* out_inf, hco_path_stats* st)
{ track_path(dHdx, dHdt, start_sol31, sp, tp, dp, cfg, v, path_key, out_track31, out_conv, out_inf, st, NULL); }

int hco_trace_path(const int* dHdx, const int* dHdt, const hco_c32* start_sol31, const hco_c32* sp, const hco_c32* tp, const hco_c32* dp,
                   const hco_settings* cfg, int cap, float* t0, float* delta_t, uint8_t* accepted,
                   hco_c32* out_track31, uint8_t* out_conv, uint8_t* out_inf, hco_path_stats* st)
{
  step_trace trace = {t0, delta_t, accepted, cap, 0};
  track_path(dHdx, dHdt, start_sol31, sp, tp, dp, cfg, NULL, 0u, out_track31, out_conv, out_inf, st, &trace);
  return trace.n;
}

void hco_track_path(const int* dHdx, const int* dHdt, const hco_c32* start_sol31, const hco_c32* sp,
                    const hco_c32* tp, const hco_c32* dp, const hco_settings* cfg,
                    hco_c32* out_track31, uint8_t* out_conv, uint8_t* out_inf, hco_path_stats* st)
{ hco_track_path_v(dHdx, dHdt, start_sol31, sp, tp, dp, cfg, NULL, 0u, out_track31, out_conv, out_inf, st); }

void hco_track_batch(const int* dHdx, const int* dHdt, const hco_c32* start_sols, const hco_c32* sp,
                     const hco_c32* target, const hco_c32* diff, int n_hyp, const hco_settings* cfg, int n_threads,
                     hco_c32* tracks, uint8_t* converged, uint8_t* infinity, hco_path_stats* stats)
{ hco_track_batch_v(dHdx, dHdt, start_sols, sp, target, diff, n_hyp, cfg, NULL, n_threads, tracks, converged, infinity, stats); }

void hco_track_batch_v(const int* dHdx, const int* dHdt, const hco_c32* start_sols, const hco_c32* sp,
                       const hco_c32* target, const hco_c32* diff, int n_hyp, const hco_settings* cfg, const hco_variant* v, int n_threads,
                       hco_c32* tracks, uint8_t* converged, uint8_t* infinity, hco_path_stats* stats)
{
  const long n_paths = (long)n_hyp * HCO_TRACKS;
#ifdef _OPENMP
  if (n_threads > 0) omp_set_num_threads(n_threads);
#endif
  #pragma omp parallel for schedule(dynamic, 4)
  for (long ix = 0; ix < n_paths; ix++) {
    const int h = (int)(ix / HCO_TRACKS), s = (int)(ix % HCO_TRACKS);
    hco_track_path_v(dHdx, dHdt, start_sols + (size_t)s * (HCO_N + 1), sp, target + (size_t)h * (HCO_NP + 1),
                     diff + (size_t)h * (HCO_NP + 1), cfg, v, (uint32_t)ix, tracks + (size_t)ix * (HCO_N + 1), converged + ix, infinity + ix,
                     stats ? stats + ix : NULL);
  }
}

#if HCO_TRIFOCAL   /* scoring and hypothesis generation know the meaning of the trifocal unknowns / parameters */
/* ------------------------------------------------------------------------------------------------------------
 * early-abort scoring: dev-trifocal_2op1p-eval.cuh:28-250 with a fixed FMA placement; rnorm3df -> 1/sqrtf,
 * hypotf -> sqrtf (both correctly rounded here and, with -prec-sqrt/-prec-div, on the device). */
static void cayley_to_R(const float r0, const float r1, const float r2, float* R)
{
  const float a00 = r0 * r0, a11 = r1 * r1, a22 = r2 * r2;
  R[0] = (1.0f + a00) - (a11 + a22);
  R[1] = 2.0f * fmaf(r0, r1, -r2);
  R[2] = 2.0f * fmaf(r0, r2, r1);
  R[3] = 2.0f * fmaf(r0, r1, r2);
  R[4] = (1.0f + a11) - (a00 + a22);
  R[5] = 2.0f * fmaf(r1, r2, -r0);
  R[6] = 2.0f * fmaf(r0, r2, -r1);
  R[7] = 2.0f * fmaf(r1, r2, r0);
  R[8] = (1.0f + a22) - (a00 + a11);
  /* :78-91 — column norms applied row-wise, exactly as the reference does */
  const float n0 = 1.0f / sqrtf(fmaf(R[0], R[0], fmaf(R[3], R[3], R[6] * R[6])));
  const float n1 = 1.0f / sqrtf(fmaf(R[1], R[1], fmaf(R[4], R[4], R[7] * R[7])));
  const float n2 = 1.0f / sqrtf(fmaf(R[2], R[2], fmaf(R[5], R[5], R[8] * R[8])));
  R[0] *= n0; R[1] *= n0; R[2] *= n0;
  R[3] *= n1; R[4] *= n1; R[5] *= n1;
  R[6] *= n2; R[7] *= n2; R[8] *= n2;
}

static inline int reproj_inlier(const float* R, const float* T, float g1x, float g1y, float gx, float gy,
                                float B, float fx, float fy, float cx, float cy)
{
  const float A = fmaf(R[2], gx, fmaf(R[5], gy, R[8]));                    /* e3' R' gamma */
  const float numer = fmaf(T[2], A, -B);
  const float C = fmaf(R[6], g1x, fmaf(R[7], g1y, R[8]));                  /* e3' R gamma1 */
  const float denom = fmaf(-C, A, 1.0f);
  const float z = fmaf(numer, C, denom * T[2]);
  const float X = fmaf(numer, fmaf(R[0], g1x, fmaf(R[1], g1y, R[2])), denom * T[0]) / z;
  const float Y = fmaf(numer, fmaf(R[3], g1x, fmaf(R[4], g1y, R[5])), denom * T[1]) / z;
  const float ex = fmaf(X, fx, cx) - fmaf(gx, fx, cx);
  const float ey = fmaf(Y, fy, cy) - fmaf(gy, fy, cy);
  return sqrtf(fmaf(ex, ex, ey * ey)) < 2.0f;                              /* REPROJ_ERROR_INLIER_THRESH */
}

int hco_score_solution(const hco_c32* x, const float* loc, int n_edgels, const float* K, int* n21, int* n31, int* gate_out)
{
  int gate = 1;
  for (int i = 18; i < 30; i++) gate &= ((double)fabsf(x[i].im) < 1e-5);   /* IMAG_PART_TOL, :41-54 */
  if (gate_out) *gate_out = gate;
  *n21 = 0; *n31 = 0;
  if (!gate) return 0;
  float R21[9], R31[9], T21[3], T31[3];
  cayley_to_R(x[24].re, x[25].re, x[26].re, R21);
  cayley_to_R(x[27].re, x[28].re, x[29].re, R31);
  for (int i = 0; i < 3; i++) { T21[i] = x[18 + i].re; T31[i] = x[21 + i].re; }
  const float fx = K[0], fy = K[4], cx = K[3], cy = K[5];                  /* …TrunRANSAC.cu:138-141 (cx = K[3]) */
  const float B21 = fmaf(R21[2], T21[0], fmaf(R21[5], T21[1], R21[8] * T21[2]));
  const float B31 = fmaf(R31[2], T31[0], fmaf(R31[5], T31[1], R31[8] * T31[2]));
  int c21 = 0, c31 = 0;
  for (int e = 0; e < n_edgels; e++) {
    const float* g = loc + (size_t)e * 6;
    c21 += reproj_inlier(R21, T21, g[0], g[1], g[2], g[3], B21, fx, fy, cx, cy);
    c31 += reproj_inlier(R31, T31, g[0], g[1], g[4], g[5], B31, fx, fy, cx, cy);
  }
  *n21 = c21; *n31 = c31;
  const float r21 = (float)c21 / (float)n_edgels, r31 = (float)c31 / (float)n_edgels;
  return ((double)r21 >= 0.90 && (double)r31 >= 0.90);                     /* PASS_RANSAC_INLIER_SUPPORT_RATIO, :241-242 */
}

/* ------------------------------------------------------------------------------------------------------------
 * GPU_HC_Solver.cpp:252-306 — one rand() stream, three draws per attempt, e0 != e1 and e1 != e2 accepted */
void hco_prepare_target_params(unsigned seed, int n_hyp, int n_edgels, const float* loc, const float* tan,
                               const hco_c32* sp, hco_c32* target, hco_c32* diff, int* picked)
{
  srand(seed);
  for (int h = 0; h < n_hyp; h++) {
    unsigned e[3];
    for (;;) {
      for (int r = 0; r < 3; r++) e[r] = (unsigned)rand() % (unsigned)n_edgels;
      if (e[0] != e[1] && e[1] != e[2]) break;
    }
    hco_c32* T = target + (size_t)h * (HCO_NP + 1);
    hco_c32* D = diff + (size_t)h * (HCO_NP + 1);
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 6; j++) T[i * 6 + j] = c_make(loc[(size_t)e[i] * 6 + j], 0.0f);
    for (int i = 0; i < 2; i++)
      for (int j = 0; j < 6; j++) T[18 + i * 6 + j] = c_make(tan[(size_t)e[i] * 6 + j], 0.0f);
    T[30] = c_make(1.0f, 0.0f); T[31] = c_make(0.5f, 0.0f); T[32] = c_make(1.0f, 0.0f); T[33] = c_make(1.0f, 0.0f);
    for (int i = 0; i <= HCO_NP; i++) D[i] = c_sub(T[i], sp[i]);
    if (picked) for (int r = 0; r < 3; r++) picked[h * 3 + r] = (int)e[r];
  }
}

#endif   /* HCO_TRIFOCAL */
/* ------------------------------------------------------------------------------------------------------------
 * double-precision Newton polish against the target system (test helper) */
typedef struct { double re, im; } zc;
static inline zc z_mul(zc a, zc b) { zc r = {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; return r; }
static inline zc z_sub(zc a, zc b) { zc r = {a.re - b.re, a.im - b.im}; return r; }
static inline zc z_add(zc a, zc b) { zc r = {a.re + b.re, a.im + b.im}; return r; }
static inline zc z_div(zc a, zc b)
{ double d = b.re * b.re + b.im * b.im; zc r = {(a.re * b.re + a.im * b.im) / d, (a.im * b.re - a.re * b.im) / d}; return r; }

/* Newton refinement in the arithmetic spec (float): what hcb200_refine_tracks does on the device.  x31 in/out. */
void hco_refine_path(const int* dHdx, const int* dHdt, const hco_c32* target34, hco_c32* x31, int iters, float* out_sum_d, float* out_sum_x)
{
  hco_c32 x[HCO_N + 1], p[HCO_NP + 1], A[HCO_N * HCO_N], b[HCO_N];
  memcpy(x, x31, sizeof(hco_c32) * HCO_N);
  x[HCO_N] = c_make(1.0f, 0.0f);
  memcpy(p, target34, sizeof p);
  float sum_d = -1.0f, sum_x = -1.0f;
  for (int it = 0; it < iters; it++) {
    hco_eval_Hx(dHdx, x, p, A);
    hco_eval_H(dHdt, x, p, b);
    hco_solve(A, b);
    float vd[HCO_N], vx[HCO_N];
    for (int i = 0; i < HCO_N; i++) {
      x[i] = c_sub(x[i], b[i]);
      vd[i] = fmaf(b[i].re, b[i].re, b[i].im * b[i].im);
      vx[i] = fmaf(x[i].re, x[i].re, x[i].im * x[i].im);
    }
    sum_d = butterfly_sum(vd);
    sum_x = butterfly_sum(vx);
  }
  memcpy(x31, x, sizeof(hco_c32) * HCO_N);
  *out_sum_d = sum_d;
  *out_sum_x = sum_x;
}


double hco_newton_refine_f64(const int* dHdx, const int* dHdt, const hco_c32* tp, const hco_c32* x_in, int iters, double* x_out)
{
  zc x[HCO_N + 1], p[HCO_NP + 1], A[HCO_N][HCO_N], b[HCO_N];
  for (int i = 0; i < HCO_N; i++) { x[i].re = x_in[i].re; x[i].im = x_in[i].im; }
  x[HCO_N].re = 1; x[HCO_N].im = 0;
  for (int i = 0; i <= HCO_NP; i++) { p[i].re = tp[i].re; p[i].im = tp[i].im; }
  double res = 0;
  for (int it = 0; it <= iters; it++) {
    res = 0;
    for (int row = 0; row < HCO_N; row++) {
      zc acc = {0, 0};
      for (int j = 0; j < HCO_HT_TERMS; j++) {
        const int base = (j * HCO_HT_PARTS) * HCO_N + row;
        if (!dHdt[base]) continue;
        zc t = {(double)dHdt[base], 0};
        t = z_mul(t, p[dHdt[base + HCO_N]]); t = z_mul(t, p[dHdt[base + 2 * HCO_N]]);
        t = z_mul(t, x[dHdt[base + 3 * HCO_N]]); t = z_mul(t, x[dHdt[base + 4 * HCO_N]]); t = z_mul(t, x[dHdt[base + 5 * HCO_N]]);
        acc = z_add(acc, t);
      }
      b[row] = acc;
      res += acc.re * acc.re + acc.im * acc.im;
    }
    if (it == iters) break;
    for (int row = 0; row < HCO_N; row++)
      for (int col = 0; col < HCO_N; col++) {
        zc acc = {0, 0};
        for (int j = 0; j < HCO_HX_TERMS; j++) {
          const int base = (col * HCO_HX_TERMS * HCO_HX_PARTS + j * HCO_HX_PARTS) * HCO_N + row;
          if (!dHdx[base]) continue;
          zc t = {(double)dHdx[base], 0};
          t = z_mul(t, p[dHdx[base + HCO_N]]); t = z_mul(t, p[dHdx[base + 2 * HCO_N]]);
          t = z_mul(t, x[dHdx[base + 3 * HCO_N]]); t = z_mul(t, x[dHdx[base + 4 * HCO_N]]);
          acc = z_add(acc, t);
        }
        A[row][col] = acc;
      }
    /* plain partial-pivot LU in double */
    for (int k = 0; k < HCO_N; k++) {
      int piv = k; double best = -1;
      for (int i = k; i < HCO_N; i++) { double v = fabs(A[i][k].re) + fabs(A[i][k].im); if (v > best) { best = v; piv = i; } }
      if (piv != k) { for (int j = 0; j < HCO_N; j++) { zc t = A[k][j]; A[k][j] = A[piv][j]; A[piv][j] = t; } zc t = b[k]; b[k] = b[piv]; b[piv] = t; }
      for (int i = k + 1; i < HCO_N; i++) {
        zc m = z_div(A[i][k], A[k][k]);
        for (int j = k + 1; j < HCO_N; j++) A[i][j] = z_sub(A[i][j], z_mul(m, A[k][j]));
        b[i] = z_sub(b[i], z_mul(m, b[k]));
      }
    }
    for (int k = HCO_N - 1; k >= 0; k--) {
      zc s = b[k];
      for (int j = k + 1; j < HCO_N; j++) s = z_sub(s, z_mul(A[k][j], b[j]));
      b[k] = z_div(s, A[k][k]);
    }
    for (int i = 0; i < HCO_N; i++) x[i] = z_sub(x[i], b[i]);
  }
  for (int i = 0; i < HCO_N; i++) { x_out[2 * i] = x[i].re; x_out[2 * i + 1] = x[i].im; }
  return sqrt(res);
}
