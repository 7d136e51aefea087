// Batched per-trait heritability fit: fitlmm (src/lmm.jl:56-86) = gridbrent (src/gridbrent.jl:9-24)
// over Optim.jl's univariate Brent minimiser of -ell(h2), ell from wls (src/wls.jl:27-97).
// One warp per trait; the n eigenvalue weights are spread over the lanes and every objective
// evaluation is a handful of warp-shuffle reductions.  All lanes carry identical scalars (the
// butterfly reduction is symmetric), so the Brent control flow is warp-uniform.
#include <float.h>
#include <math.h>
#include <stdlib.h>

#include "blmm_kernels.cuh"
#include "blmm_prep_dev.cuh"

namespace blmm {

namespace {

constexpr int FIT_WARPS = 4;

// Natural logarithm with a SHORT dependent chain (the objective is evaluated ~26 times in sequence per trait, each
// evaluation two logarithms deep): v = 2^e m, m in [0.75, 1.5); a 512-entry shared-memory table gives rcp ~ 1/c and
// log c for m's interval, r = m rcp - 1 (|r| < 2^-9), log1p(r) by five terms in Estrin form: ~8 dependent FP64
// operations instead of the ~40 of log().  Absolute error <= 1.2e-16 near 1, relative <= 5e-15 elsewhere (checked
// against 40-digit arithmetic); operands outside the positive normal range fall back to log().
constexpr int FIT_LTAB = 512;
__device__ __forceinline__ void fit_build_ln_table(double2* tab, int tid, int nthreads) {
  for (int i = tid; i < FIT_LTAB; i += nthreads) {
    double c;
    if (i == FIT_LTAB / 2 - 1 || i == FIT_LTAB / 2)
      c = 1.0;
    else if (i < FIT_LTAB / 2)
      c = 0.75 + ((double)i + 0.5) * (0.25 / (FIT_LTAB / 2));
    else
      c = 1.0 + ((double)(i - FIT_LTAB / 2) + 0.5) * (0.5 / (FIT_LTAB / 2));
    const double rcp = 1.0 / c;
    tab[i] = make_double2(rcp, (rcp == 1.0) ? 0.0 : -log(rcp));
  }
}
__device__ __forceinline__ double fit_ln(double v, const double2* __restrict__ tab) {
  const int hi = __double2hiint(v), lo = __double2loint(v);
  if ((unsigned)(hi - 0x00100000) >= 0x7fe00000u) return log(v);  // zero, subnormal, negative, inf, NaN
  const int ix = hi - 0x3fe80000;
  const int e = ix >> 20;
  const double m = __hiloint2double(hi - (e << 20), lo);
  const double2 t = tab[(ix >> 11) & (FIT_LTAB - 1)];
  const double r = fma(m, t.x, -1.0);
  const double r2 = r * r;
  const double p = fma(r, 1.0 / 5.0, -1.0 / 4.0);
  const double q = fma(r, 1.0 / 3.0, -1.0 / 2.0);
  const double lp = fma(r2, fma(r2, p, q), r);
  return fma((double)e, 0.69314718055994530942, t.y + lp);
}

struct FitData {
  const double* y;       // trait (residualised on C0, padded), length n_pad
  const double* Qc;      // [c][n_pad] orthonormal basis of the covariates: C0 = Qc R (the w = 1 weight slot)
  double ld_r;           // log det(C0'C0) = log det(R'R): REML's log det(C0'WC0) = log det(Qc'WQc) + ld_r
  const double* lambda;  // [n]
  int n, n_pad, c, lane;
  LikParams lik;
  const double* xcol;    // scan_alt: the marker column that takes the LAST covariate slot (else nullptr)
  bool sqrt_weights;     // scan_alt's final likelihoods: wls is handed sqrt(w) as its weights (src/scan.jl:440-441)
  const double2* ltab;   // shared-memory table of fit_ln
  double inv_denom;      // 1 / (n [- c] + prior_df): sigma2 = (rss + a b) * inv_denom
};

__device__ __forceinline__ double fit_inv_denom(const LikParams& lik, int n, int c) {
  const double pdf = (lik.prior_b > 0.0) ? lik.prior_b + 2.0 : lik.prior_b;  // src/wls.jl:72-76
  return 1.0 / (lik.reml ? ((double)(n - c) + pdf) : ((double)n + pdf));
}

// -ell(h2) and sigma2.  The covariate projection uses the Gram form S = C'WC, t = C'Wy,
// rss = y'Wy - t'S^-1 t, log det S = 2 log|det R|, evaluated in one pass over the n weights.  C is the orthonormal
// basis Qc (and, for scan_alt, the marker column), not C0: the projection is the same, but the Gram matrix of C0 would
// be conditioned as kappa(C0)^2 (1e10 for two near-collinear covariates, ell then off by ~1e-8 relative), that of Qc
// only by the spread of the weights.
template <int C, int UNR = 4>
__device__ double neg_loglik_c(const FitData& d, double h2, double* sigma2_out) {
  constexpr int NT = C * (C + 1) / 2;
  const double delta = h2 * fast_rcp(1.0 - h2);
  double S[NT], t[C];
#pragma unroll
  for (int i = 0; i < NT; ++i) S[i] = 0.0;
#pragma unroll
  for (int i = 0; i < C; ++i) t[i] = 0.0;
  // sum_l log w_l = -log prod_l (delta lambda_l + 1): one logarithm per lane instead of one per element (the
  // running product is folded into the sum every 8 factors; a factor is at most ~2^40 for h2 <= 1 - 1e-8)
  // Every evaluation is one link of Brent's strictly sequential chain (~26 per trait), so what counts here is the
  // LENGTH of the dependent FP64 chain, not the operation count: reciprocals by Newton steps on the hardware estimate
  // (5 dependent operations instead of the ~18 of the IEEE division sequence; last-bit differences are far below the
  // rounding noise the minimiser already sees), the loop unrolled so that the elements' chains overlap.
  double yy = 0.0, slw = 0.0, prod = 1.0;
  int since = 0;
#pragma unroll UNR
  for (int l = d.lane; l < d.n; l += 32) {
    const double dl = fma(delta, d.lambda[l], 1.0);
    const double w = d.sqrt_weights ? rsqrt(dl) : fast_rcp(dl);
    prod *= dl;
    if (++since == 8) {
      slw -= fit_ln(prod, d.ltab);
      prod = 1.0;
      since = 0;
    }
    const double y = d.y[l];
    const double wy = w * y;
    yy = fma(wy, y, yy);
    double cv[C];
#pragma unroll
    for (int a = 0; a < C; ++a) cv[a] = (a == C - 1 && d.xcol) ? d.xcol[l] : d.Qc[(int64_t)a * d.n_pad + l];
    int idx = 0;
#pragma unroll
    for (int a = 0; a < C; ++a) {
      t[a] = fma(cv[a], wy, t[a]);
      const double wc = w * cv[a];
#pragma unroll
      for (int b = 0; b <= a; ++b) {
        S[idx] = fma(wc, cv[b], S[idx]);
        ++idx;
      }
    }
  }
  slw -= fit_ln(prod, d.ltab);
  if (d.sqrt_weights) slw *= 0.5;
  yy = warp_sum(yy);
  slw = warp_sum(slw);
#pragma unroll
  for (int i = 0; i < NT; ++i) S[i] = warp_sum(S[i]);
#pragma unroll
  for (int i = 0; i < C; ++i) t[i] = warp_sum(t[i]);
  // Square-root-free Cholesky S = L D L' (packed lower, row-major; Dinv = 1/D by Newton reciprocal), forward solve:
  // t' S^-1 t = sum_a u_a^2 / D_a and log det S = sum_a log D_a (= 2 sum log of the Cholesky diagonal)
  double uu = 0.0;
  double Lm[NT], u[C], Dv[C], Dinv[C];
#pragma unroll
  for (int a = 0; a < C; ++a) {
#pragma unroll
    for (int b = 0; b <= a; ++b) {
      double s = S[a * (a + 1) / 2 + b];
#pragma unroll
      for (int k = 0; k < b; ++k) s -= Lm[a * (a + 1) / 2 + k] * Lm[b * (b + 1) / 2 + k] * Dv[k];
      if (a == b) {
        Dv[a] = s;
        Dinv[a] = fast_rcp(s);
        Lm[a * (a + 1) / 2 + a] = 1.0;
      } else {
        Lm[a * (a + 1) / 2 + b] = s * Dinv[b];
      }
    }
    double s = t[a];
#pragma unroll
    for (int k = 0; k < a; ++k) s -= Lm[a * (a + 1) / 2 + k] * u[k];
    u[a] = s;
    uu = fma(s * s, Dinv[a], uu);
  }
  const double rss = yy - uu;
  const double a = d.lik.prior_a, b = d.lik.prior_b;
  const double ab = a * b;
  const double sigma2 = (rss + ab) * d.inv_denom;  // 1 / denom: a per-call constant
  // log sigma2 and the logs of the C pivots in ONE evaluation: lane 0 takes sigma2, lane a+1 D_a
  double arg = sigma2;
#pragma unroll
  for (int i = 0; i < C; ++i)
    if (d.lane == i + 1) arg = Dv[i];
  const double lg = fit_ln(arg, d.ltab);
  const double log_s2 = __shfl_sync(0xffffffffu, lg, 0);
  double lds = 0.0;
#pragma unroll
  for (int i = 0; i < C; ++i) lds += __shfl_sync(0xffffffffu, lg, i + 1);
  // (rss + ab) / sigma2 is `denom` up to the rounding of the division that made sigma2; the reference evaluates the
  // quotient (src/wls.jl:84), so it is evaluated here too
  double ll = -0.5 * (((double)d.n + b) * log_s2 - slw + (rss + ab) * fast_rcp(sigma2));
  if (d.lik.reml) ll += 0.5 * ((double)C * log_s2 - (lds + d.ld_r));
  if (sigma2_out) *sigma2_out = sigma2;
  return -ll;
}

// Optim.jl `optimize(f, lo, hi, Brent())` with its defaults rel_tol = sqrt(eps), abs_tol = eps,
// iterations = 1000 (call site src/gridbrent.jl:16).
template <int C, int UNR = 4>
__device__ void brent(const FitData& d, double lo, double hi, double* xmin, double* fmin_out) {
  const double golden = 0.5 * (3.0 - sqrt(5.0));
  const double rel_tol = sqrt(DBL_EPSILON), abs_tol = DBL_EPSILON;
  double x = lo + golden * (hi - lo);
  double fx = neg_loglik_c<C, UNR>(d, x, nullptr);
  double step = 0.0, old_step = 0.0;
  double xo = x, xoo = x, fo = fx, foo = fx;
  for (int it = 0; it < 1000; ++it) {
    double p = 0.0, q = 0.0;
    const double tol = rel_tol * fabs(x) + abs_tol;
    const double mid = (hi + lo) / 2.0;
    if (fabs(x - mid) <= 2.0 * tol - (hi - lo) / 2.0) break;
    if (fabs(old_step) > tol) {
      const double r = (x - xo) * (fx - foo);
      q = (x - xoo) * (fx - fo);
      p = (x - xoo) * q - (x - xo) * r;
      q = 2.0 * (q - r);
      if (q > 0.0)
        p = -p;
      else
        q = -q;
    }
    if (fabs(p) < fabs(q * old_step / 2.0) && p < q * (hi - x) && p < q * (x - lo)) {
      old_step = step;
      step = p / q;
      const double xt = x + step;
      if ((xt - lo) < 2.0 * tol || (hi - xt) < 2.0 * tol) step = (x < mid) ? tol : -tol;
    } else {
      old_step = (x < mid) ? (hi - x) : (lo - x);
      step = golden * old_step;
    }
    const double xn = (fabs(step) >= tol) ? x + step : x + ((step > 0.0) ? tol : -tol);
    const double fn = neg_loglik_c<C, UNR>(d, xn, nullptr);
    if (fn < fx) {
      if (xn < x)
        hi = x;
      else
        lo = x;
      xoo = xo; foo = fo;
      xo = x; fo = fx;
      x = xn; fx = fn;
    } else {
      if (xn < x)
        lo = xn;
      else
        hi = xn;
      if (fn <= fo || xo == x) {
        xoo = xo; foo = fo;
        xo = xn; fo = fn;
      } else if (fn <= foo || xoo == x || xoo == xo) {
        xoo = xn; foo = fn;
      }
    }
  }
  *xmin = x;
  *fmin_out = fx;
}

// gridbrent over [0, 1] in optim_interval pieces (src/gridbrent.jl:9-24): points = range(0, 1, length =
// optim_interval + 1); keeps the first of equal minima
template <int C, int UNR = 4>
__device__ double fit_one(const FitData& d, int optim_interval) {
  double bx = 0.0, bf = INFINITY;
  for (int i = 0; i < optim_interval; ++i) {
    const double lo = (double)i / (double)optim_interval;
    const double hi = (i + 1 == optim_interval) ? 1.0 : (double)(i + 1) / (double)optim_interval;
    double x, f;
    brent<C, UNR>(d, lo, hi, &x, &f);
    if (i == 0 || f < bf) {
      bx = x;
      bf = f;
    }
  }
  return bx;
}

// Templated on the covariate count so that the common c = 1..3 cases keep their Gram matrices in a few
// registers (a run-time switch over all eight sizes cost 200 registers per thread: 8 warps per SM).
// BULK: many traits — occupancy hides the latency of each warp's chain (64 registers for c <= 2); otherwise (a few
// traits: the null fit of scan / permutations) nothing hides it and the registers are better spent on no spills.
template <int C, bool BULK>
__global__ void __launch_bounds__(32 * FIT_WARPS, BULK ? (C <= 2 ? 8 : (C <= 4 ? 4 : 2)) : 1)
    fit_h2_kernel(const double* __restrict__ Yr, int64_t m, int n, int n_pad, int c, const double* __restrict__ Qc,
                  const double* __restrict__ ld_r, const double* __restrict__ lambda, LikParams lik, int optim_interval, double* __restrict__ h2_out,
                  double* __restrict__ sigma2_out, double* __restrict__ ell_out, int staged) {
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t j = (int64_t)blockIdx.x * FIT_WARPS + wid;
  // Brent is a chain of ~26 dependent objective evaluations, each a pass over the n weights: with the operands in
  // shared memory (eigenvalues and covariates once per block, the trait once per warp) a pass waits on shared-memory
  // latency instead of L1/L2 latency.  `staged` is off when the block's copies would not fit (very large n).
  extern __shared__ double fit_sm[];
  double2* ltab = reinterpret_cast<double2*>(fit_sm);
  fit_build_ln_table(ltab, threadIdx.x, blockDim.x);
  const double* yv = Yr + (j < m ? j : 0) * n_pad;
  if (!staged) __syncthreads();
  if (staged) {
    double* lam_s = fit_sm + 2 * FIT_LTAB;
    double* c_s = lam_s + n_pad;
    double* y_s = c_s + (int64_t)C * n_pad + (int64_t)wid * n_pad;
    for (int l = threadIdx.x; l < n_pad; l += blockDim.x) lam_s[l] = (l < n) ? lambda[l] : 0.0;
    for (int l = threadIdx.x; l < C * n_pad; l += blockDim.x) c_s[l] = Qc[l];
    for (int l = lane; l < n_pad; l += 32) y_s[l] = yv[l];
    __syncthreads();
    lambda = lam_s;
    Qc = c_s;
    yv = y_s;
  }
  if (j >= m) return;
  FitData d{yv, Qc, *ld_r, lambda, n, n_pad, c, lane, lik, nullptr, false, ltab, fit_inv_denom(lik, n, C)};
  const double bx = fit_one<C, BULK ? 1 : 4>(d, optim_interval);
  double s2;
  const double f = neg_loglik_c<C, BULK ? 1 : 4>(d, bx, &s2);
  if (lane == 0) {
    if (h2_out) h2_out[j] = bx;
    if (sigma2_out) sigma2_out[j] = s2;
    if (ell_out) ell_out[j] = -f;
  }
}

// scan_alt (src/scan.jl:397-453), one warp per marker: covariates [C0 g_i] (C = c + 1 columns), the variance
// components re-estimated by Brent for every marker, then lod_i = (ell_alt - ell_null) / ln 10 with both
// likelihoods evaluated as the reference does — ML, and with sqrt(w) passed to wls as the weights.
// ell_null comes from scan_alt_null_kernel.
template <int C>
__global__ void __launch_bounds__(32 * FIT_WARPS, C <= 2 ? 8 : (C <= 4 ? 4 : 2))
    scan_alt_kernel(const double* __restrict__ y, const double* __restrict__ G0, int64_t p, int n, int n_pad,
                    const double* __restrict__ Qc, const double* __restrict__ ld_r, const double* __restrict__ lambda, LikParams lik,
                    int optim_interval, const double* __restrict__ ell_null, double* __restrict__ lod,
                    double* __restrict__ h2_each) {
  __shared__ double2 ltab[FIT_LTAB];
  fit_build_ln_table(ltab, threadIdx.x, blockDim.x);
  __syncthreads();
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * FIT_WARPS + wid;
  if (i >= p) return;
  FitData d{y, Qc, *ld_r, lambda, n, n_pad, C, lane, lik, G0 + i * n_pad, false, ltab, fit_inv_denom(lik, n, C)};
  const double h2 = fit_one<C>(d, optim_interval);
  d.sqrt_weights = true;
  d.lik.reml = 0;
  d.inv_denom = fit_inv_denom(d.lik, n, C);
  const double ell_alt = -neg_loglik_c<C>(d, h2, nullptr);
  if (lane == 0) {
    lod[i] = (ell_alt - ell_null[0]) / 2.30258509299404568402;
    if (h2_each) h2_each[i] = h2;
  }
}

// ell_null of scan_alt: wls(y0, X0_covar, sqrt(w(h2_null)), prior).ell, one warp
template <int C>
__global__ void scan_alt_null_kernel(const double* __restrict__ y, int n, int n_pad, const double* __restrict__ Qc,
                                     const double* __restrict__ lambda, LikParams lik,
                                     const double* __restrict__ h2_null, double* __restrict__ ell_null) {
  __shared__ double2 ltab[FIT_LTAB];
  fit_build_ln_table(ltab, threadIdx.x, blockDim.x);
  __syncthreads();
  lik.reml = 0;
  FitData d{y, Qc, 0.0, lambda, n, n_pad, C, (int)(threadIdx.x & 31), lik, nullptr, true, ltab, fit_inv_denom(lik, n, C)};
  const double e = -neg_loglik_c<C>(d, h2_null[0], nullptr);
  if (threadIdx.x == 0) ell_null[0] = e;
}

// -----------------------------------------------------------------------------------------------
// The whole single-trait prologue of scan(...; permutation_test = true) in ONE launch (one block of 128 threads):
//   rotation of the trait and the covariates by U' (src/transform_helpers.jl:1-54), the unweighted residual of the
//   trait on the covariates, fitlmm (Brent, warp 0), the weight constants at the fitted h2, and the re-weighted null
//   residual z = P (sw .* y) of transform_reweight (src/transform_helpers.jl:57-92).
// It replaces seven launches (rotate x2, weight constants x2, trait statistics, Brent, null residual) whose kernels take
// 4-12 us each and whose launch gaps are as long again: a permutation step is 0.45 ms of scan, so they were a tenth
// of it.  For small n only (null_fit_chain_applies): the rotation is done by one thread per output here.
// -----------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(128, 1)
    null_fit_chain_kernel(const double* __restrict__ U, const double* __restrict__ y, const double* __restrict__ Cov,
                          const double* __restrict__ lambda, int n, int n_pad, LikParams lik, int optim_interval,
                          double* __restrict__ C0_out, double* __restrict__ Yr_out, WeightConsts wc,
                          double* __restrict__ h2_out, double* __restrict__ sigma2_out, double* __restrict__ z_out,
                          double* __restrict__ zrss_out, int* flags) {
  extern __shared__ double cs[];
  double2* ltab = reinterpret_cast<double2*>(cs);  // [FIT_LTAB]
  double* lam_s = cs + 2 * FIT_LTAB;               // [n_pad]
  double* c_s = lam_s + n_pad;                     // [C][n_pad]  rotated covariates
  double* y_s = c_s + (int64_t)C * n_pad;          // [n_pad]     rotated, then residualised trait
  double* q_s = y_s + n_pad;                       // [C][n_pad]  orthonormal basis of the rotated covariates
  __shared__ WcShared sh;
  __shared__ double h2_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  fit_build_ln_table(ltab, tid, 128);
  // U'[Cov y]: one thread per output
  for (int idx = tid; idx < (C + 1) * n_pad; idx += 128) {
    const int col = idx / n_pad, a = idx % n_pad;
    // rotate_elem: this path and the separate kernels (and scan without permutations) see bit-identical rotated inputs
    // and hence the same Brent trajectory
    const double v = (a < n) ? rotate_elem(U, (col < C) ? Cov + (int64_t)col * n : y, n, a) : 0.0;
    if (col < C) {
      c_s[idx] = v;
      C0_out[idx] = v;
    } else {
      y_s[a] = v;
    }
  }
  for (int l = tid; l < n_pad; l += 128) lam_s[l] = (l < n) ? lambda[l] : 0.0;
  __syncthreads();
  // unweighted basis of the covariates (slot 1 of wc: w = 1), then Yr = y0 - Q Q'y0
  const WeightSlot ols = weight_slot(wc, 1, n_pad, C);
  weight_consts_block(true, 0.0, lam_s, c_s, n, n_pad, C, ols, flags, sh);
  for (int l = tid; l < C * n_pad; l += 128) q_s[l] = ols.Q[l];
  __syncthreads();
  if (warp == 0) {
    unweighted_residual(y_s, ols, n_pad, C, lane, [&](int l, double v) { Yr_out[l] = v; });
    FitData d{y_s, q_s, *ols.lds, lam_s, n, n_pad, C, lane, lik, nullptr, false, ltab, fit_inv_denom(lik, n, C)};
    const double h2 = fit_one<C>(d, optim_interval);
    double s2;
    neg_loglik_c<C>(d, h2, &s2);
    if (lane == 0) {
      h2_s = h2;
      if (h2_out) *h2_out = h2;
      if (sigma2_out) *sigma2_out = s2;
    }
  }
  __syncthreads();
  // transform_reweight at the fitted h2 (slot 0)
  const WeightSlot w0 = weight_slot(wc, 0, n_pad, C);
  weight_consts_block(false, h2_s, lam_s, c_s, n, n_pad, C, w0, flags, sh);
  if (warp == 0) {
    double coef[MAXC];
    const double ss = proj_norm2(y_s, w0, n_pad, C, lane, coef, z_out);
    if (lane == 0) *zrss_out = ss;
  }
}

}  // namespace

// one block rotates y and the covariates with one thread per output, each a length-n dot product: small n only (then
// the shared memory, 2 FIT_LTAB + (2 + 2 c) n_pad doubles, is under 30 KB for every c <= MAXC)
bool null_fit_chain_applies(int n) { return n <= 128; }

int launch_null_fit_chain(const double* U, const double* y, const double* Cov, const double* lambda, int n, int n_pad,
                          int c, LikParams lik, int optim_interval, double* C0, double* Yr, WeightConsts wc, double* h2,
                          double* sigma2, double* z, double* zrss, int* flags, cudaStream_t stream) {
  const size_t smem = ((size_t)2 * FIT_LTAB + (size_t)(2 + 2 * c) * n_pad) * sizeof(double);
  return dispatch_c<1, MAXC>(c, [&](auto C) {
    null_fit_chain_kernel<C><<<1, 128, smem, stream>>>(U, y, Cov, lambda, n, n_pad, lik, optim_interval, C0, Yr, wc, h2,
                                                       sigma2, z, zrss, flags);
  });
}

int launch_scan_alt(const double* y, const double* G0, int64_t p, int n, int n_pad, int c, const double* Qc,
                    const double* ld_r, const double* lambda, LikParams lik, int optim_interval, const double* h2_null, double* ell_null,
                    double* lod, double* h2_each, cudaStream_t stream) {
  const unsigned blocks = (unsigned)((p + FIT_WARPS - 1) / FIT_WARPS);
  const bool ok = dispatch_c<1, MAXC - 1>(c, [&](auto C) {
    scan_alt_null_kernel<C><<<1, 32, 0, stream>>>(y, n, n_pad, Qc, lambda, lik, h2_null, ell_null);
    scan_alt_kernel<C + 1><<<blocks, 32 * FIT_WARPS, 0, stream>>>(y, G0, p, n, n_pad, Qc, ld_r, lambda, lik,
                                                                  optim_interval,
                                                                  ell_null, lod, h2_each);
  });
  return ok ? 2 : 0;
}

int launch_fit_h2(const double* Yr, int64_t m, int n, int n_pad, int c, const double* Qc, const double* ld_r,
                  const double* lambda, LikParams lik, int optim_interval, double* h2, double* sigma2,
                  double* ell, int* flags, cudaStream_t stream) {
  (void)flags;
  const unsigned blocks = (unsigned)((m + FIT_WARPS - 1) / FIT_WARPS);
  const size_t tab_bytes = (size_t)FIT_LTAB * sizeof(double2);
  size_t smem = tab_bytes + (size_t)(1 + c + FIT_WARPS) * n_pad * sizeof(double);
  const int staged = smem <= 96 * 1024 ? 1 : 0;
  const int stage = staged && !getenv("BLMM_B200_FIT_UNSTAGED");  // test hook: force the unstaged kernel
  if (!stage) smem = tab_bytes;
  const bool bulk = blocks > 148 * 4;
  auto launch = [&](auto kernel) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kernel<<<blocks, 32 * FIT_WARPS, smem, stream>>>(Yr, m, n, n_pad, c, Qc, ld_r, lambda, lik, optim_interval, h2, sigma2,
                                                     ell, stage);
  };
  return dispatch_c<1, MAXC>(c, [&](auto C) {
    if (bulk)
      launch(fit_h2_kernel<C, true>);
    else
      launch(fit_h2_kernel<C, false>);
  });
}

}  // namespace blmm
