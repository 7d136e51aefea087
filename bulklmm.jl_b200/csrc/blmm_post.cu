// Post-processing of LOD scores on the device (SURVEY section 8f, ranks 1-2):
//   lod2log10p     -log10 of the chi-square tail probability of a LOD score   src/util.jl:199-206
//   thresholds     type-7 quantiles of the per-permutation maximum LODs
//                  src/analysis_helpers/single_trait_analysis.jl:13-23
//   row scaling    the observation-weight pre-scaling block                   src/bulkscan.jl:231-250
// lod2log10p is one HBM-bound elementwise pass (8 B read + 8 B written per LOD); the others are tiny.
#include <float.h>
#include <math.h>

#include <cub/device/device_radix_sort.cuh>

#include "blmm_kernels.cuh"

namespace blmm {

namespace {

// log Q(a, y), Q = regularised upper incomplete gamma, a = df/2 (df >= 1 integer), y >= 0.
// Large y: Q(a,y) = e^-y [ base + sum_j y^(a0+j)/Gamma(a0+j+1) ], base = erfcx(sqrt y) (a0 = 1/2) or 1
// (a0 = 1): every term positive, so log Q = -y + log(bracket) keeps full relative accuracy however
// small Q is.  Small y: log1p(-P) with P from its power series, accurate as Q -> 1.
__device__ double log_gamma_q(int df, double y) {
  // y <= 0: the whole mass lies above (logccdf = 0, as Distributions.jl returns); NaN passes through
  if (!(y > 0.0)) return (y <= 0.0) ? 0.0 : y;
  const double a = 0.5 * (double)df;
  if (y < 1.0 && y < a + 1.0) {
    // P(a,y) = y^a e^-y / Gamma(a+1) * sum_k y^k / ((a+1)...(a+k))
    double term = 1.0, sum = 1.0;
    for (int k = 1; k < 200; ++k) {
      term *= y / (a + (double)k);
      sum += term;
      if (term < sum * 1e-17) break;
    }
    const double logP = a * log(y) - y - lgamma(a + 1.0) + log(sum);
    return log1p(-exp(logP));
  }
  const bool half = (df & 1) != 0;
  double bracket = half ? erfcx(sqrt(y)) : 1.0;
  // terms t_j = y^(a0+j)/Gamma(a0+j+1), j = 0 .. a-a0-1
  const double a0 = half ? 0.5 : 1.0;
  const int nterm = (int)(a - a0 + 0.25);
  if (nterm > 0) {
    double tj = half ? sqrt(y) * 1.1283791670955125739 /* y^.5/Gamma(1.5) = 2 sqrt(y/pi) */ : y;
    bracket += tj;
    for (int j = 1; j < nterm; ++j) {
      tj *= y / (a0 + (double)j);
      bracket += tj;
    }
  }
  return -y + log(bracket);
}

__global__ void lod2log10p_kernel(const double* __restrict__ lod, int64_t rows, int64_t cols, int64_t ld_in,
                                  int64_t ld_out, int df, double* __restrict__ out) {
  const int64_t total = rows * cols;
  const double ln10 = 2.30258509299404568402;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t c = idx / rows, r = idx - c * rows;
    const double l = lod[c * ld_in + r];
    // lrs = 2 ln10 lod;  logccdf(Chisq(df), lrs) = log Q(df/2, lrs/2)
    const double v = -log_gamma_q(df, l * ln10) / ln10;
    out[c * ld_out + r] = v;
  }
}

__global__ void quantile7_kernel(const double* __restrict__ sorted, int64_t n, const double* __restrict__ probs,
                                 int nprob, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nprob) return;
  // Julia `quantile` default (alpha = beta = 1) = Hyndman-Fan type 7
  const double pr = probs[i];
  double h = (double)(n - 1) * pr;
  if (h < 0.0) h = 0.0;
  if (h > (double)(n - 1)) h = (double)(n - 1);
  const int64_t lo = (int64_t)floor(h);
  const int64_t hi = lo + 1 < n ? lo + 1 : lo;
  const double g = h - (double)lo;
  // a + g (b - a) with separate roundings, as Statistics.jl's quantile evaluates it (no FMA contraction)
  out[i] = __dadd_rn(sorted[lo], __dmul_rn(g, __dsub_rn(sorted[hi], sorted[lo])));
}

__global__ void scale_rows_kernel(const double* __restrict__ X, const double* __restrict__ w, int64_t n,
                                  int64_t cols, double* __restrict__ out) {
  const int64_t total = n * cols;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x)
    out[idx] = w[idx % n] * X[idx];
}

__global__ void weight_kinship_kernel(const double* __restrict__ K, const double* __restrict__ w, int n,
                                      double* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)n * n) return;
  const int a = (int)(idx % n), b = (int)(idx / n);
  out[idx] = w[a] * K[idx] * w[b];
}

// One warp per output column j: the first maximum over the column's partials (peak_key order, ties to the smaller
// marker: a total order, so the result does not depend on which lane saw which record).
__global__ void peak_reduce_kernel(const PeakRec* __restrict__ part, int64_t n_mb, int64_t m, int p,
                                   const double* __restrict__ grid, double* __restrict__ peak_lod,
                                   int64_t* __restrict__ peak_marker, double* __restrict__ h2) {
  const int64_t j = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (j >= m) return;
  const PeakRec* r = part + j * n_mb;
  double lod = 0.0;
  int row = 0x7fffffff, gi = 0;
  for (int64_t i = lane; i < n_mb; i += 32) {
    const PeakRec c = r[i];
    peak_take(lod, row, gi, c.lod, c.marker, c.gidx, p);
  }
  peak_over_lanes(lod, row, gi, p, 1);
  if (lane == 0) {
    peak_lod[j] = lod;
    if (peak_marker) peak_marker[j] = row;
    if (grid && h2) h2[j] = grid[gi];
  }
}

}  // namespace

int launch_peak_reduce(const PeakRec* part, int64_t n_mb, int64_t m, int p, const double* grid, double* peak_lod,
                       int64_t* peak_marker, double* h2, cudaStream_t stream) {
  if (m <= 0) return 0;
  peak_reduce_kernel<<<(unsigned)((m + 7) / 8), 256, 0, stream>>>(part, n_mb, m, p, grid, peak_lod, peak_marker, h2);
  return 1;
}

int launch_lod2log10p(const double* lod, int64_t rows, int64_t cols, int64_t ld_in, int64_t ld_out, int df,
                      double* out, int sm_count, cudaStream_t stream) {
  if (rows * cols <= 0) return 0;
  const int64_t want = (rows * cols + 255) / 256;
  const int64_t cap = (int64_t)sm_count * 32;
  lod2log10p_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, stream>>>(lod, rows, cols, ld_in, ld_out, df, out);
  return 1;
}

size_t thresholds_workspace_bytes(int64_t n) {
  size_t tmp = 0;
  cub::DeviceRadixSort::SortKeys(nullptr, tmp, (const double*)nullptr, (double*)nullptr, n);
  return tmp + 256;
}

int launch_thresholds(const double* maxlod, int64_t n, const double* probs_dev, int nprob, double* sorted,
                      void* tmp, size_t tmp_bytes, double* out, cudaStream_t stream) {
  cub::DeviceRadixSort::SortKeys(tmp, tmp_bytes, maxlod, sorted, n, 0, 64, stream);
  quantile7_kernel<<<(nprob + 63) / 64, 64, 0, stream>>>(sorted, n, probs_dev, nprob, out);
  return 2;
}

int launch_scale_rows(const double* X, const double* w, int64_t n, int64_t cols, double* out, int sm_count,
                      cudaStream_t stream) {
  if (n * cols <= 0) return 0;
  const int64_t want = (n * cols + 255) / 256;
  const int64_t cap = (int64_t)sm_count * 32;
  scale_rows_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, stream>>>(X, w, n, cols, out);
  return 1;
}

int launch_weight_kinship(const double* K, const double* w, int n, double* out, cudaStream_t stream) {
  const int64_t nn = (int64_t)n * n;
  weight_kinship_kernel<<<(unsigned)((nn + 255) / 256), 256, 0, stream>>>(K, w, n, out);
  return 1;
}

}  // namespace blmm
