// Device steps shared by the kernels of blmm_prep.cu and the fused single-trait kernel of blmm_fit.cu (each translation
// unit gets its own copy: anonymous namespace).  Each step exists once, so that every path that uses it computes the
// same bits.
#pragma once
#include <float.h>
#include <math.h>

#include "blmm_kernels.cuh"

namespace blmm {
namespace {

__device__ __forceinline__ double block_sum_128(double v, double* red) {
  // blockDim.x == 128; returns the sum to every thread
  v = warp_sum(v);
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  return (red[0] + red[1]) + (red[2] + red[3]);
}

// (U'x)_a with one accumulator, b ascending: rotate_kernel's summation order, so that the kernels which rotate their
// own inputs (one thread per output) and the separate rotation see bit-identical values.
__device__ __forceinline__ double rotate_elem(const double* __restrict__ U, const double* __restrict__ x, int n,
                                              int a) {
  const double* u = U + (int64_t)a * n;
  double v = 0.0;
  for (int b = 0; b < n; ++b) v = fma(u[b], x[b], v);
  return v;
}

// Weight slot k of WeightConsts: its w, sw and Q (n_pad, n_pad, c x n_pad) and its two scalars.
struct WeightSlot {
  double *w, *sw, *Q, *slw, *lds;
};
__device__ __forceinline__ WeightSlot weight_slot(const WeightConsts& wc, int k, int n_pad, int c) {
  return WeightSlot{wc.w + (int64_t)k * n_pad, wc.sw + (int64_t)k * n_pad, wc.Q + (int64_t)k * c * n_pad, wc.slw + k,
                    wc.lds + k};
}

// One weight vector's constants, by a block of 128 threads (the body of weight_consts_kernel; also called by the fused
// single-trait kernel of blmm_fit.cu): w, sw, the CholQR^2 basis Q of sw .* C0, sum log w, log det (C0' W C0).
// Ends with a __syncthreads(): the outputs are visible to the whole block on return.
struct WcShared {
  double red[4];
  double Linv[MAXC][MAXC];
  double ldsum;
};
__device__ __forceinline__ void weight_consts_block(bool ols, double h2, const double* __restrict__ lambda,
                                                    const double* __restrict__ C0, int n, int n_pad, int c,
                                                    WeightSlot out, int* flags, WcShared& sh) {
  double* __restrict__ w = out.w;
  double* __restrict__ sw = out.sw;
  double* __restrict__ Q = out.Q;
  double* red = sh.red;
  double(*Linv)[MAXC] = sh.Linv;
  double& ldsum = sh.ldsum;
  const int tid = threadIdx.x;
  const double delta = h2 / (1.0 - h2);

  double slw = 0.0;
  for (int l = tid; l < n_pad; l += 128) {
    double wv = 0.0;
    if (l < n) {
      wv = ols ? 1.0 : 1.0 / (delta * lambda[l] + 1.0);
      if (!(wv > 0.0)) atomicExch(&flags[FLAG_WEIGHTS], 1);
      slw += log(wv);
    }
    const double s = sqrt(wv);
    w[l] = wv;
    sw[l] = s;
    for (int a = 0; a < c; ++a) Q[(int64_t)a * n_pad + l] = s * C0[(int64_t)a * n_pad + l];
  }
  slw = block_sum_128(slw, red);
  if (tid == 0) {
    *out.slw = slw;
    ldsum = 0.0;
  }
  // Cholesky-QR, applied twice: Q <- Q * inv(chol(Q'Q))'.  The second pass restores orthonormality
  // to rounding level; log det(C0' W C0) accumulates over the passes.
  for (int pass = 0; pass < 2; ++pass) {
    double S[MAXC][MAXC];
    for (int a = 0; a < c; ++a)
      for (int b = 0; b <= a; ++b) {
        double s = 0.0;
        for (int l = tid; l < n_pad; l += 128) s = fma(Q[(int64_t)a * n_pad + l], Q[(int64_t)b * n_pad + l], s);
        S[a][b] = block_sum_128(s, red);
      }
    if (tid == 0) {
      // in-place lower Cholesky, then its inverse
      bool ok = true;
      double Lc[MAXC][MAXC];
      for (int a = 0; a < c; ++a) {
        for (int b = 0; b <= a; ++b) {
          double s = S[a][b];
          for (int t = 0; t < b; ++t) s -= Lc[a][t] * Lc[b][t];
          if (a == b) {
            if (!(s > 0.0)) ok = false;
            Lc[a][a] = sqrt(s);
          } else {
            Lc[a][b] = s / Lc[b][b];
          }
        }
      }
      if (!ok) atomicExch(&flags[FLAG_NOT_SPD], 1);
      double ld = 0.0;
      for (int a = 0; a < c; ++a) ld += log(Lc[a][a]);
      ldsum += 2.0 * ld;
      for (int a = 0; a < c; ++a) {
        for (int b = 0; b < c; ++b) Linv[a][b] = 0.0;
        Linv[a][a] = 1.0 / Lc[a][a];
        for (int b = 0; b < a; ++b) {
          double s = 0.0;
          for (int t = b; t < a; ++t) s -= Lc[a][t] * Linv[t][b];
          Linv[a][b] = s / Lc[a][a];
        }
      }
    }
    __syncthreads();
    for (int l = tid; l < n_pad; l += 128) {
      for (int a = c - 1; a >= 0; --a) {
        double s = 0.0;
        for (int b = 0; b <= a; ++b) s = fma(Linv[a][b], Q[(int64_t)b * n_pad + l], s);
        Q[(int64_t)a * n_pad + l] = s;
      }
    }
    __syncthreads();
  }
  if (tid == 0) *out.lds = ldsum;
  __syncthreads();
}


// z = P_k (sw_k .* x) over a warp: coef = Q_k'(sw_k .* x) to every lane; proj_elem then evaluates z_l.
__device__ __forceinline__ void proj_coefs(const double* __restrict__ xb, const double* __restrict__ sw,
                                           const double* __restrict__ Q, int n_pad, int c, int lane,
                                           double coef[MAXC]) {
#pragma unroll
  for (int a = 0; a < MAXC; ++a) {
    if (a < c) {
      double s = 0.0;
      for (int l = lane; l < n_pad; l += 32) s = fma(Q[(int64_t)a * n_pad + l], sw[l] * xb[l], s);
      coef[a] = warp_sum(s);
    }
  }
}
__device__ __forceinline__ double proj_elem(const double* __restrict__ xb, const double* __restrict__ sw,
                                            const double* __restrict__ Q, int n_pad, int c, int l,
                                            const double coef[MAXC]) {
  double z = sw[l] * xb[l];
#pragma unroll
  for (int a = 0; a < MAXC; ++a)
    if (a < c) z = fma(-Q[(int64_t)a * n_pad + l], coef[a], z);
  return z;
}

// The warp's unweighted residual of its staged vector xb on the covariates (a weight slot with w = 1): xb <- P xb in
// place, and elem(l, value) for every element (the callers' side writes).  Each lane rewrites only the elements it
// reads; ends with a __syncwarp().
template <class Elem>
__device__ __forceinline__ void unweighted_residual(double* xb, const WeightSlot& s, int n_pad, int c, int lane,
                                                    Elem&& elem) {
  double coef[MAXC];
  proj_coefs(xb, s.sw, s.Q, n_pad, c, lane, coef);
  for (int l = lane; l < n_pad; l += 32) {
    const double v = proj_elem(xb, s.sw, s.Q, n_pad, c, l, coef);
    xb[l] = v;
    elem(l, v);
  }
  __syncwarp();
}

// ||P_k (sw_k .* x)||^2 over a warp, to every lane; leaves the projection coefficients in coef and, when z is given,
// writes z = P_k (sw_k .* x).
__device__ __forceinline__ double proj_norm2(const double* __restrict__ xb, const WeightSlot& s, int n_pad, int c,
                                             int lane, double coef[MAXC], double* __restrict__ z = nullptr) {
  proj_coefs(xb, s.sw, s.Q, n_pad, c, lane, coef);
  double ss = 0.0;
  for (int l = lane; l < n_pad; l += 32) {
    const double v = proj_elem(xb, s.sw, s.Q, n_pad, c, l, coef);
    if (z) z[l] = v;
    ss = fma(v, v, ss);
  }
  return warp_sum(ss);
}

// ---- the table kernels (trait_stats_table_kernel, marker_operand_table_kernel) ----
// Lane v of a warp owns one (kind a = v / KB, grid point k = bt KB + v % KB) pair of lane batch bt < nbatch.

// The block's table T[bt][l][32] (lane-contiguous): kind 0 holds w_k[l], kind a >= 1 holds Q_k,a-1[l] sw_k[l]; lanes
// past the c + 1 kinds or the nk points, and rows l >= n, hold 0.  Tt (optional) receives the same values as
// Tt[bt][32][n_pad] (l-contiguous).  Ends with a __syncthreads().
__device__ __forceinline__ void build_weight_table(const WeightConsts& wc, int n, int n_pad, int c, int nk, int KB,
                                                   int nbatch, double* __restrict__ T, double* __restrict__ Tt) {
  for (int idx = threadIdx.x; idx < nbatch * n_pad * 32; idx += blockDim.x) {
    const int v = idx & 31, l = (idx >> 5) % n_pad, bt = (idx >> 5) / n_pad;
    const int a = v / KB, k = bt * KB + v % KB;
    double val = 0.0;
    if (a <= c && k < nk && l < n) {
      const double sw = wc.sw[(int64_t)k * n_pad + l];
      val = (a == 0) ? wc.w[(int64_t)k * n_pad + l] : wc.Q[((int64_t)k * c + (a - 1)) * n_pad + l] * sw;
    }
    T[idx] = val;
    if (Tt) Tt[((size_t)bt * 32 + v) * n_pad + l] = val;
  }
  __syncthreads();
}

// One pass of a warp over its staged vector against one lane batch Tb (= T + bt n_pad 32) of the table: src is x^2 in
// the kind-0 lanes and x in the others.  sv = sum_l Tb[l][lane] src[l] (four accumulators); red = sv - sum_{a >= 1}
// sv_(a, kk)^2, the Gram form of ||P_k(sw_k .* x)||^2 in the kind-0 lane of point kk.
struct TablePass {
  double sv, red;
};
__device__ __forceinline__ TablePass table_pass(const double* __restrict__ Tb, const double* __restrict__ src, int n,
                                                int c, int KB, int kk_lane, int lane) {
  Tb += lane;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  int l = 0;
  for (; l + 4 <= n; l += 4) {
    s0 = fma(Tb[(l + 0) * 32], src[l + 0], s0);
    s1 = fma(Tb[(l + 1) * 32], src[l + 1], s1);
    s2 = fma(Tb[(l + 2) * 32], src[l + 2], s2);
    s3 = fma(Tb[(l + 3) * 32], src[l + 3], s3);
  }
  for (; l < n; ++l) s0 = fma(Tb[l * 32], src[l], s0);
  const double sv = (s0 + s1) + (s2 + s3);
  double red = sv;
  const double t2 = sv * sv;
  for (int a = 1; a <= c; ++a) red -= __shfl_sync(0xffffffffu, t2, (a * KB + kk_lane) & 31);
  return TablePass{sv, red};
}

// Marker column i >= p of the marker operand Mop[k][q][i][kk] (nk slabs) is zero: padding to the marker tile.
__device__ __forceinline__ void zero_marker_column(double* __restrict__ Mop, int64_t i, int64_t p_pad, int n_pad,
                                                  int nk, int lane) {
  const int nq = n_pad / KC;
  for (int k = 0; k < nk; ++k)
    for (int l = lane; l < n_pad; l += 32) Mop[(((int64_t)k * nq + l / KC) * p_pad + i) * KC + (l % KC)] = 0.0;
}

}  // namespace
}  // namespace blmm
