// Preprocessing kernels of libblmm_b200: kinship, rotation by U', per-h2 weight constants, per-trait
// null statistics, the weight-folded marker operand, null-grid binning and operand packing.
// None of these is the roofline kernel (that is blmm_scan.cu); they touch each input O(1) times
// and are written for coalesced access and no host round trips.
#include <float.h>
#include <math.h>

#include <algorithm>

#include "blmm_kernels.cuh"
#include "blmm_prep_dev.cuh"

namespace blmm {

namespace {

constexpr int WARPS_PER_BLOCK = 8;

// Lane batches of the table kernels: KB grid points of (1 + c) kinds each per batch of 32 lane slots.
__host__ __device__ inline int table_kb(int c) {
  const int KB = 32 / (1 + c);
  return KB;
}
__host__ __device__ inline int table_batches(int c, int nk) { return (nk + table_kb(c) - 1) / table_kb(c); }

// Dynamic shared memory of the table kernels (the tables and two staged vectors per warp), or 0 when it is over the
// limit and the generic kernel runs instead (BXD-size grid scans: 30 KB and 51 KB).
size_t trait_table_smem(int n_pad, int c, int nk) {
  const size_t table_smem =
      ((size_t)table_batches(c, nk) * n_pad * 32 + (size_t)WARPS_PER_BLOCK * 2 * n_pad) * sizeof(double);
  if (table_smem <= 96 * 1024) return table_smem;
  return 0;
}
size_t marker_table_smem(int n_pad, int c, int nk) {  // + the transposed table and the store offsets
  const int nbatch = table_batches(c, nk);
  const size_t tsmem =
      ((size_t)2 * nbatch * n_pad * 32 + (size_t)WARPS_PER_BLOCK * 2 * n_pad + (size_t)n_pad) * sizeof(double);
  if (tsmem <= 56 * 1024) return tsmem;
  return 0;
}

// -----------------------------------------------------------------------------------------------
// FP64 SIMT GEMM tile (64 x 64 outputs, K step 16, 256 threads, 4 x 4 per thread) used by the two
// setup products: rotation (A = U', B = X, both K-contiguous) and kinship ((G-1/2)(G-1/2)').
// -----------------------------------------------------------------------------------------------
constexpr int GT = 64, GK = 16;

struct RotateOps {
  const double* U;
  const double* X;
  int64_t ldx;
  int n;
  int64_t cols;
  __device__ double a(int row, int k) const { return (row < n && k < n) ? U[(int64_t)k + (int64_t)row * n] : 0.0; }
  __device__ double b(int k, int64_t col) const { return (col < cols && k < n) ? X[(int64_t)k + col * ldx] : 0.0; }
};

// RI = output rows per thread: the row tile is 16*RI (64 .. 128), chosen by the launcher so that the padded row
// count of the result is covered without a mostly-empty second row tile (n_pad = 80 -> RI = 5, one tile).
template <int RI>
__global__ void __launch_bounds__(256) rotate_kernel(RotateOps op, double* __restrict__ out, int64_t ldo,
                                                     int64_t ldo_zero) {
  constexpr int RT = 16 * RI;
  __shared__ double As[GK][RT + 1];
  __shared__ double Bs[GK][GT + 1];
  const int tid = threadIdx.x;
  const int a0 = blockIdx.y * RT;
  const int64_t c0 = (int64_t)blockIdx.x * GT;
  const int tr = tid & 15, tc = tid >> 4;
  double acc[RI][4] = {};
  for (int k0 = 0; k0 < op.n; k0 += GK) {
    {
      const int kk = tid & 15, r = tid >> 4;
#pragma unroll
      for (int i = 0; i < RI; ++i) As[kk][r + 16 * i] = op.a(a0 + r + 16 * i, k0 + kk);
#pragma unroll
      for (int i = 0; i < 4; ++i) Bs[kk][r + 16 * i] = op.b(k0 + kk, c0 + r + 16 * i);
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < GK; ++kk) {
      double av[RI], bv[4];
#pragma unroll
      for (int i = 0; i < RI; ++i) av[i] = As[kk][tr + 16 * i];
#pragma unroll
      for (int j = 0; j < 4; ++j) bv[j] = Bs[kk][tc * 4 + j];
#pragma unroll
      for (int i = 0; i < RI; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fma(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int64_t col = c0 + tc * 4 + j;
    if (col >= op.cols) continue;
#pragma unroll
    for (int i = 0; i < RI; ++i) {
      const int row = a0 + tr + 16 * i;
      if (row < ldo_zero) out[(int64_t)row + col * ldo] = (row < op.n) ? acc[i][j] : 0.0;
    }
  }
}

__global__ void __launch_bounds__(256) kinship_partial_kernel(const double* __restrict__ G, int n, int64_t p,
                                                              int64_t chunk, double* __restrict__ partial) {
  __shared__ double As[GK][GT + 1];
  __shared__ double Bs[GK][GT + 1];
  const int tid = threadIdx.x;
  const int a0 = blockIdx.y * GT, b0 = blockIdx.x * GT;
  const int64_t i0 = (int64_t)blockIdx.z * chunk;
  const int64_t i1 = (i0 + chunk < p) ? i0 + chunk : p;
  const int tr = tid & 15, tc = tid >> 4;
  double acc[4][4] = {};
  for (int64_t k0 = i0; k0 < i1; k0 += GK) {
    {
      // the subject index is the contiguous one: let it be the fast thread index
      const int r = tid & 63, kb = tid >> 6;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int kk = kb + 4 * i;
        const bool kin = (k0 + kk) < i1;
        As[kk][r] = (kin && a0 + r < n) ? G[(int64_t)(a0 + r) + (k0 + kk) * n] - 0.5 : 0.0;
        Bs[kk][r] = (kin && b0 + r < n) ? G[(int64_t)(b0 + r) + (k0 + kk) * n] - 0.5 : 0.0;
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < GK; ++kk) {
      double av[4], bv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) av[i] = As[kk][tr + 16 * i];
#pragma unroll
      for (int j = 0; j < 4; ++j) bv[j] = Bs[kk][tc * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fma(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  double* dst = partial + (int64_t)blockIdx.z * n * n;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int col = b0 + tc * 4 + j;
    if (col >= n) continue;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int row = a0 + tr + 16 * i;
      if (row < n) dst[(int64_t)row + (int64_t)col * n] = acc[i][j];
    }
  }
}

__global__ void kinship_finish_kernel(const double* __restrict__ partial, int nsplit, int n, int64_t p,
                                      double* __restrict__ K) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nn = (int64_t)n * n;
  if (idx >= nn) return;
  double s = 0.0;
  for (int z = 0; z < nsplit; ++z) s += partial[(int64_t)z * nn + idx];  // fixed order: reproducible
  const int a = (int)(idx % n), b = (int)(idx / n);
  K[idx] = (a == b) ? 1.0 : 2.0 * s / (double)p + 0.5;
}

int kinship_nsplit(int n, int64_t p) {
  const int64_t tiles = (int64_t)((n + GT - 1) / GT) * ((n + GT - 1) / GT);
  int64_t ns = 592 / tiles;
  const int64_t maxs = (p + 255) / 256;
  if (ns > maxs) ns = maxs;
  if (ns < 1) ns = 1;
  return (int)ns;
}

// -----------------------------------------------------------------------------------------------
// weight constants
// -----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) weight_consts_kernel(const double* __restrict__ h2_dev, int nk,
                                                            const double* __restrict__ lambda,
                                                            const double* __restrict__ C0, int n, int n_pad,
                                                            int c, WeightConsts wc, int* flags) {
  __shared__ WcShared sh;
  const int k = blockIdx.x;
  const bool ols = (k == nk);
  weight_consts_block(ols, ols ? 0.0 : h2_dev[k], lambda, C0, n, n_pad, c, weight_slot(wc, k, n_pad, c), flags, sh);
}

// The same with the rotation of the covariates folded in (weight_consts_rot_applies): every block rotates the c
// covariate columns itself (rotate_elem: C0 is bit-identical) instead of waiting for a separate launch; the covariate
// rotation sat at the head of the marker-side critical path of every grid scan.
__global__ void __launch_bounds__(128) weight_consts_rot_kernel(const double* __restrict__ h2_dev, int nk,
                                                                const double* __restrict__ lambda,
                                                                const double* __restrict__ U,
                                                                const double* __restrict__ Cov, int n, int n_pad, int c,
                                                                WeightConsts wc, double* __restrict__ C0_out,
                                                                int* flags) {
  extern __shared__ double c_s[];  // [c][n_pad]
  __shared__ WcShared sh;
  for (int idx = threadIdx.x; idx < c * n_pad; idx += 128) {
    const int col = idx / n_pad, a = idx % n_pad;
    const double v = (a < n) ? rotate_elem(U, Cov + (int64_t)col * n, n, a) : 0.0;
    c_s[idx] = v;
    if (blockIdx.x == 0) C0_out[idx] = v;
  }
  __syncthreads();
  const int k = blockIdx.x;
  const bool ols = (k == nk);
  weight_consts_block(ols, ols ? 0.0 : h2_dev[k], lambda, c_s, n, n_pad, c, weight_slot(wc, k, n_pad, c), flags, sh);
}

// ell of wls / wls_multivar (src/wls.jl:72-92) from the weighted rss
__device__ __forceinline__ double null_loglik(double rss, double slw, double lds, int n, int c, LikParams lik,
                                              double* sigma2_out) {
  const double a = lik.prior_a, b = lik.prior_b;
  const double pdf = (b > 0.0) ? b + 2.0 : b;
  const double ab = a * b;
  const double denom = lik.reml ? ((double)(n - c) + pdf) : ((double)n + pdf);
  const double sigma2 = (rss + ab) / denom;
  double ll = -0.5 * (((double)n + b) * log(sigma2) - slw + (rss + ab) / sigma2);
  if (lik.reml) ll += 0.5 * ((double)c * log(sigma2) - lds);
  if (sigma2_out) *sigma2_out = sigma2;
  return ll;
}

// alt-grid weight of grid point k in the single-logarithm scan: e = exp(-2 (ell_k - max_k ell) / n)
__device__ __forceinline__ double alt_e(double ll, double llmax, int n) {
  return exp(-(ll - llmax) * (2.0 / (double)n));
}

__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK)
    trait_stats_kernel(const double* __restrict__ Y0, int64_t m, int n, int n_pad, int c, int nk, WeightConsts wc,
                       LikParams lik, const double* __restrict__ grid_dev, double* __restrict__ Yr,
                       double* __restrict__ ell, double* __restrict__ rss_out, int* __restrict__ best,
                       double* __restrict__ ellmax, double* __restrict__ h2_out, int* bin_count, int* flags) {
  extern __shared__ double smem[];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t j = (int64_t)blockIdx.x * WARPS_PER_BLOCK + wid;
  if (j >= m) return;
  double* yb = smem + (int64_t)wid * n_pad;
  for (int l = lane; l < n_pad; l += 32) yb[l] = Y0[j * n_pad + l];
  __syncwarp();
  // unweighted residual on the covariates (slot nk: w = 1)
  unweighted_residual(yb, weight_slot(wc, nk, n_pad, c), n_pad, c, lane,
                      [&](int l, double y) { Yr[j * n_pad + l] = y; });
  double bestv = -INFINITY;
  int bestk = 0;
  for (int k = 0; k < nk; ++k) {
    double coef[MAXC];
    const double rss = proj_norm2(yb, weight_slot(wc, k, n_pad, c), n_pad, c, lane, coef);
    const double ll = null_loglik(rss, wc.slw[k], wc.lds[k], n, c, lik, nullptr);
    if (lane == 0) {
      ell[(int64_t)k + j * nk] = ll;
      rss_out[(int64_t)k * m + j] = rss;
      if (!(sqrt(rss) > DBL_EPSILON)) atomicExch(&flags[FLAG_ZERO_NORM], 1);
    }
    if (k == 0 || ll > bestv) {  // strict: first maximum wins, as findmax
      bestv = ll;
      bestk = k;
    }
  }
  if (lane == 0) {
    best[j] = bestk;
    ellmax[j] = bestv;
    if (h2_out) h2_out[j] = grid_dev[bestk];
    if (bin_count) atomicAdd(&bin_count[bestk], 1);
  }
}

// Table form of trait_stats_kernel for problems whose weight tables fit in shared memory (trait_table_smem; every
// BXD-size grid scan).  Lane v of a warp owns one (kind a, grid point k) pair: a = 0 accumulates sum_l w_k[l] y_l^2,
// a >= 1 accumulates t_ka = sum_l Q_ka[l] sw_k[l] y_l, in ONE pass over the trait with no cross-lane
// reduction; then rss_k = s_k - sum_a t_ka^2 (Gram form on the trait already residualised without weights, so
// nothing large cancels), and lane k evaluates the log-likelihood of grid point k.  The block's table
// T[batch][l][32] (lane-contiguous: conflict-free) is built once and reused for every trait of the block.
// With fuse.Top (a single batch), also the alt-grid operands: Top, e and et for j < tcol_pad.
__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK, 4)
    trait_stats_table_kernel(const double* __restrict__ Y0, int64_t m, int n, int n_pad, int c, int nk, WeightConsts wc,
                             LikParams lik, const double* __restrict__ grid_dev, double* __restrict__ Yr,
                             double* __restrict__ ell, double* __restrict__ rss_out, int* __restrict__ best,
                             double* __restrict__ ellmax, double* __restrict__ h2_out, int* bin_count, int* flags,
                             TraitFuse fuse) {
  extern __shared__ double smem[];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KB = table_kb(c);
  const int nbatch = table_batches(c, nk);
  double* T = smem;                                   // [nbatch][n_pad][32]
  double* ybase = smem + (size_t)nbatch * n_pad * 32;  // [WARPS_PER_BLOCK][2][n_pad]: residual and its square
  build_weight_table(wc, n, n_pad, c, nk, KB, nbatch, T, nullptr);
  const int a_lane = lane / KB, kk_lane = lane % KB;
  double* yb = ybase + (int64_t)wid * 2 * n_pad;
  double* yb2 = yb + n_pad;
  const double* src = (a_lane == 0) ? yb2 : yb;  // this lane's kind: a = 0 sums w y^2, a >= 1 sums (Q sw) y
  const WeightSlot ols = weight_slot(wc, nk, n_pad, c);  // slot nk: w = 1
  const int64_t jend = fuse.Top ? fuse.tcol_pad : m;
  for (int64_t j = (int64_t)blockIdx.x * WARPS_PER_BLOCK + wid; j < jend; j += (int64_t)gridDim.x * WARPS_PER_BLOCK) {
    if (j >= m) {
      // padding columns of the packed operand and of the per-k scalars
      for (int l = lane; l < n_pad; l += 32) fuse.Top[((int64_t)(l / KC) * fuse.tcol_pad + j) * KC + (l % KC)] = 0.0;
      for (int k = lane; k < nk; k += 32) {
        fuse.e[(int64_t)k * fuse.tcol_pad + j] = 1.0;
        fuse.et[(int64_t)k * fuse.tcol_pad + j] = 0.0;
      }
      continue;
    }
    for (int l = lane; l < n_pad; l += 32) yb[l] = Y0[j * n_pad + l];
    __syncwarp();
    unweighted_residual(yb, ols, n_pad, c, lane, [&](int l, double y) {
      yb2[l] = y * y;
      Yr[j * n_pad + l] = y;
      if (fuse.Top) fuse.Top[((int64_t)(l / KC) * fuse.tcol_pad + j) * KC + (l % KC)] = y;
    });
    double bestv = -INFINITY;
    int bestk = 0x7fffffff;
    double ll_mine = 0.0, rss_mine = 1.0;  // lane k's values (single batch), for the fused alt-grid scalars
    for (int bt = 0; bt < nbatch; ++bt) {
      const double rss = table_pass(T + (size_t)bt * n_pad * 32, src, n, c, KB, kk_lane, lane).red;
      const int k = bt * KB + kk_lane;
      const bool valid = (a_lane == 0) && (k < nk);
      const int kc = valid ? k : 0;
      const double ll = null_loglik(rss, wc.slw[kc], wc.lds[kc], n, c, lik, nullptr);
      if (valid) {
        ll_mine = ll;
        rss_mine = rss;
        ell[(int64_t)k + j * nk] = ll;
        rss_out[(int64_t)k * m + j] = rss;
        if (!(sqrt(rss) > DBL_EPSILON)) atomicExch(&flags[FLAG_ZERO_NORM], 1);
        if (ll > bestv) {  // within a lane k only grows, so strict > keeps the first maximum
          bestv = ll;
          bestk = k;
        }
      }
    }
    // first maximum over the grid (findmax): larger value wins, equal values -> smaller k
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, bestv, o);
      const int ok = __shfl_xor_sync(0xffffffffu, bestk, o);
      if (ov > bestv || (ov == bestv && ok < bestk)) {
        bestv = ov;
        bestk = ok;
      }
    }
    if (fuse.Top && lane < nk) {
      // alt-grid scalars (as alt_scalars_kernel); one batch, so lane k still holds its own ell and rss
      const double ev = alt_e(ll_mine, bestv, n);
      fuse.e[(int64_t)lane * fuse.tcol_pad + j] = ev;
      fuse.et[(int64_t)lane * fuse.tcol_pad + j] = ev / rss_mine;
    }
    if (lane == 0) {
      if (bestk == 0x7fffffff) bestk = 0;  // every log-likelihood NaN: as findmax on NaNs, first index
      best[j] = bestk;
      ellmax[j] = bestv;
      if (h2_out) h2_out[j] = grid_dev[bestk];
      if (bin_count) atomicAdd(&bin_count[bestk], 1);
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK)
    marker_operand_kernel(const double* __restrict__ G0, int64_t p, int64_t p_pad, int n, int n_pad, int c, int nk,
                          WeightConsts wc, int fold_sw, double* __restrict__ Mop, int* flags) {
  extern __shared__ double smem[];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * WARPS_PER_BLOCK + wid;
  if (i >= p_pad) return;
  if (i >= p) {
    zero_marker_column(Mop, i, p_pad, n_pad, nk, lane);
    return;
  }
  const int nq = n_pad / KC;
  double* gb = smem + (int64_t)wid * n_pad;
  for (int l = lane; l < n_pad; l += 32) gb[l] = G0[i * n_pad + l];
  __syncwarp();
  for (int k = 0; k < nk; ++k) {
    const WeightSlot s = weight_slot(wc, k, n_pad, c);
    double coef[MAXC];
    const double nrm = sqrt(proj_norm2(gb, s, n_pad, c, lane, coef));
    if (lane == 0 && !(nrm > DBL_EPSILON)) atomicExch(&flags[FLAG_ZERO_NORM], 1);
    const double inv = 1.0 / nrm;
    for (int l = lane; l < n_pad; l += 32) {
      const double z = proj_elem(gb, s.sw, s.Q, n_pad, c, l, coef);
      Mop[(((int64_t)k * nq + l / KC) * p_pad + i) * KC + (l % KC)] = (fold_sw ? s.sw[l] * z : z) * inv;
    }
  }
}

// Table form of marker_operand_kernel for the weight-folded operand of the grid scans (fold_sw), when the
// per-block tables fit in shared memory (marker_table_smem).  As in trait_stats_table_kernel lane v owns one (kind a,
// grid point k) pair and gets s_k = sum_l w_k g_l^2 and t_ka = sum_l Q_ka sw_k g_l in one pass without cross-lane
// reductions (||P_k(sw_k g)||^2 = s_k - sum_a t_ka^2; g is first residualised without weights on the covariates, which
// P_k annihilates anyway, so nothing large cancels).  The second pass writes sw_k P_k(sw_k g) / ||.|| =
// (w_k g - sum_a (Q_ka sw_k) t_ka) / ||.|| from the same table entries, read through a transposed copy so that
// lanes walking along l do not collide on one bank.
__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK, 4)
    marker_operand_table_kernel(const double* __restrict__ G0, int64_t p, int64_t p_pad, int n, int n_pad, int c, int nk,
                                WeightConsts wc, double* __restrict__ Mop, int* flags) {
  extern __shared__ double smem[];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KB = table_kb(c);
  const int nbatch = table_batches(c, nk);
  const int nq = n_pad / KC;
  double* T = smem;                                       // [nbatch][n_pad][32]  (lane-contiguous)
  double* Tt = T + (size_t)nbatch * n_pad * 32;           // [nbatch][32][n_pad]  (l-contiguous)
  double* gbase = Tt + (size_t)nbatch * n_pad * 32;       // [WARPS_PER_BLOCK][2][n_pad]
  // [n_pad] offset of element l inside one k-slab for marker 0: (l / KC) p_pad KC + l % KC (marker i adds i KC)
  int64_t* off_s = reinterpret_cast<int64_t*>(gbase + (size_t)WARPS_PER_BLOCK * 2 * n_pad);
  for (int l = threadIdx.x; l < n_pad; l += blockDim.x) off_s[l] = (int64_t)(l / KC) * p_pad * KC + (l % KC);
  build_weight_table(wc, n, n_pad, c, nk, KB, nbatch, T, Tt);
  const int a_lane = lane / KB, kk_lane = lane % KB;
  double* gb = gbase + (int64_t)wid * 2 * n_pad;
  double* gb2 = gb + n_pad;
  const double* src = (a_lane == 0) ? gb2 : gb;
  const WeightSlot ols = weight_slot(wc, nk, n_pad, c);  // slot nk: w = 1
  for (int64_t i = (int64_t)blockIdx.x * WARPS_PER_BLOCK + wid; i < p_pad; i += (int64_t)gridDim.x * WARPS_PER_BLOCK) {
    if (i >= p) {
      zero_marker_column(Mop, i, p_pad, n_pad, nk, lane);
      continue;
    }
    for (int l = lane; l < n_pad; l += 32) gb[l] = G0[i * n_pad + l];
    __syncwarp();
    unweighted_residual(gb, ols, n_pad, c, lane, [&](int l, double g) { gb2[l] = g * g; });
    for (int bt = 0; bt < nbatch; ++bt) {
      const TablePass tp = table_pass(T + (size_t)bt * n_pad * 32, src, n, c, KB, kk_lane, lane);
      const double sv = tp.sv;  // lane (a, kk): a = 0 -> sum w g^2, a >= 1 -> t_a
      const double nrm = sqrt(tp.red);
      const bool valid0 = (a_lane == 0) && (bt * KB + kk_lane < nk);
      if (valid0 && !(nrm > DBL_EPSILON)) atomicExch(&flags[FLAG_ZERO_NORM], 1);
      const double inv_mine = 1.0 / nrm;  // meaningful in lanes (0, kk)
      const int kcount = (nk - bt * KB) < KB ? (nk - bt * KB) : KB;
      const double* Ttb = Tt + (size_t)bt * 32 * n_pad;
      // this lane's destination offsets inside one k-slab do not depend on k: no division in the store loop
      // (ncu: the kernel was bound by the integer instructions of its index arithmetic, not by FP64 or memory)
      const int64_t slab = (int64_t)nq * p_pad * KC;
      for (int kk = 0; kk < kcount; ++kk) {
        const double inv = __shfl_sync(0xffffffffu, inv_mine, kk);
        double tk[MAXC];
#pragma unroll
        for (int a = 0; a < MAXC; ++a)
          if (a < c) tk[a] = __shfl_sync(0xffffffffu, sv, ((a + 1) * KB + kk) & 31);
        double* out_k = Mop + (int64_t)(bt * KB + kk) * slab + i * KC;
        const double* wk = Ttb + (size_t)kk * n_pad;
        for (int l2 = lane; l2 < n_pad; l2 += 32) {
          double z = wk[l2] * gb[l2];  // w_k g
#pragma unroll
          for (int a = 0; a < MAXC; ++a)
            if (a < c) z = fma(-Ttb[((size_t)(a + 1) * KB + kk) * n_pad + l2], tk[a], z);
          out_k[off_s[l2]] = z * inv;
        }
      }
    }
    __syncwarp();
  }
}

// alt-grid trait scalars: e[k][j] = alt_e(ell[k,j], ellmax_j), et = e / rss; pads e = 1, et = 0.
__global__ void alt_scalars_kernel(const double* __restrict__ ell, const double* __restrict__ rss,
                                   const double* __restrict__ ellmax, int64_t m, int64_t tcol_pad, int nk, int n,
                                   double* __restrict__ e, double* __restrict__ et) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= tcol_pad) return;
  if (j >= m) {
    for (int k = 0; k < nk; ++k) {
      e[(int64_t)k * tcol_pad + j] = 1.0;
      et[(int64_t)k * tcol_pad + j] = 0.0;
    }
    return;
  }
  const double emax = ellmax[j];
  for (int k = 0; k < nk; ++k) {
    const double ev = alt_e(ell[(int64_t)k + j * nk], emax, n);
    e[(int64_t)k * tcol_pad + j] = ev;
    et[(int64_t)k * tcol_pad + j] = ev / rss[(int64_t)k * m + j];
  }
}

__global__ void bin_layout_kernel(const int* __restrict__ bin_count, int nk, int tile, int n_tiles_max,
                                  int* bin_start, int* bin_cursor, int* tile_k0, int* n_tiles) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  int pos = 0, t = 0;
  for (int b = 0; b < nk; ++b) {
    bin_start[b] = pos;
    bin_cursor[b] = 0;
    const int nt = (bin_count[b] + tile - 1) / tile;
    for (int i = 0; i < nt; ++i) tile_k0[t++] = b;
    pos += nt * tile;
  }
  *n_tiles = t;
  for (; t < n_tiles_max; ++t) tile_k0[t] = 0;
}

__global__ void bin_scatter_kernel(const int* __restrict__ best, const double* __restrict__ rss, int64_t m,
                                   const int* __restrict__ bin_start, int* bin_cursor, int* __restrict__ col_map,
                                   double* __restrict__ et) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = j < m;
  const unsigned active = __ballot_sync(0xffffffffu, live);
  if (!live) return;
  const int b = best[j];
  // one atomic per (warp, bin) instead of one per trait: the lanes of a warp that chose the same grid point
  // take consecutive slots (there are only |grid| cursors for all m traits)
  const unsigned peers = __match_any_sync(active, b);
  const int lane = threadIdx.x & 31;
  const int leader = __ffs(peers) - 1;
  int base = 0;
  if (lane == leader) base = atomicAdd(&bin_cursor[b], __popc(peers));
  base = __shfl_sync(peers, base, leader);
  const int pos = bin_start[b] + base + __popc(peers & ((1u << lane) - 1u));
  col_map[pos] = (int)j;
  et[pos] = 1.0 / rss[(int64_t)b * m + j];
}

__global__ void pack_traits_kernel(const double* __restrict__ Yr, const int* __restrict__ col_map, int64_t m,
                                   int64_t tcol_pad, int n_pad, int64_t total, const double* __restrict__ scale2,
                                   double* __restrict__ Top) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int kk = (int)(idx % KC);
  const int64_t pos = (idx / KC) % tcol_pad;
  const int q = (int)(idx / (KC * tcol_pad));
  int64_t src = col_map ? (int64_t)col_map[pos] : (pos < m ? pos : -1);
  double v = (src >= 0) ? Yr[src * n_pad + q * KC + kk] : 0.0;
  if (scale2) v *= sqrt(scale2[pos]);
  Top[idx] = v;
}

__global__ void pack_perms_kernel(const double* __restrict__ z, const double* __restrict__ rss,
                                  const int32_t* __restrict__ perm_idx, int64_t nperms, int n, int64_t tcol_pad,
                                  int64_t total, double* __restrict__ Top, double* __restrict__ et,
                                  int* __restrict__ flags) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int kk = (int)(idx % KC);
  const int64_t s = (idx / KC) % tcol_pad;
  const int q = (int)(idx / (KC * tcol_pad));
  const int l = q * KC + kk;
  double v = 0.0;
  if (s <= nperms && l < n) {
    int src = (s == 0) ? l : perm_idx[(int64_t)l + (s - 1) * n];
    if ((unsigned)src >= (unsigned)n) {  // not a 0-based index into 1:n (e.g. Julia's 1-based n): refuse, do not read
      flags[FLAG_PERM_RANGE] = 1;
      src = 0;
    }
    v = z[src] / sqrt(*rss);
  }
  Top[idx] = v;
  if (q == 0 && kk == 0) et[s] = 1.0;
}

__global__ void __launch_bounds__(32) null_residual_kernel(const double* __restrict__ Yr, int n, int n_pad, int c,
                                                           WeightConsts wc, double* __restrict__ z,
                                                           double* __restrict__ rss) {
  double coef[MAXC];
  const double s = proj_norm2(Yr, weight_slot(wc, 0, n_pad, c), n_pad, c, threadIdx.x, coef, z);
  if (threadIdx.x == 0) *rss = s;
}

// -----------------------------------------------------------------------------------------------
// Rotation for large n (n >= 128, e.g. the scaled configuration's n = 1000, where U'G is 2e11 flop): the same product
// as rotate_kernel on the FP64 tensor cores.  out(a, col) = sum_b U[b + a n] X[b + col ldx]: both operands are
// K-contiguous, exactly the DMMA m8n8k4 "row.col" fragment layout.  128 x 128 output tile per CTA, 8 warps of
// 64 x 32 (8 x 4 atoms), K streamed in chunks of KC = 20 through a [row][KC] shared-memory tile (the conflict-free
// stride of the scan kernels); the next chunk's global loads are in flight in registers while the current one is
// multiplied.
// -----------------------------------------------------------------------------------------------
constexpr int RD_T = 128;
__global__ void __launch_bounds__(256, 1)
    rotate_dmma_kernel(const double* __restrict__ U, const double* __restrict__ X, int64_t ldx, int n, int64_t cols,
                       double* __restrict__ out, int64_t ldo, int64_t ldo_zero) {
  __shared__ __align__(16) double As[RD_T * KC];
  __shared__ __align__(16) double Bs[RD_T * KC];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int wa = warp & 1, wc = warp >> 1;
  const int a0 = blockIdx.y * RD_T;
  const int64_t c0 = (int64_t)blockIdx.x * RD_T;
  constexpr int PER = RD_T * KC / 256;  // 10 elements of each operand per thread and chunk
  double ra[PER], rb[PER];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int idx = tid + i * 256;
      const int r = idx / KC, kk = idx % KC;
      const int k = k0 + kk;
      const int arow = a0 + r;
      const int64_t bcol = c0 + r;
      ra[i] = (arow < n && k < n) ? U[(int64_t)k + (int64_t)arow * n] : 0.0;
      rb[i] = (bcol < cols && k < n) ? X[(int64_t)k + bcol * ldx] : 0.0;
    }
  };
  double acc[8][4][2];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  fetch(0);
  const double* ap = As + (wa * 64 + g) * KC + t;
  const double* bp = Bs + (wc * 32 + g) * KC + t;
  for (int k0 = 0; k0 < n; k0 += KC) {
    __syncthreads();  // the previous chunk's fragments have been read
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      As[tid + i * 256] = ra[i];
      Bs[tid + i * 256] = rb[i];
    }
    __syncthreads();
    if (k0 + KC < n) fetch(k0 + KC);
#pragma unroll
    for (int s4 = 0; s4 < KC / 4; ++s4) {
      double af[8], bf[4];
#pragma unroll
      for (int i = 0; i < 8; ++i) af[i] = ap[i * 8 * KC + s4 * 4];
#pragma unroll
      for (int j = 0; j < 4; ++j) bf[j] = bp[j * 8 * KC + s4 * 4];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int cc = 0; cc < 2; ++cc) {
      const int64_t col = c0 + wc * 32 + j * 8 + 2 * t + cc;
      if (col >= cols) continue;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int row = a0 + wa * 64 + i * 8 + g;
        if (row < ldo_zero) out[(int64_t)row + col * ldo] = acc[i][j][cc];  // rows >= n multiplied zeros: 0
      }
    }
}

}  // namespace

// -----------------------------------------------------------------------------------------------
// launchers
// -----------------------------------------------------------------------------------------------
int launch_rotate(const double* U, const double* X, int64_t ldx, double* out, int64_t ldo, int64_t ldo_zero,
                  int n, int64_t cols, cudaStream_t stream) {
  if (cols <= 0) return 0;
  if (n >= 128 && cols >= 64) {
    // large n: tensor-core rotation (at n = 1000 the SIMT tile kernel ran at ~15 TF/s: 13 ms for U'G of the scaled problem)
    dim3 grid((unsigned)((cols + RD_T - 1) / RD_T), (unsigned)((ldo_zero + RD_T - 1) / RD_T));
    rotate_dmma_kernel<<<grid, 256, 0, stream>>>(U, X, ldx, n, cols, out, ldo, ldo_zero);
    return 1;
  }
  RotateOps op{U, X, ldx, n, cols};
  // row tile: the smallest of 64/80/96/112/128 that covers the padded rows in as few tiles as possible
  const int64_t tiles128 = (ldo_zero + 127) / 128;
  const int ri = (int)std::min<int64_t>(8, std::max<int64_t>(4, ((ldo_zero + tiles128 - 1) / tiles128 + 15) / 16));
  dim3 grid((unsigned)((cols + GT - 1) / GT), (unsigned)((ldo_zero + 16 * ri - 1) / (16 * ri)));
  switch (ri) {
    case 4: rotate_kernel<4><<<grid, 256, 0, stream>>>(op, out, ldo, ldo_zero); break;
    case 5: rotate_kernel<5><<<grid, 256, 0, stream>>>(op, out, ldo, ldo_zero); break;
    case 6: rotate_kernel<6><<<grid, 256, 0, stream>>>(op, out, ldo, ldo_zero); break;
    case 7: rotate_kernel<7><<<grid, 256, 0, stream>>>(op, out, ldo, ldo_zero); break;
    default: rotate_kernel<8><<<grid, 256, 0, stream>>>(op, out, ldo, ldo_zero); break;
  }
  return 1;
}

int64_t kinship_workspace_doubles(int n, int64_t p) { return (int64_t)kinship_nsplit(n, p) * n * n; }

int launch_kinship(const double* G, int n, int64_t p, double* K, double* partial, cudaStream_t stream) {
  const int ns = kinship_nsplit(n, p);
  int64_t chunk = (p + ns - 1) / ns;
  chunk = round_up(chunk, GK);
  const int nsplit = (int)((p + chunk - 1) / chunk);
  dim3 grid((n + GT - 1) / GT, (n + GT - 1) / GT, nsplit);
  kinship_partial_kernel<<<grid, 256, 0, stream>>>(G, n, p, chunk, partial);
  const int64_t nn = (int64_t)n * n;
  kinship_finish_kernel<<<(unsigned)((nn + 255) / 256), 256, 0, stream>>>(partial, nsplit, n, p, K);
  return 2;
}

int launch_weight_consts(const double* h2_dev, int nk, const double* lambda, const double* C0, int n,
                         int n_pad, int c, WeightConsts wc, int* flags, cudaStream_t stream) {
  weight_consts_kernel<<<nk + 1, 128, 0, stream>>>(h2_dev, nk, lambda, C0, n, n_pad, c, wc, flags);
  return 1;
}

// one thread per rotated covariate element, each a length-n dot product: worth folding in for small n only
bool weight_consts_rot_applies(int n) { return n <= 128; }

int launch_weight_consts_rot(const double* h2_dev, int nk, const double* lambda, const double* U, const double* Cov,
                             int n, int n_pad, int c, WeightConsts wc, double* C0, int* flags, cudaStream_t stream) {
  weight_consts_rot_kernel<<<nk + 1, 128, (size_t)c * n_pad * sizeof(double), stream>>>(h2_dev, nk, lambda, U, Cov, n,
                                                                                         n_pad, c, wc, C0, flags);
  return 1;
}

namespace {
// Blocks of a table kernel over `cols` warp columns: one resident wave (4 blocks per SM by shared memory); fewer,
// longer-lived blocks were measured slower, the kernels being bound by per-column latency, not by building the tables.
// Raises the kernel's dynamic shared-memory limit when smem needs more than the default 48 KB.
template <class Kernel>
unsigned table_wave(Kernel* kernel, size_t smem, int64_t cols, int sm_count) {
  if (smem > 48 * 1024) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  return (unsigned)std::min<int64_t>((cols + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK, (int64_t)sm_count * 4);
}
}  // namespace

int launch_trait_stats(const double* Y0, int64_t m, int n, int n_pad, int c, int nk, WeightConsts wc,
                       LikParams lik, const double* grid_dev, double* Yr, double* ell, double* rss,
                       int* best, double* ellmax, double* h2_out, int* bin_count, int* flags, const TraitFuse* fuse,
                       int sm_count, cudaStream_t stream) {
  const size_t table_smem = trait_table_smem(n_pad, c, nk);
  bool fused = false;
  if (table_smem) {
    // with one lane batch, lane k holds grid point k's ell and rss at the end: the alt-grid operands come for free
    const TraitFuse f = (fuse && table_batches(c, nk) == 1) ? *fuse : TraitFuse{};
    fused = f.Top != nullptr;
    const int64_t cols = fused ? f.tcol_pad : m;
    trait_stats_table_kernel<<<table_wave(trait_stats_table_kernel, table_smem, cols, sm_count), 32 * WARPS_PER_BLOCK,
                               table_smem, stream>>>(Y0, m, n, n_pad, c, nk, wc, lik, grid_dev, Yr, ell, rss, best,
                                                     ellmax, h2_out, bin_count, flags, f);
  } else {
    const size_t smem = (size_t)WARPS_PER_BLOCK * n_pad * sizeof(double);
    if (smem > 48 * 1024)
      cudaFuncSetAttribute(trait_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const unsigned blocks = (unsigned)((m + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK);
    trait_stats_kernel<<<blocks, 32 * WARPS_PER_BLOCK, smem, stream>>>(Y0, m, n, n_pad, c, nk, wc, lik, grid_dev, Yr,
                                                                        ell, rss, best, ellmax, h2_out, bin_count,
                                                                        flags);
  }
  if (!fuse || fused) return 1;
  alt_scalars_kernel<<<(unsigned)((fuse->tcol_pad + 255) / 256), 256, 0, stream>>>(ell, rss, ellmax, m, fuse->tcol_pad,
                                                                                   nk, n, fuse->e, fuse->et);
  return 2 + launch_pack_traits(Yr, nullptr, m, fuse->tcol_pad, n_pad, nullptr, fuse->Top, stream);
}

int launch_marker_operand(const double* G0, int64_t p, int64_t p_pad, int n, int n_pad, int c, int nk,
                          WeightConsts wc, bool fold_sw, double* Mop, int* flags, int sm_count, cudaStream_t stream) {
  if (const size_t tsmem = fold_sw ? marker_table_smem(n_pad, c, nk) : 0) {
    marker_operand_table_kernel<<<table_wave(marker_operand_table_kernel, tsmem, p_pad, sm_count), 32 * WARPS_PER_BLOCK,
                                  tsmem, stream>>>(G0, p, p_pad, n, n_pad, c, nk, wc, Mop, flags);
    return 1;
  }
  const size_t smem = (size_t)WARPS_PER_BLOCK * n_pad * sizeof(double);
  if (smem > 48 * 1024)
    cudaFuncSetAttribute(marker_operand_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  const unsigned blocks = (unsigned)((p_pad + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK);
  marker_operand_kernel<<<blocks, 32 * WARPS_PER_BLOCK, smem, stream>>>(G0, p, p_pad, n, n_pad, c, nk, wc,
                                                                         fold_sw ? 1 : 0, Mop, flags);
  return 1;
}

int launch_null_bins(const int* best, const double* rss, int64_t m, int nk, int tile, int64_t tcol_pad,
                     int* bin_count, int* bin_start, int* bin_cursor, int* tile_k0, int* n_tiles,
                     int* col_map, double* et, cudaStream_t stream) {
  cudaMemsetAsync(col_map, 0xFF, (size_t)tcol_pad * sizeof(int), stream);
  cudaMemsetAsync(et, 0, (size_t)tcol_pad * sizeof(double), stream);
  bin_layout_kernel<<<1, 32, 0, stream>>>(bin_count, nk, tile, (int)(tcol_pad / tile), bin_start, bin_cursor,
                                          tile_k0, n_tiles);
  bin_scatter_kernel<<<(unsigned)((m + 255) / 256), 256, 0, stream>>>(best, rss, m, bin_start, bin_cursor, col_map,
                                                                       et);
  return 2;
}

int launch_pack_traits(const double* Yr, const int* col_map, int64_t m, int64_t tcol_pad, int n_pad,
                       const double* scale2, double* Top, cudaStream_t stream) {
  const int64_t total = (int64_t)n_pad * tcol_pad;
  pack_traits_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(Yr, col_map, m, tcol_pad, n_pad, total,
                                                                           scale2, Top);
  return 1;
}

int launch_pack_perms(const double* z, const double* rss, const int32_t* perm_idx, int64_t nperms, int n,
                      int n_pad, int64_t tcol_pad, double* Top, double* et, int* flags, cudaStream_t stream) {
  const int64_t total = (int64_t)n_pad * tcol_pad;
  pack_perms_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(z, rss, perm_idx, nperms, n, tcol_pad,
                                                                          total, Top, et, flags);
  return 1;
}

int launch_null_residual(const double* Yr, int n, int n_pad, int c, WeightConsts wc, double* z, double* rss,
                         cudaStream_t stream) {
  null_residual_kernel<<<1, 32, 0, stream>>>(Yr, n, n_pad, c, wc, z, rss);
  return 1;
}

}  // namespace blmm
