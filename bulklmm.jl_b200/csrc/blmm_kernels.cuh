// Kernel launchers of libblmm_b200 (host-callable).  Every launcher enqueues on `stream`, never
// synchronises, and returns the number of kernels it launched (for blmm_launch_count).
//
// Internal layouts (all Float64):
//   padded column-major : X[col * n_pad + l],          l < n_pad = nq*KC, rows >= n are zero
//   K-chunked panel     : X[(q * ncol_pad + col) * KC + kk],   l = q*KC + kk      (blmm_common.cuh)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "blmm_common.cuh"

namespace blmm {

// Run-time covariate count to template argument: f(std::integral_constant<int, C>{}) for the C in [LO, HI] equal to
// c; returns false, calling nothing, when c is outside the range.
template <int LO, int HI, class F>
bool dispatch_c(int c, F&& f) {
  if constexpr (LO > HI) {
    return false;
  } else {
    if (c == LO) {
      f(std::integral_constant<int, LO>{});
      return true;
    }
    return dispatch_c<LO + 1, HI>(c, f);
  }
}

// ---- preprocessing (blmm_prep.cu) -------------------------------------------------------------

// out(a, col) = sum_b U[b + a*n] * X[b + col*ldx]   (Ut*X of src/transform_helpers.jl:34,49);
// out is column-major with leading dimension ldo >= n; rows [n, ldo_zero) are zero-filled.
int launch_rotate(const double* U, const double* X, int64_t ldx, double* out, int64_t ldo, int64_t ldo_zero,
                  int n, int64_t cols, cudaStream_t stream);

// K = 2 (G - 1/2)(G - 1/2)' / p + 1/2, diag := 1   (src/kinship.jl:4-14).  G: n x p (ld n).
// `partial` is workspace of kinship_workspace_doubles(n, p) doubles.
int64_t kinship_workspace_doubles(int n, int64_t p);
int launch_kinship(const double* G, int n, int64_t p, double* K, double* partial, cudaStream_t stream);

// Per-weight-vector constants for nk heritabilities h2[k] (device array), plus (slot nk) the
// unweighted w = 1 case used to pre-residualise traits:
//   w = 1 / (h2/(1-h2) * lambda + 1)                         makeweights, src/lmm.jl:15-33
//   sw = sqrt(w);   Q = orthonormal basis of span(sw .* C0)  (the Q of `qr(XX)`, src/wls.jl:58)
//   slw = sum log w;   lds = log det (C0' W C0) = 2 log|det R|   (src/wls.jl:66)
struct WeightConsts {
  double* w;    // [nk+1][n_pad]
  double* sw;   // [nk+1][n_pad]
  double* Q;    // [nk+1][c][n_pad]
  double* slw;  // [nk+1]
  double* lds;  // [nk+1]
};
int launch_weight_consts(const double* h2_dev, int nk, const double* lambda, const double* C0, int n,
                         int n_pad, int c, WeightConsts wc, int* flags, cudaStream_t stream);

// The same from the UNROTATED covariates (Cov: n x c, ld n), for the n where weight_consts_rot_applies: each block
// rotates them by U' itself and block 0 also writes C0.
bool weight_consts_rot_applies(int n);
int launch_weight_consts_rot(const double* h2_dev, int nk, const double* lambda, const double* U, const double* Cov,
                             int n, int n_pad, int c, WeightConsts wc, double* C0, int* flags, cudaStream_t stream);

struct LikParams {  // wls / wls_multivar scalars, src/wls.jl:72-92, 150-170
  double prior_a, prior_b;
  int reml;
};

// One warp per trait.  Reads Y0 (padded column-major), writes
//   Yr   : Y0 residualised (unweighted) on C0 — spans the same null model, less cancellation
//   ell  : [ngrid x m] column-major null log-likelihoods            src/bulkscan_helpers.jl:267-269
//   rss  : [nk][m] weighted residual sum of squares (= squared norm of the residualised trait)
//   best : [m] first arg-max over k of ell (findmax, src/bulkscan_helpers.jl:204-211)
//   ellmax: [m] max_k ell;   h2_out (optional): grid[best];   bin_count (optional): histogram of best
// `fuse` (optional, alt-grid): also the scan's trait operands for j < tcol_pad — Top[q][j][kk] = Yr (pads 0),
// e[k][j] = exp(-2 (ell[k,j] - ellmax_j) / n) (pads 1), et = e / rss (pads 0) — in the statistics kernel itself when
// its table form holds every grid point in one lane batch, else by two more kernels.
struct TraitFuse {
  double* Top;
  double* e;
  double* et;
  int64_t tcol_pad;
};
int launch_trait_stats(const double* Y0, int64_t m, int n, int n_pad, int c, int nk, WeightConsts wc,
                       LikParams lik, const double* grid_dev, double* Yr, double* ell, double* rss,
                       int* best, double* ellmax, double* h2_out, int* bin_count, int* flags, const TraitFuse* fuse,
                       int sm_count, cudaStream_t stream);

// One warp per marker: x = P_k (sw_k .* g_i) / ||P_k (sw_k .* g_i)||  (the normalised X00 column of
// weighted_liteqtl + computeR_LMM, src/bulkscan_helpers.jl:175-201, 47-64).
//   fold_sw = true : Mop[k][q][i][kk] = sw_k .* x — the trait-side sqrt(w) and projector folded in, so
//                    the trait operand (unweighted residual) is weight independent (grid scans);
//   fold_sw = false: Mop = x, for trait operands that are already weighted and projected
//                    (permutations of the re-weighted null residual, src/scan.jl:531-541; w = 1 slot).
int launch_marker_operand(const double* G0, int64_t p, int64_t p_pad, int n, int n_pad, int c, int nk,
                          WeightConsts wc, bool fold_sw, double* Mop, int* flags, int sm_count, cudaStream_t stream);

// null-grid binning: lay the traits out bin by bin, each bin padded to a multiple of `tile`.
//   tile_k0[t]  : grid index of trait tile t;  n_tiles: number of tiles in use (device scalar)
//   col_map[pos]: trait index at packed position pos, -1 for padding;  et[pos] = 1 / rss[best][j]
int launch_null_bins(const int* best, const double* rss, int64_t m, int nk, int tile, int64_t tcol_pad,
                     int* bin_count, int* bin_start, int* bin_cursor, int* tile_k0, int* n_tiles,
                     int* col_map, double* et, cudaStream_t stream);

// Top[q][pos][kk] = Yr[col_map[pos]][q*KC+kk]  (identity map when col_map == nullptr; pads zero), times
// sqrt(scale2[pos]) when scale2 is given (one-k scans fold et = 1/rss into the trait operand: d^2 et = (d sqrt et)^2)
int launch_pack_traits(const double* Yr, const int* col_map, int64_t m, int64_t tcol_pad, int n_pad,
                       const double* scale2, double* Top, cudaStream_t stream);

// Permutation operand (transform_permute + column normalisation, src/transform_helpers.jl:94-102,
// src/scan.jl:531-536): column 0 = z/||z||, column s>=1 = z[perm_idx[:,s-1]]/||z||, where z is the
// weighted null residual (padded column 0 of Zr) and rss = ||z||^2.
// Also fills et[0..tcol_pad) with 1 (the columns are already normalised).  An index outside 0..n-1 raises
// FLAG_PERM_RANGE (the entry is not read).
int launch_pack_perms(const double* z, const double* rss, const int32_t* perm_idx, int64_t nperms, int n,
                      int n_pad, int64_t tcol_pad, double* Top, double* et, int* flags, cudaStream_t stream);

// z = P (sw .* y): the re-weighted null residual `copy_r0` of transform_reweight
// (src/transform_helpers.jl:71-82) for one trait, weight slot 0 of wc.  Writes z (n_pad) and rss.
int launch_null_residual(const double* Yr, int n, int n_pad, int c, WeightConsts wc, double* z,
                         double* rss, cudaStream_t stream);

// ---- heritability fit (blmm_fit.cu) -----------------------------------------------------------
// fitlmm per trait: gridbrent over [0,1] in optim_interval pieces (src/lmm.jl:56-86,
// src/gridbrent.jl:9-24, Optim.jl Brent).  One warp per trait.  Outputs length m (nullable).
// Qc, ld_r: the w = 1 weight slot's orthonormal covariate basis (C0 = Qc R) and log det(C0'C0) = log det(R'R) (device
// scalar), which turns REML's log det(Qc'WQc) into log det(C0'WC0).
int launch_fit_h2(const double* Yr, int64_t m, int n, int n_pad, int c, const double* Qc, const double* ld_r,
                  const double* lambda, LikParams lik, int optim_interval, double* h2, double* sigma2,
                  double* ell, int* flags, cudaStream_t stream);

// The single-trait prologue of scan with permutations in one launch, for the n where null_fit_chain_applies (else the
// caller runs the separate launches): C0 = U'Cov (n_pad x c), Yr = residual of U'y on C0, h2 / sigma2 = fitlmm,
// wc slot 0 = constants at h2 (slot 1 = the unweighted ones), z = P (sw .* Yr) with zrss = ||z||^2.
// U: n x n (ld n), y: n, Cov: n x c (ld n) — unrotated device inputs.
bool null_fit_chain_applies(int n);
int launch_null_fit_chain(const double* U, const double* y, const double* Cov, const double* lambda, int n, int n_pad,
                          int c, LikParams lik, int optim_interval, double* C0, double* Yr, WeightConsts wc, double* h2,
                          double* sigma2, double* z, double* zrss, int* flags, cudaStream_t stream);

// scan_alt (src/scan.jl:397-453) for ONE trait y (residualised, padded): per-marker Brent with covariates
// [C0 g_i] (c + 1 <= MAXC columns), lod_i = (ell_alt_i - ell_null) / ln 10, h2_each[i] (nullable).
// h2_null: device scalar from launch_fit_h2; ell_null: device scalar workspace; Qc, ld_r as for launch_fit_h2.
int launch_scan_alt(const double* y, const double* G0, int64_t p, int n, int n_pad, int c, const double* Qc,
                    const double* ld_r, const double* lambda, LikParams lik, int optim_interval, const double* h2_null, double* ell_null,
                    double* lod, double* h2_each, cudaStream_t stream);

// ---- the scans (blmm_scan.cu, blmm_scan_stream.cu) -----------------------------------------------
// For every (marker i, packed trait column s):
//     d_k = sum_l Mop[k][i][l] * Top[s][l]
//     v_k = e[k][s] - d_k^2 * et[k][s]                      k in the trait tile's k-list
//     L   = -(n/2) * log10( min_k v_k )
//     h2  = grid[#strict improvements of the running min]   (tmax! counter semantics) or grid[argmin]
// = bulkscan_alt_grid (src/bulkscan.jl:445-526, tmax! src/bulkscan_helpers.jl:330-350) in its
// single-logarithm form; with a one-element k-list and e = 1 it is weighted_liteqtl + r2lod
// (src/bulkscan_helpers.jl:175-201, 22-24) for null-grid bins and permutations.
// launch_scan keeps the trait tile in shared memory (nq <= SCAN_MAX_NQ), launch_scan_stream_grid streams K; both, and
// launch_scan_exact (bulkscan_null, EXACT mode), return 0 and launch nothing for fields their kernel does not implement.
struct ScanParams {
  const double* Top;       // trait operand   [nq][tcol_pad][KC]; EXACT: c+2 column kinds per trait (launch_exact_columns)
  const double* Mop;       // marker operand  [nk_total][nq][p_pad][KC]  (EXACT: one slab, w = 1)
  const double* e;         // [nk][tcol_pad] or nullptr (=> 1)
  const double* et;        // [nk][tcol_pad], required (not read in EXACT mode)
  int et_folded;           // e == nullptr only: et is already folded into the trait operand (columns scaled by
                           // sqrt(et)), v = 1 - d^2; resident kernel only
  const int* tile_k0;      // per trait tile: first k (index into Mop); nullptr => 0
  const int* n_tiles_dev;  // device scalar: number of trait tiles in use; nullptr => n_tiles_t
  const int* col_map;      // [tcol_pad] packed column -> output column (-1 = padding); nullptr => identity
  const double* grid;      // device copy of the h2 grid (for the h2 panel), ngrid <= 255 values
  int ngrid;
  double* L;               // p x m output, ld = ldL (nullptr => not stored)
  double* L0;              // if non-null: output column 0 goes here (length p) and column s >= 1 goes to
                           // column s-1 of L / colmax (scan_perms_lite's lod vs L_perms split, src/scan.jl:545-546)
  double* H2;              // p x m h2 panel, ld = ldL (nullptr => not stored)
  uint8_t* H2idx;          // p x m panel of grid INDICES (h2 = grid[index]), ld = p, one byte each (nullptr => not
                           // stored): what host-buffer calls bring back over PCIe instead of 8-byte values; resident
                           // kernel only
  double* colmax;          // [m] max over markers per output column (nullptr => off); caller zero-fills
  int64_t ldL;
  int nq;                  // K-chunks (ceil(n / KC))
  int p;                   // markers
  int p_pad;               // padded marker count (multiple of the marker tile)
  int64_t m;               // output columns
  int64_t tcol_pad;        // padded packed-trait count (multiple of the trait tile); EXACT: operand columns of Top
  int n_tiles_t;           // trait tiles (upper bound when n_tiles_dev is given); EXACT: tiles of 64 traits
  int nk;                  // k-list length of every trait tile
  int argmax_mode;         // 0 = tmax! counter semantics, 1 = arg-max index
  double half_n;           // n / 2
  PeakRec* peaks;          // non-null: per-trait peaks instead of L / H2 / H2idx / colmax, one record per output column
                           // and warp marker block (peak_blocks; launch_peak_reduce finishes them)
  // K-streamed kernels only
  const double* dyinv;     // EXACT: [n_tiles_t * 64] 1 / (y_j' z_j)
  int band;                // trait tiles per rasterisation band (0 = default)
  unsigned long long* unit_counter;  // device scalar, zero at launch: dynamic unit scheduler (nullptr => round-robin)
};

// Per-trait peak records (ScanParams::peaks): one per output column and block of `block_rows` markers (the marker rows
// of one warp, half a marker tile).  The record of column col and block mb is col * peak_blocks(p_pad, block_rows) + mb.
__host__ __device__ inline int peak_blocks(int p_pad, int block_rows) { return p_pad / block_rows; }

constexpr int SCAN_TT = 128;  // traits per CTA tile
constexpr int SCAN_MT = 64;   // markers per CTA tile
constexpr int SCAN_MAX_NQ = 5;  // largest number of K-chunks for which launch_scan keeps the trait tile resident
int launch_scan(const ScanParams& P, int sm_count, cudaStream_t stream);
int launch_scan_stream_grid(const ScanParams& P, int sm_count, cudaStream_t stream);

// marker atoms (8 markers each, per warp) of the EXACT kernel for c covariates: its c + 2 operand kinds take registers
constexpr int exact_marker_atoms(int c) { return c + 2 <= 5 ? 4 : 2; }
constexpr int stream_exact_marker_tile(int c) { return 2 * 8 * exact_marker_atoms(c); }  // markers per CTA tile
// z_j, q_j1..q_jc, w_j columns and 1/dy_j of every trait at its own h2 (slots = n_tt*64 >= m); Qc: the unweighted
// orthonormal covariate basis (the w = 1 weight slot)
int launch_exact_columns(const double* Yr, const double* h2, const double* lambda, const double* Qc, int64_t m,
                         int64_t slots, int n, int n_pad, int c, double* Xop, int64_t xcol_pad, double* dyinv,
                         int* flags, cudaStream_t stream);
int launch_scan_exact(const ScanParams& P, int c, int sm_count, cudaStream_t stream);

// ---- post-processing (blmm_post.cu) -------------------------------------------------------------
int launch_lod2log10p(const double* lod, int64_t rows, int64_t cols, int64_t ld_in, int64_t ld_out, int df,
                      double* out, int sm_count, cudaStream_t stream);
// Per-trait peaks from the scan's partials part[j * n_mb + mb]: peak_lod[j] / peak_marker[j] = the first maximum of
// column j in findmax order (peak_key), h2[j] = grid[gidx] when both grid and h2 are given.  One warp per column.
int launch_peak_reduce(const PeakRec* part, int64_t n_mb, int64_t m, int p, const double* grid, double* peak_lod,
                       int64_t* peak_marker, double* h2, cudaStream_t stream);
size_t thresholds_workspace_bytes(int64_t n);
int launch_thresholds(const double* maxlod, int64_t n, const double* probs_dev, int nprob, double* sorted,
                      void* tmp, size_t tmp_bytes, double* out, cudaStream_t stream);
// out = diag(w) * X (X: n x cols column-major, ld n); out may alias X
int launch_scale_rows(const double* X, const double* w, int64_t n, int64_t cols, double* out, int sm_count,
                      cudaStream_t stream);
int launch_weight_kinship(const double* K, const double* w, int n, double* out, cudaStream_t stream);

}  // namespace blmm
