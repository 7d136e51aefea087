/*
 * blmm_b200.h — C-ABI of libblmm_b200.so: BulkLMM.jl's multi-trait LMM genome-scan hot path
 * on one NVIDIA B200 (sm_100a), hand-written CUDA behind plain C entry points.
 *
 * The reference (senresearch/BulkLMM.jl v1.2.0, pure Julia) has no FFI of its own; the boundary
 * is the set of Julia functions named below, whose bodies the Julia shim
 * (bulklmm.jl_b200/julia/BulkLMMB200.jl, see INTEGRATION.md) replaces by `ccall`s into this
 * library.  Every matrix is Julia-native: Float64, column-major, Int64 dimensions.  The caller
 * allocates inputs and outputs; the library never keeps a caller pointer after a call returns.
 *
 * Conventions
 *   - return value 0 = success; non-zero = BLMM_E_*; blmm_last_error(ctx) gives the message
 *     (for the conditions the reference itself reports, its exact error string).
 *   - one context = one GPU (blmm_create) or several GPUs of one box (blmm_create_multi); one call in
 *     flight per context; several contexts may coexist.  A multi-GPU context shards traits (bulkscan) or
 *     permutation columns (scan) over its GPUs inside the library — the analogue of the reference's `nb`
 *     trait blocks, src/bulkscan.jl:263-309 — and returns results bit-identical to a one-GPU context.
 *   - `mem_space` selects whether the data pointers of a call are host or device pointers.
 *     Device-pointer calls are asynchronous on the context's stream until blmm_sync().  On a multi-GPU
 *     context device pointers live on the PRIMARY GPU (devices[0]); NCCL moves the shards (see below).
 *   - host results may be ordinary pageable arrays (a Julia Array, a numpy array): large results are staged
 *     through a pinned ring and moved by host threads; pinned (cudaHostRegister-ed) arrays are written by DMA.
 *   - no C++ exception crosses the boundary; no torch / CUDA types appear in a signature.
 */
#ifndef BLMM_B200_H
#define BLMM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BLMM_ABI_VERSION 3

#if defined(__GNUC__)
#define BLMM_API __attribute__((visibility("default")))
#else
#define BLMM_API
#endif

/* status codes */
enum {
  BLMM_OK = 0,
  BLMM_E_INVALID = 1,        /* bad argument (message says which) */
  BLMM_E_DIM = 2,            /* "Dimension mismatch."                     src/transform_helpers.jl:9-11 */
  BLMM_E_H2_ONE = 3,         /* "Heritability of 1 is not allowed."       src/lmm.jl:19-21 */
  BLMM_E_ZERO_NORM = 4,      /* "Dividing by zeros: the input vector can not contain any zeros!" src/util.jl:69-71 */
  BLMM_E_ONE_TRAIT = 5,      /* "Can only handle one trait."              src/scan.jl:496-498 */
  BLMM_E_CUDA = 6,           /* CUDA / cuSOLVER runtime failure */
  BLMM_E_NOT_SPD = 7,        /* covariate Gram matrix not positive definite (rank-deficient covariates) */
  BLMM_E_NO_DEVICE = 8,      /* no usable sm_100 device */
  BLMM_E_WEIGHTS = 9         /* "Some weights are not positive." (reference only warns, src/wls.jl:35-37, then sqrt throws) */
};

/* memory space of the data pointers of one call */
enum { BLMM_MEM_HOST = 0, BLMM_MEM_DEVICE = 1 };

/* bulkscan methods — `method` keyword of bulkscan(), src/bulkscan.jl:126-152 */
enum {
  BLMM_METHOD_NULL_GRID = 0,  /* bulkscan_null_grid  src/bulkscan.jl:340-385 */
  BLMM_METHOD_ALT_GRID = 1,   /* bulkscan_alt_grid   src/bulkscan.jl:445-526 */
  BLMM_METHOD_NULL_EXACT = 2  /* bulkscan_null       src/bulkscan.jl:212-314 */
};

/* h2_panel semantics of alt-grid */
enum {
  BLMM_H2PANEL_REFERENCE = 0, /* counter semantics of tmax!, src/bulkscan_helpers.jl:340-344 (SURVEY Q1) */
  BLMM_H2PANEL_ARGMAX = 1     /* grid value at the arg-max (first maximum) */
};

/* kinship decomposition schemes — `decomp_scheme` keyword, src/transform_helpers.jl:21-49 */
enum { BLMM_DECOMP_EIGEN = 0, BLMM_DECOMP_SVD = 1 };

typedef struct blmm_ctx blmm_ctx;

/* One scan problem.  Replaces the positional arguments (Y, G, Covar, K) of
 * bulkscan(Y,G,Covar,K) src/bulkscan.jl:113 and scan(y,g,covar,K) src/scan.jl:182, with the
 * kinship already decomposed (blmm_decompose) so that the one-off eigendecomposition is timed
 * as setup and a caller may pass its own (U, lambda).                                            */
typedef struct {
  int64_t n;            /* subjects */
  int64_t p;            /* markers  */
  int64_t m;            /* traits   */
  int64_t c;            /* covariate columns INCLUDING the intercept column when wanted (>= 1) */
  const double* Y;      /* n x m, column-major, ld = n */
  const double* G;      /* n x p, column-major, ld = n */
  const double* Covar;  /* n x c, column-major, ld = n (the shim builds [1 Covar] when addIntercept) */
  const double* U;      /* n x n, column a = a-th eigenvector of K  (Ut = U', src/transform_helpers.jl:24) */
  const double* lambda; /* n eigenvalues, matching U's columns */
  const double* obs_weights; /* NULL, or n observation weights: the `weights` keyword.  Y, G and Covar are
                           row-scaled by them on the device (src/bulkscan.jl:231-250, 351-370, 457-476;
                           src/scan.jl:204-222); (U, lambda) must then decompose W*K*W (blmm_weight_kinship) */
} blmm_problem;

/* Keyword arguments shared by the entry points (defaults of src/bulkscan.jl:81-92 in comments). */
typedef struct {
  int32_t method;            /* BLMM_METHOD_*                       ("null-grid") */
  int32_t reml;              /* 0 = ML, 1 = REML                    (false) */
  double prior_variance;     /* prior[1]                            (1.0; scan: 0.0) */
  double prior_sample_size;  /* prior[2]                            (0.0) */
  const double* h2_grid;     /* HOST pointer, ngrid values in [0,1) (0.0:0.1:0.9) */
  int32_t ngrid;
  int32_t optim_interval;    /* Brent sub-intervals of [0,1]        (1) */
  int32_t h2_panel_mode;     /* BLMM_H2PANEL_*                      (reference) */
  int32_t mem_space;         /* BLMM_MEM_* for problem + output pointers */
  int64_t ld_out;            /* leading dimension of p x m outputs; 0 => p */
  int32_t chisq_df;          /* `output_pvals`/`chisq_df` keywords: 0 = no p-values; >= 1 = also write
                                -log10 p of every LOD (lod2log10p, src/util.jl:199-206) to log10p_out (1) */
  int32_t reserved;
  double* log10p_out;        /* p x m (ld = ld_out or p), same memory space as the other outputs */
} blmm_opts;

/* ---- context ------------------------------------------------------------------------------ */
BLMM_API int blmm_abi_version(void);
BLMM_API int blmm_create(blmm_ctx** out, int device);
/* One context over `ndev` distinct GPUs of this box (ndev == 1 is blmm_create).  Replaces the `nb` keyword's trait
 * blocks (Threads.@threads, src/bulkscan.jl:263-309) by one host thread + GPU per block:
 *   blmm_bulkscan, blmm_bulkscan_peaks, blmm_scan_null, blmm_fit_h2, blmm_grid_loglik   shard the m traits,
 *   blmm_scan_perms                                                shards the permutation columns,
 * into contiguous column blocks (cut at the kernel's 128-column tile); G, Covar, U, lambda are replicated.
 *   BLMM_MEM_HOST  : every GPU reads its block of the caller's arrays and writes its slab of the caller's
 *                    column-major results over its own PCIe link; no collective.
 *   BLMM_MEM_DEVICE: (blmm_bulkscan, blmm_scan_perms) the pointers are memory of devices[0]; NCCL over NVLink
 *                    broadcasts the replicated inputs, scatters the column blocks and gathers the result slabs
 *                    (LOD, h2 panel / h2_null_list, per-permutation max LOD) into the primary's output arrays;
 *                    needs ld_out == p.  libnccl.so.2 is loaded at the first such call.
 * Every other entry point runs on devices[0].                                                          */
BLMM_API int blmm_create_multi(blmm_ctx** out, const int* devices, int ndev);
/* Number of GPUs behind the context (1 for blmm_create). */
BLMM_API int blmm_device_count(const blmm_ctx* ctx);
BLMM_API void blmm_destroy(blmm_ctx* ctx);
BLMM_API const char* blmm_last_error(const blmm_ctx* ctx);
/* Wait for all work queued on the context's stream. */
BLMM_API int blmm_sync(blmm_ctx* ctx);
/* The context's CUDA stream as an opaque integer (cudaStream_t), for event timing by the host. */
BLMM_API uint64_t blmm_stream(blmm_ctx* ctx);
/* Number of kernels this library launched on the context since creation (bench's gpu_launches). */
BLMM_API int64_t blmm_launch_count(const blmm_ctx* ctx);

/* Optional device timing of the dominant kernel (the fused scan, blmm_scan.cu): when switched on,
 * CUDA events are recorded on the context's stream around that launch; blmm_last_scan_ms() waits
 * for the launch and returns its duration in milliseconds (-1 if none was timed).              */
BLMM_API int blmm_set_profiling(blmm_ctx* ctx, int on);
BLMM_API double blmm_last_scan_ms(blmm_ctx* ctx);
/* Multi-GPU device-resident calls: device time (ms, CUDA events on the primary's stream) of the NCCL gather of the
 * last call, from the end of the primary's own scan to the last slab received; valid after blmm_sync(); -1 if none. */
BLMM_API double blmm_last_gather_ms(const blmm_ctx* ctx);
/* Measurement aid (needs no context, no GPU): GB/s at which `nthreads` host threads (0 = the library's default drain
 * thread count) fill a `bytes`-sized pageable buffer with streaming stores — the rate at which this host can take
 * Float64 results at all, i.e. the ceiling of host-buffer calls next to the PCIe rate (bench.py reports both). */
BLMM_API double blmm_host_write_gbs(int nthreads, int64_t bytes);

/* ---- setup -------------------------------------------------------------------------------- */
/* calcKinship(geno), src/kinship.jl:4-14.  G: n x p.  K_out: n x n. */
BLMM_API int blmm_kinship(blmm_ctx* ctx, int64_t n, int64_t p, const double* G, double* K_out, int mem_space);

/* The factorisation inside transform_rotation, src/transform_helpers.jl:21-49 (cuSOLVER syevd;
 * for a symmetric PSD K the SVD scheme is the same decomposition in descending order).
 * U_out: n x n (columns = eigenvectors), lambda_out: n (ascending for EIGEN, descending for SVD).
 * nneg_out (may be NULL): number of eigenvalues < -1e-7 (the reference warns, :27-30).          */
BLMM_API int blmm_decompose(blmm_ctx* ctx, int64_t n, const double* K, int scheme, double* U_out,
                   double* lambda_out, int* nneg_out, int mem_space);

/* transform_rotation, src/transform_helpers.jl:1-54, given (U, lambda):
 * Y0_out = U'Y (n x m), X0_out = U'[Covar G] (n x (c+p)).  Either output may be NULL.          */
BLMM_API int blmm_rotate(blmm_ctx* ctx, const blmm_problem* prob, double* Y0_out, double* X0_out, int mem_space);

/* ---- the hot path ------------------------------------------------------------------------- */
/* bulkscan(Y,G,Covar,K; method=...), src/bulkscan.jl:113-162.
 *   L_out : p x m LOD matrix (ld = opts->ld_out or p), marker index fastest.
 *   h2_out: m heritabilities (null-grid / null-exact: h2_null_list), or
 *           p x m h2_panel (alt-grid; may be NULL to skip the second output).                   */
BLMM_API int blmm_bulkscan(blmm_ctx* ctx, const blmm_problem* prob, const blmm_opts* opts, double* L_out,
                  double* h2_out);

/* Per-trait LOD peaks of bulkscan(Y,G,Covar,K; method=...) without the p x m outputs.  For every trait j:
 *   peak_lod_out[j]    = L[i*, j]  with i* = findmax(L[:, j]) (first index on ties; NaN ranks above every number)
 *   peak_marker_out[j] = i* (0-based)
 *   h2_out[j]          = alt-grid: h2_panel[i*, j] (per opts->h2_panel_mode); null-grid / null-exact: h2_null_list[j]
 * L and h2_panel are the values blmm_bulkscan returns for the same arguments, bit for bit.
 * opts->chisq_df > 0: opts->log10p_out receives m values, -log10 p of peak_lod_out.  ld_out is ignored.
 * peak_marker_out and h2_out may be NULL.  On a multi-GPU context: host buffers only, traits sharded.
 * The scan keeps one 16-byte record per trait and block of 16 or 32 markers on the device instead of the p x m
 * matrices, so problems whose L would not fit in device memory can be scanned.                        */
BLMM_API int blmm_bulkscan_peaks(blmm_ctx* ctx, const blmm_problem* prob, const blmm_opts* opts,
                                 double* peak_lod_out, int64_t* peak_marker_out, double* h2_out);

/* The |grid| x m matrix of null log-likelihoods `ell_results`, src/bulkscan_helpers.jl:267-269
 * (wls_multivar(...).Ell per grid point, src/wls.jl:103-176).  ell_out: ngrid x m, column-major. */
BLMM_API int blmm_grid_loglik(blmm_ctx* ctx, const blmm_problem* prob, const blmm_opts* opts, double* ell_out);

/* fitlmm per trait, src/lmm.jl:56-86 (gridbrent src/gridbrent.jl:9-24 + Optim Brent), batched over
 * the m traits of `prob` (markers unused).  Outputs (each length m, any may be NULL):
 * h2_out, sigma2_out, ell_out.                                                                  */
BLMM_API int blmm_fit_h2(blmm_ctx* ctx, const blmm_problem* prob, const blmm_opts* opts, double* h2_out,
                double* sigma2_out, double* ell_out);

/* scan(y,g,covar,K; permutation_test=true), src/scan.jl:485-557 (scan_perms_lite).  prob->m must
 * be 1.  perm_idx: n x nperms int32, column-major, 0-based — column s is the shuffle
 * r0[perm_idx[:,s]] the shim drew with the reference's RNG (src/transform_helpers.jl:94-102); an entry outside
 * 0..n-1 (e.g. Julia's 1-based n) is refused with BLMM_E_INVALID.
 *   lod_out      : p            LODs of the un-permuted trait
 *   Lperms_out   : p x nperms   (ld = opts->ld_out or p), or NULL to skip materialising it
 *   maxlod_out   : nperms       per-permutation max LOD (what get_thresholds consumes,
 *                               src/analysis_helpers/single_trait_analysis.jl:13-23), or NULL
 *   sigma2_out, h2_out : scalars (sigma2_e, h2_null)                                            */
BLMM_API int blmm_scan_perms(blmm_ctx* ctx, const blmm_problem* prob, const blmm_opts* opts,
                    const int32_t* perm_idx, int64_t nperms, double* lod_out, double* Lperms_out,
                    double* maxlod_out, double* sigma2_out, double* h2_out);

/* scan(y,g,covar,K) null scan of single traits, src/scan.jl:310-360 (scan_null), evaluated in the
 * LiteQTL correlation form the reference's own tests equate it with (test/bulkscan_test.jl:60-80);
 * sqrt(w) without abs() as in scan_null (SURVEY Q2).  lod_out: p x m, sigma2_out/h2_out: m.     */
BLMM_API int blmm_scan_null(blmm_ctx* ctx, const blmm_problem* prob, const blmm_opts* opts, double* lod_out,
                   double* sigma2_out, double* h2_out);

/* scan(y, g, covar, K; assumption = "alt"), src/scan.jl:397-453, prob->m == 1: the variance components are
 * re-estimated by Brent for every marker (covariates [Covar g_i], so c + 1 <= 8), and
 * lod_i = (ell_alt_i - ell_null) / ln 10 with both likelihoods evaluated exactly as the reference does (ML, and
 * with sqrt(w) handed to wls as the weights, src/scan.jl:436-442).  lod_out: p; h2_each_marker_out: p or NULL;
 * sigma2_out, h2_out: the null fit, one value each or NULL.                                          */
BLMM_API int blmm_scan_alt(blmm_ctx* ctx, const blmm_problem* prob, const blmm_opts* opts, double* lod_out,
                  double* h2_each_marker_out, double* sigma2_out, double* h2_out);

/* ---- post-processing ------------------------------------------------------------------------ */
/* lod2log10p.(L, df), src/util.jl:199-206: out = -logccdf(Chisq(df), 2 ln10 lod) / ln10, elementwise over a
 * rows x cols matrix (ld_in / ld_out leading dimensions, 0 => rows).  out may alias lod.            */
BLMM_API int blmm_lod2log10p(blmm_ctx* ctx, const double* lod, int64_t rows, int64_t cols, int64_t ld_in,
                    int64_t ld_out, int df, double* out, int mem_space);

/* get_thresholds, src/analysis_helpers/single_trait_analysis.jl:13-23, from the per-permutation maximum
 * LODs that blmm_scan_perms returns (maxlod_out): thrs_out[i] = quantile(maxlod, 1 - signif_level[i])
 * (Julia's default quantile definition, type 7).  maxlod: nperms values in `mem_space`;
 * signif_level / thrs_out: HOST arrays of nlev values.                                            */
BLMM_API int blmm_thresholds(blmm_ctx* ctx, const double* maxlod, int64_t nperms, const double* signif_level,
                    int nlev, double* thrs_out, int mem_space);

/* K_st = W*K*W for observation weights w (src/bulkscan.jl:239, src/scan.jl:213): K_out[a,b] = w[a] K[a,b] w[b]. */
BLMM_API int blmm_weight_kinship(blmm_ctx* ctx, int64_t n, const double* K, const double* w, double* K_out,
                        int mem_space);

/* ---- data ingest (SURVEY 8f rank 4) ------------------------------------------------------------ */
/* The delimited-text matrices the reference reads with readdlm, parsed by host threads into a column-major
 * Float64 matrix: rows = data lines after `skip_rows`, columns = fields first_col, first_col + col_step, ... up to
 * (not including) the last `drop_last_cols` fields (0-based field numbers).
 *   readBXDpheno(file)                    src/readData.jl:159-161   skip 1, first_col 1, step 1, drop_last 1
 *   readBXDgeno(file; skipstart = 1)      src/readData.jl:163-165   skip 1, first_col 1, step 2, drop_last 0
 *   readGenoProb_ExcludeComplements(file) src/readData.jl:85-96     skip 1, first_col 1, step 2, drop_last 0
 * device < 0: *data_out is host memory (malloc);  device >= 0: device memory on that GPU (one H2D copy), ready
 * for BLMM_MEM_DEVICE calls.  Release with blmm_free_matrix(data, device).  Needs no context; the message of a
 * failure (missing file, non-numeric field, ragged row) is returned by blmm_io_last_error() (thread-local).   */
BLMM_API int blmm_read_csv(const char* path, char delim, int64_t skip_rows, int64_t first_col, int64_t col_step,
                  int64_t drop_last_cols, int device, int64_t* rows_out, int64_t* cols_out, double** data_out);
BLMM_API void blmm_free_matrix(double* data, int device);
BLMM_API const char* blmm_io_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* BLMM_B200_H */
