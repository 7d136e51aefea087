// C-ABI of libblmm_b200.so (include/blmm_b200.h): argument checking, workspace management, the
// launch sequences of the scan methods, host<->device staging for BLMM_MEM_HOST calls.
// No exception crosses the boundary; every entry point returns a BLMM_E_* status.
#include <cuda_runtime.h>
#include <cusolverDn.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <string>
#include <vector>

#include "../../include/blmm_b200.h"
#include "blmm_ctx.cuh"
#include "blmm_kernels.cuh"

using namespace blmm;

namespace {

HostPipe* host_pipe(blmm_ctx* ctx);

// device view of an input matrix: the caller's pointer (device mode) or a staged copy (host mode).  Large pageable
// inputs are first gathered into a pinned arena by the drain threads (see hostpipe_gather_input); the arena is reset
// at the start of every call (host-buffer calls return only when all their copies are complete).
const double* stage_in(blmm_ctx* ctx, Slot s, const double* p, size_t count, int mem_space,
                       cudaStream_t stream = nullptr) {
  if (mem_space == BLMM_MEM_DEVICE) return p;
  double* d = ws<double>(ctx, s, count);
  const size_t bytes = count * sizeof(double);
  cudaStream_t st = stream ? stream : ctx->stream;
  const void* src = p;
  if (bytes >= ((size_t)2 << 20) && !host_ptr_is_pinned(p)) {
    const size_t need = ctx->h_in_off + bytes;
    if (need > ctx->h_in_cap) {
      // earlier regions may still be feeding copies: let them finish before the arena moves
      CUDA_TRY(cudaStreamSynchronize(ctx->stream));
      CUDA_TRY(cudaStreamSynchronize(ctx->copy_stream));
      CUDA_TRY(cudaStreamSynchronize(ctx->aux_stream));
      if (ctx->h_in) CUDA_TRY(cudaFreeHost(ctx->h_in));
      ctx->h_in = nullptr;
      ctx->h_in_cap = 0;
      ctx->h_in_off = 0;
      const size_t cap = std::max(bytes + bytes / 2, (size_t)32 << 20);
      CUDA_TRY(cudaMallocHost(&ctx->h_in, cap));
      ctx->h_in_cap = cap;
    }
    uint8_t* region = ctx->h_in + ctx->h_in_off;
    ctx->h_in_off += (bytes + 255) & ~(size_t)255;
    hostpipe_gather_input(host_pipe(ctx), region, p, bytes);
    src = region;
  }
  CUDA_TRY(cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, st));
  return d;
}

// Device status flags are raised by kernels and collected HERE: they are cleared only after they have been read, so
// that a condition raised by an asynchronous (device-pointer) call is reported by the next blmm_sync or host-buffer
// call instead of being wiped by the next call's entry.
void finish_and_check(blmm_ctx* ctx) {
  CUDA_TRY(cudaMemcpyAsync(ctx->h_flags, ctx->d_flags, FLAG_COUNT * sizeof(int), cudaMemcpyDeviceToHost,
                           ctx->stream));
  CUDA_TRY(cudaMemsetAsync(ctx->d_flags, 0, FLAG_COUNT * sizeof(int), ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  CUDA_TRY(cudaGetLastError());
  if (ctx->h_flags[FLAG_PERM_RANGE])
    throw Fail{BLMM_E_INVALID, "perm_idx entries must be 0-based indices in 0..n-1"};
  if (ctx->h_flags[FLAG_WEIGHTS]) throw Fail{BLMM_E_WEIGHTS, "Some weights are not positive."};
  if (ctx->h_flags[FLAG_NOT_SPD])
    throw Fail{BLMM_E_NOT_SPD, "Covariate matrix is rank deficient (weighted Gram matrix not positive definite)."};
  if (ctx->h_flags[FLAG_ZERO_NORM])
    throw Fail{BLMM_E_ZERO_NORM, "Dividing by zeros: the input vector can not contain any zeros!"};
}

HostPipe* host_pipe(blmm_ctx* ctx) {
  if (!ctx->pipe) ctx->pipe = hostpipe_create(ctx->device, ctx->host_threads > 0 ? ctx->host_threads : default_host_threads());
  return ctx->pipe;
}

// A p x cols result (device, leading dimension p) into the caller's host matrix (leading dimension ld), queued on
// `stream`: one DMA when the destination is pinned, the bounce ring + drain threads when it is pageable.
void matrix_to_host(blmm_ctx* ctx, cudaStream_t stream, double* dst, int64_t ld, const double* src_dev, int64_t p,
                    int64_t cols, bool pinned) {
  if (!dst || cols <= 0) return;
  if (pinned && ld == p)
    CUDA_TRY(cudaMemcpyAsync(dst, src_dev, (size_t)p * cols * sizeof(double), cudaMemcpyDeviceToHost, stream));
  else if (pinned)
    CUDA_TRY(cudaMemcpy2DAsync(dst, ld * sizeof(double), src_dev, p * sizeof(double), p * sizeof(double), cols,
                               cudaMemcpyDeviceToHost, stream));
  else
  {
    hostpipe_set_active(host_pipe(ctx), 1 << 30);
    hostpipe_push(host_pipe(ctx), stream, dst, ld, src_dev, p, p, cols, nullptr);
  }
}

void copy_out(blmm_ctx* ctx, double* dst, const double* src_dev, size_t count, int mem_space) {
  if (!dst || dst == src_dev) return;
  CUDA_TRY(cudaMemcpyAsync(dst, src_dev, count * sizeof(double),
                           mem_space == BLMM_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost,
                           ctx->stream));
}

// Where the results of a scan call are computed and how they reach the caller.  Device mode: the kernels write into the
// caller's arrays, or into workspace for an output the caller passed NULL for that the kernels write anyway.  Host
// mode: they write into workspace, and deliver() queues the copies into the caller's arrays in the order the outputs
// were bound, then collects the device flags and waits for the drain threads.
class Results {
 public:
  Results(blmm_ctx* ctx, int mem_space) : dev(mem_space == BLMM_MEM_DEVICE), ctx_(ctx) {}
  const bool dev;
  // `count` results
  double* vec(double* user, Slot s, size_t count) { return bind(user, s, Copy{user, nullptr, (int64_t)count, 1, 0}); }
  // a p x cols result: leading dimension ld in the caller's array, p in workspace
  double* panel(double* user, Slot s, int64_t p, int64_t cols, int64_t ld) {
    return bind(user, s, Copy{user, nullptr, p, cols, ld});
  }
  // `count` results the kernels always write into workspace (device mode: copied device-to-device right away)
  void copy(double* user, const double* src, size_t count) {
    if (dev)
      copy_out(ctx_, user, src, count, BLMM_MEM_DEVICE);
    else if (user)
      add(Copy{user, src, (int64_t)count, 1, 0});
  }
  void deliver() {
    if (dev) return;
    for (int i = 0; i < n_; ++i) {
      const Copy& c = q_[i];
      if (c.ld == 0)
        copy_out(ctx_, c.dst, c.src, (size_t)c.rows, BLMM_MEM_HOST);
      else  // large pageable results go through the ring; small ones are not worth the hand-over
        matrix_to_host(ctx_, ctx_->stream, c.dst, c.ld, c.src, c.rows, c.cols,
                       (double)c.rows * (double)c.cols * 8.0 < 8e6 || host_ptr_is_pinned(c.dst));
    }
    finish_and_check(ctx_);
    hostpipe_wait(ctx_->pipe);
  }

 private:
  struct Copy { double* dst; const double* src; int64_t rows, cols, ld; };  // ld == 0: a vector
  double* bind(double* user, Slot s, Copy c) {
    if (dev && user) return user;
    double* d = ws<double>(ctx_, s, (size_t)c.rows * c.cols);
    c.src = d;
    if (!dev && user) add(c);
    return d;
  }
  void add(const Copy& c) {
    if (n_ == 5) throw Fail{BLMM_E_INVALID, "internal: more results than Results holds"};
    q_[n_++] = c;
  }
  blmm_ctx* ctx_;
  Copy q_[5];  // a call has at most five outputs
  int n_ = 0;
};

void check_problem(const blmm_problem* pr, bool need_markers, bool need_decomp = true) {
  if (!pr) throw Fail{BLMM_E_INVALID, "problem is NULL"};
  if (pr->n <= 0 || pr->m < 0 || pr->p < 0) throw Fail{BLMM_E_DIM, "Dimension mismatch."};
  if (pr->c < 1 || pr->c > MAXC)
    throw Fail{BLMM_E_INVALID, "covariate count c (including the intercept) must be in 1.." + std::to_string(MAXC)};
  if (pr->c >= pr->n) throw Fail{BLMM_E_INVALID, "more covariates than subjects"};
  if (!pr->Y && pr->m > 0) throw Fail{BLMM_E_INVALID, "Y is NULL"};
  if (!pr->Covar) throw Fail{BLMM_E_INVALID, "Covar is NULL"};
  if (need_markers && (!pr->G || pr->p <= 0)) throw Fail{BLMM_E_INVALID, "G is NULL or p == 0"};
  if (need_decomp && (!pr->U || !pr->lambda)) throw Fail{BLMM_E_INVALID, "U / lambda is NULL (call blmm_decompose)"};
  if (pr->n > (int64_t)1 << 20 || pr->p > (int64_t)1 << 30 || pr->m > (int64_t)1 << 30)
    throw Fail{BLMM_E_INVALID, "problem too large"};
}

// leading dimension of the caller's p-row result matrices
int64_t out_ld(const blmm_opts* o, int64_t p) {
  const int64_t ld = o->ld_out ? o->ld_out : p;
  if (ld < p) throw Fail{BLMM_E_INVALID, "ld_out < p"};
  return ld;
}

void check_optim_interval(const blmm_opts* o) {
  if (o->optim_interval < 1) throw Fail{BLMM_E_INVALID, "optim_interval must be >= 1"};
}

LikParams lik_of(const blmm_opts* o) { return LikParams{o->prior_variance, o->prior_sample_size, o->reml ? 1 : 0}; }

// Inputs of one call on the device (rotated ones padded, column-major).
struct Rotated {
  int n, n_pad, nq, c;
  int64_t m;
  const double* lambda;
  const double* dU;  // the rotation matrix (observation weights folded in)
  const double* dC;  // the unrotated covariates
  double *C0, *Y0 = nullptr, *G0 = nullptr;  // U'C, U'Y, U'G: rotate_covariates, rotate_traits, rotate_markers_aside
};

// Stages U, lambda and the covariates; rotates nothing.
Rotated stage_inputs(blmm_ctx* ctx, const blmm_problem* pr, int mem_space) {
  Rotated R;
  R.n = (int)pr->n;
  R.nq = num_kchunks(pr->n);
  R.n_pad = R.nq * KC;
  R.c = (int)pr->c;
  R.m = pr->m;
  const size_t n = (size_t)pr->n;
  const double* dU = stage_in(ctx, S_U_IN, pr->U, n * n, mem_space);
  if (pr->obs_weights) {
    // U'(w .* X) = (w .* U)'X: fold the observation weights into the rotation matrix once
    const double* dw = stage_in(ctx, S_OBSW, pr->obs_weights, n, mem_space);
    double* Uw = ws<double>(ctx, S_UW, n * n);
    ctx->launches += launch_scale_rows(dU, dw, pr->n, pr->n, Uw, ctx->sm_count, ctx->stream);
    dU = Uw;
  }
  R.dU = dU;
  R.lambda = stage_in(ctx, S_LAM, pr->lambda, n, mem_space);
  R.dC = stage_in(ctx, S_C_IN, pr->Covar, n * R.c, mem_space);
  R.C0 = ws<double>(ctx, S_C0, (size_t)R.n_pad * R.c);
  return R;
}

void rotate_covariates(blmm_ctx* ctx, const Rotated& R, cudaStream_t stream) {
  ctx->launches += launch_rotate(R.dU, R.dC, R.n, R.C0, R.n_pad, R.n_pad, R.n, R.c, stream);
}

void rotate_traits(blmm_ctx* ctx, const blmm_problem* pr, Rotated& R, int mem_space) {
  if (R.m <= 0) return;
  const double* dY = stage_in(ctx, S_Y_IN, pr->Y, (size_t)pr->n * (size_t)R.m, mem_space);
  R.Y0 = ws<double>(ctx, S_Y0, (size_t)R.n_pad * R.m);
  ctx->launches += launch_rotate(R.dU, dY, pr->n, R.Y0, R.n_pad, R.n_pad, R.n, R.m, ctx->stream);
}

// Reallocating a workspace slot frees the old buffer, and cudaFree synchronises the device: the marker slots are sized
// before a call's first fork, so that no allocation serialises the streams mid-overlap.
void reserve_marker_ws(blmm_ctx* ctx, const blmm_problem* pr, int mem_space) {
  ws<double>(ctx, S_G_IN, mem_space == BLMM_MEM_HOST ? (size_t)pr->n * pr->p : 1);
  ws<double>(ctx, S_G0, (size_t)num_kchunks(pr->n) * KC * pr->p);
}

// Staging and rotating the markers depends on nothing but G and U: it runs on the third stream, forked from the main
// stream, beside whatever the other two are doing (trait rotation / statistics / Brent fit; covariates and weight
// constants); the consumer is made to wait for it by wait_markers() right before the first kernel that reads G0.
void rotate_markers_aside(blmm_ctx* ctx, const blmm_problem* pr, Rotated& R, int mem_space) {
  CUDA_TRY(cudaEventRecord(ctx->aux_fork_ev, ctx->stream));  // dU (and a previous call's readers of G0) are ordered before
  CUDA_TRY(cudaStreamWaitEvent(ctx->aux_stream, ctx->aux_fork_ev, 0));
  const double* dG = stage_in(ctx, S_G_IN, pr->G, (size_t)pr->n * (size_t)pr->p, mem_space, ctx->aux_stream);
  R.G0 = ws<double>(ctx, S_G0, (size_t)R.n_pad * pr->p);
  ctx->launches += launch_rotate(R.dU, dG, pr->n, R.G0, R.n_pad, R.n_pad, R.n, pr->p, ctx->aux_stream);
  CUDA_TRY(cudaEventRecord(ctx->aux_done_ev, ctx->aux_stream));
}
void wait_markers(blmm_ctx* ctx, cudaStream_t consumer) { CUDA_TRY(cudaStreamWaitEvent(consumer, ctx->aux_done_ev, 0)); }

WeightConsts weight_ws(blmm_ctx* ctx, int nk, int n_pad, int c) {
  WeightConsts wc;
  wc.w = ws<double>(ctx, S_W, (size_t)(nk + 1) * n_pad);
  wc.sw = ws<double>(ctx, S_SW, (size_t)(nk + 1) * n_pad);
  wc.Q = ws<double>(ctx, S_Q, (size_t)(nk + 1) * c * n_pad);
  wc.slw = ws<double>(ctx, S_SLW, nk + 1);
  wc.lds = ws<double>(ctx, S_LDS, nk + 1);
  return wc;
}

const double* upload_grid(blmm_ctx* ctx, const blmm_opts* o) {
  if (!o->h2_grid || o->ngrid < 1) throw Fail{BLMM_E_INVALID, "h2_grid is NULL or empty"};
  if (o->ngrid > 255) throw Fail{BLMM_E_INVALID, "h2 grids longer than 255 points are not supported"};
  for (int k = 0; k < o->ngrid; ++k) {
    const double h = o->h2_grid[k];
    if (isinf(h / (1.0 - h))) throw Fail{BLMM_E_H2_ONE, "Heritability of 1 is not allowed."};
  }
  double* d = ws<double>(ctx, S_GRID, o->ngrid);
  CUDA_TRY(cudaMemcpyAsync(d, o->h2_grid, o->ngrid * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  return d;
}

// output_pvals: -log10 p of every LOD into dP, computed on the device before anything is copied back
void pvals_after_scan(blmm_ctx* ctx, const blmm_opts* o, const double* dL, double* dP, int64_t p, int64_t m,
                      int64_t ldL) {
  if (o->chisq_df <= 0) return;
  if (o->chisq_df > 1000) throw Fail{BLMM_E_INVALID, "chisq_df must be in 1..1000"};
  if (!o->log10p_out) throw Fail{BLMM_E_INVALID, "chisq_df > 0 but log10p_out is NULL"};
  ctx->launches += launch_lod2log10p(dL, p, m, ldL, ldL, o->chisq_df, dP, ctx->sm_count, ctx->stream);
}

// zeroed device counter for the stream kernels' dynamic unit scheduler
unsigned long long* fresh_unit_counter(blmm_ctx* ctx) {
  unsigned long long* c = ws<unsigned long long>(ctx, S_UNITCTR, 1);
  CUDA_TRY(cudaMemsetAsync(c, 0, sizeof(unsigned long long), ctx->stream));
  return c;
}

// The scan launch(es) of a call between the two profiling events blmm_last_scan_ms reads.
template <typename F>
void timed_scan(blmm_ctx* ctx, F&& launch) {
  if (ctx->profiling) CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
  launch();
  if (ctx->profiling) {
    CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->scan_timed = true;
  }
}

void run_scan(blmm_ctx* ctx, ScanParams P) {
  // L2 residency of the marker operand: every trait tile re-reads all of it (47 MB at BXD size with 10 grid points), and
  // while 4 GB of LOD / h2 panels stream through L2 the per-copy evict_last hint alone did not keep it there (ncu:
  // 2.1 GB of DRAM reads per scan).  A persisting access-policy window over it for the duration of the launch does:
  // 0.30 GB (profiles/l2_persist_r02.json).  BLMM_B200_L2_PERSIST = 0 switches it off (dropping the per-copy hint as well, mode 2 of the experiment, kept 1.0 GB of reads).
  static const int l2_mode = getenv("BLMM_B200_L2_PERSIST") ? atoi(getenv("BLMM_B200_L2_PERSIST")) : 1;
  bool window = false;
  // (k-loop scans only: a one-k scan reads each marker slab once per trait tile of its bin and measured 1-3 % slower
  // with 64 MB of L2 set aside)
  if (l2_mode > 0 && P.e && P.nq <= scan_max_nq(P.nk)) {
    int maxw = 0, maxp = 0;
    cudaDeviceGetAttribute(&maxw, cudaDevAttrMaxAccessPolicyWindowSize, ctx->device);
    cudaDeviceGetAttribute(&maxp, cudaDevAttrMaxPersistingL2CacheSize, ctx->device);
    const size_t bytes = (size_t)P.nk * P.nq * P.p_pad * KC * 8;  // every slab a tile may use
    if (!ctx->l2_limit_set) {  // per device: a multi-GPU process holds one context per GPU
      cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, std::min<size_t>((size_t)maxp, (size_t)64 << 20));
      ctx->l2_limit_set = true;
      if (getenv("BLMM_B200_TRACE"))
        fprintf(stderr, "[blmm trace] L2 persisting max %d MB, window max %d MB, marker operand %.1f MB\n", maxp >> 20, maxw >> 20, bytes / 1048576.0);
    }
    cudaStreamAttrValue av;
    memset(&av, 0, sizeof av);
    av.accessPolicyWindow.base_ptr = const_cast<double*>(P.Mop);
    av.accessPolicyWindow.num_bytes = std::min<size_t>(bytes, (size_t)maxw);
    av.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)std::min<size_t>((size_t)maxp, (size_t)64 << 20) / (double)bytes);
    av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    window = cudaStreamSetAttribute(ctx->stream, cudaStreamAttributeAccessPolicyWindow, &av) == cudaSuccess;
    cudaGetLastError();
  }
  timed_scan(ctx, [&] {
    if (P.nq <= scan_max_nq(P.nk)) {
      const int launched = launch_scan(P, ctx->sm_count, ctx->stream);
      if (!launched) throw Fail{BLMM_E_INVALID, "scan kernel: unsupported parameter combination"};
      ctx->launches += launched;
    } else {
      // n too large for the shared-memory-resident trait tile: same arithmetic, K streamed
      static_assert(SCAN_TT == 128 && SCAN_MT == 64, "packing shared with the streamed GRID kernel");
      StreamParams Q{};
      Q.Mop = P.Mop; Q.Xop = P.Top; Q.e = P.e; Q.et = P.et; Q.tile_k0 = P.tile_k0; Q.n_tiles_dev = P.n_tiles_dev;
      Q.col_map = P.col_map; Q.grid = P.grid; Q.ngrid = P.ngrid; Q.L = P.L; Q.L0 = P.L0;
      Q.H2 = P.H2; Q.colmax = P.colmax; Q.ldL = P.ldL; Q.nq = P.nq; Q.p = P.p; Q.p_pad = P.p_pad; Q.m = P.m;
      Q.xcol_pad = P.tcol_pad; Q.tcol_pad = P.tcol_pad; Q.n_tt = P.n_tiles_t; Q.nk = P.nk;
      Q.argmax_mode = P.argmax_mode; Q.half_n = P.half_n; Q.peaks = P.peaks;
      Q.unit_counter = fresh_unit_counter(ctx);  // n > 100: operands beyond L2 are the normal case here
      ctx->launches += launch_scan_stream_grid(Q, ctx->sm_count, ctx->stream);
    }
  });
  if (window) {
    cudaStreamAttrValue av;
    memset(&av, 0, sizeof av);
    cudaStreamSetAttribute(ctx->stream, cudaStreamAttributeAccessPolicyWindow, &av);  // num_bytes = 0: window off
  }
  CUDA_TRY(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------
double trace_now() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// Chunk boundaries in trait tiles, tbeg[0..nchunk].  The link idles until the first chunk exists, so the first two
// chunks are small (1/4 and 1/2 of an even share, at least one tile) and the rest share what is left evenly.
void chunk_tiles(int n_tiles, int nchunk, int* tbeg) {
  const int even = n_tiles / nchunk;
  const int first = std::max(1, even / 4), second = std::max(1, even / 2);
  tbeg[0] = 0;
  tbeg[1] = std::min(n_tiles, first);
  tbeg[2] = std::min(n_tiles, first + second);
  const int rest = n_tiles - tbeg[2];
  for (int ch = 3; ch <= nchunk; ++ch) tbeg[ch] = tbeg[2] + (int)((int64_t)rest * (ch - 2) / (nchunk - 2));
}

// Host-buffer alt-grid: the p x m panels (2 x 2 GB at BXD size) leave over PCIe, which takes ~4x the scan itself.  The
// trait tiles are scanned in chunks, and each chunk's columns are copied back on the second stream while the next
// chunks are scanned.  The h2 panel holds one of <= 255 grid values per entry, so it crosses PCIe as one-byte grid
// indices (1/8 of the bytes) through the pinned ring and is expanded to grid[index] in the caller's Float64 array by
// the drain threads; L goes straight into a pinned destination, or through the same ring into a pageable one
// (blmm_hostpipe.cu).  dL / dH: the p x m workspace panels (dH NULL without an h2 panel).
void alt_grid_to_host_chunked(blmm_ctx* ctx, const ScanParams& P, const blmm_opts* o, double* L_out, double* h2_out,
                              double* dL, double* dH, int64_t ld, double t_enter) {
  const int64_t p = P.p, m = P.m;
  const int n_tiles = P.n_tiles_t;
  // PCIe is the bottleneck, so what matters is how soon the first copy starts: more, smaller chunks for big panels
  const int nchunk = n_tiles >= 64 ? MAX_CHUNK : 8;
  // The index encoding is worth it when the panel is large (PCIe time saved > host expansion time): >= 1e8
  // entries by default.  BLMM_B200_H2_TRANSFER = index | f64 overrides; BLMM_B200_HOST_THREADS sets the drain
  // thread count (default min(16, cores - 1), divided between the GPUs of a multi-GPU context).
  const char* h2_mode = getenv("BLMM_B200_H2_TRANSFER");
  const bool want_idx = h2_mode ? (h2_mode[0] == 'i') : (ctx->idx_hint >= 0 ? ctx->idx_hint == 1 : (double)p * (double)m >= 1e8);
  const bool idx_panel = dH && want_idx && P.nq <= scan_max_nq(P.nk);
  uint8_t* dI = idx_panel ? ws<uint8_t>(ctx, S_H2IDX, (size_t)p * m) : nullptr;
  if (idx_panel && ctx->h_idx_cap < (size_t)p * m) {
    // the whole index panel has its own pinned staging (1 byte per entry), so that queueing its copies never
    // waits for a ring slot: every copy of the call is in the stream before the first one has finished
    if (ctx->h_idx) CUDA_TRY(cudaFreeHost(ctx->h_idx));
    ctx->h_idx = nullptr;
    ctx->h_idx_cap = 0;
    CUDA_TRY(cudaMallocHost(&ctx->h_idx, (size_t)p * m));
    ctx->h_idx_cap = (size_t)p * m;
  }
  const bool L_pinned = host_ptr_is_pinned(L_out);
  const bool H_pinned = h2_out && host_ptr_is_pinned(h2_out);
  HostPipe* pipe = (idx_panel || !L_pinned || (dH && !H_pinned)) ? host_pipe(ctx) : nullptr;
  // only index expansion to do (every Float64 copy is a direct DMA): a few drain threads, not all of them
  hostpipe_set_active(pipe, (L_pinned && (idx_panel || !dH || H_pinned)) ? 6 : 1 << 30);
  int tbeg[MAX_CHUNK + 1];
  chunk_tiles(n_tiles, nchunk, tbeg);
  int64_t cbeg[MAX_CHUNK + 1];
  for (int ch = 0; ch <= nchunk; ++ch) cbeg[ch] = std::min<int64_t>((int64_t)tbeg[ch] * SCAN_TT, m);
  // every chunk's scan is queued first: the copy loop below may block on ring slots
  for (int ch = 0; ch < nchunk; ++ch) {
    const int t0 = tbeg[ch], t1 = tbeg[ch + 1];
    if (t1 == t0) continue;
    const int64_t c0 = cbeg[ch];
    ScanParams Pc = P;
    Pc.Top = P.Top + (int64_t)t0 * SCAN_TT * KC;
    Pc.e = P.e + (int64_t)t0 * SCAN_TT;
    Pc.et = P.et + (int64_t)t0 * SCAN_TT;
    Pc.L = dL + c0 * p;
    Pc.H2 = (dH && !idx_panel) ? dH + c0 * p : nullptr;
    Pc.H2idx = idx_panel ? dI + c0 * p : nullptr;
    Pc.m = m - c0;
    Pc.n_tiles_t = t1 - t0;
    run_scan(ctx, Pc);
    CUDA_TRY(cudaEventRecord(ctx->chunk_ev[ch], ctx->stream));
  }
  for (int ch = 0; ch < nchunk; ++ch) {
    const int64_t c0 = cbeg[ch], c1 = cbeg[ch + 1];
    if (c1 == c0) continue;
    CUDA_TRY(cudaStreamWaitEvent(ctx->copy_stream, ctx->chunk_ev[ch], 0));
    // indices first: their expansion then overlaps the (8x larger) copy of the chunk's LOD columns
    if (idx_panel) {
      CUDA_TRY(cudaMemcpyAsync(ctx->h_idx + c0 * p, dI + c0 * p, (size_t)(c1 - c0) * p, cudaMemcpyDeviceToHost,
                               ctx->copy_stream));
      CUDA_TRY(cudaEventRecord(ctx->idx_ev[ch], ctx->copy_stream));
      hostpipe_push_staged(pipe, ctx->idx_ev[ch], h2_out + c0 * ld, ld, ctx->h_idx + c0 * p, p, c1 - c0, o->h2_grid);
    }
    matrix_to_host(ctx, ctx->copy_stream, L_out + c0 * ld, ld, dL + c0 * p, p, c1 - c0, L_pinned);
    if (dH && !idx_panel) matrix_to_host(ctx, ctx->copy_stream, h2_out + c0 * ld, ld, dH + c0 * p, p, c1 - c0, H_pinned);
  }
  const double t_queued = trace_now();
  finish_and_check(ctx);
  const double t_scanned = trace_now();
  CUDA_TRY(cudaStreamSynchronize(ctx->copy_stream));
  const double t_copied = trace_now();
  hostpipe_wait(pipe);
  if (getenv("BLMM_B200_TRACE"))
    fprintf(stderr, "[blmm trace] dev %d alt-grid host call: queued %.2f ms, scans done %.2f, copies done %.2f, drained %.2f\n",
            ctx->device, (t_queued - t_enter) * 1e3, (t_scanned - t_enter) * 1e3, (t_copied - t_enter) * 1e3,
            (trace_now() - t_enter) * 1e3);
}

// The output side of a bulk scan when it is not the p x m panels: the per-trait peaks of blmm_bulkscan_peaks.
struct PeakOut {
  double* lod;
  int64_t* marker;  // may be NULL
  double* h2;       // may be NULL
};

// Per-trait peaks occupy the vector results of a call; Results moves 8-byte elements, the int64 markers included.
int64_t* marker_vec(Results& out, int64_t* user, int64_t m) {
  return reinterpret_cast<int64_t*>(out.vec(reinterpret_cast<double*>(user), S_PKMARK, m));
}

// pk == nullptr: L_out / h2_out receive the p x m panels.  pk != nullptr: the same scan keeps one record per trait and
// 32-marker block (PeakRec) instead, and launch_peak_reduce leaves the m peaks in pk.
int bulkscan_grid(blmm_ctx* ctx, const blmm_problem* pr, const blmm_opts* o, double* L_out, double* h2_out,
                  const PeakOut* pk = nullptr) {
  const double t_enter = trace_now();
  check_problem(pr, true);
  if (pk && !pk->lod) throw Fail{BLMM_E_INVALID, "peak_lod_out is NULL"};
  if (!pk && !L_out) throw Fail{BLMM_E_INVALID, "L_out is NULL"};
  const bool alt = o->method == BLMM_METHOD_ALT_GRID;
  const int ms = o->mem_space;
  const int nk = o->ngrid;
  const int64_t p = pr->p, m = pr->m;
  const int64_t ld = pk ? p : out_ld(o, p);
  if (m == 0) return BLMM_OK;
  const double* d_grid = upload_grid(ctx, o);
  Results out(ctx, ms);
  if (pk) h2_out = pk->h2;
  // peaks: dL, dP and dH are m-vectors of the values at the peak
  double* dL = pk ? out.vec(pk->lod, S_L, m) : out.panel(L_out, S_L, p, m, ld);
  double* dP = o->chisq_df <= 0 ? nullptr
               : pk             ? out.vec(o->log10p_out, S_PVAL, m)
                                : out.panel(o->log10p_out, S_PVAL, p, m, ld);
  // alt-grid: the p x m h2 panel; null-grid: h2_null_list, written by the trait statistics
  double* dH = (alt && h2_out) ? (pk ? out.vec(h2_out, S_H2P, m) : out.panel(h2_out, S_H2P, p, m, ld)) : nullptr;
  double* h2v = (!alt && h2_out) ? out.vec(h2_out, S_H2V, m) : nullptr;
  int64_t* dM = pk ? marker_vec(out, pk->marker, m) : nullptr;
  const int64_t ldL = out.dev ? ld : p;
  const int64_t p_pad = round_up(p, SCAN_MT);
  const int64_t n_mb = p_pad / (SCAN_MT / 2);  // the 32-marker blocks of both grid kernels
  reserve_marker_ws(ctx, pr, ms);
  double* Mop = ws<double>(ctx, S_MOP, (size_t)nk * num_kchunks(pr->n) * KC * p_pad);
  PeakRec* parts = pk ? ws<PeakRec>(ctx, S_PEAKS, (size_t)n_mb * m) : nullptr;
  WeightConsts wc = weight_ws(ctx, nk, num_kchunks(pr->n) * KC, (int)pr->c);
  Rotated R = stage_inputs(ctx, pr, ms);
  // The marker side of a grid scan (G -> U'G -> weight-folded marker operand) depends only on G, U and the per-h2
  // weight constants, the trait side only on Y: the two chains are latency-bound on their own, so the covariate
  // rotation, the weight constants and the marker operand run on the second stream (U'G on the third) while the main
  // stream does the trait rotation and then (after the weight constants) the trait statistics.
  CUDA_TRY(cudaEventRecord(ctx->fork_ev, ctx->stream));
  CUDA_TRY(cudaStreamWaitEvent(ctx->copy_stream, ctx->fork_ev, 0));
  const bool rot_in_wc = pr->n <= 128;  // small n: the covariate rotation is folded into the weight-constant blocks
  if (!rot_in_wc) rotate_covariates(ctx, R, ctx->copy_stream);
  rotate_markers_aside(ctx, pr, R, ms);
  if (rot_in_wc)
    ctx->launches += launch_weight_consts_rot(d_grid, nk, R.lambda, R.dU, R.dC, R.n, R.n_pad, R.c, wc, R.C0,
                                              ctx->d_flags, ctx->copy_stream);
  else
    ctx->launches += launch_weight_consts(d_grid, nk, R.lambda, R.C0, R.n, R.n_pad, R.c, wc, ctx->d_flags,
                                          ctx->copy_stream);
  CUDA_TRY(cudaEventRecord(ctx->wc_ev, ctx->copy_stream));
  wait_markers(ctx, ctx->copy_stream);
  ctx->launches += launch_marker_operand(R.G0, p, p_pad, R.n, R.n_pad, R.c, nk, wc, true, Mop, ctx->d_flags,
                                         ctx->copy_stream);
  CUDA_TRY(cudaEventRecord(ctx->join_ev, ctx->copy_stream));
  rotate_traits(ctx, pr, R, ms);
  CUDA_TRY(cudaStreamWaitEvent(ctx->stream, ctx->wc_ev, 0));

  double* Yr = ws<double>(ctx, S_YR, (size_t)R.n_pad * m);
  double* ell = ws<double>(ctx, S_ELL, (size_t)nk * m);
  double* rss = ws<double>(ctx, S_RSS, (size_t)nk * m);
  int* best = ws<int>(ctx, S_BEST, m);
  double* ellmax = ws<double>(ctx, S_ELLMAX, m);
  int* bins = ws<int>(ctx, S_BINS, 3 * 256 + 8);  // count[256] start[256] cursor[256] n_tiles
  int* bin_count = bins, *bin_start = bins + 256, *bin_cursor = bins + 512, *n_tiles = bins + 768;
  CUDA_TRY(cudaMemsetAsync(bins, 0, (3 * 256 + 8) * sizeof(int), ctx->stream));

  // alt-grid: the statistics kernel also writes the packed trait operand and the per-k scalars when it can
  TraitFuse fuse{nullptr, nullptr, nullptr, 0, false};
  if (alt) {
    fuse.tcol_pad = round_up(m, SCAN_TT);
    fuse.e = ws<double>(ctx, S_E, (size_t)nk * fuse.tcol_pad);
    fuse.et = ws<double>(ctx, S_ET, (size_t)nk * fuse.tcol_pad);
    fuse.Top = ws<double>(ctx, S_TOP, (size_t)R.n_pad * fuse.tcol_pad);
  }
  ctx->launches += launch_trait_stats(R.Y0, m, R.n, R.n_pad, R.c, nk, wc, lik_of(o), d_grid, Yr, ell, rss, best,
                                      ellmax, h2v, alt ? nullptr : bin_count, ctx->d_flags, ctx->stream,
                                      alt ? &fuse : nullptr);

  ScanParams P{};
  P.Mop = Mop;
  P.grid = d_grid;
  P.ngrid = nk;
  P.nq = R.nq;
  P.p = (int)p;
  P.p_pad = (int)p_pad;
  P.m = m;
  P.half_n = (double)R.n / 2.0;
  P.argmax_mode = (o->h2_panel_mode == BLMM_H2PANEL_ARGMAX) ? 1 : 0;
  P.L = pk ? nullptr : dL;
  P.ldL = ldL;
  P.peaks = parts;
  if (alt) {
    if (!fuse.done) {
      ctx->launches += launch_alt_scalars(ell, rss, ellmax, m, fuse.tcol_pad, nk, R.n, fuse.e, fuse.et, ctx->stream);
      ctx->launches += launch_pack_traits(Yr, nullptr, m, fuse.tcol_pad, R.n_pad, nullptr, fuse.Top, ctx->stream);
    }
    P.Top = fuse.Top;
    P.e = fuse.e;
    P.et = fuse.et;
    P.tcol_pad = fuse.tcol_pad;
    P.n_tiles_t = (int)(fuse.tcol_pad / SCAN_TT);
    P.nk = nk;
    P.H2 = pk ? nullptr : dH;
  } else {
    const int64_t tcol_pad = round_up(m, SCAN_TT) + (int64_t)nk * SCAN_TT;
    int* tile_k0 = ws<int>(ctx, S_TILEK0, tcol_pad / SCAN_TT);
    int* col_map = ws<int>(ctx, S_COLMAP, tcol_pad);
    double* et = ws<double>(ctx, S_ET, tcol_pad);
    ctx->launches += launch_null_bins(best, rss, m, nk, SCAN_TT, tcol_pad, bin_count, bin_start, bin_cursor,
                                      tile_k0, n_tiles, col_map, et, ctx->stream);
    double* Top = ws<double>(ctx, S_TOP, (size_t)R.n_pad * tcol_pad);
    // shared-memory-resident kernel: 1/rss is folded into the packed trait columns (one FP64 operation less
    // per output); the K-streamed fallback for n > 100 keeps it as the per-column scalar et
    const bool fold = R.nq <= scan_max_nq(1);
    ctx->launches += launch_pack_traits(Yr, col_map, m, tcol_pad, R.n_pad, fold ? et : nullptr, Top, ctx->stream);
    P.et_folded = fold ? 1 : 0;
    P.Top = Top;
    P.et = et;
    P.tile_k0 = tile_k0;
    P.n_tiles_dev = n_tiles;
    P.col_map = col_map;
    P.tcol_pad = tcol_pad;
    P.n_tiles_t = (int)(tcol_pad / SCAN_TT);
    P.nk = 1;
  }
  CUDA_TRY(cudaStreamWaitEvent(ctx->stream, ctx->join_ev, 0));  // marker operand ready
  if (!pk && !out.dev && alt && P.n_tiles_t >= 16 && o->chisq_df <= 0) {
    alt_grid_to_host_chunked(ctx, P, o, L_out, h2_out, dL, dH, ld, t_enter);  // delivers L and the h2 panel itself
    return BLMM_OK;
  }
  run_scan(ctx, P);
  if (pk) {
    ctx->launches += launch_peak_reduce(parts, n_mb, m, (int)p, alt ? d_grid : nullptr, dL, dM, dH, ctx->stream);
    pvals_after_scan(ctx, o, dL, dP, m, 1, m);
  } else {
    pvals_after_scan(ctx, o, dL, dP, p, m, ldL);
  }
  out.deliver();
  return BLMM_OK;
}

int grid_loglik(blmm_ctx* ctx, const blmm_problem* pr, const blmm_opts* o, double* ell_out) {
  check_problem(pr, false);
  if (!ell_out) throw Fail{BLMM_E_INVALID, "ell_out is NULL"};
  const int ms = o->mem_space, nk = o->ngrid;
  const int64_t m = pr->m;
  if (m == 0) return BLMM_OK;
  const double* d_grid = upload_grid(ctx, o);
  Results out(ctx, ms);
  double* ell = out.vec(ell_out, S_ELL, (size_t)nk * m);
  Rotated R = stage_inputs(ctx, pr, ms);
  rotate_covariates(ctx, R, ctx->stream);
  rotate_traits(ctx, pr, R, ms);
  WeightConsts wc = weight_ws(ctx, nk, R.n_pad, R.c);
  ctx->launches += launch_weight_consts(d_grid, nk, R.lambda, R.C0, R.n, R.n_pad, R.c, wc, ctx->d_flags, ctx->stream);
  double* Yr = ws<double>(ctx, S_YR, (size_t)R.n_pad * m);
  double* rss = ws<double>(ctx, S_RSS, (size_t)nk * m);
  int* best = ws<int>(ctx, S_BEST, m);
  double* ellmax = ws<double>(ctx, S_ELLMAX, m);
  ctx->launches += launch_trait_stats(R.Y0, m, R.n, R.n_pad, R.c, nk, wc, lik_of(o), d_grid, Yr, ell, rss, best,
                                      ellmax, nullptr, nullptr, ctx->d_flags, ctx->stream);
  // a zero-norm trait is only an error for the scans (colDivide!), not for wls_multivar (a device-mode call leaves
  // the flag for the next blmm_sync)
  if (!out.dev) CUDA_TRY(cudaMemsetAsync(ctx->d_flags + FLAG_ZERO_NORM, 0, sizeof(int), ctx->stream));
  out.deliver();
  return BLMM_OK;
}

// Yr for m traits: rotation + unweighted residual on the covariates (weight slot 0 = OLS)
double* residualised_traits(blmm_ctx* ctx, const Rotated& R, const blmm_opts* o) {
  WeightConsts wc0 = weight_ws(ctx, 0, R.n_pad, R.c);
  ctx->launches += launch_weight_consts(nullptr, 0, R.lambda, R.C0, R.n, R.n_pad, R.c, wc0, ctx->d_flags, ctx->stream);
  double* Yr = ws<double>(ctx, S_YR, (size_t)R.n_pad * R.m);
  double* ell = ws<double>(ctx, S_ELL, 1);
  double* rss = ws<double>(ctx, S_RSS, 1);
  int* best = ws<int>(ctx, S_BEST, R.m);
  double* ellmax = ws<double>(ctx, S_ELLMAX, R.m);
  ctx->launches += launch_trait_stats(R.Y0, R.m, R.n, R.n_pad, R.c, 0, wc0, lik_of(o), nullptr, Yr, ell, rss, best,
                                      ellmax, nullptr, nullptr, ctx->d_flags, ctx->stream);
  return Yr;
}

int fit_h2(blmm_ctx* ctx, const blmm_problem* pr, const blmm_opts* o, double* h2_out, double* sigma2_out,
           double* ell_out) {
  check_problem(pr, false);
  const int ms = o->mem_space;
  const int64_t m = pr->m;
  if (m == 0) return BLMM_OK;
  check_optim_interval(o);
  Results out(ctx, ms);
  double* h2 = out.vec(h2_out, S_H2V, m);
  double* s2 = out.vec(sigma2_out, S_SIG2, m);
  double* el = out.vec(ell_out, S_ELLV, m);
  Rotated R = stage_inputs(ctx, pr, ms);
  rotate_covariates(ctx, R, ctx->stream);
  rotate_traits(ctx, pr, R, ms);
  double* Yr = residualised_traits(ctx, R, o);
  ctx->launches += launch_fit_h2(Yr, m, R.n, R.n_pad, R.c, R.C0, R.lambda, lik_of(o), o->optim_interval, h2, s2, el,
                                 ctx->d_flags, ctx->stream);
  out.deliver();
  return BLMM_OK;
}

// bulkscan_null (src/bulkscan.jl:212-314): per-trait Brent h2, then univar_liteqtl with the trait's own
// weights as c+2 operand columns (blmm_scan_stream.cu, EXACT mode).  sigma2_out is optional (scan_null).
// pk: per-trait peaks instead of the p x m panels, as in bulkscan_grid.
int bulkscan_exact(blmm_ctx* ctx, const blmm_problem* pr, const blmm_opts* o, double* L_out, double* h2_out,
                   double* sigma2_out, const PeakOut* pk = nullptr) {
  check_problem(pr, true);
  if (pk && !pk->lod) throw Fail{BLMM_E_INVALID, "peak_lod_out is NULL"};
  if (!pk && !L_out) throw Fail{BLMM_E_INVALID, "L_out is NULL"};
  check_optim_interval(o);
  const int ms = o->mem_space;
  const int64_t p = pr->p, m = pr->m;
  const int64_t ld = pk ? p : out_ld(o, p);
  if (m == 0) return BLMM_OK;
  Results out(ctx, ms);
  if (pk) h2_out = pk->h2;
  double* dL = pk ? out.vec(pk->lod, S_L, m) : out.panel(L_out, S_L, p, m, ld);
  double* dP = o->chisq_df <= 0 ? nullptr
               : pk             ? out.vec(o->log10p_out, S_PVAL, m)
                                : out.panel(o->log10p_out, S_PVAL, p, m, ld);
  double* h2 = out.vec(h2_out, S_H2V, m);
  double* s2 = out.vec(sigma2_out, S_SIG2, m);
  int64_t* dM = pk ? marker_vec(out, pk->marker, m) : nullptr;
  reserve_marker_ws(ctx, pr, ms);
  Rotated R = stage_inputs(ctx, pr, ms);
  rotate_covariates(ctx, R, ctx->stream);
  rotate_traits(ctx, pr, R, ms);
  rotate_markers_aside(ctx, pr, R, ms);
  double* Yr = residualised_traits(ctx, R, o);  // also leaves the w = 1 constants in weight slot 0
  ctx->launches += launch_fit_h2(Yr, m, R.n, R.n_pad, R.c, R.C0, R.lambda, lik_of(o), o->optim_interval, h2, s2,
                                 nullptr, ctx->d_flags, ctx->stream);
  // markers residualised (unweighted) on the covariates and normalised: r^2 is invariant to both
  const int mt = stream_exact_marker_tile(R.c);
  const int64_t p_pad = round_up(p, mt);
  WeightConsts wc0 = weight_ws(ctx, 0, R.n_pad, R.c);
  double* Mop = ws<double>(ctx, S_MOP, (size_t)R.n_pad * p_pad);
  wait_markers(ctx, ctx->stream);  // U'G was computed on the third stream meanwhile
  ctx->launches += launch_marker_operand(R.G0, p, p_pad, R.n, R.n_pad, R.c, 1, wc0, false, Mop, ctx->d_flags, ctx->stream);
  const int cg = R.c + 2;
  const int64_t n_tt = (m + 63) / 64;
  const int64_t slots = n_tt * 64;
  const int64_t xcol_pad = slots * cg;
  double* Xop = ws<double>(ctx, S_XOP, (size_t)R.n_pad * xcol_pad);
  double* dyinv = ws<double>(ctx, S_DYINV, slots);
  ctx->launches += launch_exact_columns(Yr, h2, R.lambda, R.C0, m, slots, R.n, R.n_pad, R.c, Xop, xcol_pad, dyinv,
                                        ctx->d_flags, ctx->stream);
  StreamParams P{};
  P.Mop = Mop;
  P.Xop = Xop;
  P.dyinv = dyinv;
  P.L = pk ? nullptr : dL;
  P.ldL = out.dev ? ld : p;
  const int64_t n_mb = p_pad / (mt / 2);
  P.peaks = pk ? ws<PeakRec>(ctx, S_PEAKS, (size_t)n_mb * m) : nullptr;
  P.nq = R.nq;
  P.p = (int)p;
  P.p_pad = (int)p_pad;
  P.m = m;
  P.xcol_pad = xcol_pad;
  P.n_tt = (int)n_tt;
  P.nk = 1;
  P.half_n = (double)R.n / 2.0;
  if (const char* b = getenv("BLMM_STREAM_BAND")) P.band = atoi(b);  // development knob (L2 rasterisation study)
  // dynamic unit hand-out when the operands do not fit in L2 (it costs one global atomic per unit)
  const double operand_bytes = 8.0 * R.n_pad * ((double)p_pad + (double)xcol_pad);
  bool dynamic = operand_bytes > 100e6;
  if (const char* d = getenv("BLMM_STREAM_DYNAMIC")) dynamic = d[0] == '1';  // test hook: force either scheduler
  P.unit_counter = dynamic ? fresh_unit_counter(ctx) : nullptr;
  timed_scan(ctx, [&] { ctx->launches += launch_scan_exact(P, R.c, ctx->sm_count, ctx->stream); });
  CUDA_TRY(cudaGetLastError());
  if (pk) {
    ctx->launches += launch_peak_reduce(P.peaks, n_mb, m, (int)p, nullptr, dL, dM, nullptr, ctx->stream);
    pvals_after_scan(ctx, o, dL, dP, m, 1, m);
  } else {
    pvals_after_scan(ctx, o, dL, dP, p, m, P.ldL);
  }
  out.deliver();
  return BLMM_OK;
}

// scan(...; assumption = "alt"), src/scan.jl:397-453: one trait, variance components re-estimated per marker
int scan_alt(blmm_ctx* ctx, const blmm_problem* pr, const blmm_opts* o, double* lod_out, double* h2_each_out,
             double* sigma2_out, double* h2_out) {
  if (pr && pr->m != 1) throw Fail{BLMM_E_ONE_TRAIT, "Can only handle one trait."};
  check_problem(pr, true);
  if (!lod_out) throw Fail{BLMM_E_INVALID, "lod_out is NULL"};
  check_optim_interval(o);
  if (pr->c + 1 > MAXC) throw Fail{BLMM_E_INVALID, "scan_alt supports at most " + std::to_string(MAXC - 1) + " covariates"};
  const int64_t p = pr->p;
  Results out(ctx, o->mem_space);
  double* dlod = out.vec(lod_out, S_L, p);
  double* dh2 = h2_each_out ? out.vec(h2_each_out, S_H2P, p) : nullptr;
  reserve_marker_ws(ctx, pr, o->mem_space);
  Rotated R = stage_inputs(ctx, pr, o->mem_space);
  rotate_covariates(ctx, R, ctx->stream);
  rotate_traits(ctx, pr, R, o->mem_space);
  rotate_markers_aside(ctx, pr, R, o->mem_space);
  double* Yr = residualised_traits(ctx, R, o);
  double* misc = ws<double>(ctx, S_MISC, 8);  // [0] h2_null, [1] sigma2, [2] ell_null
  ctx->launches += launch_fit_h2(Yr, 1, R.n, R.n_pad, R.c, R.C0, R.lambda, lik_of(o), o->optim_interval, misc, misc + 1,
                                 nullptr, ctx->d_flags, ctx->stream);
  wait_markers(ctx, ctx->stream);  // U'G was computed on the third stream meanwhile
  const int launched = launch_scan_alt(Yr, R.G0, p, R.n, R.n_pad, R.c, R.C0, R.lambda, lik_of(o), o->optim_interval,
                                       misc, misc + 2, dlod, dh2, ctx->stream);
  if (!launched) throw Fail{BLMM_E_INVALID, "unsupported covariate count"};
  ctx->launches += launched;
  CUDA_TRY(cudaGetLastError());
  out.copy(h2_out, misc, 1);
  out.copy(sigma2_out, misc + 1, 1);
  out.deliver();
  return BLMM_OK;
}

int scan_perms(blmm_ctx* ctx, const blmm_problem* pr, const blmm_opts* o, const int32_t* perm_idx, int64_t nperms,
               double* lod_out, double* Lperms_out, double* maxlod_out, double* sigma2_out, double* h2_out) {
  if (pr && pr->m != 1) throw Fail{BLMM_E_ONE_TRAIT, "Can only handle one trait."};
  check_problem(pr, true);
  if (nperms < 0 || (nperms > 0 && !perm_idx)) throw Fail{BLMM_E_INVALID, "perm_idx is NULL"};
  if (!lod_out) throw Fail{BLMM_E_INVALID, "lod_out is NULL"};
  check_optim_interval(o);
  const int ms = o->mem_space;
  const int64_t p = pr->p;
  const int64_t ld = out_ld(o, p);
  Results out(ctx, ms);
  double* d_lod = out.vec(lod_out, S_L, p);
  // (the h2-panel slot is free in a permutation scan)
  double* d_Lp = (Lperms_out && nperms > 0) ? out.panel(Lperms_out, S_H2P, p, nperms, ld) : nullptr;
  double* d_max = (maxlod_out && nperms > 0) ? out.vec(maxlod_out, S_COLMAX, nperms) : nullptr;
  double* h2 = out.vec(h2_out, S_H2V, 1);
  double* s2 = out.vec(sigma2_out, S_SIG2, 1);
  reserve_marker_ws(ctx, pr, ms);
  Rotated R = stage_inputs(ctx, pr, ms);
  WeightConsts wc = weight_ws(ctx, 1, R.n_pad, R.c);
  double* z = ws<double>(ctx, S_Z, R.n_pad + 8);
  double* zrss = z + R.n_pad;
  // Small n: rotation of y and the covariates, residualisation, Brent, weight constants and the null residual are ONE
  // launch (null_fit_chain_kernel), with the markers rotated beside it; otherwise the same steps as separate kernels,
  // the markers forked after the trait rotation.
  const bool fused = pr->n <= 128 && !getenv("BLMM_B200_NO_CHAIN");  // test hook: force the separate kernels
  bool chained = false;
  if (fused) {
    rotate_markers_aside(ctx, pr, R, ms);
    const double* dY = stage_in(ctx, S_Y_IN, pr->Y, (size_t)pr->n, ms);
    double* Yr1 = ws<double>(ctx, S_YR, (size_t)R.n_pad);
    const int launched = launch_null_fit_chain(R.dU, dY, R.dC, R.lambda, R.n, R.n_pad, R.c, lik_of(o), o->optim_interval,
                                               R.C0, Yr1, wc, h2, s2, z, zrss, ctx->d_flags, ctx->stream);
    ctx->launches += launched;
    chained = launched > 0;  // 0: does not apply (shared memory)
  }
  if (!chained) {
    rotate_covariates(ctx, R, ctx->stream);
    rotate_traits(ctx, pr, R, ms);
    if (!fused) rotate_markers_aside(ctx, pr, R, ms);
    double* Yr = residualised_traits(ctx, R, o);
    ctx->launches += launch_fit_h2(Yr, 1, R.n, R.n_pad, R.c, R.C0, R.lambda, lik_of(o), o->optim_interval, h2, s2,
                                   nullptr, ctx->d_flags, ctx->stream);
    // transform_reweight at the fitted h2 (weight slot 0)
    ctx->launches += launch_weight_consts(h2, 1, R.lambda, R.C0, R.n, R.n_pad, R.c, wc, ctx->d_flags, ctx->stream);
    ctx->launches += launch_null_residual(Yr, R.n, R.n_pad, R.c, wc, z, zrss, ctx->stream);
  }
  const int64_t p_pad = round_up(p, SCAN_MT);
  double* Mop = ws<double>(ctx, S_MOP, (size_t)R.n_pad * p_pad);
  wait_markers(ctx, ctx->stream);  // U'G was computed on the third stream meanwhile
  ctx->launches += launch_marker_operand(R.G0, p, p_pad, R.n, R.n_pad, R.c, 1, wc, false, Mop, ctx->d_flags, ctx->stream);

  const int64_t ncol = nperms + 1;
  const int64_t tcol_pad = round_up(ncol, SCAN_TT);
  const int32_t* d_perm = nperms > 0 ? perm_idx : nullptr;
  if (nperms > 0 && !out.dev) {
    int32_t* dp = ws<int32_t>(ctx, S_PERM, (size_t)R.n * nperms);
    CUDA_TRY(cudaMemcpyAsync(dp, perm_idx, (size_t)R.n * nperms * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    d_perm = dp;
  }
  double* Top = ws<double>(ctx, S_TOP, (size_t)R.n_pad * tcol_pad);
  double* et1 = ws<double>(ctx, S_ET, tcol_pad);
  ctx->launches += launch_pack_perms(z, zrss, d_perm, nperms, R.n, R.n_pad, tcol_pad, Top, et1, ctx->d_flags, ctx->stream);

  ScanParams P{};
  P.Top = Top;
  P.Mop = Mop;
  P.et = et1;
  P.et_folded = (R.nq <= scan_max_nq(1)) ? 1 : 0;  // columns are normalised: v = 1 - d^2
  P.nq = R.nq;
  P.p = (int)p;
  P.p_pad = (int)p_pad;
  P.m = ncol;
  P.tcol_pad = tcol_pad;
  P.n_tiles_t = (int)(tcol_pad / SCAN_TT);
  P.nk = 1;
  P.half_n = (double)R.n / 2.0;
  P.L0 = d_lod;
  P.L = d_Lp;
  P.ldL = out.dev ? ld : p;
  if (d_max) {
    CUDA_TRY(cudaMemsetAsync(d_max, 0, nperms * sizeof(double), ctx->stream));
    P.colmax = d_max;
  }
  run_scan(ctx, P);
  out.deliver();
  return BLMM_OK;
}

int kinship(blmm_ctx* ctx, int64_t n, int64_t p, const double* G, double* K_out, int ms) {
  if (n <= 0 || p <= 0 || !G || !K_out) throw Fail{BLMM_E_INVALID, "bad kinship arguments"};
  const double* dG = stage_in(ctx, S_G_IN, G, (size_t)n * p, ms);
  double* part = ws<double>(ctx, S_KPART, kinship_workspace_doubles((int)n, p));
  double* dK = (ms == BLMM_MEM_DEVICE) ? K_out : ws<double>(ctx, S_KIN, (size_t)n * n);
  ctx->launches += launch_kinship(dG, (int)n, p, dK, part, ctx->stream);
  CUDA_TRY(cudaGetLastError());
  copy_out(ctx, K_out, dK, (size_t)n * n, ms);
  if (ms == BLMM_MEM_HOST) CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return BLMM_OK;
}

__global__ void permute_eig_kernel(const double* __restrict__ V, const double* __restrict__ lam,
                                   const int* __restrict__ order, int n, int take_abs, double* __restrict__ U,
                                   double* __restrict__ lam_out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)n * n) return;
  const int a = (int)(idx / n), b = (int)(idx % n);
  U[idx] = V[(int64_t)order[a] * n + b];
  if (b == 0) lam_out[a] = take_abs ? fabs(lam[order[a]]) : lam[order[a]];
}

int decompose(blmm_ctx* ctx, int64_t n, const double* K, int scheme, double* U_out, double* lambda_out,
              int* nneg_out, int ms) {
  if (n <= 0 || !K || !U_out || !lambda_out) throw Fail{BLMM_E_INVALID, "bad decompose arguments"};
  if (scheme != BLMM_DECOMP_EIGEN && scheme != BLMM_DECOMP_SVD)
    throw Fail{BLMM_E_INVALID, "Please choose either `eigen` or `svd` for decomposition of the kinship matrix."};
  if (!ctx->solver) {
    if (cusolverDnCreate(&ctx->solver) != CUSOLVER_STATUS_SUCCESS) throw Fail{BLMM_E_CUDA, "cusolverDnCreate failed"};
    cusolverDnSetStream(ctx->solver, ctx->stream);
  }
  const size_t nn = (size_t)n * n;
  double* V = ws<double>(ctx, S_EIGV, nn + n + 8);
  double* lam = V + nn;
  int* info = reinterpret_cast<int*>(lam + n);
  CUDA_TRY(cudaMemcpyAsync(V, K, nn * sizeof(double),
                           ms == BLMM_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
  int lwork = 0;
  if (cusolverDnDsyevd_bufferSize(ctx->solver, CUSOLVER_EIG_MODE_VECTOR, CUBLAS_FILL_MODE_LOWER, (int)n, V, (int)n,
                                  lam, &lwork) != CUSOLVER_STATUS_SUCCESS)
    throw Fail{BLMM_E_CUDA, "cusolverDnDsyevd_bufferSize failed"};
  double* work = ws<double>(ctx, S_SOLVER, lwork);
  if (cusolverDnDsyevd(ctx->solver, CUSOLVER_EIG_MODE_VECTOR, CUBLAS_FILL_MODE_LOWER, (int)n, V, (int)n, lam, work,
                       lwork, info) != CUSOLVER_STATUS_SUCCESS)
    throw Fail{BLMM_E_CUDA, "cusolverDnDsyevd failed"};
  ctx->launches += 1;
  std::vector<double> hl(n);
  int hinfo = 0;
  CUDA_TRY(cudaMemcpyAsync(hl.data(), lam, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaMemcpyAsync(&hinfo, info, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  if (hinfo != 0) throw Fail{BLMM_E_CUDA, "syevd did not converge (info = " + std::to_string(hinfo) + ")"};
  if (nneg_out) {
    // the reference warns on eigen values < -1e-7 (src/transform_helpers.jl:27-30); its svd branch tests the
    // singular values, which are never negative (:42-45), so it never warns there
    int c = 0;
    if (scheme == BLMM_DECOMP_EIGEN)
      for (int64_t i = 0; i < n; ++i) c += hl[i] < -1e-7;
    *nneg_out = c;
  }
  // eigen: ascending eigenvalues (LAPACK order).  svd: singular values |lambda| descending.
  std::vector<int> order(n);
  for (int64_t i = 0; i < n; ++i) order[i] = (int)i;
  if (scheme == BLMM_DECOMP_SVD)
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return fabs(hl[a]) > fabs(hl[b]); });
  int* d_order = ws<int>(ctx, S_MISC, n);
  CUDA_TRY(cudaMemcpyAsync(d_order, order.data(), n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  double* dU = (ms == BLMM_MEM_DEVICE) ? U_out : ws<double>(ctx, S_U_IN, nn);
  double* dl = (ms == BLMM_MEM_DEVICE) ? lambda_out : ws<double>(ctx, S_LAM, n);
  permute_eig_kernel<<<(unsigned)((nn + 255) / 256), 256, 0, ctx->stream>>>(V, lam, d_order, (int)n,
                                                                             scheme == BLMM_DECOMP_SVD, dU, dl);
  ctx->launches += 1;
  CUDA_TRY(cudaGetLastError());
  copy_out(ctx, U_out, dU, nn, ms);
  copy_out(ctx, lambda_out, dl, n, ms);
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));  // `order` is a host temporary
  return BLMM_OK;
}

int rotate(blmm_ctx* ctx, const blmm_problem* pr, double* Y0_out, double* X0_out, int ms) {
  // transform_rotation accepts any number of columns in its second matrix (X = [1 g])
  if (!pr || pr->n <= 0 || pr->m < 0 || pr->c < 0 || !pr->U) throw Fail{BLMM_E_DIM, "Dimension mismatch."};
  if ((Y0_out && pr->m > 0 && !pr->Y) || (X0_out && pr->c > 0 && !pr->Covar))
    throw Fail{BLMM_E_INVALID, "input matrix is NULL"};
  const size_t n = (size_t)pr->n;
  const double* dU = stage_in(ctx, S_U_IN, pr->U, n * n, ms);
  if (Y0_out && pr->m > 0) {
    const double* dY = stage_in(ctx, S_Y_IN, pr->Y, n * pr->m, ms);
    double* out = (ms == BLMM_MEM_DEVICE) ? Y0_out : ws<double>(ctx, S_Y0, n * pr->m);
    ctx->launches += launch_rotate(dU, dY, pr->n, out, pr->n, pr->n, (int)pr->n, pr->m, ctx->stream);
    copy_out(ctx, Y0_out, out, n * pr->m, ms);
  }
  if (X0_out) {
    const double* dC = stage_in(ctx, S_C_IN, pr->Covar, n * pr->c, ms);
    const int64_t cols = pr->c + ((pr->G && pr->p > 0) ? pr->p : 0);
    double* out = (ms == BLMM_MEM_DEVICE) ? X0_out : ws<double>(ctx, S_G0, n * cols);
    ctx->launches += launch_rotate(dU, dC, pr->n, out, pr->n, pr->n, (int)pr->n, pr->c, ctx->stream);
    if (cols > pr->c) {
      const double* dG = stage_in(ctx, S_G_IN, pr->G, n * pr->p, ms);
      ctx->launches += launch_rotate(dU, dG, pr->n, out + n * pr->c, pr->n, pr->n, (int)pr->n, pr->p, ctx->stream);
    }
    copy_out(ctx, X0_out, out, n * cols, ms);
  }
  CUDA_TRY(cudaGetLastError());
  if (ms == BLMM_MEM_HOST) CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return BLMM_OK;
}

int lod2log10p(blmm_ctx* ctx, const double* lod, int64_t rows, int64_t cols, int64_t ld_in, int64_t ld_out, int df,
               double* out, int ms) {
  if (rows < 0 || cols < 0 || (rows * cols > 0 && (!lod || !out))) throw Fail{BLMM_E_INVALID, "bad lod2log10p arguments"};
  if (df < 1 || df > 1000) throw Fail{BLMM_E_INVALID, "chisq_df must be in 1..1000"};
  if (rows * cols == 0) return BLMM_OK;
  if (!ld_in) ld_in = rows;
  if (!ld_out) ld_out = rows;
  if (ld_in < rows || ld_out < rows) throw Fail{BLMM_E_INVALID, "leading dimension < rows"};
  if (ms == BLMM_MEM_DEVICE) {
    ctx->launches += launch_lod2log10p(lod, rows, cols, ld_in, ld_out, df, out, ctx->sm_count, ctx->stream);
    CUDA_TRY(cudaGetLastError());
    return BLMM_OK;
  }
  double* d = ws<double>(ctx, S_PVAL, (size_t)rows * cols);
  CUDA_TRY(cudaMemcpy2DAsync(d, rows * sizeof(double), lod, ld_in * sizeof(double), rows * sizeof(double), cols,
                             cudaMemcpyHostToDevice, ctx->stream));
  ctx->launches += launch_lod2log10p(d, rows, cols, rows, rows, df, d, ctx->sm_count, ctx->stream);
  CUDA_TRY(cudaMemcpy2DAsync(out, ld_out * sizeof(double), d, rows * sizeof(double), rows * sizeof(double), cols,
                             cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  CUDA_TRY(cudaGetLastError());
  return BLMM_OK;
}

int thresholds(blmm_ctx* ctx, const double* maxlod, int64_t nperms, const double* signif, int nlev, double* thrs,
               int ms) {
  if (nperms < 1 || !maxlod || nlev < 0 || (nlev > 0 && (!signif || !thrs)))
    throw Fail{BLMM_E_INVALID, "bad thresholds arguments"};
  if (nlev == 0) return BLMM_OK;
  const double* dmax = stage_in(ctx, S_COLMAX, maxlod, nperms, ms);
  std::vector<double> probs(nlev);
  for (int i = 0; i < nlev; ++i) probs[i] = 1.0 - signif[i];
  double* d_probs = ws<double>(ctx, S_PROBS, 2 * (size_t)nlev);
  CUDA_TRY(cudaMemcpyAsync(d_probs, probs.data(), nlev * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  double* sorted = ws<double>(ctx, S_SORT, nperms);
  const size_t tmp_bytes = thresholds_workspace_bytes(nperms);
  void* tmp = ws<unsigned char>(ctx, S_SORTTMP, tmp_bytes);
  ctx->launches += launch_thresholds(dmax, nperms, d_probs, nlev, sorted, tmp, tmp_bytes, d_probs + nlev, ctx->stream);
  CUDA_TRY(cudaMemcpyAsync(thrs, d_probs + nlev, nlev * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));  // `probs` is a host temporary; thrs is a host array
  CUDA_TRY(cudaGetLastError());
  return BLMM_OK;
}

int weight_kinship(blmm_ctx* ctx, int64_t n, const double* K, const double* w, double* K_out, int ms) {
  if (n <= 0 || !K || !w || !K_out) throw Fail{BLMM_E_INVALID, "bad weight_kinship arguments"};
  const double* dK = stage_in(ctx, S_KIN, K, (size_t)n * n, ms);
  const double* dw = stage_in(ctx, S_OBSW, w, n, ms);
  double* out = (ms == BLMM_MEM_DEVICE) ? K_out : ws<double>(ctx, S_EIGV, (size_t)n * n + n + 8);
  ctx->launches += launch_weight_kinship(dK, dw, (int)n, out, ctx->stream);
  CUDA_TRY(cudaGetLastError());
  copy_out(ctx, K_out, out, (size_t)n * n, ms);
  if (ms == BLMM_MEM_HOST) CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return BLMM_OK;
}

template <typename F>
int guarded(blmm_ctx* ctx, F&& f) {
  if (!ctx) return BLMM_E_INVALID;
  try {
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) throw Fail{BLMM_E_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e)};
    ctx->err.clear();
    ctx->h_in_off = 0;  // every earlier host-buffer call has completed its copies
    return f();
  } catch (const Fail& fl) {
    ctx->err = fl.msg;
    // leave nothing in flight that still writes into the caller's arrays, and no stale device flag
    cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    if (ctx->aux_stream) cudaStreamSynchronize(ctx->aux_stream);
    try {
      hostpipe_wait(ctx->pipe);
    } catch (...) {
    }
    if (ctx->d_flags) cudaMemset(ctx->d_flags, 0, FLAG_COUNT * sizeof(int));
    cudaGetLastError();
    return fl.code;
  } catch (const std::exception& ex) {
    ctx->err = ex.what();
    return BLMM_E_INVALID;
  } catch (...) {
    ctx->err = "unknown failure";
    return BLMM_E_INVALID;
  }
}

// the scan entry points: guarded() with the options checked first
template <typename F>
int guarded(blmm_ctx* ctx, const blmm_opts* opts, F&& f) {
  return guarded(ctx, [&] {
    if (!opts) throw Fail{BLMM_E_INVALID, "opts is NULL"};
    return f();
  });
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// extern "C" surface
// ---------------------------------------------------------------------------------------------
extern "C" {

int blmm_abi_version(void) { return BLMM_ABI_VERSION; }

int blmm_create(blmm_ctx** out, int device) {
  if (!out) return BLMM_E_INVALID;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) {
    cudaGetLastError();
    return BLMM_E_NO_DEVICE;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return BLMM_E_NO_DEVICE;
  if (prop.major != 10) return BLMM_E_NO_DEVICE;  // kernels are built for sm_100a only
  blmm_ctx* ctx = new (std::nothrow) blmm_ctx();
  if (!ctx) return BLMM_E_INVALID;
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  bool ok = cudaSetDevice(device) == cudaSuccess &&
            cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaEventCreateWithFlags(&ctx->aux_fork_ev, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&ctx->aux_done_ev, cudaEventDisableTiming) == cudaSuccess &&
            cudaMalloc(&ctx->d_flags, FLAG_COUNT * sizeof(int)) == cudaSuccess &&
            cudaMemset(ctx->d_flags, 0, FLAG_COUNT * sizeof(int)) == cudaSuccess &&
            cudaMallocHost(&ctx->h_flags, FLAG_COUNT * sizeof(int)) == cudaSuccess &&
            cudaEventCreate(&ctx->ev0) == cudaSuccess && cudaEventCreate(&ctx->ev1) == cudaSuccess;
  ok = ok && cudaEventCreateWithFlags(&ctx->fork_ev, cudaEventDisableTiming) == cudaSuccess &&
       cudaEventCreateWithFlags(&ctx->join_ev, cudaEventDisableTiming) == cudaSuccess &&
       cudaEventCreateWithFlags(&ctx->wc_ev, cudaEventDisableTiming) == cudaSuccess;
  for (int i = 0; ok && i < MAX_CHUNK; ++i)
    ok = cudaEventCreateWithFlags(&ctx->chunk_ev[i], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&ctx->idx_ev[i], cudaEventDisableTiming | cudaEventBlockingSync) == cudaSuccess;
  if (!ok) {
    blmm_destroy(ctx);
    return BLMM_E_CUDA;
  }
  *out = ctx;
  return BLMM_OK;
}

int blmm_create_multi(blmm_ctx** out, const int* devices, int ndev) {
  if (!out) return BLMM_E_INVALID;
  *out = nullptr;
  if (!devices || ndev < 1 || ndev > 64) return BLMM_E_INVALID;
  for (int a = 0; a < ndev; ++a)
    for (int b = a + 1; b < ndev; ++b)
      if (devices[a] == devices[b]) return BLMM_E_INVALID;
  if (ndev == 1) return blmm_create(out, devices[0]);
  blmm_ctx* ctx = new (std::nothrow) blmm_ctx();
  if (!ctx) return BLMM_E_INVALID;
  const int st = multi_create(ctx, devices, ndev);
  if (st != BLMM_OK) {
    blmm_destroy(ctx);
    return st;
  }
  *out = ctx;
  return BLMM_OK;
}

int blmm_device_count(const blmm_ctx* ctx) { return ctx ? multi_ndev(ctx) : 0; }

void blmm_destroy(blmm_ctx* ctx) {
  if (!ctx) return;
  if (ctx->multi) {
    multi_destroy(ctx);
    delete ctx;
    return;
  }
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
  if (ctx->aux_stream) cudaStreamSynchronize(ctx->aux_stream);
  hostpipe_destroy(ctx->pipe);
  for (int s = 0; s < S_COUNT; ++s)
    if (ctx->buf[s]) cudaFree(ctx->buf[s]);
  if (ctx->d_flags) cudaFree(ctx->d_flags);
  if (ctx->h_flags) cudaFreeHost(ctx->h_flags);
  if (ctx->solver) cusolverDnDestroy(ctx->solver);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (ctx->fork_ev) cudaEventDestroy(ctx->fork_ev);
  if (ctx->join_ev) cudaEventDestroy(ctx->join_ev);
  if (ctx->wc_ev) cudaEventDestroy(ctx->wc_ev);
  for (int i = 0; i < MAX_CHUNK; ++i) {
    if (ctx->chunk_ev[i]) cudaEventDestroy(ctx->chunk_ev[i]);
    if (ctx->idx_ev[i]) cudaEventDestroy(ctx->idx_ev[i]);
  }
  if (ctx->h_idx) cudaFreeHost(ctx->h_idx);
  if (ctx->h_in) cudaFreeHost(ctx->h_in);
  if (ctx->aux_fork_ev) cudaEventDestroy(ctx->aux_fork_ev);
  if (ctx->aux_done_ev) cudaEventDestroy(ctx->aux_done_ev);
  if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* blmm_last_error(const blmm_ctx* ctx) { return ctx ? ctx->err.c_str() : "context is NULL"; }

int blmm_sync(blmm_ctx* ctx) {
  if (ctx && ctx->multi) return multi_sync(ctx);
  return guarded(ctx, [&] {
    finish_and_check(ctx);
    return BLMM_OK;
  });
}

uint64_t blmm_stream(blmm_ctx* ctx) {
  if (ctx && ctx->multi) ctx = multi_primary(ctx);
  return ctx ? (uint64_t)(uintptr_t)ctx->stream : 0;
}

int64_t blmm_launch_count(const blmm_ctx* ctx) {
  if (ctx && ctx->multi) return multi_launch_count(ctx);
  return ctx ? ctx->launches : 0;
}

int blmm_set_profiling(blmm_ctx* ctx, int on) {
  if (!ctx) return BLMM_E_INVALID;
  if (ctx->multi) return multi_set_profiling(ctx, on);
  ctx->profiling = on;
  ctx->scan_timed = false;
  return BLMM_OK;
}

double blmm_last_scan_ms(blmm_ctx* ctx) {
  if (ctx && ctx->multi) return multi_last_scan_ms(ctx);
  if (!ctx || !ctx->scan_timed) return -1.0;
  float ms = -1.f;
  if (cudaEventSynchronize(ctx->ev1) != cudaSuccess) return -1.0;
  if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) != cudaSuccess) return -1.0;
  return (double)ms;
}

double blmm_last_gather_ms(const blmm_ctx* ctx) { return ctx ? ctx->gather_ms : -1.0; }

double blmm_host_write_gbs(int nthreads, int64_t bytes) {
  if (bytes < 4096) return -1.0;
  return host_write_gbs(nthreads > 0 ? nthreads : default_host_threads(), (size_t)bytes);
}

// entry points that do not shard run on the primary GPU of a multi-GPU context
#define PRIMARY(ctx) ((ctx) && (ctx)->multi ? multi_primary(ctx) : (ctx))
#define FORWARD_ERR(parent, call)                                  \
  do {                                                             \
    blmm_ctx* _p = PRIMARY(parent);                                \
    const int _st = (call);                                        \
    if ((parent) && _p != (parent)) (parent)->err = _p->err;       \
    return _st;                                                    \
  } while (0)

int blmm_kinship(blmm_ctx* ctx, int64_t n, int64_t p, const double* G, double* K_out, int mem_space) {
  FORWARD_ERR(ctx, guarded(_p, [&] { return kinship(_p, n, p, G, K_out, mem_space); }));
}

int blmm_decompose(blmm_ctx* ctx, int64_t n, const double* K, int scheme, double* U_out, double* lambda_out,
                   int* nneg_out, int mem_space) {
  FORWARD_ERR(ctx, guarded(_p, [&] { return decompose(_p, n, K, scheme, U_out, lambda_out, nneg_out, mem_space); }));
}

int blmm_rotate(blmm_ctx* ctx, const blmm_problem* prob, double* Y0_out, double* X0_out, int mem_space) {
  FORWARD_ERR(ctx, guarded(_p, [&] { return rotate(_p, prob, Y0_out, X0_out, mem_space); }));
}

int blmm_bulkscan(blmm_ctx* ctx, const blmm_problem* prob, const blmm_opts* opts, double* L_out, double* h2_out) {
  if (ctx && ctx->multi) return multi_bulkscan(ctx, prob, opts, L_out, h2_out);
  return guarded(ctx, opts, [&] {
    switch (opts->method) {
      case BLMM_METHOD_NULL_GRID:
      case BLMM_METHOD_ALT_GRID:
        return bulkscan_grid(ctx, prob, opts, L_out, h2_out);
      case BLMM_METHOD_NULL_EXACT:
        return bulkscan_exact(ctx, prob, opts, L_out, h2_out, nullptr);
      default:
        throw Fail{BLMM_E_INVALID, "unknown method"};
    }
  });
}

int blmm_bulkscan_peaks(blmm_ctx* ctx, const blmm_problem* prob, const blmm_opts* opts, double* peak_lod_out,
                        int64_t* peak_marker_out, double* h2_out) {
  if (ctx && ctx->multi) return multi_bulkscan_peaks(ctx, prob, opts, peak_lod_out, peak_marker_out, h2_out);
  return guarded(ctx, opts, [&] {
    const PeakOut pk{peak_lod_out, peak_marker_out, h2_out};
    switch (opts->method) {
      case BLMM_METHOD_NULL_GRID:
      case BLMM_METHOD_ALT_GRID:
        return bulkscan_grid(ctx, prob, opts, nullptr, nullptr, &pk);
      case BLMM_METHOD_NULL_EXACT:
        return bulkscan_exact(ctx, prob, opts, nullptr, nullptr, nullptr, &pk);
      default:
        throw Fail{BLMM_E_INVALID, "unknown method"};
    }
  });
}

int blmm_grid_loglik(blmm_ctx* ctx, const blmm_problem* prob, const blmm_opts* opts, double* ell_out) {
  if (ctx && ctx->multi) return multi_grid_loglik(ctx, prob, opts, ell_out);
  return guarded(ctx, opts, [&] { return grid_loglik(ctx, prob, opts, ell_out); });
}

int blmm_fit_h2(blmm_ctx* ctx, const blmm_problem* prob, const blmm_opts* opts, double* h2_out, double* sigma2_out,
                double* ell_out) {
  if (ctx && ctx->multi) return multi_fit_h2(ctx, prob, opts, h2_out, sigma2_out, ell_out);
  return guarded(ctx, opts, [&] { return fit_h2(ctx, prob, opts, h2_out, sigma2_out, ell_out); });
}

int blmm_scan_perms(blmm_ctx* ctx, const blmm_problem* prob, const blmm_opts* opts, const int32_t* perm_idx,
                    int64_t nperms, double* lod_out, double* Lperms_out, double* maxlod_out, double* sigma2_out,
                    double* h2_out) {
  if (ctx && ctx->multi)
    return multi_scan_perms(ctx, prob, opts, perm_idx, nperms, lod_out, Lperms_out, maxlod_out, sigma2_out, h2_out);
  return guarded(ctx, opts, [&] {
    return scan_perms(ctx, prob, opts, perm_idx, nperms, lod_out, Lperms_out, maxlod_out, sigma2_out, h2_out);
  });
}

int blmm_scan_null(blmm_ctx* ctx, const blmm_problem* prob, const blmm_opts* opts, double* lod_out,
                   double* sigma2_out, double* h2_out) {
  if (ctx && ctx->multi) return multi_scan_null(ctx, prob, opts, lod_out, sigma2_out, h2_out);
  return guarded(ctx, opts, [&] { return bulkscan_exact(ctx, prob, opts, lod_out, h2_out, sigma2_out); });
}

int blmm_scan_alt(blmm_ctx* ctx, const blmm_problem* prob, const blmm_opts* opts, double* lod_out,
                  double* h2_each_marker_out, double* sigma2_out, double* h2_out) {
  FORWARD_ERR(ctx, guarded(_p, opts, [&] {
    return scan_alt(_p, prob, opts, lod_out, h2_each_marker_out, sigma2_out, h2_out);
  }));
}

int blmm_lod2log10p(blmm_ctx* ctx, const double* lod, int64_t rows, int64_t cols, int64_t ld_in, int64_t ld_out, int df,
                    double* out, int mem_space) {
  FORWARD_ERR(ctx, guarded(_p, [&] { return lod2log10p(_p, lod, rows, cols, ld_in, ld_out, df, out, mem_space); }));
}

int blmm_thresholds(blmm_ctx* ctx, const double* maxlod, int64_t nperms, const double* signif_level, int nlev,
                    double* thrs_out, int mem_space) {
  FORWARD_ERR(ctx, guarded(_p, [&] { return thresholds(_p, maxlod, nperms, signif_level, nlev, thrs_out, mem_space); }));
}

int blmm_weight_kinship(blmm_ctx* ctx, int64_t n, const double* K, const double* w, double* K_out, int mem_space) {
  FORWARD_ERR(ctx, guarded(_p, [&] { return weight_kinship(_p, n, K, w, K_out, mem_space); }));
}

}  // extern "C"
