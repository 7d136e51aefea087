// Private to the library: the context behind the opaque `blmm_ctx` of include/blmm_b200.h, shared by the API
// translation units (blmm_api.cu: one GPU; blmm_multi.cu: several GPUs behind one context; blmm_hostpipe.cu:
// pageable host results).
#pragma once
#include <cuda_runtime.h>
#include <cusolverDn.h>
#include <stdint.h>

#include <algorithm>
#include <string>

#include "../../include/blmm_b200.h"
#include "blmm_common.cuh"

namespace blmm {

// workspace slots (grow-only device buffers owned by the context)
enum Slot {
  S_Y_IN, S_G_IN, S_C_IN, S_U_IN, S_LAM, S_GRID, S_Y0, S_C0, S_G0, S_YR, S_W, S_SW, S_Q, S_SLW, S_LDS,
  S_ELL, S_RSS, S_BEST, S_ELLMAX, S_MOP, S_TOP, S_E, S_ET, S_BINS, S_TILEK0, S_COLMAP, S_L, S_H2P, S_H2V,
  S_SIG2, S_ELLV, S_Z, S_PERM, S_COLMAX, S_KPART, S_KIN, S_SOLVER, S_EIGV, S_MISC, S_XOP, S_DYINV, S_PVAL,
  S_OBSW, S_UW, S_SORT, S_SORTTMP, S_PROBS, S_H2IDX, S_UNITCTR, S_PEAKS, S_PKMARK,
  S_COUNT
};

struct Fail {
  int code;
  std::string msg;
};

#define CUDA_TRY(expr)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess)                                                                      \
      throw ::blmm::Fail{BLMM_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)};      \
  } while (0)

struct HostPipe;    // blmm_hostpipe.cu
struct MultiState;  // blmm_multi.cu

constexpr int MAX_CHUNK = 16;

}  // namespace blmm

struct blmm_ctx {
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;  // device->host result copies that overlap the scan (host-buffer calls)
  cudaStream_t aux_stream = nullptr;   // staging + rotation of the markers, beside the other two
  cudaEvent_t aux_fork_ev = nullptr, aux_done_ev = nullptr;
  cudaEvent_t chunk_ev[blmm::MAX_CHUNK] = {};
  cudaEvent_t idx_ev[blmm::MAX_CHUNK] = {};  // chunk's h2 index panel has landed in h_idx
  uint8_t* h_idx = nullptr;                   // pinned staging of the h2 index panel (host-buffer alt-grid calls)
  size_t h_idx_cap = 0;
  uint8_t* h_in = nullptr;                    // pinned arena for large pageable inputs of the current call
  size_t h_in_cap = 0, h_in_off = 0;
  cudaEvent_t fork_ev = nullptr, join_ev = nullptr, wc_ev = nullptr;  // marker-side preprocessing on copy_stream
  cusolverDnHandle_t solver = nullptr;
  void* buf[blmm::S_COUNT] = {};
  size_t cap[blmm::S_COUNT] = {};
  int* d_flags = nullptr;
  int* h_flags = nullptr;  // pinned
  std::string err;
  int64_t launches = 0;
  int profiling = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool scan_timed = false;
  bool l2_limit_set = false;  // persisting-L2 carve-out requested on this device
  // host results: pinned bounce ring + drain threads for pageable destinations and the h2 index panel
  blmm::HostPipe* pipe = nullptr;
  int idx_hint = -1;     // multi-GPU parent: encode the h2 panel as indices (1) or not (0), decided on the WHOLE panel
  int host_threads = 0;  // 0 = default (min(16, cores - 1)); a multi-GPU parent divides the cores between its GPUs
  // several GPUs behind one context (blmm_create_multi): this context is then only the dispatcher
  blmm::MultiState* multi = nullptr;
  double gather_ms = -1.0;  // device time of the last NCCL gather (multi-GPU device-resident calls)
};

namespace blmm {

template <typename T>
T* ws(blmm_ctx* ctx, Slot s, size_t count) {
  const size_t bytes = std::max<size_t>(count * sizeof(T), 256);
  if (ctx->cap[s] < bytes) {
    if (ctx->buf[s]) CUDA_TRY(cudaFree(ctx->buf[s]));
    ctx->buf[s] = nullptr;
    ctx->cap[s] = 0;
    CUDA_TRY(cudaMalloc(&ctx->buf[s], bytes));
    ctx->cap[s] = bytes;
  }
  return reinterpret_cast<T*>(ctx->buf[s]);
}

// ---- blmm_hostpipe.cu -------------------------------------------------------------------------------------
// Results that end in ordinary (pageable) host arrays — what a Julia `Array{Float64}` or a numpy array is — cannot be
// the target of an asynchronous device-to-host DMA: the runtime stages such copies through its own buffer on the
// calling thread, one at a time.  The pipe does the staging itself: device -> pinned ring slot (DMA on `stream`)
// -> caller's array (drain threads, non-temporal stores), so the PCIe link never waits for a host copy.  The same
// ring carries the alt-grid h2 panel as one-byte grid indices, expanded to grid[index] by the drain threads.
bool host_ptr_is_pinned(const void* p);
int default_host_threads();
HostPipe* hostpipe_create(int device, int nthreads);
void hostpipe_destroy(HostPipe* hp);
// Queue `cols` columns of `rows` elements from device memory (leading dimension ld_src elements) into the host
// matrix dst (Float64, leading dimension ld_dst).  grid == nullptr: the source elements are Float64 and are copied;
// otherwise they are one-byte indices and dst gets grid[index].  The device-to-host copies are issued on `stream` in
// call order (the caller orders `stream` after the producer); returns when everything is issued, not when it landed.
void hostpipe_push(HostPipe* hp, cudaStream_t stream, double* dst, int64_t ld_dst, const void* src_dev, int64_t ld_src,
                   int64_t rows, int64_t cols, const double* grid);
// The same for a piece the caller has already copied (asynchronously) into its own pinned staging at `staged`
// (`rows` x `cols`, packed) and marked with `ev`: nothing blocks, the drain threads pick it up when `ev` completes.
void hostpipe_push_staged(HostPipe* hp, cudaEvent_t ev, double* dst, int64_t ld_dst, const void* staged, int64_t rows,
                          int64_t cols, const double* grid);
// Input side of the same problem: a host-to-device copy from pageable memory is staged by the runtime on the calling
// thread (one memcpy thread, ~7 GB/s: 3 ms for the 22 MB trait matrix in front of everything else).  The drain threads
// copy `bytes` from `src` into the pinned buffer `pinned_dst` in parallel; returns when the copy is complete (nothing
// else may be queued on the pipe meanwhile).
void hostpipe_gather_input(HostPipe* hp, void* pinned_dst, const void* src, size_t bytes);
// At most `n` drain threads take work from now on (the others sleep): expanding the index panel next to a DMA into
// pinned result arrays needs ~6 threads and more of them only compete with the DMA for the host's memory system
// (1 GPU: 45.3 ms with 6, 48.7 ms with 15), while moving ring slots into pageable arrays wants all of them.
void hostpipe_set_active(HostPipe* hp, int n);
// Blocks until every queued piece is in the caller's arrays; throws Fail on a CUDA error.
void hostpipe_wait(HostPipe* hp);

double host_write_gbs(int nthreads, size_t bytes);

// ---- blmm_multi.cu ----------------------------------------------------------------------------------------
int multi_create(blmm_ctx* parent, const int* devices, int ndev);
void multi_destroy(blmm_ctx* parent);
int multi_ndev(const blmm_ctx* parent);
blmm_ctx* multi_primary(blmm_ctx* parent);
int multi_sync(blmm_ctx* parent);
int64_t multi_launch_count(const blmm_ctx* parent);
int multi_set_profiling(blmm_ctx* parent, int on);
double multi_last_scan_ms(blmm_ctx* parent);
int multi_bulkscan(blmm_ctx* parent, const blmm_problem* prob, const blmm_opts* opts, double* L_out, double* h2_out);
int multi_scan_perms(blmm_ctx* parent, const blmm_problem* prob, const blmm_opts* opts, const int32_t* perm_idx,
                     int64_t nperms, double* lod_out, double* Lperms_out, double* maxlod_out, double* sigma2_out,
                     double* h2_out);
int multi_fit_h2(blmm_ctx* parent, const blmm_problem* prob, const blmm_opts* opts, double* h2_out, double* sigma2_out,
                 double* ell_out);
int multi_scan_null(blmm_ctx* parent, const blmm_problem* prob, const blmm_opts* opts, double* lod_out,
                    double* sigma2_out, double* h2_out);
int multi_grid_loglik(blmm_ctx* parent, const blmm_problem* prob, const blmm_opts* opts, double* ell_out);
int multi_bulkscan_peaks(blmm_ctx* parent, const blmm_problem* prob, const blmm_opts* opts, double* peak_lod_out,
                         int64_t* peak_marker_out, double* h2_out);

}  // namespace blmm
