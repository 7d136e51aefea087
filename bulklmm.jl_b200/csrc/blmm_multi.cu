// Several GPUs behind ONE context (blmm_create_multi): the analogue of the reference's `nb` trait blocks
// (Threads.@threads over column blocks of Y, src/bulkscan.jl:263-309), with a GPU per block.
//
//   * one persistent host thread per GPU; each drives an ordinary single-GPU context through the public entry points;
//   * bulkscan shards TRAITS, scan-with-permutations shards PERMUTATION columns, into contiguous column blocks cut at
//     multiples of the 128-column trait tile; G, Covar, (U, lambda) are replicated; there is no exchange step in the
//     arithmetic, so the sharded result is bit-identical to the single-GPU one;
//   * BLMM_MEM_HOST: every GPU reads its block of the caller's host arrays and writes its contiguous slab of the
//     caller's column-major results over its own PCIe link;
//   * BLMM_MEM_DEVICE: the caller's pointers live on the PRIMARY GPU (devices[0]).  NCCL over NVLink broadcasts the
//     replicated inputs, scatters the column blocks, and gathers the result slabs (LOD, h2 panel / h2_null_list,
//     per-permutation maximum LOD) into the primary's output arrays; the device time of that gather is reported by
//     blmm_last_gather_ms().  NCCL is loaded at first use (dlopen "libnccl.so.2"): host-buffer calls never need it.
#include <dlfcn.h>
#include <nccl.h>

#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

#include "blmm_ctx.cuh"
#include "blmm_kernels.cuh"

namespace blmm {

namespace {

struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
};

struct Worker {
  std::thread th;
  std::mutex mu;
  std::condition_variable cv;
  std::function<int()> job;
  bool has_job = false, quit = false;
  int rc = 0;
};

// grow-only device buffers of one GPU for device-resident multi-GPU calls
enum MBuf { MB_G, MB_C, MB_U, MB_LAM, MB_W, MB_Y, MB_L, MB_H, MB_P, MB_PERM, MB_LOD, MB_MAX, MB_SCAL, MB_COUNT };

struct DevBufs {
  void* p[MB_COUNT] = {};
  size_t cap[MB_COUNT] = {};
};

}  // namespace

struct MultiState {
  int ndev = 0;
  std::vector<int> devices;
  std::vector<blmm_ctx*> sub;
  std::vector<Worker*> workers;
  std::vector<DevBufs> bufs;
  NcclApi nccl;
  std::vector<ncclComm_t> comms;
  cudaEvent_t g0 = nullptr, g1 = nullptr;  // primary: around the gather
  bool gather_timed = false;
  std::vector<std::vector<double>> scratch;  // per GPU host scratch (outputs only the primary reports)
};

namespace {

void worker_loop(Worker* w, int device) {
  cudaSetDevice(device);
  for (;;) {
    std::function<int()> job;
    {
      std::unique_lock<std::mutex> lk(w->mu);
      w->cv.wait(lk, [&] { return w->quit || w->has_job; });
      if (w->quit) return;
      job = w->job;
    }
    int rc;
    try {
      rc = job();
    } catch (...) {
      rc = BLMM_E_INVALID;
    }
    {
      std::lock_guard<std::mutex> lk(w->mu);
      w->rc = rc;
      w->has_job = false;
    }
    w->cv.notify_all();
  }
}

// Runs f(r) on GPU r's thread for every r, waits for all; returns the status of the lowest failing r (-1: none).
int run_all(MultiState* M, const std::function<int(int)>& f, int* fail_rank = nullptr) {
  for (int r = 0; r < M->ndev; ++r) {
    Worker* w = M->workers[r];
    {
      std::lock_guard<std::mutex> lk(w->mu);
      w->job = [&f, r] { return f(r); };
      w->has_job = true;
    }
    w->cv.notify_all();
  }
  int rc = BLMM_OK;
  for (int r = M->ndev - 1; r >= 0; --r) {
    Worker* w = M->workers[r];
    std::unique_lock<std::mutex> lk(w->mu);
    w->cv.wait(lk, [&] { return !w->has_job; });
    if (w->rc != BLMM_OK) {
      rc = w->rc;
      if (fail_rank) *fail_rank = r;
    }
  }
  return rc;
}

int fail(blmm_ctx* parent, int code, const std::string& msg) {
  parent->err = msg;
  return code;
}

// status of a sharded call: the failing GPU's own message (the reference's string where it has one)
int finish(blmm_ctx* parent, int rc, int fail_rank) {
  if (rc == BLMM_OK) {
    parent->err.clear();
    return rc;
  }
  MultiState* M = parent->multi;
  const char* m = (fail_rank >= 0 && fail_rank < M->ndev) ? blmm_last_error(M->sub[fail_rank]) : "";
  parent->err = (m && *m) ? m : "multi-GPU call failed";
  return rc;
}

// columns [j0, j1) of GPU r when `total` columns are cut at multiples of `align`
void shard_cols(int64_t total, int ndev, int r, int64_t align, int64_t* j0, int64_t* j1) {
  const int64_t tiles = (total + align - 1) / align;
  *j0 = std::min<int64_t>(total, tiles * r / ndev * align);
  *j1 = std::min<int64_t>(total, tiles * (r + 1) / ndev * align);
}

// permutation columns [s0[r], s1[r]) of every GPU: each GPU also scans the un-permuted trait as its column 0, so
// blocks of 128 - 1 permutations fill whole 128-column tiles; the first GPUs get the tiles when there are fewer
// tiles than GPUs (the primary always has work: it reports the un-permuted LODs)
void shard_perms(int64_t nperms, int ndev, std::vector<int64_t>& s0, std::vector<int64_t>& s1) {
  const int64_t tiles = (nperms + ndev + SCAN_TT - 1) / SCAN_TT;
  int64_t pos = 0;
  for (int r = 0; r < ndev; ++r) {
    const int64_t tr = tiles * (ndev - r) / ndev - tiles * (ndev - r - 1) / ndev;
    const int64_t cnt = std::min<int64_t>(tr > 0 ? tr * SCAN_TT - 1 : 0, nperms - pos);
    s0[r] = pos;
    s1[r] = pos + cnt;
    pos += cnt;
  }
}

template <typename T>
T* mbuf(MultiState* M, int r, MBuf b, size_t count) {
  DevBufs& B = M->bufs[r];
  const size_t bytes = std::max<size_t>(count * sizeof(T), 256);
  if (B.cap[b] < bytes) {
    if (B.p[b]) CUDA_TRY(cudaFree(B.p[b]));
    B.p[b] = nullptr;
    B.cap[b] = 0;
    CUDA_TRY(cudaMalloc(&B.p[b], bytes));
    B.cap[b] = bytes;
  }
  return reinterpret_cast<T*>(B.p[b]);
}

#define NCCL_TRY(expr)                                                                                         \
  do {                                                                                                         \
    ncclResult_t _r = (expr);                                                                                  \
    if (_r != ncclSuccess)                                                                                     \
      throw Fail{BLMM_E_CUDA, std::string(#expr) + ": " + (M->nccl.GetErrorString ? M->nccl.GetErrorString(_r) : "NCCL error")}; \
  } while (0)

void ensure_nccl(MultiState* M) {
  if (!M->comms.empty()) return;
  NcclApi& N = M->nccl;
  if (!N.lib) {
    N.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!N.lib) N.lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!N.lib) throw Fail{BLMM_E_CUDA, std::string("NCCL is not loadable (device-resident multi-GPU calls need it): ") + dlerror()};
    bool ok = true;
    auto sym = [&](const char* name) {
      void* s = dlsym(N.lib, name);
      ok = ok && s;
      return s;
    };
    N.CommInitAll = reinterpret_cast<decltype(N.CommInitAll)>(sym("ncclCommInitAll"));
    N.CommDestroy = reinterpret_cast<decltype(N.CommDestroy)>(sym("ncclCommDestroy"));
    N.GetErrorString = reinterpret_cast<decltype(N.GetErrorString)>(sym("ncclGetErrorString"));
    N.Broadcast = reinterpret_cast<decltype(N.Broadcast)>(sym("ncclBroadcast"));
    N.Send = reinterpret_cast<decltype(N.Send)>(sym("ncclSend"));
    N.Recv = reinterpret_cast<decltype(N.Recv)>(sym("ncclRecv"));
    N.GroupStart = reinterpret_cast<decltype(N.GroupStart)>(sym("ncclGroupStart"));
    N.GroupEnd = reinterpret_cast<decltype(N.GroupEnd)>(sym("ncclGroupEnd"));
    if (!ok) throw Fail{BLMM_E_CUDA, "libnccl.so.2 lacks a required symbol"};
  }
  std::vector<ncclComm_t> comms(M->ndev);
  NCCL_TRY(N.CommInitAll(comms.data(), M->ndev, M->devices.data()));
  M->comms = comms;
}

// One replicated input: broadcast from the primary's pointer into GPU r's buffer (in place on the primary).
struct Bcast {
  const void* root_ptr;
  MBuf buf;
  size_t bytes;
};

}  // namespace

// ---------------------------------------------------------------------------------------------------------
int multi_create(blmm_ctx* parent, const int* devices, int ndev) {
  MultiState* M = new MultiState();
  parent->multi = M;
  M->ndev = ndev;
  M->devices.assign(devices, devices + ndev);
  M->bufs.resize(ndev);
  M->scratch.resize(ndev);
  // drain threads per GPU: BLMM_B200_HOST_THREADS is per GPU; by default the host's cores are divided between them
  int host_threads = default_host_threads();
  if (!getenv("BLMM_B200_HOST_THREADS")) {
    const unsigned hc = std::thread::hardware_concurrency();
    host_threads = std::max(1, std::min(16, ((int)hc - 1) / ndev));
  }
  for (int r = 0; r < ndev; ++r) {
    blmm_ctx* c = nullptr;
    const int st = blmm_create(&c, devices[r]);
    if (st != BLMM_OK) return st;
    c->host_threads = host_threads;
    M->sub.push_back(c);
  }
  for (int r = 0; r < ndev; ++r) {
    Worker* w = new Worker();
    M->workers.push_back(w);
    w->th = std::thread(worker_loop, w, devices[r]);
  }
  parent->device = devices[0];
  parent->sm_count = M->sub[0]->sm_count;
  if (cudaSetDevice(devices[0]) != cudaSuccess || cudaEventCreate(&M->g0) != cudaSuccess ||
      cudaEventCreate(&M->g1) != cudaSuccess)
    return BLMM_E_CUDA;
  return BLMM_OK;
}

void multi_destroy(blmm_ctx* parent) {
  MultiState* M = parent->multi;
  if (!M) return;
  for (Worker* w : M->workers) {
    {
      std::lock_guard<std::mutex> lk(w->mu);
      w->quit = true;
    }
    w->cv.notify_all();
    if (w->th.joinable()) w->th.join();
    delete w;
  }
  for (blmm_ctx* c : M->sub)
    if (c) blmm_sync(c);
  if (M->nccl.CommDestroy)
    for (ncclComm_t c : M->comms) M->nccl.CommDestroy(c);
  for (int r = 0; r < (int)M->bufs.size(); ++r) {
    cudaSetDevice(M->devices[r]);
    for (int b = 0; b < MB_COUNT; ++b)
      if (M->bufs[r].p[b]) cudaFree(M->bufs[r].p[b]);
  }
  if (M->g0) cudaEventDestroy(M->g0);
  if (M->g1) cudaEventDestroy(M->g1);
  for (blmm_ctx* c : M->sub) blmm_destroy(c);
  delete M;
  parent->multi = nullptr;
}

int multi_ndev(const blmm_ctx* parent) { return parent->multi ? parent->multi->ndev : 1; }
blmm_ctx* multi_primary(blmm_ctx* parent) { return parent->multi->sub[0]; }

int multi_sync(blmm_ctx* parent) {
  MultiState* M = parent->multi;
  int fr = -1;
  const int rc = run_all(M, [&](int r) { return blmm_sync(M->sub[r]); }, &fr);
  if (rc == BLMM_OK && M->gather_timed) {
    float ms = -1.f;
    cudaSetDevice(M->devices[0]);
    if (cudaEventElapsedTime(&ms, M->g0, M->g1) == cudaSuccess) parent->gather_ms = (double)ms;
    M->gather_timed = false;
  }
  return finish(parent, rc, fr);
}

int64_t multi_launch_count(const blmm_ctx* parent) {
  int64_t s = 0;
  for (blmm_ctx* c : parent->multi->sub) s += c->launches;
  return s;
}

int multi_set_profiling(blmm_ctx* parent, int on) {
  for (blmm_ctx* c : parent->multi->sub) blmm_set_profiling(c, on);
  return BLMM_OK;
}

double multi_last_scan_ms(blmm_ctx* parent) {
  MultiState* M = parent->multi;
  std::vector<double> ms(M->ndev, -1.0);
  run_all(M, [&](int r) {
    ms[r] = blmm_last_scan_ms(M->sub[r]);
    return BLMM_OK;
  });
  double mx = -1.0;
  for (double v : ms) mx = std::max(mx, v);
  return mx;
}

// ---------------------------------------------------------------------------------------------------------
// bulkscan: traits sharded
// ---------------------------------------------------------------------------------------------------------
int multi_bulkscan(blmm_ctx* parent, const blmm_problem* pr, const blmm_opts* o, double* L_out, double* h2_out) {
  MultiState* M = parent->multi;
  if (!pr || !o) return fail(parent, BLMM_E_INVALID, "problem / opts is NULL");
  if (pr->n <= 0 || pr->m < 0 || pr->p <= 0) return fail(parent, BLMM_E_DIM, "Dimension mismatch.");
  if (!L_out) return fail(parent, BLMM_E_INVALID, "L_out is NULL");
  const int64_t n = pr->n, p = pr->p, m = pr->m;
  const int64_t ld = o->ld_out ? o->ld_out : p;
  const bool alt = o->method == BLMM_METHOD_ALT_GRID;
  const bool dev = o->mem_space == BLMM_MEM_DEVICE;
  const int nd = M->ndev;
  std::vector<int64_t> j0(nd), j1(nd);
  for (int r = 0; r < nd; ++r) shard_cols(m, nd, r, SCAN_TT, &j0[r], &j1[r]);
  int fr = -1;

  if (!dev) {
    // the h2 panel's PCIe encoding is decided on the whole panel: what limits a multi-GPU host call is the host's
    // ingest rate (all GPUs feed one memory system), and one-byte indices halve the bytes that cross it
    const int idx_hint = ((double)p * (double)m >= 1e8) ? 1 : 0;
    const int rc = run_all(M, [&](int r) -> int {
      if (j1[r] == j0[r]) return BLMM_OK;
      M->sub[r]->idx_hint = idx_hint;
      blmm_problem sp = *pr;
      sp.Y = pr->Y + j0[r] * n;
      sp.m = j1[r] - j0[r];
      blmm_opts so = *o;
      if (o->log10p_out) so.log10p_out = o->log10p_out + j0[r] * ld;
      double* h = h2_out ? (alt ? h2_out + j0[r] * ld : h2_out + j0[r]) : nullptr;
      return blmm_bulkscan(M->sub[r], &sp, &so, L_out + j0[r] * ld, h);
    }, &fr);
    return finish(parent, rc, fr);
  }

  // device-resident: pointers on the primary GPU; NCCL moves the shards
  if (ld != p) return fail(parent, BLMM_E_INVALID, "multi-GPU device-resident calls need ld_out == p (contiguous slabs)");
  if (pr->c < 1 || pr->c > MAXC || !pr->Y || !pr->G || !pr->Covar || !pr->U || !pr->lambda)
    return fail(parent, BLMM_E_INVALID, "bad problem (NULL input or covariate count)");
  const bool pv = o->chisq_df > 0;
  if (pv && !o->log10p_out) return fail(parent, BLMM_E_INVALID, "chisq_df > 0 but log10p_out is NULL");
  try {
    ensure_nccl(M);
  } catch (const Fail& f) {
    return fail(parent, f.code, f.msg);
  }
  // phase A: buffers on every GPU (a failure here must not leave the others waiting inside NCCL)
  int rc = run_all(M, [&](int r) -> int {
    if (r == 0) return BLMM_OK;
    try {
      const size_t mr = (size_t)(j1[r] - j0[r]);
      mbuf<double>(M, r, MB_G, (size_t)n * p);
      mbuf<double>(M, r, MB_C, (size_t)n * pr->c);
      mbuf<double>(M, r, MB_U, (size_t)n * n);
      mbuf<double>(M, r, MB_LAM, n);
      if (pr->obs_weights) mbuf<double>(M, r, MB_W, n);
      mbuf<double>(M, r, MB_Y, (size_t)n * mr);
      mbuf<double>(M, r, MB_L, (size_t)p * mr);
      if (h2_out) mbuf<double>(M, r, MB_H, alt ? (size_t)p * mr : mr);
      if (pv) mbuf<double>(M, r, MB_P, (size_t)p * mr);
    } catch (const Fail& f) {
      M->sub[r]->err = f.msg;
      return f.code;
    }
    return BLMM_OK;
  }, &fr);
  if (rc != BLMM_OK) return finish(parent, rc, fr);

  const std::vector<Bcast> bc = {{pr->G, MB_G, (size_t)n * p * 8},   {pr->Covar, MB_C, (size_t)n * pr->c * 8},
                                 {pr->U, MB_U, (size_t)n * n * 8},   {pr->lambda, MB_LAM, (size_t)n * 8},
                                 {pr->obs_weights, MB_W, (size_t)n * 8}};
  rc = run_all(M, [&](int r) -> int {
    blmm_ctx* c = M->sub[r];
    cudaStream_t st = c->stream;
    NcclApi& N = M->nccl;
    ncclComm_t comm = M->comms[r];
    int status = BLMM_OK;
    try {
      DevBufs& B = M->bufs[r];
      // scatter / broadcast
      NCCL_TRY(N.GroupStart());
      for (const Bcast& b : bc) {
        if (!b.root_ptr) continue;
        void* mine = r == 0 ? const_cast<void*>(b.root_ptr) : B.p[b.buf];
        NCCL_TRY(N.Broadcast(mine, mine, b.bytes, ncclChar, 0, comm, st));
      }
      if (r == 0) {
        for (int q = 1; q < nd; ++q)
          if (j1[q] > j0[q]) NCCL_TRY(N.Send(pr->Y + j0[q] * n, (size_t)(j1[q] - j0[q]) * n, ncclDouble, q, comm, st));
      } else if (j1[r] > j0[r]) {
        NCCL_TRY(N.Recv(B.p[MB_Y], (size_t)(j1[r] - j0[r]) * n, ncclDouble, 0, comm, st));
      }
      NCCL_TRY(N.GroupEnd());
      // compute on the local block
      const int64_t mr = j1[r] - j0[r];
      double *Lr, *Hr = nullptr, *Pr = nullptr;
      blmm_problem sp = *pr;
      blmm_opts so = *o;
      sp.m = mr;
      if (r == 0) {
        sp.Y = pr->Y;  // j0[0] == 0
        Lr = L_out;
        Hr = h2_out;
        Pr = o->log10p_out;
      } else {
        sp.Y = (const double*)B.p[MB_Y];
        sp.G = (const double*)B.p[MB_G];
        sp.Covar = (const double*)B.p[MB_C];
        sp.U = (const double*)B.p[MB_U];
        sp.lambda = (const double*)B.p[MB_LAM];
        if (pr->obs_weights) sp.obs_weights = (const double*)B.p[MB_W];
        Lr = (double*)B.p[MB_L];
        if (h2_out) Hr = (double*)B.p[MB_H];
        if (pv) Pr = (double*)B.p[MB_P];
      }
      so.log10p_out = Pr;
      so.ld_out = p;
      if (mr > 0) status = blmm_bulkscan(c, &sp, &so, Lr, Hr);
      // gather the slabs on the primary (always entered, so that no GPU waits for a failed one)
      if (r == 0) {
        CUDA_TRY(cudaEventRecord(M->g0, st));
        NCCL_TRY(N.GroupStart());
        for (int q = 1; q < nd; ++q) {
          const size_t mq = (size_t)(j1[q] - j0[q]);
          if (!mq) continue;
          NCCL_TRY(N.Recv(L_out + j0[q] * p, mq * p, ncclDouble, q, comm, st));
          if (h2_out) NCCL_TRY(N.Recv(alt ? h2_out + j0[q] * p : h2_out + j0[q], alt ? mq * p : mq, ncclDouble, q, comm, st));
          if (pv) NCCL_TRY(N.Recv(o->log10p_out + j0[q] * p, mq * p, ncclDouble, q, comm, st));
        }
        NCCL_TRY(N.GroupEnd());
        CUDA_TRY(cudaEventRecord(M->g1, st));
        M->gather_timed = true;
      } else if (mr > 0) {
        NCCL_TRY(N.GroupStart());
        NCCL_TRY(N.Send(Lr, (size_t)mr * p, ncclDouble, 0, comm, st));
        if (h2_out) NCCL_TRY(N.Send(Hr, alt ? (size_t)mr * p : (size_t)mr, ncclDouble, 0, comm, st));
        if (pv) NCCL_TRY(N.Send(Pr, (size_t)mr * p, ncclDouble, 0, comm, st));
        NCCL_TRY(N.GroupEnd());
      }
    } catch (const Fail& f) {
      c->err = f.msg;
      return f.code;
    }
    return status;
  }, &fr);
  return finish(parent, rc, fr);
}

// ---------------------------------------------------------------------------------------------------------
// scan with permutations: permutation columns sharded; every GPU repeats the (cheap) null fit of the one trait
// ---------------------------------------------------------------------------------------------------------
int multi_scan_perms(blmm_ctx* parent, const blmm_problem* pr, const blmm_opts* o, const int32_t* perm_idx,
                     int64_t nperms, double* lod_out, double* Lperms_out, double* maxlod_out, double* sigma2_out,
                     double* h2_out) {
  MultiState* M = parent->multi;
  if (!pr || !o) return fail(parent, BLMM_E_INVALID, "problem / opts is NULL");
  if (pr->m != 1) return fail(parent, BLMM_E_ONE_TRAIT, "Can only handle one trait.");
  if (pr->n <= 0 || pr->p <= 0) return fail(parent, BLMM_E_DIM, "Dimension mismatch.");
  if (nperms < 0 || (nperms > 0 && !perm_idx)) return fail(parent, BLMM_E_INVALID, "perm_idx is NULL");
  if (!lod_out) return fail(parent, BLMM_E_INVALID, "lod_out is NULL");
  const int64_t n = pr->n, p = pr->p;
  const int64_t ld = o->ld_out ? o->ld_out : p;
  const bool dev = o->mem_space == BLMM_MEM_DEVICE;
  const int nd = M->ndev;
  std::vector<int64_t> s0(nd), s1(nd);
  shard_perms(nperms, nd, s0, s1);
  int fr = -1;

  if (!dev) {
    const int rc = run_all(M, [&](int r) -> int {
      const int64_t np = s1[r] - s0[r];
      if (r > 0 && np == 0) return BLMM_OK;
      double *lod = lod_out, *s2 = sigma2_out, *h2 = h2_out;
      if (r > 0) {  // the un-permuted LODs and the null fit are reported by the primary only
        M->scratch[r].resize((size_t)p + 2);
        lod = M->scratch[r].data();
        s2 = lod + p;
        h2 = lod + p + 1;
      }
      return blmm_scan_perms(M->sub[r], pr, o, perm_idx ? perm_idx + s0[r] * n : nullptr, np, lod,
                             Lperms_out ? Lperms_out + s0[r] * ld : nullptr, maxlod_out ? maxlod_out + s0[r] : nullptr,
                             s2, h2);
    }, &fr);
    return finish(parent, rc, fr);
  }

  if (ld != p) return fail(parent, BLMM_E_INVALID, "multi-GPU device-resident calls need ld_out == p (contiguous slabs)");
  if (pr->c < 1 || pr->c > MAXC || !pr->Y || !pr->G || !pr->Covar || !pr->U || !pr->lambda)
    return fail(parent, BLMM_E_INVALID, "bad problem (NULL input or covariate count)");
  try {
    ensure_nccl(M);
  } catch (const Fail& f) {
    return fail(parent, f.code, f.msg);
  }
  int rc = run_all(M, [&](int r) -> int {
    if (r == 0) return BLMM_OK;
    try {
      const size_t np = (size_t)(s1[r] - s0[r]);
      mbuf<double>(M, r, MB_G, (size_t)n * p);
      mbuf<double>(M, r, MB_C, (size_t)n * pr->c);
      mbuf<double>(M, r, MB_U, (size_t)n * n);
      mbuf<double>(M, r, MB_LAM, n);
      if (pr->obs_weights) mbuf<double>(M, r, MB_W, n);
      mbuf<double>(M, r, MB_Y, n);
      mbuf<int32_t>(M, r, MB_PERM, (size_t)n * np);
      mbuf<double>(M, r, MB_LOD, p);
      if (Lperms_out) mbuf<double>(M, r, MB_L, (size_t)p * np);
      if (maxlod_out) mbuf<double>(M, r, MB_MAX, np);
      mbuf<double>(M, r, MB_SCAL, 2);
    } catch (const Fail& f) {
      M->sub[r]->err = f.msg;
      return f.code;
    }
    return BLMM_OK;
  }, &fr);
  if (rc != BLMM_OK) return finish(parent, rc, fr);

  const std::vector<Bcast> bc = {{pr->G, MB_G, (size_t)n * p * 8},   {pr->Covar, MB_C, (size_t)n * pr->c * 8},
                                 {pr->U, MB_U, (size_t)n * n * 8},   {pr->lambda, MB_LAM, (size_t)n * 8},
                                 {pr->obs_weights, MB_W, (size_t)n * 8}, {pr->Y, MB_Y, (size_t)n * 8}};
  rc = run_all(M, [&](int r) -> int {
    blmm_ctx* c = M->sub[r];
    cudaStream_t st = c->stream;
    NcclApi& N = M->nccl;
    ncclComm_t comm = M->comms[r];
    int status = BLMM_OK;
    try {
      DevBufs& B = M->bufs[r];
      NCCL_TRY(N.GroupStart());
      for (const Bcast& b : bc) {
        if (!b.root_ptr) continue;
        void* mine = r == 0 ? const_cast<void*>(b.root_ptr) : B.p[b.buf];
        NCCL_TRY(N.Broadcast(mine, mine, b.bytes, ncclChar, 0, comm, st));
      }
      if (r == 0) {
        for (int q = 1; q < nd; ++q)
          if (s1[q] > s0[q]) NCCL_TRY(N.Send(perm_idx + s0[q] * n, (size_t)(s1[q] - s0[q]) * n, ncclInt32, q, comm, st));
      } else if (s1[r] > s0[r]) {
        NCCL_TRY(N.Recv(B.p[MB_PERM], (size_t)(s1[r] - s0[r]) * n, ncclInt32, 0, comm, st));
      }
      NCCL_TRY(N.GroupEnd());
      const int64_t np = s1[r] - s0[r];
      blmm_opts so = *o;
      so.ld_out = p;
      if (r == 0) {
        status = blmm_scan_perms(c, pr, &so, perm_idx, np, lod_out, Lperms_out, maxlod_out, sigma2_out, h2_out);
      } else if (np > 0) {
        blmm_problem sp = *pr;
        sp.Y = (const double*)B.p[MB_Y];
        sp.G = (const double*)B.p[MB_G];
        sp.Covar = (const double*)B.p[MB_C];
        sp.U = (const double*)B.p[MB_U];
        sp.lambda = (const double*)B.p[MB_LAM];
        if (pr->obs_weights) sp.obs_weights = (const double*)B.p[MB_W];
        double* sc = (double*)B.p[MB_SCAL];
        status = blmm_scan_perms(c, &sp, &so, (const int32_t*)B.p[MB_PERM], np, (double*)B.p[MB_LOD],
                                 Lperms_out ? (double*)B.p[MB_L] : nullptr, maxlod_out ? (double*)B.p[MB_MAX] : nullptr,
                                 sc, sc + 1);
      }
      // NCCL gather of the per-permutation maxima (and the L_perms slabs when they are materialised)
      if (r == 0) {
        CUDA_TRY(cudaEventRecord(M->g0, st));
        NCCL_TRY(N.GroupStart());
        for (int q = 1; q < nd; ++q) {
          const size_t nq = (size_t)(s1[q] - s0[q]);
          if (!nq) continue;
          if (maxlod_out) NCCL_TRY(N.Recv(maxlod_out + s0[q], nq, ncclDouble, q, comm, st));
          if (Lperms_out) NCCL_TRY(N.Recv(Lperms_out + s0[q] * p, nq * p, ncclDouble, q, comm, st));
        }
        NCCL_TRY(N.GroupEnd());
        CUDA_TRY(cudaEventRecord(M->g1, st));
        M->gather_timed = true;
      } else if (np > 0) {
        NCCL_TRY(N.GroupStart());
        if (maxlod_out) NCCL_TRY(N.Send(B.p[MB_MAX], (size_t)np, ncclDouble, 0, comm, st));
        if (Lperms_out) NCCL_TRY(N.Send(B.p[MB_L], (size_t)np * p, ncclDouble, 0, comm, st));
        NCCL_TRY(N.GroupEnd());
      }
    } catch (const Fail& f) {
      c->err = f.msg;
      return f.code;
    }
    return status;
  }, &fr);
  return finish(parent, rc, fr);
}

// ---------------------------------------------------------------------------------------------------------
// the other per-trait entry points: host buffers, traits sharded
// ---------------------------------------------------------------------------------------------------------
namespace {
int host_only(blmm_ctx* parent, const blmm_problem* pr, const blmm_opts* o) {
  if (!pr || !o) return fail(parent, BLMM_E_INVALID, "problem / opts is NULL");
  if (pr->n <= 0 || pr->m < 0) return fail(parent, BLMM_E_DIM, "Dimension mismatch.");
  if (o->mem_space != BLMM_MEM_HOST)
    return fail(parent, BLMM_E_INVALID,
                "multi-GPU contexts take device pointers in blmm_bulkscan and blmm_scan_perms only");
  return BLMM_OK;
}
}  // namespace

int multi_fit_h2(blmm_ctx* parent, const blmm_problem* pr, const blmm_opts* o, double* h2_out, double* sigma2_out,
                 double* ell_out) {
  MultiState* M = parent->multi;
  if (int e = host_only(parent, pr, o)) return e;
  int fr = -1;
  const int rc = run_all(M, [&](int r) -> int {
    int64_t j0, j1;
    shard_cols(pr->m, M->ndev, r, 32, &j0, &j1);
    if (j1 == j0) return BLMM_OK;
    blmm_problem sp = *pr;
    sp.Y = pr->Y + j0 * pr->n;
    sp.m = j1 - j0;
    return blmm_fit_h2(M->sub[r], &sp, o, h2_out ? h2_out + j0 : nullptr, sigma2_out ? sigma2_out + j0 : nullptr,
                       ell_out ? ell_out + j0 : nullptr);
  }, &fr);
  return finish(parent, rc, fr);
}

int multi_scan_null(blmm_ctx* parent, const blmm_problem* pr, const blmm_opts* o, double* lod_out, double* sigma2_out,
                    double* h2_out) {
  MultiState* M = parent->multi;
  if (int e = host_only(parent, pr, o)) return e;
  if (!lod_out) return fail(parent, BLMM_E_INVALID, "lod_out is NULL");
  const int64_t ld = o->ld_out ? o->ld_out : pr->p;
  int fr = -1;
  const int rc = run_all(M, [&](int r) -> int {
    int64_t j0, j1;
    shard_cols(pr->m, M->ndev, r, 64, &j0, &j1);
    if (j1 == j0) return BLMM_OK;
    blmm_problem sp = *pr;
    sp.Y = pr->Y + j0 * pr->n;
    sp.m = j1 - j0;
    blmm_opts so = *o;
    if (o->log10p_out) so.log10p_out = o->log10p_out + j0 * ld;
    return blmm_scan_null(M->sub[r], &sp, &so, lod_out + j0 * ld, sigma2_out ? sigma2_out + j0 : nullptr,
                          h2_out ? h2_out + j0 : nullptr);
  }, &fr);
  return finish(parent, rc, fr);
}

int multi_bulkscan_peaks(blmm_ctx* parent, const blmm_problem* pr, const blmm_opts* o, double* peak_lod_out,
                         int64_t* peak_marker_out, double* h2_out) {
  MultiState* M = parent->multi;
  if (int e = host_only(parent, pr, o)) return e;
  if (!peak_lod_out) return fail(parent, BLMM_E_INVALID, "peak_lod_out is NULL");
  int fr = -1;
  const int rc = run_all(M, [&](int r) -> int {
    int64_t j0, j1;
    shard_cols(pr->m, M->ndev, r, SCAN_TT, &j0, &j1);
    if (j1 == j0) return BLMM_OK;
    blmm_problem sp = *pr;
    sp.Y = pr->Y + j0 * pr->n;
    sp.m = j1 - j0;
    blmm_opts so = *o;
    if (o->log10p_out) so.log10p_out = o->log10p_out + j0;
    return blmm_bulkscan_peaks(M->sub[r], &sp, &so, peak_lod_out + j0, peak_marker_out ? peak_marker_out + j0 : nullptr,
                               h2_out ? h2_out + j0 : nullptr);
  }, &fr);
  return finish(parent, rc, fr);
}

int multi_grid_loglik(blmm_ctx* parent, const blmm_problem* pr, const blmm_opts* o, double* ell_out) {
  MultiState* M = parent->multi;
  if (int e = host_only(parent, pr, o)) return e;
  if (!ell_out) return fail(parent, BLMM_E_INVALID, "ell_out is NULL");
  int fr = -1;
  const int rc = run_all(M, [&](int r) -> int {
    int64_t j0, j1;
    shard_cols(pr->m, M->ndev, r, 32, &j0, &j1);
    if (j1 == j0) return BLMM_OK;
    blmm_problem sp = *pr;
    sp.Y = pr->Y + j0 * pr->n;
    sp.m = j1 - j0;
    return blmm_grid_loglik(M->sub[r], &sp, o, ell_out + j0 * o->ngrid);
  }, &fr);
  return finish(parent, rc, fr);
}

}  // namespace blmm
