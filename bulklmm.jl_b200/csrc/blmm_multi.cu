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

// grow-only device buffers of one GPU for device-resident multi-GPU calls, one per array of a DeviceCall
struct DevBufs {
  std::vector<void*> p;
  std::vector<size_t> cap;
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

// run_all, then the parent's status and message are those of the lowest failing GPU
int run_ranks(blmm_ctx* parent, const std::function<int(int)>& f) {
  int fr = -1;
  const int rc = run_all(parent->multi, f, &fr);
  return finish(parent, rc, fr);
}

// f(), with a Fail thrown inside reported as c's message and the returned status
template <typename F>
int catch_fail(blmm_ctx* c, F&& f) {
  try {
    return f();
  } catch (const Fail& e) {
    c->err = e.msg;
    return e.code;
  }
}

// the contiguous column block [b[r], e[r]) of every GPU r
struct Shards {
  std::vector<int64_t> b, e;
  explicit Shards(int ndev) : b(ndev), e(ndev) {}
  int64_t count(int r) const { return e[r] - b[r]; }
};

// `total` columns cut at multiples of `align`
Shards shard_cols(int64_t total, int ndev, int64_t align) {
  Shards s(ndev);
  const int64_t tiles = (total + align - 1) / align;
  for (int r = 0; r < ndev; ++r) {
    s.b[r] = std::min<int64_t>(total, tiles * r / ndev * align);
    s.e[r] = std::min<int64_t>(total, tiles * (r + 1) / ndev * align);
  }
  return s;
}

// permutation columns: each GPU also scans the un-permuted trait as its column 0, so blocks of 128 - 1 permutations
// fill whole 128-column tiles; the first GPUs get the tiles when there are fewer tiles than GPUs (the primary always
// has work: it reports the un-permuted LODs)
Shards shard_perms(int64_t nperms, int ndev) {
  Shards s(ndev);
  const int64_t tiles = (nperms + ndev + SCAN_TT - 1) / SCAN_TT;
  int64_t pos = 0;
  for (int r = 0; r < ndev; ++r) {
    const int64_t tr = tiles * (ndev - r) / ndev - tiles * (ndev - r - 1) / ndev;
    const int64_t cnt = std::min<int64_t>(tr > 0 ? tr * SCAN_TT - 1 : 0, nperms - pos);
    s.b[r] = pos;
    s.e[r] = pos + cnt;
    pos += cnt;
  }
  return s;
}

// the problem restricted to GPU r's block of traits
blmm_problem trait_block(const blmm_problem* pr, const Shards& s, int r) {
  blmm_problem sp = *pr;
  sp.Y = pr->Y + s.b[r] * pr->n;
  sp.m = s.count(r);
  return sp;
}

// buffer b of GPU r, at least `bytes` long
void* mbuf(MultiState* M, int r, size_t b, size_t bytes) {
  DevBufs& B = M->bufs[r];
  if (B.p.size() <= b) {
    B.p.resize(b + 1, nullptr);
    B.cap.resize(b + 1, 0);
  }
  bytes = std::max<size_t>(bytes, 256);
  if (B.cap[b] < bytes) {
    if (B.p[b]) CUDA_TRY(cudaFree(B.p[b]));
    B.p[b] = nullptr;
    B.cap[b] = 0;
    CUDA_TRY(cudaMalloc(&B.p[b], bytes));
    B.cap[b] = bytes;
  }
  return B.p[b];
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

// One array of a device-resident call: the caller's pointer on the primary GPU (NULL: the call has no such array)
// and its element count, on every GPU (replicated inputs) or per column (scattered input, gathered outputs).
struct Part {
  const void* root;
  size_t count;
};

// What a device-resident call moves between the GPUs.  The primary works on the caller's arrays; every other GPU
// works on grow-only buffers of its own, one per array, indexed by the array's position in this description.
struct DeviceCall {
  std::vector<Part> replicated;  // doubles, broadcast from the primary
  Part scattered;                // column-sharded input: every GPU receives its own columns from the primary
  ncclDataType_t scattered_type;
  size_t scattered_size;         // bytes per element
  std::vector<Part> gathered;    // doubles: every GPU's column slab lands in the primary's array (count 0: no array)
  std::vector<size_t> scratch;   // doubles of results that stay on the GPUs other than the primary
};

// one GPU's pointers to the arrays of a DeviceCall, in the order of the description (NULL where there is no array)
struct RankPtrs {
  std::vector<const void*> in;
  const void* scattered = nullptr;
  std::vector<double*> out;
  std::vector<double*> scratch;
};

// the inputs of the model every GPU holds a copy of, in the order local_problem() reads them
std::vector<Part> model_inputs(const blmm_problem* pr) {
  const size_t n = (size_t)pr->n;
  return {{pr->G, n * pr->p}, {pr->Covar, n * pr->c}, {pr->U, n * n}, {pr->lambda, n}, {pr->obs_weights, n}};
}

// the problem with GPU r's copies of the model inputs
blmm_problem local_problem(const blmm_problem* pr, const RankPtrs& x) {
  blmm_problem sp = *pr;
  sp.G = (const double*)x.in[0];
  sp.Covar = (const double*)x.in[1];
  sp.U = (const double*)x.in[2];
  sp.lambda = (const double*)x.in[3];
  sp.obs_weights = (const double*)x.in[4];
  return sp;
}

// multi-GPU device-resident calls: pointers on the primary GPU; NCCL moves the shards
int device_checks(blmm_ctx* parent, const blmm_problem* pr, const blmm_opts* o) {
  if ((o->ld_out ? o->ld_out : pr->p) != pr->p)
    return fail(parent, BLMM_E_INVALID, "multi-GPU device-resident calls need ld_out == p (contiguous slabs)");
  if (pr->c < 1 || pr->c > MAXC || !pr->Y || !pr->G || !pr->Covar || !pr->U || !pr->lambda)
    return fail(parent, BLMM_E_INVALID, "bad problem (NULL input or covariate count)");
  return BLMM_OK;
}

// Runs a device-resident call: broadcast the replicated inputs and scatter the column blocks `s` of the sharded one,
// call(r, pointers) on every GPU, gather the result slabs into the primary's arrays.
int run_device(blmm_ctx* parent, const Shards& s, const DeviceCall& d,
               const std::function<int(int, const RankPtrs&)>& call) {
  MultiState* M = parent->multi;
  const int nd = M->ndev;
  int rc = catch_fail(parent, [&] {
    ensure_nccl(M);
    return BLMM_OK;
  });
  if (rc != BLMM_OK) return rc;
  const auto gathers = [](const Part& g) { return g.root && g.count; };
  // buffers on every GPU (a failure here must not leave the others waiting inside NCCL)
  std::vector<RankPtrs> ptrs(nd);
  rc = run_ranks(parent, [&](int r) -> int {
    RankPtrs& x = ptrs[r];
    if (r == 0) {
      for (const Part& a : d.replicated) x.in.push_back(a.root);
      x.scattered = d.scattered.root;
      for (const Part& g : d.gathered) x.out.push_back((double*)g.root);
      return BLMM_OK;
    }
    return catch_fail(M->sub[r], [&] {
      const size_t cols = (size_t)s.count(r);
      size_t b = 0;  // position in the description
      const auto next = [&](bool used, size_t bytes) {
        void* q = used ? mbuf(M, r, b, bytes) : nullptr;
        ++b;
        return q;
      };
      for (const Part& a : d.replicated) x.in.push_back(next(a.root, a.count * 8));
      x.scattered = next(true, d.scattered.count * cols * d.scattered_size);
      for (const Part& g : d.gathered) x.out.push_back((double*)next(gathers(g), g.count * cols * 8));
      for (size_t count : d.scratch) x.scratch.push_back((double*)next(true, count * 8));
      return BLMM_OK;
    });
  });
  if (rc != BLMM_OK) return rc;

  return run_ranks(parent, [&](int r) -> int {
    blmm_ctx* c = M->sub[r];
    return catch_fail(c, [&] {
      const RankPtrs& x = ptrs[r];
      cudaStream_t st = c->stream;
      NcclApi& N = M->nccl;
      ncclComm_t comm = M->comms[r];
      const size_t cols = (size_t)s.count(r);
      // broadcast / scatter
      NCCL_TRY(N.GroupStart());
      for (size_t k = 0; k < d.replicated.size(); ++k) {
        if (!d.replicated[k].root) continue;
        void* mine = const_cast<void*>(x.in[k]);
        NCCL_TRY(N.Broadcast(mine, mine, d.replicated[k].count * 8, ncclChar, 0, comm, st));
      }
      const Part& sc = d.scattered;
      if (r == 0) {
        for (int q = 1; q < nd; ++q)
          if (s.count(q) > 0)
            NCCL_TRY(N.Send((const char*)sc.root + s.b[q] * sc.count * d.scattered_size, s.count(q) * sc.count,
                            d.scattered_type, q, comm, st));
      } else if (cols > 0) {
        NCCL_TRY(N.Recv(const_cast<void*>(x.scattered), cols * sc.count, d.scattered_type, 0, comm, st));
      }
      NCCL_TRY(N.GroupEnd());
      // compute on the local block
      const int status = call(r, x);
      // gather the slabs on the primary (always entered, so that no GPU waits for a failed one)
      if (r == 0) {
        CUDA_TRY(cudaEventRecord(M->g0, st));
        NCCL_TRY(N.GroupStart());
        for (int q = 1; q < nd; ++q) {
          const size_t mq = (size_t)s.count(q);
          if (!mq) continue;
          for (const Part& g : d.gathered)
            if (gathers(g))
              NCCL_TRY(N.Recv((double*)g.root + s.b[q] * g.count, mq * g.count, ncclDouble, q, comm, st));
        }
        NCCL_TRY(N.GroupEnd());
        CUDA_TRY(cudaEventRecord(M->g1, st));
        M->gather_timed = true;
      } else if (cols > 0) {
        NCCL_TRY(N.GroupStart());
        for (size_t k = 0; k < d.gathered.size(); ++k)
          if (gathers(d.gathered[k])) NCCL_TRY(N.Send(x.out[k], cols * d.gathered[k].count, ncclDouble, 0, comm, st));
        NCCL_TRY(N.GroupEnd());
      }
      return status;
    });
  });
}

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
    for (void* b : M->bufs[r].p)
      if (b) cudaFree(b);
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
  const int rc = run_ranks(parent, [&](int r) { return blmm_sync(M->sub[r]); });
  if (rc == BLMM_OK && M->gather_timed) {
    float ms = -1.f;
    cudaSetDevice(M->devices[0]);
    if (cudaEventElapsedTime(&ms, M->g0, M->g1) == cudaSuccess) parent->gather_ms = (double)ms;
    M->gather_timed = false;
  }
  return rc;
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
  const int64_t n = pr->n, p = pr->p;
  const int64_t ld = o->ld_out ? o->ld_out : p;
  const bool alt = o->method == BLMM_METHOD_ALT_GRID;
  const Shards s = shard_cols(pr->m, M->ndev, SCAN_TT);

  if (o->mem_space != BLMM_MEM_DEVICE) {
    // the h2 panel's PCIe encoding is decided on the whole panel: what limits a multi-GPU host call is the host's
    // ingest rate (all GPUs feed one memory system), and one-byte indices halve the bytes that cross it
    const int idx_hint = ((double)p * (double)pr->m >= 1e8) ? 1 : 0;
    return run_ranks(parent, [&](int r) -> int {
      if (!s.count(r)) return BLMM_OK;
      const int64_t j = s.b[r];
      M->sub[r]->idx_hint = idx_hint;
      const blmm_problem sp = trait_block(pr, s, r);
      blmm_opts so = *o;
      if (o->log10p_out) so.log10p_out = o->log10p_out + j * ld;
      double* h = h2_out ? (alt ? h2_out + j * ld : h2_out + j) : nullptr;
      return blmm_bulkscan(M->sub[r], &sp, &so, L_out + j * ld, h);
    });
  }

  if (int e = device_checks(parent, pr, o)) return e;
  const bool pv = o->chisq_df > 0;
  if (pv && !o->log10p_out) return fail(parent, BLMM_E_INVALID, "chisq_df > 0 but log10p_out is NULL");
  // gathered: L, h2 (a panel or one value per trait), -log10 p (the primary gets the caller's pointer either way)
  const DeviceCall d{model_inputs(pr), {pr->Y, (size_t)n}, ncclDouble, sizeof(double),
                     {{L_out, (size_t)p}, {h2_out, alt ? (size_t)p : 1}, {o->log10p_out, pv ? (size_t)p : 0}}, {}};
  return run_device(parent, s, d, [&](int r, const RankPtrs& x) -> int {
    if (!s.count(r)) return BLMM_OK;
    blmm_problem sp = local_problem(pr, x);
    sp.Y = (const double*)x.scattered;
    sp.m = s.count(r);
    blmm_opts so = *o;
    so.log10p_out = x.out[2];
    so.ld_out = p;
    return blmm_bulkscan(M->sub[r], &sp, &so, x.out[0], x.out[1]);
  });
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
  const Shards s = shard_perms(nperms, M->ndev);

  if (o->mem_space != BLMM_MEM_DEVICE) {
    return run_ranks(parent, [&](int r) -> int {
      const int64_t j = s.b[r];
      if (r > 0 && !s.count(r)) return BLMM_OK;
      double *lod = lod_out, *s2 = sigma2_out, *h2 = h2_out;
      if (r > 0) {  // the un-permuted LODs and the null fit are reported by the primary only
        M->scratch[r].resize((size_t)p + 2);
        lod = M->scratch[r].data();
        s2 = lod + p;
        h2 = lod + p + 1;
      }
      return blmm_scan_perms(M->sub[r], pr, o, perm_idx ? perm_idx + j * n : nullptr, s.count(r), lod,
                             Lperms_out ? Lperms_out + j * ld : nullptr, maxlod_out ? maxlod_out + j : nullptr, s2,
                             h2);
    });
  }

  if (int e = device_checks(parent, pr, o)) return e;
  std::vector<Part> replicated = model_inputs(pr);
  replicated.push_back({pr->Y, (size_t)n});
  // gathered: the per-permutation maxima and L_perms; the other GPUs' un-permuted LODs and null fit (sigma2, h2) stay
  const DeviceCall d{replicated, {perm_idx, (size_t)n}, ncclInt32, sizeof(int32_t),
                     {{maxlod_out, 1}, {Lperms_out, (size_t)p}}, {(size_t)p, 2}};
  return run_device(parent, s, d, [&](int r, const RankPtrs& x) -> int {
    if (r > 0 && !s.count(r)) return BLMM_OK;
    blmm_problem sp = local_problem(pr, x);
    sp.Y = (const double*)x.in[5];
    blmm_opts so = *o;
    so.ld_out = p;
    double *lod = lod_out, *s2 = sigma2_out, *h2 = h2_out;
    if (r > 0) {
      lod = x.scratch[0];
      s2 = x.scratch[1];
      h2 = x.scratch[1] + 1;
    }
    return blmm_scan_perms(M->sub[r], &sp, &so, (const int32_t*)x.scattered, s.count(r), lod, x.out[1], x.out[0], s2,
                           h2);
  });
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
  const Shards s = shard_cols(pr->m, M->ndev, 32);
  return run_ranks(parent, [&](int r) -> int {
    if (!s.count(r)) return BLMM_OK;
    const int64_t j = s.b[r];
    const blmm_problem sp = trait_block(pr, s, r);
    return blmm_fit_h2(M->sub[r], &sp, o, h2_out ? h2_out + j : nullptr, sigma2_out ? sigma2_out + j : nullptr,
                       ell_out ? ell_out + j : nullptr);
  });
}

int multi_scan_null(blmm_ctx* parent, const blmm_problem* pr, const blmm_opts* o, double* lod_out, double* sigma2_out,
                    double* h2_out) {
  MultiState* M = parent->multi;
  if (int e = host_only(parent, pr, o)) return e;
  if (!lod_out) return fail(parent, BLMM_E_INVALID, "lod_out is NULL");
  const int64_t ld = o->ld_out ? o->ld_out : pr->p;
  const Shards s = shard_cols(pr->m, M->ndev, 64);
  return run_ranks(parent, [&](int r) -> int {
    if (!s.count(r)) return BLMM_OK;
    const int64_t j = s.b[r];
    const blmm_problem sp = trait_block(pr, s, r);
    blmm_opts so = *o;
    if (o->log10p_out) so.log10p_out = o->log10p_out + j * ld;
    return blmm_scan_null(M->sub[r], &sp, &so, lod_out + j * ld, sigma2_out ? sigma2_out + j : nullptr,
                          h2_out ? h2_out + j : nullptr);
  });
}

int multi_bulkscan_peaks(blmm_ctx* parent, const blmm_problem* pr, const blmm_opts* o, double* peak_lod_out,
                         int64_t* peak_marker_out, double* h2_out) {
  MultiState* M = parent->multi;
  if (int e = host_only(parent, pr, o)) return e;
  if (!peak_lod_out) return fail(parent, BLMM_E_INVALID, "peak_lod_out is NULL");
  const Shards s = shard_cols(pr->m, M->ndev, SCAN_TT);
  return run_ranks(parent, [&](int r) -> int {
    if (!s.count(r)) return BLMM_OK;
    const int64_t j = s.b[r];
    const blmm_problem sp = trait_block(pr, s, r);
    blmm_opts so = *o;
    if (o->log10p_out) so.log10p_out = o->log10p_out + j;
    return blmm_bulkscan_peaks(M->sub[r], &sp, &so, peak_lod_out + j, peak_marker_out ? peak_marker_out + j : nullptr,
                               h2_out ? h2_out + j : nullptr);
  });
}

int multi_grid_loglik(blmm_ctx* parent, const blmm_problem* pr, const blmm_opts* o, double* ell_out) {
  MultiState* M = parent->multi;
  if (int e = host_only(parent, pr, o)) return e;
  if (!ell_out) return fail(parent, BLMM_E_INVALID, "ell_out is NULL");
  const Shards s = shard_cols(pr->m, M->ndev, 32);
  return run_ranks(parent, [&](int r) -> int {
    if (!s.count(r)) return BLMM_OK;
    const blmm_problem sp = trait_block(pr, s, r);
    return blmm_grid_loglik(M->sub[r], &sp, o, ell_out + s.b[r] * o->ngrid);
  });
}

}  // namespace blmm
