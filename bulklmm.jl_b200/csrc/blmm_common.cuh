// Shared device helpers for libblmm_b200 (sm_100a only): mbarrier / bulk-async-copy (TMA engine)
// PTX wrappers, the FP64 tensor-core atom, warp reductions, and the operand layout constants.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace blmm {

// ---------------------------------------------------------------------------------------------
// Operand layout ("K-chunked panels").
// Both GEMM operands are K-contiguous vectors of length n (a trait or a marker).  They are stored
// as [q][col][KC] with KC = 20 doubles per K-chunk: a tile of consecutive columns of one chunk is
// ONE contiguous block (a single bulk async copy), and a row stride of 20 doubles makes the DMMA
// fragment loads (8 rows x 4 consecutive doubles per warp) shared-memory bank-conflict free
// (20*2 mod 32 = 8: the four rows of a half-warp land on four disjoint 8-bank groups).
// ---------------------------------------------------------------------------------------------
constexpr int KC = 20;
constexpr int MAXC = 8;      // covariate columns incl. intercept handled by the register paths
constexpr int NTRI = MAXC * (MAXC + 1) / 2;

// device-side status flags (one int each), raised by kernels, read back by the host API
enum Flag { FLAG_WEIGHTS = 0, FLAG_NOT_SPD = 1, FLAG_ZERO_NORM = 2, FLAG_PERM_RANGE = 3, FLAG_COUNT = 8 };

__host__ __device__ inline int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }
__host__ __device__ inline int num_kchunks(int64_t n) { return (int)((n + KC - 1) / KC); }

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// Counter arrive for "last consumer refills the stage": acq_rel at CTA scope orders this warp's shared-memory
// reads of the stage before the increment and the last arriver's bulk copy after it — what the separate
// __threadfence_block() (a sequentially consistent MEMBAR) + relaxed atomic paid more for.
__device__ __forceinline__ int smem_counter_arrive(int* cnt) {
  int old;
  asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(smem_u32(cnt)) : "memory");
  return old;
}

// 1-D bulk asynchronous copy global -> shared through the TMA engine (SASS: UBLKCP), completion
// counted in bytes on an mbarrier.  dst/src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// The same copy with an L2 cache-policy hint (createpolicy), e.g. evict_last for operands that are
// re-read many times while large outputs stream through L2.
__device__ __forceinline__ uint64_t l2_evict_last_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bulk_g2s_hint(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar,
                                              uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}

// FP64 tensor-core atom: D(8x8) += A(8x4, row) * B(4x8, col).  Lane l = 4*g + t holds
// a = A[g][t], b = B[t][g], c0/c1 = C[g][2t], C[g][2t+1].  SASS: DMMA.8x8x4.
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// streaming (evict-first) 8-byte store: the LOD / h2 panels are written once and never re-read
// by the kernel, so they should not push the L2-resident marker operand out.
__device__ __forceinline__ void st_stream(double* p, double v) {
  asm volatile("st.global.cs.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}

// max over non-negative doubles (bit pattern order == numeric order); NaN propagates as "large".
__device__ __forceinline__ void atomic_max_nonneg(double* addr, double v) {
  atomicMax(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)__double_as_longlong(v));
}

// ---------------------------------------------------------------------------------------------
// The scan kernels' LOD: a 512-entry table built in shared memory by the kernel itself, scaled by n/2.
// ---------------------------------------------------------------------------------------------
constexpr int LTAB = 512;  // entries of the in-kernel logarithm table

// tab[i] = {rcp, (n/2) log10(rcp)} for the i-th interval of m in [0.75, 1.5): 256 intervals over [0.75, 1), 256 over
// [1, 1.5); the two intervals touching 1 use rcp = 1 exactly.  Called by all threads of the block (nthreads >= 1).
__device__ __forceinline__ void build_lod_table(double2* tab, int tid, int nthreads, double half_n) {
  for (int i = tid; i < LTAB; i += nthreads) {
    double c;
    if (i == LTAB / 2 - 1 || i == LTAB / 2)
      c = 1.0;
    else if (i < LTAB / 2)
      c = 0.75 + ((double)i + 0.5) * (0.25 / (LTAB / 2));
    else
      c = 1.0 + ((double)(i - LTAB / 2) + 0.5) * (0.5 / (LTAB / 2));
    const double rcp = 1.0 / c;
    tab[i] = make_double2(rcp, (rcp == 1.0) ? 0.0 : half_n * log10(rcp));
  }
}

// LOD = -(n/2) log10(v) for the final epilogue, ~8 FP64 operations (the FP64 pipe is shared with DMMA).
// v = 2^e * m, m in [0.75, 1.5); the table gives rcp ~ 1/c and (n/2) log10(rcp) for m's interval
// (256 intervals over [0.75, 1), 256 over [1, 1.5)); r = m*rcp - 1, |r| < 2^-9; log1p(r) by a 5-term
// series.  The two intervals touching 1 use rcp = 1 exactly, so LODs keep full relative accuracy as
// v -> 1 (LOD -> 0): relative error <= r^5/6 ~ 1e-16 there, absolute error ~1e-19 * n elsewhere.
// `special` is raised for operands outside the positive normal range (fixed up by the caller).
__device__ __forceinline__ double fast_lod(double v, const double2* __restrict__ tab, double c_ln, double c_e,
                                           bool& special) {
  const int hi = __double2hiint(v), lo = __double2loint(v);
  const int ix = hi - 0x3fe80000;
  const int e = ix >> 20;
  const double m = __hiloint2double(hi - (e << 20), lo);
  const double2 t = tab[(ix >> 11) & (LTAB - 1)];
  const double r = fma(m, t.x, -1.0);
  // -(n/2) log10(e) * log1p(r) = r * (k1 + r (k2 + r (k3 + r (k4 + r k5)))), k_i = c_ln * (-1)^(i+1) / i: the
  // scale is folded into the coefficients and the last multiply into the final FMA (8 FP64 operations in all)
  double q = fma(r, c_ln * (1.0 / 5.0), c_ln * (-1.0 / 4.0));
  q = fma(q, r, c_ln * (1.0 / 3.0));
  q = fma(q, r, c_ln * (-1.0 / 2.0));
  q = fma(q, r, c_ln);
  special |= (unsigned)(hi - 0x00100000) >= 0x7fe00000u;
  // c_ln = -(n/2) log10(e), c_e = -(n/2) log10(2), t.y = -(n/2) * (-log10 rcp)
  return fma(q, r, fma((double)e, c_e, t.y));
}

// IEEE results for the operands fast_lod flags: v = 0 (r^2 = 1) -> LOD = +inf (a subnormal v,
// unreachable as 1 - r^2, is treated as 0); v < 0 -> NaN (Julia's log10 throws there); v = +inf ->
// -inf; NaN passes through.
__device__ __forceinline__ double fix_lod(double v, double res) {
  const int hi = __double2hiint(v);
  res = ((unsigned)hi < 0x00100000u) ? INFINITY : res;
  res = (hi < 0) ? __longlong_as_double(0x7ff8000000000000LL) : res;
  res = (hi >= 0x7ff00000) ? -v : res;
  return res;
}


// ---------------------------------------------------------------------------------------------
// Per-trait peaks (findmax of an LOD column over the markers) reduced in the scan epilogues.
// ---------------------------------------------------------------------------------------------
// The first maximum of one output column within one warp's block of markers.
struct __align__(16) PeakRec {
  double lod;  // the LOD itself, bit for bit (NaN payload included)
  int marker;  // 0-based marker index; >= p when the block holds only padding rows
  int gidx;    // alt-grid: index of that marker's h2 in the grid; otherwise 0
};

// Julia's findmax order as an integer: every NaN above +Inf (so the first NaN wins), -0.0 below +0.0, numeric order
// otherwise.  Padding rows (row >= p) get the smallest key and never win.
__device__ __forceinline__ long long peak_key(double v, int row, int p) {
  const long long b = __double_as_longlong(v);
  long long k = b >= 0 ? b : (b ^ 0x7fffffffffffffffLL);
  k = ((b & 0x7fffffffffffffffLL) > 0x7ff0000000000000LL) ? 0x7fffffffffffffffLL : k;
  return row < p ? k : (-0x7fffffffffffffffLL - 1);
}

// (lod, row, gidx) := the candidate (l2, r2, g2) when it ranks higher: a larger key, or the same key at a smaller row
__device__ __forceinline__ void peak_take(double& lod, int& row, int& gidx, double l2, int r2, int g2, int p) {
  const long long k1 = peak_key(lod, row, p), k2 = peak_key(l2, r2, p);
  const bool take = k2 > k1 || (k2 == k1 && r2 < row);
  lod = take ? l2 : lod;
  row = take ? r2 : row;
  gidx = take ? g2 : gidx;
}

// The same over the lanes lane ^ o, o = o0, 2 o0, ..., 16 (o0 = 4: the 8 marker rows g of a DMMA fragment column)
__device__ __forceinline__ void peak_over_lanes(double& lod, int& row, int& gidx, int p, int o0) {
  for (int o = o0; o < 32; o <<= 1) {
    const double l2 = __shfl_xor_sync(0xffffffffu, lod, o);
    const int r2 = __shfl_xor_sync(0xffffffffu, row, o);
    const int g2 = __shfl_xor_sync(0xffffffffu, gidx, o);
    peak_take(lod, row, gidx, l2, r2, g2, p);
  }
}

// 1 / a to full double precision without the division sequence: the hardware's ~20-bit reciprocal estimate and two
// Newton steps (4 FP64 operations; the result may differ from the correctly rounded quotient in the last bit).
__device__ __forceinline__ double fast_rcp(double a) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(a));
  double e = fma(-a, r, 1.0);
  r = fma(r, e, r);
  e = fma(-a, r, 1.0);
  return fma(r, e, r);
}

}  // namespace blmm
