// The output side of the scan kernels scan_kernel (blmm_scan.cu) and scan_stream_kernel (blmm_scan_stream.cu), and
// their launch.  Register arrays are passed by reference with compile-time extents and indexed only with loop indices
// that unrolling makes constant: a run-time index would move an array to local memory under the kernels' register caps.
#pragma once
#include "blmm_kernels.cuh"

namespace blmm {

constexpr int SCAN_SMEM_LIMIT = 227 * 1024;  // dynamic shared memory of one scan CTA

// Output column of packed trait position pos (-1 = padding): with a column map, its entry map[i] (map is P.col_map or
// a copy of part of it), else pos itself, with the positions past the m columns as padding.
__device__ __forceinline__ int64_t out_column(const ScanParams& P, const int* map, int64_t i, int64_t pos) {
  return P.col_map ? (int64_t)map[i] : (pos < P.m ? pos : -1);
}

// Where output column col is stored, from marker row row0 on; nullptr for what is not stored (everything when col < 0).
// Column 0 may be split off (ScanParams::L0): then column s >= 1 is column s-1 of L and colmax.
struct OutColumn {
  double* L;
  double* H2;
  double* colmax;
  uint8_t* H2idx;
};
__device__ __forceinline__ OutColumn out_column_ptrs(const ScanParams& P, int64_t col, int row0, bool with_colmax,
                                                     bool with_h2) {
  OutColumn o{nullptr, nullptr, nullptr, nullptr};
  if (col >= 0) {
    if (P.L0) {
      if (col == 0) {
        o.L = P.L0 + row0;
      } else {
        if (P.L) o.L = P.L + (col - 1) * P.ldL + row0;
        if (with_colmax) o.colmax = P.colmax + (col - 1);
      }
    } else {
      if (P.L) o.L = P.L + col * P.ldL + row0;
      if (with_colmax) o.colmax = P.colmax + col;
    }
    if (with_h2 && P.H2) o.H2 = P.H2 + col * P.ldL + row0;
    if (with_h2 && P.H2idx) o.H2idx = P.H2idx + col * (int64_t)P.p + row0;
  }
  return o;
}

// Byte o of the packed tmax! counters, four per word: output o = (a * NB + b) * 2 + cc of a warp's register block.
template <int NC>
__device__ __forceinline__ int counter_byte(const uint32_t (&cnt)[NC], int o) {
  return (int)((cnt[o >> 2] >> ((o & 3) * 8)) & 0xFFu);
}

// One k of the running minimum over the grid (tmax!, src/bulkscan_helpers.jl:330-350), integer pipe only: a strict `<`
// as `max .< to_compare`, on the bit patterns (equivalent for the non-negative v that occur; a negative v, r^2 > 1 by
// rounding, orders below every positive one, as it should).  The counter byte of each output counts the strict
// improvements after k = 0, or with ARGMAX holds the k of the minimum.
template <bool ARGMAX, int MA, int NB, int NC>
__device__ __forceinline__ void running_min_step(const double (&v)[MA][NB][2], double (&vmin)[MA][NB][2],
                                                 uint32_t (&cnt)[NC], int kk) {
  static_assert(NC * 4 >= MA * NB * 2, "one counter byte per output");
  const bool first = (kk == 0);
#pragma unroll
  for (int a = 0; a < MA; ++a)
#pragma unroll
    for (int b = 0; b < NB; ++b)
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const double x = v[a][b][cc];
        const bool better = __double_as_longlong(x) < __double_as_longlong(vmin[a][b][cc]);
        const bool upd = first || better;
        vmin[a][b][cc] = upd ? x : vmin[a][b][cc];
        const int o = (a * NB + b) * 2 + cc;
        const int sh = (o & 3) * 8;
        if (ARGMAX) {
          if (upd) cnt[o >> 2] = (cnt[o >> 2] & ~(0xFFu << sh)) | ((uint32_t)kk << sh);
        } else {
          if (better && !first) cnt[o >> 2] += (1u << sh);
        }
      }
}

// lod = -(n/2) log10(v) for the first NBO trait columns of v: one table logarithm each (fast_lod), and the IEEE results
// (fix_lod) when any lane of the warp holds an operand outside the positive normal range.
template <int MA, int NB, int NBO>
__device__ __forceinline__ void lod_finish(const double (&v)[MA][NB][2], double (&lod)[MA][NBO][2],
                                           const double2* logtab, double half_n) {
  static_assert(NBO <= NB, "trait columns of v");
  const double c_ln = -half_n * 0.43429448190325182765;
  const double c_e = -half_n * 0.30102999566398119521;
  bool special = false;
#pragma unroll
  for (int a = 0; a < MA; ++a)
#pragma unroll
    for (int b = 0; b < NBO; ++b)
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) lod[a][b][cc] = fast_lod(v[a][b][cc], logtab, c_ln, c_e, special);
  if (__any_sync(0xffffffffu, special)) {
#pragma unroll
    for (int a = 0; a < MA; ++a)
#pragma unroll
      for (int b = 0; b < NBO; ++b)
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) lod[a][b][cc] = fix_lod(v[a][b][cc], lod[a][b][cc]);
  }
}

// Per-trait peaks of a warp's register block (the LOD of marker row0 + 8a and output column column(b, cc) in
// lod[a][b][cc]): for every column, the first maximum over the register rows a and then over the lanes g, compared on
// integer keys (peak_take, peak_over_lanes).  With GIDX the record carries the grid index kbase + counter byte of the
// entry that wins.  Lane g = 0 stores it as record mb of the column.
template <bool GIDX, int MA, int NB, int NC, typename ColumnOf>
__device__ __forceinline__ void peak_store(const double (&lod)[MA][NB][2], const uint32_t (&cnt)[NC], int kbase,
                                           int row0, int g, const ScanParams& P, int block_rows, int mb,
                                           ColumnOf column) {
#pragma unroll
  for (int b = 0; b < NB; ++b)
#pragma unroll
    for (int cc = 0; cc < 2; ++cc) {
      double pl = lod[0][b][cc];
      int row = row0, gi = 0;
#pragma unroll
      for (int a = 0; a < MA; ++a) {
        const int ga = GIDX ? kbase + counter_byte(cnt, (a * NB + b) * 2 + cc) : 0;
        if (a == 0)
          gi = ga;
        else
          peak_take(pl, row, gi, lod[a][b][cc], row0 + a * 8, ga, P.p);
      }
      peak_over_lanes(pl, row, gi, P.p, 4);
      const int64_t col = column(b, cc);
      if (g == 0 && col >= 0) P.peaks[col * peak_blocks(P.p_pad, block_rows) + mb] = PeakRec{pl, row, gi};
    }
}

// Per-trait peaks replace every per-marker output: no scan kernel writes both.
inline bool peaks_with_panels(const ScanParams& P) {
  return P.peaks && (P.colmax || P.L || P.L0 || P.H2 || P.H2idx);
}

// A persistent scan kernel: one CTA per SM, with more dynamic shared memory than the default limit allows.
inline void launch_scan_kernel(void (*kernel)(ScanParams), int threads, size_t smem, const ScanParams& P, int sm_count,
                               cudaStream_t stream) {
  cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SCAN_SMEM_LIMIT);
  kernel<<<sm_count, threads, smem, stream>>>(P);
}

}  // namespace blmm
