// The fused marker x trait scan kernel (see ScanParams in blmm_kernels.cuh for the arithmetic).
//
// Structure (sm_100a): persistent CTAs, one per SM, 16 warps (4 per SM sub-partition, <= 128
// registers per thread).  A CTA owns a contiguous range of (trait tile, marker tile) units.  The trait
// tile (128 traits x whole K) stays resident in shared memory; for every unit the k-list's marker
// tiles (64 markers x whole K, plus that k's per-trait scalars e/et) stream through a 2-3 stage ring
// filled with 1-D bulk asynchronous copies (cp.async.bulk -> UBLKCP, the TMA engine; mbarrier
// transaction counts); the last warp to release a stage refills it.
// Each warp owns a 32 marker x 16 trait block: FP64 tensor-core mma.sync m8n8k4 (DMMA.8x8x4) over the
// K-chunked operands, then the per-k epilogue in registers (v = e - d^2*et, running min, tmax!
// counter), and ONE logarithm per output after the last k.  LOD / h2 panels are written once with
// streaming stores; nothing per-grid-point touches HBM.
//
// Ping-pong ordering.  On B200 DMMA and scalar FP64 share one pipe that a single warp per
// sub-partition can saturate, so what costs time is every warp of a sub-partition leaving the DMMA
// loop together (they consume the same stage and are served round-robin, so they run in lock step)
// and the pipe idling through the epilogues.  The warps are therefore split into two groups
// (marker rows 0-31 / 32-63 of the tile) that take turns in the DMMA loop, per sub-partition, by passing
// a token through a pair of mbarriers: while one group multiplies, the other runs its epilogue
// (running-min update, logarithm, stores) and the scalar FP64 work fills DMMA issue gaps instead of
// serialising with it.  (bar.sync / bar.arrive pairs with a thread count do NOT order the groups on this
// part: measured, both groups pass at once; tools/scratch notes in DESIGN.md.)
#include <math.h>
#include <stdlib.h>

#include "blmm_kernels.cuh"

namespace blmm {

namespace {

constexpr int TT = SCAN_TT;  // traits per CTA tile
constexpr int MT = SCAN_MT;  // markers per CTA tile
constexpr int BT = 2;        // 8-trait atoms per warp: 16 warps of 32 markers x 16 traits
constexpr int WT_WARPS = TT / (8 * BT);
constexpr int NWARPS = 2 * WT_WARPS;
constexpr int NTHREADS = 32 * NWARPS;
constexpr int SMEM_LIMIT = 227 * 1024;
constexpr int GRID_MAX = 256;

static_assert(NWARPS == 16 && NTHREADS == 512, "ping-pong barrier counts assume 16 warps");

// Development aid (tools/scan_timing.py builds a second library with -DBLMM_SCAN_TIMING): per-warp clock64
// time in each phase of the kernel.  Not compiled into the product library.
#ifdef BLMM_SCAN_TIMING
__device__ long long g_scan_timing[256 * NWARPS * 8];
__device__ long long g_scan_trace[NWARPS * 64 * 4];  // CTA 0: per warp, first 64 iterations: t(full), t(turn), t(dmma end), t(epi end)
#define TCK(i)                      \
  {                                 \
    const long long t_now = clock64(); \
    tacc[i] += t_now - tlast;       \
    tlast = t_now;                  \
  }
#else
#define TCK(i)
#endif

struct SmemPlan {
  int nstage;
  size_t top_doubles;    // nq*TT*KC
  size_t stage_doubles;  // nq*MT*KC + 2*TT
  size_t bytes;
};

constexpr size_t FIXED_SMEM = (size_t)LTAB * 16 + GRID_MAX * 8 + 2 * TT * 4 + 128;

__host__ __device__ inline SmemPlan plan_smem(int nq) {
  SmemPlan s;
  s.top_doubles = (size_t)nq * TT * KC;
  s.stage_doubles = (size_t)nq * MT * KC + 2 * TT;
  s.nstage = 3;
  s.bytes = (s.top_doubles + 3 * s.stage_doubles) * 8 + FIXED_SMEM;
  if (s.bytes > SMEM_LIMIT) {
    s.nstage = 2;
    s.bytes = (s.top_doubles + 2 * s.stage_doubles) * 8 + FIXED_SMEM;
  }
  return s;
}

// first k-step of a tile: C = 0 (no separate zeroing of the accumulators)
__device__ __forceinline__ void dmma884_zero(double& c0, double& c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%4,%4};"
      : "=d"(c0), "=d"(c1)
      : "d"(a), "d"(b), "d"(0.0));
}

// HAS_E = false: one-element k-lists with e = 1 (null-grid bins, permutations) — no running minimum,
// no counter, no h2 panel.  COLMAX: also reduce the per-column maximum (permutation thresholds).
// PEAK: store nothing per marker; every warp reduces its 32 markers of each column to one PeakRec instead.
template <int NQ, bool ARGMAX, bool HAS_E, bool COLMAX, bool PEAK>
__global__ void __launch_bounds__(NTHREADS, 1) scan_kernel(const ScanParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const SmemPlan plan = plan_smem(NQ);
  const int NS = plan.nstage;
  double* top = reinterpret_cast<double*>(smem_raw);
  double* stages = top + plan.top_doubles;
  double2* logtab = reinterpret_cast<double2*>(stages + NS * plan.stage_doubles);
  double* grid_s = reinterpret_cast<double*>(logtab + LTAB);
  int* colmap_s = reinterpret_cast<int*>(grid_s + GRID_MAX);  // [2][TT], by trait-tile parity
  uint64_t* bars = reinterpret_cast<uint64_t*>(colmap_s + 2 * TT);
  uint64_t* full = bars;  // [NS]
  uint64_t* top_full = bars + 3;
  uint64_t* top_empty = bars + 4;
  int* rel_cnt = reinterpret_cast<int*>(bars + 5);  // [NS] consumers done with a stage
  uint64_t* turn = bars + 8;                         // [4 sub-partitions][2 groups] ping-pong tokens

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  // The marker operand (all k) is re-read by every trait tile: ask L2 to keep it while the LOD /
  // h2 panels stream through (they are written with evict-first stores).
  if (tid == 0) {
    for (int s = 0; s < NS; ++s) {
      mbar_init(&full[s], 1);
      rel_cnt[s] = 0;
    }
    mbar_init(top_full, 1);
    mbar_init(top_empty, NWARPS);
    for (int i = 0; i < 8; ++i) mbar_init(&turn[i], 2);  // the two warps of the other group on the sub-partition
    mbar_fence_init();
  }
  build_lod_table(logtab, tid, NTHREADS, P.half_n);
  if (P.grid && tid < P.ngrid) grid_s[tid] = P.grid[tid];
  __syncthreads();

  const int n_tiles = P.n_tiles_dev ? *P.n_tiles_dev : P.n_tiles_t;
  const int n_mt = P.p_pad / MT;
  const int64_t units = (int64_t)n_tiles * n_mt;  // < 2^31 (checked by the launcher)
  const int u0 = (int)(units * blockIdx.x / gridDim.x);
  const int u1 = (int)(units * (blockIdx.x + 1) / gridDim.x);
  const int nk = HAS_E ? P.nk : 1;
  const int total_it = (u1 - u0) * nk;
  constexpr uint32_t marker_chunk_bytes = MT * KC * 8;
  constexpr uint32_t trait_chunk_bytes = TT * KC * 8;
  constexpr uint32_t stage_bytes = (uint32_t)NQ * marker_chunk_bytes + (HAS_E ? 2 * TT * 8 : 0);

  // Fill stage s with the operands of iteration (tt, mt, kk): the k-th marker tile and that k's
  // per-trait scalars.  Called by one thread; completion is counted on full[s].
  auto issue_stage = [&](int s, int tt, int mt, int kk) {
    const int k0 = P.tile_k0 ? P.tile_k0[tt] : 0;
    double* st = stages + (size_t)s * plan.stage_doubles;
    mbar_arrive_expect_tx(&full[s], stage_bytes);
    const double* src = P.Mop + (((size_t)(k0 + kk) * NQ) * P.p_pad + (size_t)mt * MT) * KC;
    const uint64_t keep_policy = l2_evict_last_policy();
#pragma unroll
    for (int q = 0; q < NQ; ++q)
      bulk_g2s_hint(st + (size_t)q * MT * KC, src + (size_t)q * P.p_pad * KC, marker_chunk_bytes, &full[s], keep_policy);
    double* sc = st + (size_t)NQ * MT * KC;
    if (HAS_E) {
      bulk_g2s(sc + TT, P.et + (size_t)kk * P.tcol_pad + (size_t)tt * TT, TT * 8, &full[s]);
      bulk_g2s(sc, P.e + (size_t)kk * P.tcol_pad + (size_t)tt * TT, TT * 8, &full[s]);
    }
  };
  // (tt, mt, kk) advanced by `steps` iterations
  auto advance = [&](int& tt, int& mt, int& kk, int steps) {
    kk += steps;
    while (kk >= nk) {
      kk -= nk;
      if (++mt == n_mt) {
        mt = 0;
        ++tt;
      }
    }
  };

  int tt = u0 / n_mt, mt = u0 % n_mt;
  if (tid == 0) {
    int ptt = tt, pmt = mt, pkk = 0;
    for (int i = 0; i < NS && i < total_it; ++i) {
      issue_stage(i, ptt, pmt, pkk);
      advance(ptt, pmt, pkk, 1);
    }
  }

  const int g = lane >> 2, t = lane & 3;
  const int wm = warp / WT_WARPS;  // marker sub-block (0..1) = ping-pong group
  const int wt = warp % WT_WARPS;  // trait sub-block
  const int aoff = (wm * 32 + g) * KC + t;
  const int boff = (wt * (8 * BT) + g) * KC + t;
  // Ping-pong: the two groups alternate in the DMMA loop, independently on every SM sub-partition
  // (warps w, w+4 of a group share sub-partition w & 3).  turn[2*(w&3) + grp] completes phase i when
  // both warps of the other group have granted group grp its i-th turn.
  uint64_t* my_turn = &turn[2 * (warp & 3) + wm];
  uint64_t* their_turn = &turn[2 * (warp & 3) + (wm ^ 1)];
  if (wm == 1 && lane == 0) mbar_arrive(their_turn);  // group 0 goes first

  int it = 0, s = 0;
  uint32_t sphase = 0;  // parity of the ring round
  int ntop = 0, cur_tt = -1;
#ifdef BLMM_SCAN_TIMING
  long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  long long tlast = clock64();
#endif
  for (int u = u0; u < u1; ++u) {
    if (tt != cur_tt) {
      if (tid == 0) {
        if (ntop > 0) mbar_wait(top_empty, (ntop - 1) & 1);
        mbar_arrive_expect_tx(top_full, (uint32_t)NQ * trait_chunk_bytes + (P.col_map ? TT * 4 : 0));
#pragma unroll
        for (int q = 0; q < NQ; ++q)
          bulk_g2s(top + (size_t)q * TT * KC, P.Top + ((size_t)q * P.tcol_pad + (size_t)tt * TT) * KC,
                   trait_chunk_bytes, top_full);
        // The packed-column -> output-column map of the tile is read by the final epilogue, which can
        // still be running for the previous tile in other warps: two copies, by tile parity.
        if (P.col_map) bulk_g2s(colmap_s + (ntop & 1) * TT, P.col_map + (size_t)tt * TT, TT * 4, top_full);
      }
      mbar_wait(top_full, ntop & 1);
      ++ntop;
      cur_tt = tt;
    }
    TCK(5)
    const bool last_of_tt = (u + 1 == u1) || (mt + 1 == n_mt);

    constexpr int VM = HAS_E ? 1 : 0;  // index multiplier: the one-k variants keep no running minimum
    double acc[4][BT][2];
    double vmin[HAS_E ? 4 : 1][BT][2];
    uint32_t cnt[HAS_E ? 2 * BT : 1];
    if (HAS_E) {
#pragma unroll
      for (int i = 0; i < 2 * BT; ++i) cnt[i] = 0u;
    }

    for (int kk = 0; kk < nk; ++kk, ++it) {
      mbar_wait(&full[s], sphase);
      TCK(0)
#ifdef BLMM_SCAN_TIMING
      if (blockIdx.x == 0 && lane == 0 && it >= 64 && it < 128) g_scan_trace[(warp * 64 + it - 64) * 4 + 0] = tlast;
#endif
      const double* ms = stages + (size_t)s * plan.stage_doubles;
      // first fragments of the K loop, fetched before the turn starts
      const double* ap = ms + aoff;
      const double* bp = top + boff;
      double af[2][4], bf[2][BT];
#pragma unroll
      for (int a = 0; a < 4; ++a) af[0][a] = ap[a * 8 * KC];
#pragma unroll
      for (int b = 0; b < BT; ++b) bf[0][b] = bp[b * 8 * KC];
      mbar_wait(my_turn, (uint32_t)it & 1u);
      TCK(1)
#ifdef BLMM_SCAN_TIMING
      if (blockIdx.x == 0 && lane == 0 && it >= 64 && it < 128) g_scan_trace[(warp * 64 + it - 64) * 4 + 1] = tlast;
#endif
      {
        // K loop, fully unrolled, fragments double-buffered in registers
#pragma unroll
        for (int st = 0; st < NQ * (KC / 4); ++st) {
          const int cur = st & 1;
          if (st + 1 < NQ * (KC / 4)) {
            const int q1 = (st + 1) / (KC / 4), s1 = (st + 1) % (KC / 4);
#pragma unroll
            for (int a = 0; a < 4; ++a) af[cur ^ 1][a] = ap[q1 * (MT * KC) + a * 8 * KC + s1 * 4];
#pragma unroll
            for (int b = 0; b < BT; ++b) bf[cur ^ 1][b] = bp[q1 * (TT * KC) + b * 8 * KC + s1 * 4];
          }
#pragma unroll
          for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < BT; ++b) {
              if (st == 0)
                dmma884_zero(acc[a][b][0], acc[a][b][1], af[cur][a], bf[cur][b]);
              else
                dmma884(acc[a][b][0], acc[a][b][1], af[cur][a], bf[cur][b]);
            }
        }
      }
      TCK(2)
#ifdef BLMM_SCAN_TIMING
      if (blockIdx.x == 0 && lane == 0 && it >= 64 && it < 128) g_scan_trace[(warp * 64 + it - 64) * 4 + 2] = tlast;
#endif
      // Still inside this group's turn: every scalar FP64 operation of the epilogue.  Issued while the
      // other group multiplies they would sit behind its DMMA stream until it ends (measured: the pipe
      // serves two back-to-back DMMA warps and starves a third warp's DFMA), so they go here, in the
      // order the last k-step finishes the accumulators.  v overwrites the accumulator.
      if (HAS_E) {
        double ek[BT][2], etk[BT][2];  // per-k trait scalars for this lane's 2*BT trait columns
        const double* sc = ms + (size_t)NQ * MT * KC + wt * (8 * BT) + 2 * t;
#pragma unroll
        for (int b = 0; b < BT; ++b) {
          const double2 v = *reinterpret_cast<const double2*>(sc + b * 8);
          ek[b][0] = v.x; ek[b][1] = v.y;
          const double2 w = *reinterpret_cast<const double2*>(sc + TT + b * 8);
          etk[b][0] = w.x; etk[b][1] = w.y;
        }
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < BT; ++b)
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {
              const double d = acc[a][b][cc];
              acc[a][b][cc] = fma(-(d * d), etk[b][cc], ek[b][cc]);
            }
      } else {
        // one-k scans: et = 1/rss is folded into the packed trait columns (ScanParams::et_folded), e = 1
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < BT; ++b)
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {
              const double d = acc[a][b][cc];
              acc[a][b][cc] = fma(-d, d, 1.0);
            }
      }
      // tmax! bookkeeping of this k: integer pipe only (strict `<` as `max .< to_compare`, on the bit
      // patterns: equivalent for the non-negative v that occur; a negative v (r^2 > 1 by rounding)
      // orders below every positive one, as it should)
      auto update_min = [&]() {
        if (HAS_E) {
          const bool first = (kk == 0);
#pragma unroll
          for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < BT; ++b)
#pragma unroll
              for (int cc = 0; cc < 2; ++cc) {
                const double v = acc[a][b][cc];
                const bool better = __double_as_longlong(v) < __double_as_longlong(vmin[a * VM][b][cc]);
                const bool upd = first || better;
                vmin[a * VM][b][cc] = upd ? v : vmin[a * VM][b][cc];
                const int o = (a * BT + b) * 2 + cc;
                const int sh = (o & 3) * 8;
                if (ARGMAX) {
                  if (upd) cnt[(o >> 2) * VM] = (cnt[(o >> 2) * VM] & ~(0xFFu << sh)) | ((uint32_t)kk << sh);
                } else {
                  if (better && !first) cnt[(o >> 2) * VM] += (1u << sh);
                }
              }
        }
      };
      const bool last_k = (kk == nk - 1);
      if (last_k) {
        // last k of the unit: one logarithm per output; the LOD replaces the accumulator
        update_min();
        const double c_ln = -P.half_n * 0.43429448190325182765;
        const double c_e = -P.half_n * 0.30102999566398119521;
        bool special = false;
        double lod[4][BT][2];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < BT; ++b)
#pragma unroll
            for (int cc = 0; cc < 2; ++cc)
              lod[a][b][cc] = fast_lod(HAS_E ? vmin[a * VM][b][cc] : acc[a][b][cc], logtab, c_ln, c_e, special);
        if (__any_sync(0xffffffffu, special)) {
#pragma unroll
          for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < BT; ++b)
#pragma unroll
              for (int cc = 0; cc < 2; ++cc)
                lod[a][b][cc] = fix_lod(HAS_E ? vmin[a * VM][b][cc] : acc[a][b][cc], lod[a][b][cc]);
        }
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < BT; ++b)
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) acc[a][b][cc] = lod[a][b][cc];
      }
      // the FP64 work above is issued before the turn is handed over
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < BT; ++b) asm volatile("" ::"d"(acc[a][b][0]), "d"(acc[a][b][1]));
      __syncwarp();
      if (lane == 0) mbar_arrive(their_turn);
      // Release the stage.  The last of the NWARPS consumers refills it at once with the operands
      // of iteration it + NS, so the copy is in flight as early as the ring allows.
      if (lane == 0) {
        if (last_of_tt && last_k) mbar_arrive(top_empty);
        if (smem_counter_arrive(&rel_cnt[s]) == NWARPS - 1) {
          rel_cnt[s] = 0;
          if (it + NS < total_it) {
            int ntt = tt, nmt = mt, nkk = kk;
            advance(ntt, nmt, nkk, NS);
            issue_stage(s, ntt, nmt, nkk);
          }
        }
      }
      if (++s == NS) {
        s = 0;
        sphase ^= 1u;
      }
      if (!last_k) update_min();
      TCK(3)
#ifdef BLMM_SCAN_TIMING
      if (blockIdx.x == 0 && lane == 0 && it >= 64 && it < 128) g_scan_trace[(warp * 64 + it - 64) * 4 + 3] = tlast;
#endif
    }

    // stores of the unit (LOD in the accumulator registers), outside the turn
    const int kbase = (HAS_E && ARGMAX && P.tile_k0) ? P.tile_k0[tt] : 0;
    const int row0 = mt * MT + wm * 32 + g;
    if (PEAK) {
      // per-trait peaks: the first maximum of each column over the warp's 32 markers, over a in registers and then
      // over g across the lanes, compared on integer keys (this runs outside the turn, like the stores it replaces)
      const int* cmap = colmap_s + ((ntop - 1) & 1) * TT;
#pragma unroll
      for (int b = 0; b < BT; ++b)
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          double lod = acc[0][b][cc];
          int row = row0, gi = 0;
#pragma unroll
          for (int a = 0; a < 4; ++a) {
            const int o = (a * BT + b) * 2 + cc;
            const int ga = HAS_E ? kbase + (int)((cnt[(o >> 2) * VM] >> ((o & 3) * 8)) & 0xFFu) : 0;
            if (a == 0)
              gi = ga;
            else
              peak_take(lod, row, gi, acc[a][b][cc], row0 + a * 8, ga, P.p);
          }
          peak_over_lanes(lod, row, gi, P.p, 4);
          const int posl = wt * (8 * BT) + b * 8 + 2 * t + cc;
          const int64_t pos = (int64_t)tt * TT + posl;
          const int64_t col = P.col_map ? (int64_t)cmap[posl] : (pos < P.m ? pos : -1);
          if (g == 0 && col >= 0) P.peaks[col * (P.p_pad / 32) + mt * 2 + wm] = PeakRec{lod, row, gi};
        }
      if (++mt == n_mt) {
        mt = 0;
        ++tt;
      }
      TCK(4)
      continue;
    }
    const bool full_rows = (mt + 1) * MT <= P.p;  // every marker row of the tile exists
    const int* cmap = colmap_s + ((ntop - 1) & 1) * TT;
#pragma unroll
    for (int b = 0; b < BT; ++b)
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const int posl = wt * (8 * BT) + b * 8 + 2 * t + cc;
        const int64_t pos = (int64_t)tt * TT + posl;
        const int64_t col = P.col_map ? (int64_t)cmap[posl] : (pos < P.m ? pos : -1);
        // output column pointers (column 0 may be split off, see ScanParams::L0)
        double* Lc = nullptr;
        double* Hc = nullptr;
        double* Mc = nullptr;
        uint8_t* Ic = nullptr;
        if (col >= 0) {
          if (P.L0) {
            if (col == 0) {
              Lc = P.L0 + row0;
            } else {
              if (P.L) Lc = P.L + (col - 1) * P.ldL + row0;
              if (COLMAX) Mc = P.colmax + (col - 1);
            }
          } else {
            if (P.L) Lc = P.L + col * P.ldL + row0;
            if (COLMAX) Mc = P.colmax + col;
          }
          if (HAS_E && P.H2) Hc = P.H2 + col * P.ldL + row0;
          if (HAS_E && P.H2idx) Ic = P.H2idx + col * (int64_t)P.p + row0;
        }
        if (full_rows) {
          if (Lc) {
#pragma unroll
            for (int a = 0; a < 4; ++a) st_stream(Lc + a * 8, acc[a][b][cc]);
          }
          if (HAS_E && Hc) {
#pragma unroll
            for (int a = 0; a < 4; ++a) {
              const int o = (a * BT + b) * 2 + cc;
              const int cv = (int)((cnt[(o >> 2) * VM] >> ((o & 3) * 8)) & 0xFFu);
              st_stream(Hc + a * 8, grid_s[kbase + cv]);
            }
          }
          if (HAS_E && Ic) {
#pragma unroll
            for (int a = 0; a < 4; ++a) {
              const int o = (a * BT + b) * 2 + cc;
              Ic[a * 8] = (uint8_t)(kbase + (int)((cnt[(o >> 2) * VM] >> ((o & 3) * 8)) & 0xFFu));
            }
          }
        } else {
#pragma unroll
          for (int a = 0; a < 4; ++a) {
            if (row0 + a * 8 < P.p) {
              if (Lc) st_stream(Lc + a * 8, acc[a][b][cc]);
              if (HAS_E && (Hc || Ic)) {
                const int o = (a * BT + b) * 2 + cc;
                const int cv = (int)((cnt[(o >> 2) * VM] >> ((o & 3) * 8)) & 0xFFu);
                if (Hc) st_stream(Hc + a * 8, grid_s[kbase + cv]);
                if (Ic) Ic[a * 8] = (uint8_t)(kbase + cv);
              }
            } else {
              acc[a][b][cc] = 0.0;  // padded marker rows stay out of the column maximum
            }
          }
        }
        if (COLMAX) {
          // maximum on the bit patterns (LODs are >= 0, so integer order = numeric order; a NaN is the largest
          // and propagates like Julia's maximum): integer pipe only — this runs outside the group's turn, where
          // FP64 instructions would sit behind the other group's DMMAs
          long long cm = max(max(__double_as_longlong(acc[0][b][cc]), __double_as_longlong(acc[1][b][cc])),
                             max(__double_as_longlong(acc[2][b][cc]), __double_as_longlong(acc[3][b][cc])));
          cm = max(cm, 0LL);  // -0.0 and anything negative count as 0
          cm = max(cm, __shfl_xor_sync(0xffffffffu, cm, 4));
          cm = max(cm, __shfl_xor_sync(0xffffffffu, cm, 8));
          cm = max(cm, __shfl_xor_sync(0xffffffffu, cm, 16));
          if (g == 0 && Mc) atomicMax(reinterpret_cast<unsigned long long*>(Mc), (unsigned long long)cm);
        }
      }
    if (++mt == n_mt) {
      mt = 0;
      ++tt;
    }
    TCK(4)
  }
#ifdef BLMM_SCAN_TIMING
  if (lane == 0 && blockIdx.x < 256)
    for (int i = 0; i < 8; ++i) g_scan_timing[((size_t)blockIdx.x * NWARPS + warp) * 8 + i] = tacc[i];
#endif
}

template <int NQ, bool ARGMAX, bool HAS_E, bool COLMAX, bool PEAK = false>
void launch_one(const ScanParams& P, int sm_count, cudaStream_t stream) {
  const SmemPlan plan = plan_smem(NQ);
  cudaFuncSetAttribute(scan_kernel<NQ, ARGMAX, HAS_E, COLMAX, PEAK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       SMEM_LIMIT);
  scan_kernel<NQ, ARGMAX, HAS_E, COLMAX, PEAK><<<sm_count, NTHREADS, plan.bytes, stream>>>(P);
}

template <int NQ>
void launch_nq(const ScanParams& P, int sm_count, cudaStream_t stream) {
  if (P.peaks) {
    if (!P.e)
      launch_one<NQ, false, false, false, true>(P, sm_count, stream);
    else if (P.argmax_mode)
      launch_one<NQ, true, true, false, true>(P, sm_count, stream);
    else
      launch_one<NQ, false, true, false, true>(P, sm_count, stream);
  } else if (P.e) {
    if (P.argmax_mode)
      launch_one<NQ, true, true, false>(P, sm_count, stream);
    else
      launch_one<NQ, false, true, false>(P, sm_count, stream);
  } else {
    // one-element k-lists (null-grid bins, permutations): the h2 panel is not produced
    if (P.colmax)
      launch_one<NQ, false, false, true>(P, sm_count, stream);
    else
      launch_one<NQ, false, false, false>(P, sm_count, stream);
  }
}

}  // namespace

int scan_max_nq(int nk) {
  (void)nk;
  return 5;
}

#ifdef BLMM_SCAN_TIMING
extern "C" __attribute__((visibility("default"))) int blmm_debug_scan_timing(long long* out, int nblocks) {
  return (int)cudaMemcpyFromSymbol(out, g_scan_timing, sizeof(long long) * (size_t)nblocks * NWARPS * 8);
}
extern "C" __attribute__((visibility("default"))) int blmm_debug_scan_trace(long long* out) {
  return (int)cudaMemcpyFromSymbol(out, g_scan_trace, sizeof(g_scan_trace));
}
#endif

int launch_scan(const ScanParams& P, int sm_count, cudaStream_t stream) {
  // combinations the kernel variants do not cover
  if ((!P.e && (P.nk != 1 || !P.et_folded)) || (P.e && P.colmax)) return 0;
  // peaks replace every per-marker output
  if (P.peaks && (P.colmax || P.L || P.L0 || P.H2 || P.H2idx)) return 0;
  // the kernel indexes its (unit, k) iterations with 32-bit integers
  if ((int64_t)P.n_tiles_t * (P.p_pad / MT) * (int64_t)(P.nk > 0 ? P.nk : 1) >= 2147483647LL) return 0;
  switch (P.nq) {
    case 1: launch_nq<1>(P, sm_count, stream); break;
    case 2: launch_nq<2>(P, sm_count, stream); break;
    case 3: launch_nq<3>(P, sm_count, stream); break;
    case 4: launch_nq<4>(P, sm_count, stream); break;
    case 5: launch_nq<5>(P, sm_count, stream); break;
    default: return 0;
  }
  return 1;
}

}  // namespace blmm
