// K-streamed marker x trait scan kernels: any number of subjects n (the shared-memory-resident
// kernel of blmm_scan.cu needs n <= 100), and the per-trait-weight scan of bulkscan_null.
//
// Structure (sm_100a): persistent CTAs, one per SM, 16 warps (4 per SM sub-partition).  A CTA
// walks its units (64-trait-group tile x marker tile) round-robin (unit = blockIdx + r*gridDim), in
// an order that sweeps the marker tiles of a band of 8 trait tiles, so the 148 CTAs running at
// any moment share ~8 trait tiles and ~19 marker tiles in L2 whatever n is.  Both operands stream
// through K in chunks of KC = 20: one ring stage = one marker chunk + one trait chunk, filled by
// two 1-D bulk asynchronous copies (TMA engine, mbarrier byte counts) issued by the last warp
// that released the stage.  Accumulators stay in registers across the K loop; FP64 tensor-core
// mma.sync m8n8k4 (DMMA.8x8x4) does the contraction.
//
// EXACT mode = univar_liteqtl for every trait (src/bulkscan_helpers.jl:127-150, driver
// bulkscan_null src/bulkscan.jl:212-314).  Trait j has its own weights w_j = w(h2_j), so the
// marker operand cannot carry them; instead trait j contributes c+2 columns against the
// un-weighted rotated markers g_i (SURVEY appendix A5):
//     num = g'z_j,  t_a = g'q_ja (a = 1..c),  s = (g o g)'w_j,   r^2 = num^2 / ((s - sum t_a^2) dy_j)
// with W_j = diag(w_j), C0'W_jC0 = LL', Q_j = W_j C0 L^-T, z_j = W_j y_j - Q_j (Q_j'y_j), dy_j = y_j'z_j.
// g o g is squared in registers from the marker fragment.  A warp owns 8 traits x (c+2) column
// kinds x 8*MA markers, so all accumulators of one (marker, trait) pair sit in one thread.
//
// GRID mode = the arithmetic of blmm_scan.cu (see ScanParams) with the K loop streamed.
#include <float.h>
#include <math.h>

#include "blmm_kernels.cuh"

namespace blmm {

namespace {

constexpr int SMEM_LIMIT = 227 * 1024;
constexpr int GRID_MAX = 256;
constexpr int ST_TG = 8;                  // warps along the trait dimension
constexpr int ST_WARPS = 2 * ST_TG;       // x 2 along the marker dimension
constexpr int BAND_DEFAULT = 8;           // trait tiles per rasterisation band (StreamParams::band overrides)
constexpr size_t ST_FIXED_SMEM = (size_t)LTAB * 16 + GRID_MAX * 8 + 128;

enum { MODE_EXACT = 0, MODE_GRID = 1 };

struct StreamPlan {
  int nstage;
  size_t stage_doubles;
  size_t bytes;
};

__host__ __device__ inline StreamPlan stream_plan(int NB, int MA) {
  StreamPlan s;
  s.stage_doubles = (size_t)(2 * 8 * MA + ST_TG * 8 * NB) * KC;
  int ns = (int)((SMEM_LIMIT - ST_FIXED_SMEM) / (s.stage_doubles * 8));
  s.nstage = ns > 4 ? 4 : ns;
  s.bytes = (size_t)s.nstage * s.stage_doubles * 8 + ST_FIXED_SMEM;
  return s;
}

// PEAK: store nothing per marker; every warp reduces its 8 * MA markers of each column to one PeakRec instead.
template <int NB, int MA, int MODE, bool ARGMAX, bool PEAK>
__global__ void __launch_bounds__(32 * ST_WARPS, 1) scan_stream_kernel(const StreamParams P) {
  constexpr int MT = 2 * 8 * MA;        // markers per CTA tile
  constexpr int TCOLS = ST_TG * 8 * NB;  // operand columns per CTA tile
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const StreamPlan plan = stream_plan(NB, MA);
  // ring depth, capped by the items of one unit so that the prefetch never looks more than one unit ahead
  const int ipu_cap = ((MODE == MODE_GRID) ? P.nk : 1) * P.nq;
  const int NS = plan.nstage < ipu_cap ? plan.nstage : ipu_cap;
  double* stages = reinterpret_cast<double*>(smem_raw);
  double2* logtab = reinterpret_cast<double2*>(stages + NS * plan.stage_doubles);
  double* grid_s = reinterpret_cast<double*>(logtab + LTAB);
  uint64_t* full = reinterpret_cast<uint64_t*>(grid_s + GRID_MAX);  // [4]
  int* rel_cnt = reinterpret_cast<int*>(full + 4);                  // [4]

  // Units are handed out dynamically (one atomic per unit): CTAs that become free take CONSECUTIVE units, so the
  // CTAs sharing a marker tile stream it within microseconds of each other and it is read from DRAM once.  With a
  // static round-robin the persistent CTAs drift apart over thousands of rounds and every CTA fetched its own copy
  // (ncu at n = 1000: 212 GB of DRAM reads, = units x marker tile, whatever the band size).  uq[r & 3] is the unit
  // of this CTA's r-th turn (fetched two turns ahead: the stage prefetch crosses into the next unit and warps may be a
  // unit apart).
  volatile long long* uq = reinterpret_cast<volatile long long*>(full + 8);  // inside the 128-byte barrier block
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int s = 0; s < NS; ++s) {
      mbar_init(&full[s], 1);
      rel_cnt[s] = 0;
    }
    mbar_fence_init();
    for (int o = 0; o < 3; ++o)
      uq[o] = P.unit_counter ? (long long)atomicAdd(P.unit_counter, 1ULL) : (long long)blockIdx.x + (long long)o * gridDim.x;
  }
  build_lod_table(logtab, tid, 32 * ST_WARPS, P.half_n);  // scaled by n/2: the epilogue yields the LOD directly
  if (MODE == MODE_GRID && P.grid && tid < P.ngrid) grid_s[tid] = P.grid[tid];
  __syncthreads();

  const int n_tt = P.n_tiles_dev ? *P.n_tiles_dev : P.n_tt;
  const int n_mt = P.p_pad / MT;
  const int nq = P.nq;
  const int nk = (MODE == MODE_GRID) ? P.nk : 1;
  const int64_t units = (int64_t)n_tt * n_mt;
  const int64_t ipu = (int64_t)nk * nq;  // ring items per unit
  constexpr uint32_t marker_bytes = MT * KC * 8;
  constexpr uint32_t trait_bytes = TCOLS * KC * 8;

  const int BAND = P.band > 0 ? P.band : BAND_DEFAULT;
  auto decode = [&](int64_t u, int& tt, int& mt) {
    const int64_t per_band = (int64_t)BAND * n_mt;
    const int band = (int)(u / per_band);
    const int rem = (int)(u - (int64_t)band * per_band);
    const int left = n_tt - band * BAND;
    const int bw = left < BAND ? left : BAND;
    mt = rem / bw;
    tt = band * BAND + rem % bw;
  };
  // Fill stage s with the operands of flat iteration `item` = ((r * nk) + k) * nq + q of this CTA's r-th unit
  // (r is the current or the next turn); nothing to do past the last unit.
  auto issue_stage = [&](int s, int64_t item) {
    const int q = (int)(item % nq);
    const int64_t rk = item / nq;
    const int k = (int)(rk % nk);
    const int64_t u = uq[(rk / nk) & 3];
    if (u >= units) return;
    int tt, mt;
    decode(u, tt, mt);
    const int k0 = (MODE == MODE_GRID && P.tile_k0) ? P.tile_k0[tt] : 0;
    double* st = stages + (size_t)s * plan.stage_doubles;
    mbar_arrive_expect_tx(&full[s], marker_bytes + trait_bytes);
    // L2 residency: a band's trait tiles are re-read every round of units for the whole sweep over the marker
    // tiles (keep them), a marker chunk is read by the band's <= 8 CTAs within one round and then dead (let it
    // go first).  Without the hints the streaming marker fills push the trait tiles out of a 63 MB L2
    // partition at n = 1000 (ncu: 210 GB of DRAM reads for ~35 GB of operands).
    bulk_g2s_hint(st, P.Mop + ((((size_t)(k0 + k) * nq + q) * P.p_pad) + (size_t)mt * MT) * KC, marker_bytes, &full[s],
                  l2_evict_first_policy());
    bulk_g2s_hint(st + MT * KC, P.Xop + (((size_t)q * P.xcol_pad) + (size_t)tt * TCOLS) * KC, trait_bytes, &full[s],
                  l2_evict_last_policy());
  };

  if (tid == 0)
    for (int i = 0; i < NS; ++i) issue_stage(i, i);

  const int g = lane >> 2, t = lane & 3;
  const int wm = warp / ST_TG;  // marker half (0..1)
  const int wt = warp % ST_TG;  // trait group
  const int aoff = (wm * 8 * MA + g) * KC + t;
  const int boff = MT * KC + (wt * 8 * NB + g) * KC + t;

  int64_t it = 0;
  int s = 0;
  uint32_t sphase = 0;
  for (int r = 0;; ++r) {
    const int64_t u = uq[r & 3];
    if (u >= units) break;
    // Fetch the unit two turns ahead.  Warps are at most one unit apart in either direction of warp 0 (the ring is
    // no longer than a unit), so ordinals r-1 .. r+1 are being read while r+2 is written: four slots, and the
    // fetch runs two ahead so that a warp that is a unit AHEAD of warp 0 already finds its next unit.
    // (unit_counter == nullptr: static round-robin, for problems whose operands fit in L2 anyway)
    if (tid == 0 && r > 0)
      uq[(r + 2) & 3] = P.unit_counter ? (long long)atomicAdd(P.unit_counter, 1ULL)
                                       : (long long)blockIdx.x + (long long)(r + 2) * gridDim.x;
    int tt, mt;
    decode(u, tt, mt);

    double vmin[MA][NB][2];       // GRID: running minimum;  EXACT: unused
    uint32_t cnt[(MA * NB * 2 + 3) / 4];
    double dyi[2] = {1.0, 1.0};
    if (MODE == MODE_EXACT) {
      const int64_t tr = (int64_t)tt * (ST_TG * 8) + wt * 8 + 2 * t;
      dyi[0] = P.dyinv[tr];
      dyi[1] = P.dyinv[tr + 1];
    } else {
#pragma unroll
      for (int i = 0; i < (MA * NB * 2 + 3) / 4; ++i) cnt[i] = 0u;
    }
    double lod[MA][(MODE == MODE_EXACT) ? 1 : NB][2];

    for (int kk = 0; kk < nk; ++kk) {
      double ek[NB][2], etk[NB][2];
      if (MODE == MODE_GRID) {
        const int64_t pos = (int64_t)kk * P.tcol_pad + (int64_t)tt * (ST_TG * 8 * NB) + wt * (8 * NB) + 2 * t;
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          const double2 w = *reinterpret_cast<const double2*>(P.et + pos + b * 8);
          etk[b][0] = w.x; etk[b][1] = w.y;
          if (P.e) {
            const double2 v = *reinterpret_cast<const double2*>(P.e + pos + b * 8);
            ek[b][0] = v.x; ek[b][1] = v.y;
          } else {
            ek[b][0] = ek[b][1] = 1.0;
          }
        }
      }
      double acc[MA][NB][2];
#pragma unroll
      for (int a = 0; a < MA; ++a)
#pragma unroll
        for (int b = 0; b < NB; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;

      for (int q = 0; q < nq; ++q, ++it) {
        mbar_wait(&full[s], sphase);
        const double* st = stages + (size_t)s * plan.stage_doubles;
        const double* ap = st + aoff;
        const double* bp = st + boff;
        double af[2][MA], bf[2][NB];
#pragma unroll
        for (int a = 0; a < MA; ++a) af[0][a] = ap[a * 8 * KC];
#pragma unroll
        for (int b = 0; b < NB; ++b) bf[0][b] = bp[b * 8 * KC];
#pragma unroll
        for (int ks = 0; ks < KC / 4; ++ks) {
          const int cur = ks & 1;
          if (ks + 1 < KC / 4) {
#pragma unroll
            for (int a = 0; a < MA; ++a) af[cur ^ 1][a] = ap[a * 8 * KC + (ks + 1) * 4];
#pragma unroll
            for (int b = 0; b < NB; ++b) bf[cur ^ 1][b] = bp[b * 8 * KC + (ks + 1) * 4];
          }
#pragma unroll
          for (int a = 0; a < MA; ++a) {
#pragma unroll
            for (int b = 0; b < NB; ++b) {
              if (MODE == MODE_EXACT && b == NB - 1) {
                const double a2 = af[cur][a] * af[cur][a];
                dmma884(acc[a][b][0], acc[a][b][1], a2, bf[cur][b]);
              } else {
                dmma884(acc[a][b][0], acc[a][b][1], af[cur][a], bf[cur][b]);
              }
            }
          }
        }
        // Release the stage; the last of the ST_WARPS consumers refills it with iteration it + NS.
        __syncwarp();
        if (lane == 0) {
          if (smem_counter_arrive(&rel_cnt[s]) == ST_WARPS - 1) {
            rel_cnt[s] = 0;
            issue_stage(s, it + NS);
          }
        }
        if (++s == NS) {
          s = 0;
          sphase ^= 1u;
        }
      }

      if (MODE == MODE_GRID) {
        const bool first = (kk == 0);
#pragma unroll
        for (int a = 0; a < MA; ++a)
#pragma unroll
          for (int b = 0; b < NB; ++b)
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {
              const double d = acc[a][b][cc];
              const double v = fma(-(d * d), etk[b][cc], ek[b][cc]);
              const bool better = __double_as_longlong(v) < __double_as_longlong(vmin[a][b][cc]);
              const bool upd = first || better;
              vmin[a][b][cc] = upd ? v : vmin[a][b][cc];
              const int o = (a * NB + b) * 2 + cc;
              const int sh = (o & 3) * 8;
              if (ARGMAX) {
                if (upd) cnt[o >> 2] = (cnt[o >> 2] & ~(0xFFu << sh)) | ((uint32_t)kk << sh);
              } else {
                if (better && !first) cnt[o >> 2] += (1u << sh);
              }
            }
      } else {
        // EXACT: combine the c+2 accumulators of each (marker, trait) pair
#pragma unroll
        for (int a = 0; a < MA; ++a)
#pragma unroll
          for (int cc = 0; cc < 2; ++cc) {
            double dg = acc[a][NB - 1][cc];
#pragma unroll
            for (int b = 1; b < NB - 1; ++b) dg = fma(-acc[a][b][cc], acc[a][b][cc], dg);
            // v = 1 - r^2 = 1 - num^2 dyinv / dg through a Newton reciprocal (4 FP64 operations) instead of the
            // division sequence: the FP64 pipe is shared with the DMMAs of the other warps
            const double num = acc[a][0][cc];
            vmin[a][0][cc] = fma(-((num * num) * dyi[cc]), fast_rcp(dg), 1.0);
          }
      }
    }

    // final epilogue: one logarithm per output, streaming stores
    constexpr int NBO = (MODE == MODE_EXACT) ? 1 : NB;
    bool special = false;
    const double c_ln = -P.half_n * 0.43429448190325182765;
    const double c_e = -P.half_n * 0.30102999566398119521;
#pragma unroll
    for (int a = 0; a < MA; ++a)
#pragma unroll
      for (int b = 0; b < NBO; ++b)
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) lod[a][b][cc] = fast_lod(vmin[a][b][cc], logtab, c_ln, c_e, special);
    if (__any_sync(0xffffffffu, special)) {
#pragma unroll
      for (int a = 0; a < MA; ++a)
#pragma unroll
        for (int b = 0; b < NBO; ++b)
#pragma unroll
          for (int cc = 0; cc < 2; ++cc) lod[a][b][cc] = fix_lod(vmin[a][b][cc], lod[a][b][cc]);
    }
    const int k0 = (MODE == MODE_GRID && P.tile_k0) ? P.tile_k0[tt] : 0;
    const int kbase = ARGMAX ? k0 : 0;
    const int i_base = mt * MT + wm * 8 * MA + g;
    if (PEAK) {
      // per-trait peaks: the first maximum of each column over the warp's 8 * MA markers (over a in registers, then
      // over g across the lanes); units write disjoint records, so the dynamic scheduler needs no ordering
#pragma unroll
      for (int b = 0; b < NBO; ++b)
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          double pl = lod[0][b][cc];
          int row = i_base, gi = 0;
#pragma unroll
          for (int a = 0; a < MA; ++a) {
            int ga = 0;
            if (MODE == MODE_GRID) {
              const int o = (a * NB + b) * 2 + cc;
              ga = kbase + (int)((cnt[o >> 2] >> ((o & 3) * 8)) & 0xFFu);
            }
            if (a == 0)
              gi = ga;
            else
              peak_take(pl, row, gi, lod[a][b][cc], i_base + a * 8, ga, P.p);
          }
          peak_over_lanes(pl, row, gi, P.p, 4);
          const int64_t pos = (int64_t)tt * (ST_TG * 8 * NBO) + wt * (8 * NBO) + b * 8 + 2 * t + cc;
          const int64_t col = P.col_map ? (int64_t)P.col_map[pos] : (pos < P.m ? pos : -1);
          if (g == 0 && col >= 0) P.peaks[col * (P.p_pad / (8 * MA)) + mt * 2 + wm] = PeakRec{pl, row, gi};
        }
      continue;
    }
#pragma unroll
    for (int b = 0; b < NBO; ++b)
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const int64_t pos = (int64_t)tt * (ST_TG * 8 * NBO) + wt * (8 * NBO) + b * 8 + 2 * t + cc;
        const int64_t col = P.col_map ? (int64_t)P.col_map[pos] : (pos < P.m ? pos : -1);
        double* Lc = nullptr;
        double* Hc = nullptr;
        double* Mc = nullptr;
        if (col >= 0) {
          if (P.L0) {
            if (col == 0) {
              Lc = P.L0;
            } else {
              if (P.L) Lc = P.L + (col - 1) * P.ldL;
              if (P.colmax) Mc = P.colmax + (col - 1);
            }
          } else {
            if (P.L) Lc = P.L + col * P.ldL;
            if (P.colmax) Mc = P.colmax + col;
          }
          if (MODE == MODE_GRID && P.H2) Hc = P.H2 + col * P.ldL;
        }
        double cmax = 0.0;
#pragma unroll
        for (int a = 0; a < MA; ++a) {
          const int i = i_base + a * 8;
          const double l = lod[a][b][cc];
          if (i < P.p) {
            if (Lc) st_stream(Lc + i, l);
            if (MODE == MODE_GRID && Hc) {
              const int o = (a * NB + b) * 2 + cc;
              const int cv = (int)((cnt[o >> 2] >> ((o & 3) * 8)) & 0xFFu);
              st_stream(Hc + i, grid_s[kbase + cv]);
            }
            cmax = fmax(cmax, l);
          }
        }
        if (P.colmax) {
          cmax = fmax(cmax, __shfl_xor_sync(0xffffffffu, cmax, 4));
          cmax = fmax(cmax, __shfl_xor_sync(0xffffffffu, cmax, 8));
          cmax = fmax(cmax, __shfl_xor_sync(0xffffffffu, cmax, 16));
          if (g == 0 && Mc) atomic_max_nonneg(Mc, cmax + 0.0);
        }
      }
  }
}

// -----------------------------------------------------------------------------------------------
// Per-trait columns of the EXACT mode.  One warp per trait slot j < n_tt*64 (slots >= m are
// zero-filled).  Column kind a of trait j lands at packed column ((j/8)*(C+2) + a)*8 + j%8:
// a = 0: z_j,  a = 1..C: q_ja,  a = C+1: w_j.
// -----------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(256) exact_columns_kernel(const double* __restrict__ Yr, const double* __restrict__ h2,
                                                            const double* __restrict__ lambda,
                                                            const double* __restrict__ C0, int64_t m, int64_t slots,
                                                            int n, int n_pad, double* __restrict__ Xop,
                                                            int64_t xcol_pad, double* __restrict__ dyinv, int* flags) {
  constexpr int CG = C + 2;
  constexpr int NT = C * (C + 1) / 2;
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t j = (int64_t)blockIdx.x * 8 + wid;
  if (j >= slots) return;
  const int64_t colbase = (j / 8) * CG * 8 + (j % 8);
  if (j >= m) {
    for (int l = lane; l < n_pad; l += 32)
#pragma unroll
      for (int a = 0; a < CG; ++a) Xop[(((int64_t)(l / KC)) * xcol_pad + colbase + a * 8) * KC + (l % KC)] = 0.0;
    if (lane == 0) dyinv[j] = 1.0;
    return;
  }
  const double hv = h2[j];
  const double delta = hv / (1.0 - hv);
  const double* y = Yr + j * n_pad;
  double S[NT], tc[C];
#pragma unroll
  for (int i = 0; i < NT; ++i) S[i] = 0.0;
#pragma unroll
  for (int i = 0; i < C; ++i) tc[i] = 0.0;
  bool bad = false;
  for (int l = lane; l < n; l += 32) {
    const double w = 1.0 / (delta * lambda[l] + 1.0);
    bad |= !(w > 0.0);
    const double wy = w * y[l];
    double cv[C];
#pragma unroll
    for (int a = 0; a < C; ++a) cv[a] = C0[(int64_t)a * n_pad + l];
    int idx = 0;
#pragma unroll
    for (int a = 0; a < C; ++a) {
      tc[a] = fma(cv[a], wy, tc[a]);
      const double wc = w * cv[a];
#pragma unroll
      for (int b = 0; b <= a; ++b) {
        S[idx] = fma(wc, cv[b], S[idx]);
        ++idx;
      }
    }
  }
  if (bad) atomicExch(&flags[FLAG_WEIGHTS], 1);
#pragma unroll
  for (int i = 0; i < NT; ++i) S[i] = warp_sum(S[i]);
#pragma unroll
  for (int i = 0; i < C; ++i) tc[i] = warp_sum(tc[i]);
  // S = L L' (packed lower, row-major), Linv = L^-1, u = Linv * tc = Q'y
  double Lm[NT], Li[NT], u[C];
  bool spd = true;
#pragma unroll
  for (int a = 0; a < C; ++a)
#pragma unroll
    for (int b = 0; b <= a; ++b) {
      double sv = S[a * (a + 1) / 2 + b];
#pragma unroll
      for (int k = 0; k < b; ++k) sv -= Lm[a * (a + 1) / 2 + k] * Lm[b * (b + 1) / 2 + k];
      if (a == b) {
        spd &= (sv > 0.0);
        Lm[a * (a + 1) / 2 + a] = sqrt(sv);
      } else {
        Lm[a * (a + 1) / 2 + b] = sv / Lm[b * (b + 1) / 2 + b];
      }
    }
  if (!spd && lane == 0) atomicExch(&flags[FLAG_NOT_SPD], 1);
#pragma unroll
  for (int a = 0; a < C; ++a) {
    Li[a * (a + 1) / 2 + a] = 1.0 / Lm[a * (a + 1) / 2 + a];
#pragma unroll
    for (int b = 0; b < a; ++b) {
      double sv = 0.0;
#pragma unroll
      for (int k = b; k < a; ++k) sv -= Lm[a * (a + 1) / 2 + k] * Li[k * (k + 1) / 2 + b];
      Li[a * (a + 1) / 2 + b] = sv / Lm[a * (a + 1) / 2 + a];
    }
  }
#pragma unroll
  for (int a = 0; a < C; ++a) {
    double sv = 0.0;
#pragma unroll
    for (int b = 0; b <= a; ++b) sv = fma(Li[a * (a + 1) / 2 + b], tc[b], sv);
    u[a] = sv;
  }
  double dy = 0.0;
  for (int l = lane; l < n_pad; l += 32) {
    double w = 0.0, z = 0.0, qa[C];
#pragma unroll
    for (int a = 0; a < C; ++a) qa[a] = 0.0;
    if (l < n) {
      w = 1.0 / (delta * lambda[l] + 1.0);
      const double yl = y[l];
      z = w * yl;
#pragma unroll
      for (int a = 0; a < C; ++a) {
        double sv = 0.0;
#pragma unroll
        for (int b = 0; b <= a; ++b) sv = fma(Li[a * (a + 1) / 2 + b], C0[(int64_t)b * n_pad + l], sv);
        qa[a] = w * sv;
        z = fma(-qa[a], u[a], z);
      }
      dy = fma(yl, z, dy);
    }
    const int64_t base = (((int64_t)(l / KC)) * xcol_pad + colbase) * KC + (l % KC);
    Xop[base] = z;
#pragma unroll
    for (int a = 0; a < C; ++a) Xop[base + (int64_t)(a + 1) * 8 * KC] = qa[a];
    Xop[base + (int64_t)(C + 1) * 8 * KC] = w;
  }
  dy = warp_sum(dy);
  if (lane == 0) {
    if (!(sqrt(dy) > DBL_EPSILON)) atomicExch(&flags[FLAG_ZERO_NORM], 1);
    dyinv[j] = 1.0 / dy;
  }
}

template <int NB, int MA, int MODE, bool PEAK>
void launch_stream_peak(const StreamParams& P, int sm_count, cudaStream_t stream) {
  const StreamPlan plan = stream_plan(NB, MA);
  if (MODE == MODE_GRID && P.argmax_mode) {
    cudaFuncSetAttribute(scan_stream_kernel<NB, MA, MODE, true, PEAK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         SMEM_LIMIT);
    scan_stream_kernel<NB, MA, MODE, true, PEAK><<<sm_count, 32 * ST_WARPS, plan.bytes, stream>>>(P);
  } else {
    cudaFuncSetAttribute(scan_stream_kernel<NB, MA, MODE, false, PEAK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         SMEM_LIMIT);
    scan_stream_kernel<NB, MA, MODE, false, PEAK><<<sm_count, 32 * ST_WARPS, plan.bytes, stream>>>(P);
  }
}

template <int NB, int MA, int MODE>
void launch_stream_one(const StreamParams& P, int sm_count, cudaStream_t stream) {
  if (P.peaks)
    launch_stream_peak<NB, MA, MODE, true>(P, sm_count, stream);
  else
    launch_stream_peak<NB, MA, MODE, false>(P, sm_count, stream);
}

}  // namespace

int stream_exact_marker_tile(int c) { return (c + 2 <= 5) ? 64 : 32; }
int stream_grid_marker_tile() { return 64; }
int stream_grid_trait_tile() { return ST_TG * 8 * 2; }

int launch_exact_columns(const double* Yr, const double* h2, const double* lambda, const double* C0, int64_t m,
                         int64_t slots, int n, int n_pad, int c, double* Xop, int64_t xcol_pad, double* dyinv,
                         int* flags, cudaStream_t stream) {
  const unsigned blocks = (unsigned)((slots + 7) / 8);
#define BLMM_EXCOL(C) \
  case C: exact_columns_kernel<C><<<blocks, 256, 0, stream>>>(Yr, h2, lambda, C0, m, slots, n, n_pad, Xop, xcol_pad, dyinv, flags); break;
  switch (c) {
    BLMM_EXCOL(1) BLMM_EXCOL(2) BLMM_EXCOL(3) BLMM_EXCOL(4) BLMM_EXCOL(5) BLMM_EXCOL(6) BLMM_EXCOL(7) BLMM_EXCOL(8)
    default: return 0;
  }
#undef BLMM_EXCOL
  return 1;
}

int launch_scan_exact(const StreamParams& P, int c, int sm_count, cudaStream_t stream) {
  switch (c + 2) {
    case 3: launch_stream_one<3, 4, MODE_EXACT>(P, sm_count, stream); break;
    case 4: launch_stream_one<4, 4, MODE_EXACT>(P, sm_count, stream); break;
    case 5: launch_stream_one<5, 4, MODE_EXACT>(P, sm_count, stream); break;
    case 6: launch_stream_one<6, 2, MODE_EXACT>(P, sm_count, stream); break;
    case 7: launch_stream_one<7, 2, MODE_EXACT>(P, sm_count, stream); break;
    case 8: launch_stream_one<8, 2, MODE_EXACT>(P, sm_count, stream); break;
    case 9: launch_stream_one<9, 2, MODE_EXACT>(P, sm_count, stream); break;
    case 10: launch_stream_one<10, 2, MODE_EXACT>(P, sm_count, stream); break;
    default: return 0;
  }
  return 1;
}

int launch_scan_stream_grid(const StreamParams& P, int sm_count, cudaStream_t stream) {
  launch_stream_one<2, 4, MODE_GRID>(P, sm_count, stream);
  return 1;
}

}  // namespace blmm
