// kernels_recon.cuh — intra prediction + residual (dequant, inverse DCT/DST, transform-skip, bypass,
// PCM) for one picture in three launches, one WARP per transform unit / intra task.
//
//   k_residual<P>   every TU of a non-intra CU that carries work (inter residual, PCM): no dependencies,
//                   fully parallel.  Runs after k_inter_pred (it adds onto the prediction).
//   k_mark_pending  flags the 4x4 units covered by intra TUs as "pending" in a per-plane map.
//   k_intra<P>      every intra TU: border gather + substitution + smoothing, DC/planar/angular prediction,
//                   then the TU's residual.  Intra TUs are serially dependent through their neighbours
//                   (SURVEY §3.2), so the kernel executes the dependency DAG directly: warps claim *tasks*
//                   through an atomic ticket in a topological order (DAG level, then decode order; engine.cu
//                   plan_intra_levels).  A task = the TUs (<= 8x8) of one plane inside one aligned 16x16-luma /
//                   8x8-chroma region, run in decode order on a shared-memory tile, or one larger TU.  Everything that
//                   does not depend on the neighbours (TU records, coefficient lists, dequant + inverse
//                   transform into an int32 residual buffer) is done BEFORE the warp polls the pending flags
//                   of the neighbour units its availability masks let it read; the dependent part is only
//                   gather -> predict -> add.  After the store: fence, clear own flags.  The lowest unfinished
//                   ticket never waits on a later one, so the launch cannot deadlock.
//
// Replaces decode_TU (slice.cc:3460), decode_intra_prediction (intrapred.cc:277-345) incl. border
// fetch/substitution/smoothing (intrapred.h:185-258,529-674), scale_coefficients (transform.cc:361-642)
// and the transform_* / add_residual / dequant entries of the DSP table (fallback-dct.cc).
#pragma once
#include "dev_common.cuh"
#include "kernels_residual.cuh"

#define RC_WARPS 8
#define RC_THREADS (RC_WARPS * 32)
#define RC_GSTRIDE 34      // int16 row stride of the first-stage buffer
#define RC_LG_REGION 4     // intra region task: 16x16 luma / 8x8 chroma samples (the planner's tasks and k_intra's tile)
#define RC_REGION (1 << RC_LG_REGION)
#define RC_TILE_STRIDE 40  // region tile: rows -1..2G-1 (only column -1 below row G-1), columns -1..2G-1 (G <= 16)
#define RC_BLK (33 * RC_TILE_STRIDE + 8)
#define RC_FULL 0xffffffffu

struct ReconArgs {
  const b200_tu* tus;         // decode order, as recorded
  const uint32_t* list;       // TU indices this launch works on (k_residual: any order; k_intra: grouped by task)
  int n_list;
  int poll_ns;                // k_intra: cap of the polling back-off
  int n_task;                 // k_intra: number of tasks
  int n_listw, n_list8;       // k_residual: list = [n_listw warp-per-TU entries | n_list8 8x8 TUs | the rest: 4x4 TUs]
  const uint32_t* task_start; // k_intra: [n_task + 1] offsets into list, tasks in topological order
  const b200_coeff* coeffs;
  const uint8_t* scaling;     // B200_SCALING_FACTOR_BYTES or null
  unsigned int* ticket;       // zeroed before launch (k_intra)
  unsigned long long* trace;  // optional [n_task][4]: globaltimer at claim, cycles waiting, cycles working, #TUs (debug)
  uint8_t* pend[3];           // per plane, one byte per 4x4 samples: 1 = covered by an intra TU that is not finished
  int pend_w[3];
  const uint32_t* mark_list;  // k_residual: intra TU indices whose pending flags it sets on the way (k_mark_pending's work), or null
  int n_mark;
  unsigned int* err;          // k_intra: set (task index + 1) when a dependency wait exceeded spin_limit_ns: records whose avail bits name
  unsigned int* err_host;     //          units of LATER tasks (or of the task itself) can never be satisfied; err_host = mapped host copy
  unsigned long long spin_limit_ns;
};

struct ResidualSmem {  // k_residual
  int16_t coef[RC_WARPS][32 * RC_GSTRIDE];  // column-major coefficients (tu_residual) / scratch of the sub-warp paths
  int16_t g[RC_WARPS][32 * RC_GSTRIDE];
  ResTables tb;
};

template <typename P>
struct IntraSmem {  // k_intra
  P blk[RC_WARPS][RC_BLK];            // a region tile, or a large TU's samples (row stride nT)
  int16_t coef[RC_WARPS][32 * RC_GSTRIDE];
  int16_t g[RC_WARPS][32 * RC_GSTRIDE];
  res_t res[RC_WARPS][32 * 32];       // the task's residuals (saturated int16), TU after TU (row stride nT inside a TU)
  P border[RC_WARPS][2][4 * 32 + 4];  // large TUs: [0] gathered/substituted, [1] filtered / angular ref
  b200_tu tu_s[RC_WARPS][16];
  ResTables tb;
};

// -------------------------------------------------------------------------------------------------
// Residual of one LARGE TU (16x16 or 32x32) by one warp; smaller TUs take the sub-warp paths of
// kernels_residual.cuh.  TO_RES: write the residual r(x,y), saturated to int16, to res[x + y*nT] (the caller adds it later); else
// dst(x,y) = Clip(dst + r) on samples at `dst` (row stride dstride, in GLOBAL memory: each sample is read and written
// by the same lane exactly once).
//   coefT  dequantised coefficients, COLUMN-major int16: coefficient (row j, column c) at coefT[c*RC_GSTRIDE + j], so a
//          32-bit word holds a vertical pair and one dp2a performs two MACs of the column pass;
//   g      first-stage output, row-major int16 g[y*RC_GSTRIDE + j]: horizontal pairs for the row pass.
// Both passes are register-blocked 4 outputs per lane (one 16-byte load of packed matrix bytes + two operand words per
// 8 dp2a) and only touch the rows / columns up to the last significant coefficient.
// -------------------------------------------------------------------------------------------------
template <typename P, bool TO_RES>
__device__ void tu_residual(const b200_tu& tu, const b200_coeff* co, const uint8_t* __restrict__ scaling, P* dst, int dstride, res_t* res,
                            int bd, int16_t* coefT, int16_t* g, const ResTables& tb, int lane)
{
  const int log2 = tu.log2_size, nT = 1 << log2, n = tu.n_coeff;
  const int flags = tu.flags;
  const bool special = flags & (B200_TU_BYPASS | B200_TU_TSKIP);
  const Dequant dq = dequant_setup(tu, scaling, bd);
  // ---- extent of the significant coefficients ----
  int max_row = 0, max_col = 0;
  if (special) {
    max_row = max_col = nT - 1;
  } else {
    for (int i = lane; i < n; i += 32) {
      const int pos = co[i].pos;
      max_row = max(max_row, pos >> log2);
      max_col = max(max_col, pos & (nT - 1));
    }
    max_row = __reduce_max_sync(RC_FULL, max_row) & (nT - 1);
    max_col = __reduce_max_sync(RC_FULL, max_col) & (nT - 1);
  }
  const int nq = (max_row >> 2) + 1;  // groups of 4 coefficient rows in use
  uint32_t* cw = reinterpret_cast<uint32_t*>(coefT);
  uint32_t* gw = reinterpret_cast<uint32_t*>(g);
  constexpr int CW = RC_GSTRIDE / 2;  // words per column / row (odd: conflict-free across columns)
  for (int o = lane; o < (max_col + 1) * 2 * nq; o += 32) cw[(o / (2 * nq)) * CW + o % (2 * nq)] = 0;
  __syncwarp();
  // ---- dequant + scatter (transform.cc:452-525) ----
  for (int i = lane; i < n; i += 32) {
    const b200_coeff c = co[i];
    const int v = dequant_level(dq, c);
    const int pos = (dq.rotate ? (nT * nT - 1 - c.pos) : c.pos) & (nT * nT - 1);
    coefT[(pos & (nT - 1)) * RC_GSTRIDE + (pos >> log2)] = (int16_t)v;
  }
  __syncwarp();

  auto emit4 = [&](int x, int y, const int (&r)[4]) {  // 4 horizontally adjacent samples, x % 4 == 0
    if (TO_RES) res_store4(res + x + (y << log2), r[0], r[1], r[2], r[3]);
    else add_row<P, 4>(dst + x + (size_t)y * dstride, r, bd);
  };

  if (special) {
    // transform.cc:408-448 / :548-596 with fallback-dct.cc:81-91,161-225
    const bool ts = !(flags & B200_TU_BYPASS);
    const int bd_shift = 20 - bd, ts_shift = 5 + log2, rnd = 1 << (bd_shift - 1);
    auto value = [&](int x, int y) {
      int c = coefT[x * RC_GSTRIDE + y];
      if (ts) c = ((int)((unsigned)c << ts_shift) + rnd) >> bd_shift;
      return c;
    };
    if (flags & (B200_TU_RDPCM_H | B200_TU_RDPCM_V)) {
      const bool vert = flags & B200_TU_RDPCM_V;
      if (lane < nT) {
        int sum = 0;
        for (int k = 0; k < nT; k++) {
          const int x = vert ? lane : k, y = vert ? k : lane;
          sum += value(x, y);
          if (TO_RES) res[x + (y << log2)] = (res_t)clip16(sum);
          else dst[x + (size_t)y * dstride] = (P)clip_bd((int)dst[x + (size_t)y * dstride] + sum, bd);
        }
      }
    } else {
      for (int o = lane; o < nT * nT / 4; o += 32) {
        const int x = (o & (nT / 4 - 1)) * 4, y = o >> (log2 - 2);
        const int r[4] = {value(x, y), value(x + 1, y), value(x + 2, y), value(x + 3, y)};
        emit4(x, y, r);
      }
    }
    __syncwarp();
    return;
  }

  // ---- inverse DCT (fallback-dct.cc:550-691) ----
  const uint32_t* mt = (nT == 32) ? &tb.m32[0][0] : &tb.m16[0][0];  // [jq][i], nT words per jq
  const int post_shift = 20 - bd, rnd2 = 1 << (post_shift - 1);
  // pass 1 (columns): item = (column c <= max_col, block ib of 4 output rows); lanes run over ib first
  for (int o = lane; o < (max_col + 1) << (log2 - 2); o += 32) {
    const int ib = o & (nT / 4 - 1), c = o >> (log2 - 2);
    int acc[4] = {64, 64, 64, 64};
    const uint32_t* cp = cw + c * CW;
    for (int jq = 0; jq < nq; jq++) {
      const uint32_t c0 = cp[2 * jq], c1 = cp[2 * jq + 1];
      const uint4 m = *reinterpret_cast<const uint4*>(mt + jq * nT + 4 * ib);
      acc[0] = dp2a_hi(c1, m.x, dp2a_lo(c0, m.x, acc[0]));
      acc[1] = dp2a_hi(c1, m.y, dp2a_lo(c0, m.y, acc[1]));
      acc[2] = dp2a_hi(c1, m.z, dp2a_lo(c0, m.z, acc[2]));
      acc[3] = dp2a_hi(c1, m.w, dp2a_lo(c0, m.w, acc[3]));
    }
#pragma unroll
    for (int r = 0; r < 4; r++) g[(4 * ib + r) * RC_GSTRIDE + c] = (int16_t)clip16(acc[r] >> 7);
  }
  if ((max_col & 3) != 3) {  // the row pass reads whole groups of 4 columns: clear the rest of the last group
    const int c0 = max_col + 1, nc = 3 - (max_col & 3);
    for (int o = lane; o < nT * nc; o += 32) g[(o / nc) * RC_GSTRIDE + c0 + o % nc] = 0;
  }
  __syncwarp();
  // pass 2 (rows): item = (row y, block ib of 4 output columns)
  const int nq2 = (max_col >> 2) + 1;
  for (int o = lane; o < nT << (log2 - 2); o += 32) {
    const int ib = o & (nT / 4 - 1), y = o >> (log2 - 2);
    int acc[4] = {rnd2, rnd2, rnd2, rnd2};
    const uint32_t* gp = gw + y * CW;
    for (int jq = 0; jq < nq2; jq++) {
      const uint32_t g0 = gp[2 * jq], g1 = gp[2 * jq + 1];
      const uint4 m = *reinterpret_cast<const uint4*>(mt + jq * nT + 4 * ib);
      acc[0] = dp2a_hi(g1, m.x, dp2a_lo(g0, m.x, acc[0]));
      acc[1] = dp2a_hi(g1, m.y, dp2a_lo(g0, m.y, acc[1]));
      acc[2] = dp2a_hi(g1, m.z, dp2a_lo(g0, m.z, acc[2]));
      acc[3] = dp2a_hi(g1, m.w, dp2a_lo(g0, m.w, acc[3]));
    }
    const int r[4] = {acc[0] >> post_shift, acc[1] >> post_shift, acc[2] >> post_shift, acc[3] >> post_shift};
    emit4(4 * ib, y, r);
  }
  __syncwarp();
}

// -------------------------------------------------------------------------------------------------
__constant__ int8_t k_intra_angle[35] = {0,   0,   32,  26,  21,  17, 13, 9,  5,  2,  0,  -2, -5, -9, -13, -17, -21, -26,
                                         -32, -26, -21, -17, -13, -9, -5, -2, 0,  2,  5,  9,  13, 17, 21,  26,  32};
__constant__ int16_t k_inv_angle[15] = {-4096, -1638, -910, -630, -482, -390, -315, -256, -315, -390, -482, -630, -910, -1638, -4096};

// -------------------------------------------------------------------------------------------------
// Small TUs (nT = 4 or 8) on a shared-memory tile: the whole border lives in registers (lane s holds scan
// sample s: s = 0 -> border[-2nT] ... 2nT -> border[0] ... 4nT -> border[2nT]; the 33rd sample of an 8x8 TU is
// replicated in `ve`), neighbours are exchanged with shuffles only.  dst = the TU's top-left sample in the tile.
// res = this TU's precomputed residual (row stride nT) or nullptr.  intrapred.h:185-433,529-674.
// -------------------------------------------------------------------------------------------------
template <typename P>
__device__ __forceinline__ void tu_intra_small(const b200_tu& tu, P* dst, int ts, int bd, bool filter_plane, const res_t* res, int lane)
{
  const int log2 = tu.log2_size, nT = 1 << log2, mode = tu.intra_mode, cidx = tu.cidx;
  const uint64_t avail = tu.avail;
  const int total = 4 * nT + 1;
  // ---- gather ----
  int v = 0, ve = 0;
  bool av = false, av_e = false;
  {
    const int i = lane - 2 * nT;
    if (lane < total) {
      if (i < 0) { const int r = -i - 1; av = (avail >> (r >> 2)) & 1; if (av) v = dst[-1 + r * ts]; }
      else if (i == 0) { av = (avail >> B200_AVAIL_CORNER_BIT) & 1; if (av) v = dst[-1 - ts]; }
      else { const int c = i - 1; av = (avail >> (B200_AVAIL_TOP_BIT0 + (c >> 2))) & 1; if (av) v = dst[c - ts]; }
    }
    if (nT == 8) {  // scan sample 32 = border[16] = top row column 15
      av_e = (avail >> (B200_AVAIL_TOP_BIT0 + 3)) & 1;
      if (av_e) ve = dst[15 - ts];
    }
  }
  // ---- substitution (intrapred.h:637-674) ----
  {
    const unsigned m = __ballot_sync(RC_FULL, av);
    if (m == 0 && !av_e) {
      v = ve = 1 << (bd - 1);
    } else {
      const int first_lane = m ? __ffs(m) - 1 : 0;
      const int fv = __shfl_sync(RC_FULL, v, first_lane);
      const int first = m ? fv : ve;
      const unsigned below = m & ((2u << lane) - 1u);
      const int sv = __shfl_sync(RC_FULL, v, below ? 31 - __clz(below) : 0);
      v = below ? sv : first;
      const int last = __shfl_sync(RC_FULL, v, 31);
      if (!av_e) ve = last;
    }
  }
  // ---- smoothing (intrapred.h:185-258): only nT == 8 can get here with a filter (nT == 4 never filters) ----
  if (filter_plane && nT == 8 && mode != 1) {
    const int d = min(abs(mode - 26), abs(mode - 10));
    if (d > 7) {
      const int vm = __shfl_up_sync(RC_FULL, v, 1);
      int vp = __shfl_down_sync(RC_FULL, v, 1);
      if (lane == 31) vp = ve;
      if (lane != 0) v = (vp + 2 * v + vm + 2) >> 2;
    }
  }
  // border sample at index i in [-2nT, 2nT]; must be called by all lanes (uniform control flow)
  auto B = [&](int i) -> int {
    const int s = i + 2 * nT;
    const int r = __shfl_sync(RC_FULL, v, s & 31);
    return (s == 32) ? ve : r;
  };
  const int npass = (nT == 4) ? 1 : 2;
  // ---- prediction ----
  if (mode == 0) {  // planar, intrapred.h:261-285
    const int tr = B(1 + nT), bl = B(-1 - nT);
    for (int p = 0; p < npass; p++) {
      const int o = lane + 32 * p, x = o & (nT - 1), y = (o >> log2) & (nT - 1);
      const int l = B(-1 - y), t = B(1 + x);
      int px = ((nT - 1 - x) * l + (x + 1) * tr + (nT - 1 - y) * t + (y + 1) * bl + nT) >> (log2 + 1);
      if (o < nT * nT) {
        if (res) px = clip_bd(px + res[o], bd);
        dst[x + y * ts] = (P)px;
      }
    }
  } else if (mode == 1) {  // DC, intrapred.h:288-322
    const int i = lane - 2 * nT;
    const bool in = (i >= 1 && i <= nT) || (i <= -1 && i >= -nT);
    const int dc = (__reduce_add_sync(RC_FULL, in ? v : 0) + nT) >> (log2 + 1);
    const bool edge = (cidx == 0);  // nT < 32 always here
    const int b1 = B(1), bm1 = B(-1);
    for (int p = 0; p < npass; p++) {
      const int o = lane + 32 * p, x = o & (nT - 1), y = (o >> log2) & (nT - 1);
      const int t = B(x + 1), l = B(-y - 1);
      int px = dc;
      if (edge) {
        if (x == 0 && y == 0) px = (bm1 + 2 * dc + b1 + 2) >> 2;
        else if (y == 0) px = (t + 3 * dc + 2) >> 2;
        else if (x == 0) px = (l + 3 * dc + 2) >> 2;
      }
      if (o < nT * nT) {
        if (res) px = clip_bd(px + res[o], bd);
        dst[x + y * ts] = (P)px;
      }
    }
  } else {  // angular, intrapred.h:330-433
    const int angle = k_intra_angle[mode];
    const bool vert = mode >= 18;
    const int sgn = vert ? 1 : -1;
    const int inv = (angle < 0) ? (int)k_inv_angle[mode - 11] : 0;
    const bool bfilt = (cidx == 0 && !(tu.flags & B200_TU_NO_BOUNDARY_FILTER) && (mode == 26 || mode == 10));
    const int b0 = B(0), b1 = B(1), bm1 = B(-1);
    // ref[k] = border[sgn*k] for k >= 0, border[-sgn*((k*inv+128)>>8)] for the projected part k < 0
    auto R = [&](int k) -> int { return B(k >= 0 ? sgn * k : -sgn * ((k * inv + 128) >> 8)); };
    for (int p = 0; p < npass; p++) {
      const int o = lane + 32 * p, x = o & (nT - 1), y = (o >> log2) & (nT - 1);
      const int a = vert ? y : x, b = vert ? x : y;
      const int idx = ((a + 1) * angle) >> 5, fact = ((a + 1) * angle) & 31;
      const int r1 = R(b + idx + 1), r2 = R(b + idx + 2);
      const int l = B(-1 - y), t = B(1 + x);
      int px = fact ? ((32 - fact) * r1 + fact * r2 + 16) >> 5 : r1;
      if (bfilt) {
        if (mode == 26 && x == 0) px = clip_bd(b1 + ((l - b0) >> 1), bd);
        if (mode == 10 && y == 0) px = clip_bd(bm1 + ((t - b0) >> 1), bd);
      }
      if (o < nT * nT) {
        if (res) px = clip_bd(px + res[o], bd);
        dst[x + y * ts] = (P)px;
      }
    }
  }
  __syncwarp();
}

// -------------------------------------------------------------------------------------------------
// Fast path of the small TUs: when the left column, the corner and the top row of the TU are all available (every TU
// that does not touch a picture / slice / tile boundary or a constrained-intra hole), the substitution process
// (intrapred.h:637-674) degenerates to index clamping: a missing bottom-left part repeats border[-nT], a missing
// top-right part repeats border[nT].  Every lane then reads the border samples its pixels need straight from the
// shared-memory tile (no gather, ballot or shuffle chain); the [1 2 1] smoothing of 8x8 luma TUs is applied on the fly.
// This is the dependent part of the intra DAG, so what counts is its latency: ~50 mostly independent instructions.
// -------------------------------------------------------------------------------------------------
template <typename P, int LOG2>
__device__ __forceinline__ void tu_intra_fast(const b200_tu& tu, P* dst, int ts, int bd, bool filter_plane, const res_t* res, int lane)
{
  constexpr int nT = 1 << LOG2;
  const int mode = tu.intra_mode, cidx = tu.cidx;
  const uint64_t avail = tu.avail;
  const int lo = ((avail >> (nT / 4)) & 1) ? -2 * nT : -nT;                          // first bottom-left group available?
  const int hi = ((avail >> (B200_AVAIL_TOP_BIT0 + nT / 4)) & 1) ? 2 * nT : nT;      // first top-right group available?
  // (groups are 4 samples; for nT == 8 the second bottom-left / top-right group may be missing on its own)
  const int lo2 = (nT == 8 && lo < -nT && !((avail >> 3) & 1)) ? -12 : lo;
  const int hi2 = (nT == 8 && hi > nT && !((avail >> (B200_AVAIL_TOP_BIT0 + 3)) & 1)) ? 12 : hi;
  auto S = [&](int i) -> int {  // substituted border sample
    i = min(max(i, lo2), hi2);
    return (int)dst[(i < 0) ? (-i - 1) * ts - 1 : i - 1 - ts];
  };
  bool smooth = false;
  if (nT == 8 && filter_plane && mode != 1) smooth = min(abs(mode - 26), abs(mode - 10)) > 7;
  auto B = [&](int i) -> int {  // border sample after the optional smoothing (intrapred.h:185-258)
    if (nT == 8 && smooth && i > -2 * nT && i < 2 * nT) return (S(i - 1) + 2 * S(i) + S(i + 1) + 2) >> 2;
    return S(i);
  };
  constexpr int NP = (nT == 4) ? 1 : 2;  // pixels per lane (4x4: lanes 16..31 idle)
  int px[NP];
  if (mode == 0) {  // planar, intrapred.h:261-285
    const int tr = B(1 + nT), bl = B(-1 - nT);
#pragma unroll
    for (int p = 0; p < NP; p++) {
      const int o = lane + 32 * p, x = o & (nT - 1), y = (o >> LOG2) & (nT - 1);
      px[p] = ((nT - 1 - x) * B(-1 - y) + (x + 1) * tr + (nT - 1 - y) * B(1 + x) + (y + 1) * bl + nT) >> (LOG2 + 1);
    }
  } else if (mode == 1) {  // DC, intrapred.h:288-322 (never smoothed)
    const int i = lane - nT;  // lanes 0..2nT-1 <-> border[-nT..-1], border[1..nT]
    const int mine = (lane < 2 * nT) ? S(i < 0 ? i : i + 1) : 0;
    const int dc = (__reduce_add_sync(RC_FULL, mine) + nT) >> (LOG2 + 1);
#pragma unroll
    for (int p = 0; p < NP; p++) {
      const int o = lane + 32 * p, x = o & (nT - 1), y = (o >> LOG2) & (nT - 1);
      int v = dc;
      if (cidx == 0) {
        if (x == 0 && y == 0) v = (S(-1) + 2 * dc + S(1) + 2) >> 2;
        else if (y == 0) v = (S(x + 1) + 3 * dc + 2) >> 2;
        else if (x == 0) v = (S(-y - 1) + 3 * dc + 2) >> 2;
      }
      px[p] = v;
    }
  } else {  // angular, intrapred.h:330-433
    const int angle = k_intra_angle[mode];
    const bool vert = mode >= 18;
    const int sgn = vert ? 1 : -1;
    const int inv = (angle < 0) ? (int)k_inv_angle[mode - 11] : 0;
    const bool bfilt = (cidx == 0 && !(tu.flags & B200_TU_NO_BOUNDARY_FILTER) && (mode == 26 || mode == 10));
    // ref[k] = border[sgn*k] for k >= 0, border[-sgn*((k*inv+128)>>8)] for the projected part k < 0
    auto R = [&](int k) -> int { return B(k >= 0 ? sgn * k : -sgn * ((k * inv + 128) >> 8)); };
#pragma unroll
    for (int p = 0; p < NP; p++) {
      const int o = lane + 32 * p, x = o & (nT - 1), y = (o >> LOG2) & (nT - 1);
      const int a = vert ? y : x, b = vert ? x : y;
      const int idx = ((a + 1) * angle) >> 5, fact = ((a + 1) * angle) & 31;
      const int r1 = R(b + idx + 1), r2 = R(b + idx + 2);
      int v = fact ? ((32 - fact) * r1 + fact * r2 + 16) >> 5 : r1;
      if (bfilt) {
        if (mode == 26 && x == 0) v = clip_bd(B(1) + ((B(-1 - y) - B(0)) >> 1), bd);
        if (mode == 10 && y == 0) v = clip_bd(B(-1) + ((B(1 + x) - B(0)) >> 1), bd);
      }
      px[p] = v;
    }
  }
  __syncwarp();  // all border reads done before the block is overwritten (the border does not overlap the block, but keeps the
                 // read/write phases of consecutive TUs apart)
#pragma unroll
  for (int p = 0; p < NP; p++) {
    const int o = lane + 32 * p, x = o & (nT - 1), y = (o >> LOG2) & (nT - 1);
    if (o < nT * nT) {
      int v = px[p];
      if (res) v = clip_bd(v + res[o], bd);
      dst[x + y * ts] = (P)v;
    }
  }
  __syncwarp();
}

// fast path applicable?  left column, corner and top row (of the TU itself) available
__device__ __forceinline__ bool intra_fast_ok(const b200_tu& tu)
{
  const int g = 1 << (tu.log2_size - 2);  // groups of 4 samples per side
  const uint64_t need = ((1ull << g) - 1) | (1ull << B200_AVAIL_CORNER_BIT) | (((1ull << g) - 1) << B200_AVAIL_TOP_BIT0);
  if ((tu.avail & need) != need) return false;
  if (g == 2) {  // 8x8: the outer bottom-left / top-right group must not be available without the inner one (clamping
                 // reproduces the substitution only for availability that ends once)
    const unsigned bl = (unsigned)(tu.avail >> 2) & 3, tr = (unsigned)(tu.avail >> (B200_AVAIL_TOP_BIT0 + 2)) & 3;
    if (bl == 2 || tr == 2) return false;
  }
  return true;
}

// -------------------------------------------------------------------------------------------------
// Large TUs (nT = 16 or 32): neighbour samples straight from the picture plane in global memory (`gsrc` = the
// TU's top-left sample, row stride gstride; .cg loads: written by other SMs during this launch), prediction to
// `dst` in shared memory (row stride nT), border arrays in shared memory.
// -------------------------------------------------------------------------------------------------
template <typename P>
__device__ void tu_intra_large(const b200_tu& tu, const P* gsrc, int gstride, P* dst, int bd, int bd_luma, uint32_t pic_flags, bool filter_plane,
                               P* b0mem, P* b1mem, int lane)
{
  const int log2 = tu.log2_size, nT = 1 << log2, mode = tu.intra_mode, cidx = tu.cidx, dstride = nT;
  const uint64_t avail = tu.avail;
  P* b0 = b0mem + 2 * 32 + 2;  // centre element; valid [-2nT, 2nT]
  P* b1 = b1mem + 2 * 32 + 2;
  const int total = 4 * nT + 1;
  // ---- gather + substitution (intrapred.h:529-674); scan index s: 0 -> border[-2nT], 2nT -> border[0], 4nT -> border[2nT]
  // All (up to 129) neighbour samples are requested FIRST — up to five independent loads per lane, one L2 round trip — and the
  // availability scan / substitution then runs on registers.  (The loads used to sit inside the two chunk loops, each chunk's
  // ballot waiting for its load: ten dependent round trips per large TU, ~8 us of the task's dependent latency.)
  {
    constexpr int MAXC = 5;  // ceil((4 * 32 + 1) / 32)
    int v[MAXC];
    bool av[MAXC];
#pragma unroll
    for (int c5 = 0; c5 < MAXC; c5++) {
      const int s = 32 * c5 + lane, i = s - 2 * nT;
      av[c5] = false;
      v[c5] = 0;
      if (s < total) {
        const P* addr;
        if (i < 0) { const int r = -i - 1; av[c5] = (avail >> (r >> 2)) & 1; addr = gsrc - 1 + r * gstride; }
        else if (i == 0) { av[c5] = (avail >> B200_AVAIL_CORNER_BIT) & 1; addr = gsrc - 1 - gstride; }
        else { const int c = i - 1; av[c5] = (avail >> (B200_AVAIL_TOP_BIT0 + (c >> 2))) & 1; addr = gsrc + c - gstride; }
        if (av[c5]) v[c5] = (int)__ldcg(addr);
      }
    }
    // first available sample in scan order (firstValue)
    int first_val = 1 << (bd - 1);
    bool any = false;
#pragma unroll
    for (int c5 = 0; c5 < MAXC; c5++) {
      const unsigned m = __ballot_sync(0xffffffffu, av[c5]);
      if (!any && m) { first_val = __shfl_sync(0xffffffffu, v[c5], __ffs(m) - 1); any = true; }
    }
    if (!any) {
      for (int s = lane; s < total; s += 32) b0[s - 2 * nT] = (P)(1 << (bd - 1));
    } else {
      int carry = first_val;  // value of the last sample of the previous chunk after substitution
#pragma unroll
      for (int c5 = 0; c5 < MAXC; c5++) {
        if (32 * c5 < total) {  // warp-uniform
          const int s = 32 * c5 + lane, i = s - 2 * nT;
          const unsigned m = __ballot_sync(0xffffffffu, av[c5]);
          const unsigned below = m & ((2u << lane) - 1u);  // available lanes <= this one
          const int src = below ? 31 - __clz(below) : 0;
          const int sv = __shfl_sync(0xffffffffu, v[c5], src);
          const int outv = below ? sv : carry;
          if (s < total) b0[i] = (P)outv;
          carry = __shfl_sync(0xffffffffu, outv, 31);
        }
      }
    }
  }
  __syncwarp();
  // ---- smoothing (intrapred.h:185-258) ----
  const P* bsrc = b0;
  if (filter_plane && mode != 1) {
    const int d = min(abs(mode - 26), abs(mode - 10));
    const bool filt = d > ((nT == 8) ? 7 : (nT == 16) ? 1 : 0);  // intraHorVerDistThres, intrapred.h:196-203
    if (filt) {
      const bool strong = (pic_flags & B200_PIC_STRONG_INTRA_SMOOTHING) && cidx == 0 && nT == 32 &&
                          abs((int)b0[0] + (int)b0[64] - 2 * (int)b0[32]) < (1 << (bd_luma - 5)) &&
                          abs((int)b0[0] + (int)b0[-64] - 2 * (int)b0[-32]) < (1 << (bd_luma - 5));
      for (int s = lane; s < total; s += 32) {
        const int i = s - 2 * nT;
        int v;
        if (i == -2 * nT || i == 2 * nT) v = b0[i];
        else if (strong) {
          if (i == 0) v = b0[0];
          else if (i < 0) v = (int)b0[0] + (((-i) * ((int)b0[-64] - (int)b0[0]) + 32) >> 6);
          else v = (int)b0[0] + ((i * ((int)b0[64] - (int)b0[0]) + 32) >> 6);
        } else v = ((int)b0[i + 1] + 2 * (int)b0[i] + (int)b0[i - 1] + 2) >> 2;
        b1[i] = (P)v;
      }
      __syncwarp();
      bsrc = b1;
    }
  }
  P* bfree = (bsrc == b0) ? b1 : b0;  // scratch for the angular reference array
  // ---- prediction (intrapred.h:261-433) ----
  if (mode == 0) {
    for (int o = lane; o < nT * nT; o += 32) {
      const int x = o & (nT - 1), y = o >> log2;
      dst[x + y * dstride] = (P)(((nT - 1 - x) * (int)bsrc[-1 - y] + (x + 1) * (int)bsrc[1 + nT] + (nT - 1 - y) * (int)bsrc[1 + x] +
                                  (y + 1) * (int)bsrc[-1 - nT] + nT) >> (log2 + 1));
    }
  } else if (mode == 1) {
    int part = 0;
    for (int i = lane; i < nT; i += 32) part += (int)bsrc[i + 1] + (int)bsrc[-i - 1];
    const int dc = (__reduce_add_sync(RC_FULL, part) + nT) >> (log2 + 1);
    const bool edge = (cidx == 0 && nT < 32);
    for (int o = lane; o < nT * nT; o += 32) {
      const int x = o & (nT - 1), y = o >> log2;
      int v = dc;
      if (edge) {
        if (x == 0 && y == 0) v = ((int)bsrc[-1] + 2 * dc + (int)bsrc[1] + 2) >> 2;
        else if (y == 0) v = ((int)bsrc[x + 1] + 3 * dc + 2) >> 2;
        else if (x == 0) v = ((int)bsrc[-y - 1] + 3 * dc + 2) >> 2;
      }
      dst[x + y * dstride] = (P)v;
    }
  } else {
    const int angle = k_intra_angle[mode];
    const bool vert = mode >= 18;
    const int sgn = vert ? 1 : -1;
    P* ref = bfree;  // ref[x] valid on [-nT, 2nT]
    const int last = (nT * angle) >> 5;
    const int inv = (angle < 0) ? (int)k_inv_angle[mode - 11] : 0;
    const bool project = (angle < 0) && (last < -1);
    for (int s = lane; s <= 3 * nT; s += 32) {
      const int x = s - nT;
      // ref[x] = border[sgn*x] for 0 <= x <= nT (and up to 2nT for non-negative angles); for negative angles the part
      // x in [last, -1] is projected from the other border through the inverse angle (intrapred.h:352-364,392-404)
      const bool w = (x >= 0) ? (x <= nT || angle >= 0) : (project && x >= last);
      const int idx = (x >= 0) ? sgn * x : -sgn * ((x * inv + 128) >> 8);
      if (w) ref[x] = bsrc[idx];
    }
    __syncwarp();
    const bool bfilt = (cidx == 0 && nT < 32 && !(tu.flags & B200_TU_NO_BOUNDARY_FILTER) && (mode == 26 || mode == 10));
    for (int o = lane; o < nT * nT; o += 32) {
      const int x = o & (nT - 1), y = o >> log2;
      const int a = vert ? y : x, b = vert ? x : y;
      const int idx = ((a + 1) * angle) >> 5, fact = ((a + 1) * angle) & 31;
      int v = fact ? ((32 - fact) * (int)ref[b + idx + 1] + fact * (int)ref[b + idx + 2] + 16) >> 5 : (int)ref[b + idx + 1];
      if (bfilt) {
        if (mode == 26 && x == 0) v = clip_bd((int)bsrc[1] + (((int)bsrc[-1 - y] - (int)bsrc[0]) >> 1), bd);
        if (mode == 10 && y == 0) v = clip_bd((int)bsrc[-1] + (((int)bsrc[1 + x] - (int)bsrc[0]) >> 1), bd);
      }
      dst[x + y * dstride] = (P)v;
    }
  }
  __syncwarp();
}

// TU block -> picture plane, 4-byte units (TU rows are 4-byte aligned: x multiple of 4 samples)
template <typename P>
__device__ __forceinline__ void block_store(const P* blk, uint8_t* plane, int pitch, int x, int y, int nT, int lane)
{
  const int upr = nT * (int)sizeof(P) / 4;
  for (int o = lane; o < nT * upr; o += 32) {
    const int r = o / upr, u = o % upr;
    *reinterpret_cast<uint32_t*>(plane + (size_t)(y + r) * pitch + (size_t)x * sizeof(P) + 4 * u) = reinterpret_cast<const uint32_t*>(blk + r * nT)[u];
  }
}

// -------------------------------------------------------------------------------------------------
// Persistent CTAs; work items per warp, heaviest class first: one large / PCM TU, then four 8x8 TUs, then 32 4x4 TUs.
template <typename P>
__global__ void __launch_bounds__(RC_THREADS) k_residual(DevPic pic, ReconArgs args)
{
  __shared__ ResidualSmem sm;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < (int)(sizeof(ResTables) / 4); i += RC_THREADS) reinterpret_cast<uint32_t*>(&sm.tb)[i] = reinterpret_cast<const uint32_t*>(&c_res)[i];
  // the intra DAG's pending flags (k_intra runs after this kernel): one launch less per picture than a separate k_mark_pending
  for (int i = blockIdx.x * RC_THREADS + tid; i < args.n_mark; i += gridDim.x * RC_THREADS) {
    const b200_tu tu = args.tus[args.mark_list[i]];
    const int c = tu.cidx, n4u = 1 << (tu.log2_size - 2);
    uint8_t* p = args.pend[c] + (tu.y >> 2) * args.pend_w[c] + (tu.x >> 2);
    for (int j = 0; j < n4u; j++)
      for (int k = 0; k < n4u; k++) p[j * args.pend_w[c] + k] = 1;
  }
  __syncthreads();
  const int n4 = args.n_list - args.n_listw - args.n_list8;
  const int Ww = args.n_listw, W8 = (args.n_list8 + 3) >> 2, W4 = (n4 + 31) >> 5;
  uint32_t* scratch = reinterpret_cast<uint32_t*>(sm.coef[warp]);  // 256 words are enough for the sub-warp paths
  for (int wi = blockIdx.x * RC_WARPS + warp; wi < Ww + W8 + W4; wi += gridDim.x * RC_WARPS) {
    if (wi < Ww) {
      const b200_tu tu = args.tus[args.list[wi]];
      const int c = tu.cidx, nT = 1 << tu.log2_size;
      P* dst = row_ptr<P>(pic.cur[c], pic.pitch[c], tu.y) + tu.x;
      const int dstride = pic.pitch[c] / (int)sizeof(P);
      if (tu.flags & B200_TU_PCM) {  // slice.cc:4211-4255
        for (int i = lane; i < tu.n_coeff; i += 32) {
          const b200_coeff co = args.coeffs[tu.coeff_off + i];
          dst[(co.pos & (nT - 1)) + (co.pos >> tu.log2_size) * dstride] = (P)(uint16_t)co.level;
        }
      } else {
        tu_residual<P, false>(tu, args.coeffs + tu.coeff_off, args.scaling, dst, dstride, nullptr, c ? pic.bd_c : pic.bd_y, sm.coef[warp], sm.g[warp],
                              sm.tb, lane);
      }
    } else if (wi < Ww + W8) {
      const int idx = Ww + (wi - Ww) * 4 + (lane >> 3);
      const bool active = idx < Ww + args.n_list8;
      b200_tu tu;
      if (active) tu = args.tus[args.list[idx]];
      else { tu.x = tu.y = 0; tu.cidx = 0; tu.coeff_off = 0; }
      const int c = tu.cidx;
      P* dst = row_ptr<P>(pic.cur[c], pic.pitch[c], tu.y) + tu.x;
      res8_quarter<P, false>(active, tu, args.coeffs + tu.coeff_off, args.scaling, dst, pic.pitch[c] / (int)sizeof(P), nullptr, c ? pic.bd_c : pic.bd_y,
                             scratch + (lane >> 3) * 64, lane & 7, sm.tb);
    } else {
      const int idx = Ww + args.n_list8 + (wi - Ww - W8) * 32 + lane;
      if (idx < args.n_list) {
        const b200_tu tu = args.tus[args.list[idx]];
        const int c = tu.cidx;
        P* dst = row_ptr<P>(pic.cur[c], pic.pitch[c], tu.y) + tu.x;
        res4_lane<P, false>(tu, args.coeffs + tu.coeff_off, args.scaling, dst, pic.pitch[c] / (int)sizeof(P), nullptr, c ? pic.bd_c : pic.bd_y, scratch, lane,
                            sm.tb);
      }
    }
    __syncwarp();
  }
}

__global__ void k_mark_pending(ReconArgs args)
{
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= args.n_list) return;
  const b200_tu tu = args.tus[args.list[idx]];
  const int c = tu.cidx, n4 = 1 << (tu.log2_size - 2);
  uint8_t* p = args.pend[c] + (tu.y >> 2) * args.pend_w[c] + (tu.x >> 2);
  for (int j = 0; j < n4; j++)
    for (int i = 0; i < n4; i++) p[j * args.pend_w[c] + i] = 1;
}

// Dependency set of a task = the distinct 4x4 units OUTSIDE its frame (region, or the single large TU) that its
// TUs' availability masks let them read: at most `span` units left of it (top-down), the corner and `span`
// units above it (left-to-right), span = 2G/4 for a region, nT/2 for a large TU.
// One TU's contribution (bit masks, span <= 16): left units bit u = unit row u left of the frame, top units bit u = unit
// column u above it, corner.  Lanes compute their own TU's masks and the warp ORs them.
__device__ __forceinline__ void dep_units_of(const b200_tu& tu, int rx, int ry, int span, unsigned& left, bool& corner, unsigned& top)
{
  const int half = 1 << (tu.log2_size - 1);  // availability groups per side (nT/2 groups of 4 samples = 2nT samples)
  const int ux0 = (tu.x - rx) >> 2, uy0 = (tu.y - ry) >> 2;  // TU position inside the frame, in units
  const uint64_t avail = tu.avail;
  const unsigned gm = (half >= 32) ? 0xffffffffu : ((1u << half) - 1u), sm = (1u << span) - 1u;
  const bool cb = (avail >> B200_AVAIL_CORNER_BIT) & 1;
  if (ux0 == 0) {  // left neighbours are outside the frame
    left |= (((unsigned)avail & gm) << uy0) & sm;
    if (cb) { if (uy0 == 0) corner = true; else left |= 1u << (uy0 - 1); }
  } else if (uy0 == 0 && cb) {
    top |= 1u << (ux0 - 1);
  }
  if (uy0 == 0) top |= (((unsigned)(avail >> B200_AVAIL_TOP_BIT0) & gm) << ux0) & sm;
}

template <typename P>
__global__ void __launch_bounds__(RC_THREADS, 3) k_intra(DevPic pic, ReconArgs args)
{
  extern __shared__ __align__(16) uint8_t smem_raw[];
  IntraSmem<P>& sm = *reinterpret_cast<IntraSmem<P>*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < (int)(sizeof(ResTables) / 4); i += RC_THREADS) reinterpret_cast<uint32_t*>(&sm.tb)[i] = reinterpret_cast<const uint32_t*>(&c_res)[i];
  __syncthreads();
  b200_tu* tus = sm.tu_s[warp];
  res_t* res = sm.res[warp];
  P* blk = sm.blk[warp];
  // Persistent warps: each warp keeps claiming the next task of the topological order.
  for (;;) {
    unsigned t = 0;
    if (lane == 0) t = atomicAdd(args.ticket, 1u);
    t = __shfl_sync(RC_FULL, t, 0);
    if (t >= (unsigned)args.n_task) return;
    unsigned long long tr_t0 = 0, tr_c0 = 0, tr_c1 = 0;
    if (args.trace) { asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr_t0)); tr_c0 = clock64(); }
    const uint32_t first = args.task_start[t], count = min(args.task_start[t + 1] - first, 16u);
    // ---- everything that does not depend on the neighbours: TU records, coefficient lists, residuals ----
    if (lane < (int)count) tus[lane] = args.tus[args.list[first + lane]];
    __syncwarp();
    const b200_tu tu0 = tus[0];
    // A task is one large TU, or the small TUs of one plane inside one region
    const int c = tu0.cidx, G = RC_REGION >> (c ? 1 : 0);
    const bool region = (1 << tu0.log2_size) <= min(G, 8);  // small TUs on a shared-memory tile; larger ones straight from the picture
    const int rx = region ? tu0.x & ~(G - 1) : tu0.x, ry = region ? tu0.y & ~(G - 1) : tu0.y;  // dependency frame origin
    {
      // residuals of all the task's TUs, in parallel where the sizes allow: lane i owns TU i's record; 4x4 TUs run one
      // per lane, 8x8 TUs one per quarter-warp, larger ones one after the other on the whole warp.  res holds the TUs'
      // residual blocks back to back (exclusive prefix sum of nT^2 over the lanes).
      const bool mine = lane < (int)count;
      const b200_tu& mytu = tus[mine ? lane : 0];
      const int l2 = mytu.log2_size, sz = mine ? 1 << (2 * l2) : 0;
      const int mybd = mytu.cidx ? pic.bd_c : pic.bd_y;
      int incl = sz;
#pragma unroll
      for (int d = 1; d < 16; d <<= 1) {
        const int up = __shfl_up_sync(RC_FULL, incl, d);
        if (lane >= d) incl += up;
      }
      const int my_rbase = incl - sz;
      const bool cbf = mine && (mytu.flags & B200_TU_CBF);
      const unsigned m8 = __ballot_sync(RC_FULL, cbf && l2 == 3), mw = __ballot_sync(RC_FULL, cbf && l2 > 3);
      uint32_t* scratch = reinterpret_cast<uint32_t*>(sm.coef[warp]);
      if (cbf && l2 == 2) res4_lane<P, true>(mytu, args.coeffs + mytu.coeff_off, args.scaling, nullptr, 0, res + my_rbase, mybd, scratch, lane, sm.tb);
      __syncwarp();
      for (unsigned rem = m8; rem;) {
        const int q = lane >> 3;
        const unsigned idx = __fns(rem, 0, q + 1);  // q-th pending 8x8 TU (0xffffffff: none)
        const bool active = idx < 32u;
        const b200_tu& tu = tus[active ? idx : 0];
        const int rb = __shfl_sync(RC_FULL, my_rbase, active ? idx : 0);
        res8_quarter<P, true>(active, tu, args.coeffs + tu.coeff_off, args.scaling, nullptr, 0, res + rb, tu.cidx ? pic.bd_c : pic.bd_y, scratch + q * 64,
                              lane & 7, sm.tb);
#pragma unroll
        for (int k = 0; k < 4; k++) rem &= rem - 1;  // (0 & -1 stays 0)
      }
      for (unsigned rem = mw; rem; rem &= rem - 1) {
        const int idx = __ffs(rem) - 1;
        const b200_tu& tu = tus[idx];
        const int rb = __shfl_sync(RC_FULL, my_rbase, idx);
        tu_residual<P, true>(tu, args.coeffs + tu.coeff_off, args.scaling, nullptr, 0, res + rb, tu.cidx ? pic.bd_c : pic.bd_y, sm.coef[warp], sm.g[warp],
                             sm.tb, lane);
      }
    }
    // ---- wait: one flag per distinct external neighbour unit, one lane each ----
    {
      const int span = region ? (2 * G) >> 2 : (1 << tu0.log2_size) >> 1;
      unsigned left = 0, top = 0;
      bool corner = false;
      if (lane < (int)count) dep_units_of(tus[lane], rx, ry, span, left, corner, top);
      left = __reduce_or_sync(RC_FULL, left);
      top = __reduce_or_sync(RC_FULL, top);
      corner = __any_sync(RC_FULL, corner);
      const int pw = args.pend_w[c];
      const uint8_t* pend = args.pend[c] + (ry >> 2) * pw + (rx >> 2);
      const volatile uint8_t* f = nullptr;
      if (lane < span) { if ((left >> lane) & 1) f = pend + lane * pw - 1; }
      else if (lane == span) { if (corner) f = pend - pw - 1; }
      else if (lane - span - 1 < span) { if ((top >> (lane - span - 1)) & 1) f = pend - pw + (lane - span - 1); }
      const volatile uint8_t* f2 = nullptr;  // 32x32 TU: 33 units, lane 0 takes the last top unit as well
      if (span == 16 && lane == 0 && ((top >> 15) & 1)) f2 = pend - pw + 15;
      unsigned ns = 32, spins = 0;
      unsigned long long t_wait0 = 0;
      for (;;) {
        const bool busy = (f && *f) || (f2 && *f2);
        if (!__any_sync(RC_FULL, busy)) break;
        __nanosleep(ns);
        if (ns < (unsigned)args.poll_ns) ns *= 2;
        else if ((++spins & 63u) == 0) {
          // Bounded: in a well-formed picture every dependency belongs to an earlier task, so the wait ends.  A record whose avail
          // bits name a unit of a later task (or its own) would spin forever: give up after spin_limit_ns (and at once when another
          // task already gave up), flag the picture and go on with whatever the neighbours hold.  The host reports
          // B200_ERR_INVALID at the next synchronisation point.  Checked every 64th poll (~60 us): nothing on the polling path.
          unsigned long long now;
          asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
          if (!t_wait0) t_wait0 = now;
          bool give_up = now - t_wait0 > args.spin_limit_ns || *(volatile unsigned int*)args.err != 0;
          give_up = __shfl_sync(RC_FULL, give_up, 0);
          if (give_up) {
            if (lane == 0) {
              atomicCAS(args.err, 0u, t + 1);
              *(volatile unsigned int*)args.err_host = t + 1;
              __threadfence_system();
            }
            break;
          }
        }
      }
    }
    __threadfence();  // acquire: the neighbours' samples were published before their flags were cleared
    if (args.trace) tr_c1 = clock64();

    const int bd = c ? pic.bd_c : pic.bd_y;
    const bool filter_plane = !(pic.flags & B200_PIC_INTRA_SMOOTHING_OFF) && (c == 0 || pic.chroma == 3);
    if (!region) {
      // ---- one large TU: borders straight from the picture ----
      const int nT = 1 << tu0.log2_size;
      const int gstride = pic.pitch[c] / (int)sizeof(P);
      const P* gsrc = row_ptr<P>(pic.cur[c], pic.pitch[c], tu0.y) + tu0.x;
      tu_intra_large<P>(tu0, gsrc, gstride, blk, bd, pic.bd_y, pic.flags, filter_plane, sm.border[warp][0], sm.border[warp][1], lane);
      if (tu0.flags & B200_TU_CBF) {
        for (int o = lane; o < nT * nT; o += 32) blk[o] = (P)clip_bd((int)blk[o] + res[o], bd);
        __syncwarp();
      }
      block_store<P>(blk, pic.cur[c], pic.pitch[c], tu0.x, tu0.y, nT, lane);
    } else {
      // ---- regions of small TUs: stage region + top row (2G) + left column (2G) in shared memory, run the TUs in order ----
      const int pwid = c ? pic.cw : pic.w, phei = c ? pic.ch : pic.h;
      int covered = 0;  // samples this task writes
      for (int i = 0; i < (int)count; i++) covered += 1 << (2 * tus[i].log2_size);
      const int TS = RC_TILE_STRIDE;
      P* tile = blk + TS + 4;  // tile(0,0) = region origin, 4-byte aligned; tile(-1,-1) is blk[3]
      const int gw = min(G, pwid - rx), gh = min(G, phei - ry);
      const bool full = (gw == G) && (gh == G);
      // the interior is only needed where this task does not write it itself (regions partly covered by inter blocks)
      if (covered < gw * gh) {
        if (full) {  // whole rows as 4-byte words, like the store below
          const int wpr = G * (int)sizeof(P) / 4;
          for (int o = lane; o < G * wpr; o += 32) {
            const int y = o / wpr, u = o % wpr;  // wpr is a power of two
            reinterpret_cast<uint32_t*>(tile + y * TS)[u] = __ldcg(reinterpret_cast<const uint32_t*>(row_ptr<P>(pic.cur[c], pic.pitch[c], ry + y) + rx) + u);
          }
        } else {
          for (int o = lane; o < gw * gh; o += 32) {
            const int x = o % gw, y = o / gw;
            tile[y * TS + x] = __ldcg(row_ptr<P>(pic.cur[c], pic.pitch[c], ry + y) + rx + x);
          }
        }
      }
      if (ry > 0)
        for (int x = lane - 1; x < 2 * G; x += 32)
          if (rx + x >= 0 && rx + x < pwid) tile[-TS + x] = __ldcg(row_ptr<P>(pic.cur[c], pic.pitch[c], ry - 1) + rx + x);
      if (rx > 0)  // left column incl. the bottom-left reach (available when the region is a top-left child of its parent block)
        for (int y = lane; y < 2 * G; y += 32)
          if (ry + y < phei) tile[y * TS - 1] = __ldcg(row_ptr<P>(pic.cur[c], pic.pitch[c], ry + y) + rx - 1);
      __syncwarp();
      int rbase = 0;
      for (int i = 0; i < (int)count; i++) {
        const b200_tu& tu = tus[i];
        P* tdst = tile + (tu.y - ry) * TS + (tu.x - rx);
        const res_t* tres = (tu.flags & B200_TU_CBF) ? res + rbase : nullptr;
        if (!intra_fast_ok(tu)) tu_intra_small<P>(tu, tdst, TS, bd, filter_plane, tres, lane);
        else if (tu.log2_size == 2) tu_intra_fast<P, 2>(tu, tdst, TS, bd, filter_plane, tres, lane);
        else tu_intra_fast<P, 3>(tu, tdst, TS, bd, filter_plane, tres, lane);
        rbase += 1 << (2 * tu.log2_size);
      }
      if (full) {  // whole rows as 4-byte words (tile rows are 4-byte aligned: TS * sizeof(P) and the origin offset are multiples of 4)
        const int wpr = G * (int)sizeof(P) / 4;  // words per row
        for (int o = lane; o < G * wpr; o += 32) {
          const int y = o / wpr, u = o % wpr;  // wpr is a power of two
          reinterpret_cast<uint32_t*>(row_ptr<P>(pic.cur[c], pic.pitch[c], ry + y) + rx)[u] = reinterpret_cast<const uint32_t*>(tile + y * TS)[u];
        }
      } else {
        for (int o = lane; o < gw * gh; o += 32) {
          const int x = o % gw, y = o / gw;
          row_ptr<P>(pic.cur[c], pic.pitch[c], ry + y)[rx + x] = tile[y * TS + x];
        }
      }
    }
    __threadfence();  // release: samples before flags
    __syncwarp();
    if (lane < (int)count) {  // one lane per TU clears the TU's pending units
      const b200_tu& tu = tus[lane];
      const int n4 = 1 << (tu.log2_size - 2), pw = args.pend_w[tu.cidx];
      volatile uint8_t* pend = args.pend[tu.cidx] + (tu.y >> 2) * pw + (tu.x >> 2);
      for (int j = 0; j < n4; j++)
        for (int i = 0; i < n4; i++) pend[j * pw + i] = 0;
    }
    __syncwarp();
    if (args.trace && lane == 0) {
      const unsigned long long c2 = clock64();
      unsigned long long* tr = args.trace + 4ull * t;
      tr[0] = tr_t0; tr[1] = tr_c1 - tr_c0; tr[2] = c2 - tr_c1; tr[3] = count | ((unsigned long long)tu0.cidx << 8) | ((unsigned long long)tu0.log2_size << 16);
    }
  }
}
