// direction.cu -- D8 steepest-descent flow direction for sm_100a.
//
// Replaces flow_direction_for_tile + calculate_slope
// (reference src/overflow/flow_direction.py:14-96).
//
// Layout.  The raster is cut into column bands of 128 cells and row chunks of
// `chunk_rows`; one warp owns one (band, chunk) work item at a time and streams
// down its rows.  Each warp runs a private TMA pipeline: lane 0 issues
// cp.async.bulk.tensor.2d loads of [8 rows x 136 floats] boxes (the band plus a
// 4-float apron each side, so every lane's float4 stays 16-byte aligned) into a
// ring of shared-memory stages guarded by mbarriers; out-of-raster box elements
// are zero-filled by TMA and replaced in registers by the nodata fill.  A lane
// owns 4 adjacent cells.  Per new input row it forms the 19 float32 differences
// its cells share with their south / south-east / south-west / east neighbours
// once (a - b == -(b - a) exactly in IEEE arithmetic), so every cell costs
// 4.75 subtractions instead of 8, and writes its four uint8 codes as one 32-bit
// store: a warp stores one full 128-byte line per output row.
//
// Arithmetic (bit-exact with the reference).  The reference subtracts in
// float32, divides diagonals by sqrt(2) in float64 and keeps the first strict
// maximum in scan order E,NE,N,NW,W,SW,S,SE; a nodata neighbour is slope +inf.
//  * nodata inputs are rewritten to -inf on load, so (z - n) is +inf for them;
//  * within the four cardinals (or the four diagonals) the float64 slopes order
//    exactly like the float32 differences (division by a positive constant is
//    monotone and injective on float32 inputs), so each class maximum and its
//    first index come from float32 max / compares;
//  * cardinal best c against diagonal best d: the float64 test d/sqrt(2) > c is
//    decided by u = fma(d, 1/sqrt(2), -c) whenever |u| > 2^-19 |c|, which implies
//    |u| > 2^-21 |d| (the float32 evaluation error is below 2^-23 |d|); an exact tie d/sqrt(2) == c cannot
//    happen for finite non-zero float32 inputs (sqrt(2) is irrational and the
//    float64 constant is 2^-53-close to it);
//  * everything else -- +inf in both classes or among the cardinals (nodata neighbours),
//    a NODATA or non-finite centre, or |u| inside the guard band -- takes d8_exact(), which re-reads the
//    3x3 window from shared memory and runs the reference algorithm literally in
//    float64.
#include <math.h>

#include <atomic>
#include <stdlib.h>

#include "common.cuh"

namespace ofl {

#ifndef OFL_DIR_L2PROMO
#define OFL_DIR_L2PROMO 0
#endif
#ifndef OFL_DIR_RB
#define OFL_DIR_RB 4
#endif
#ifndef OFL_DIR_STAGES
#define OFL_DIR_STAGES 4
#endif
#ifndef OFL_DIR_WARPS
#define OFL_DIR_WARPS 4
#endif
#ifndef OFL_DIR_CTAS_PER_SM
#define OFL_DIR_CTAS_PER_SM 3
#endif
constexpr int DIR_RB = OFL_DIR_RB;          // rows per TMA box / pipeline stage
constexpr int DIR_STAGES = OFL_DIR_STAGES;  // stages per warp
#ifndef OFL_DIR_NC
#define OFL_DIR_NC 4
#endif
constexpr int NC = OFL_DIR_NC;   // adjacent cells per lane (4, or 2: half the per-thread state, twice the warps)
static_assert(NC == 2 || NC == 4, "a lane owns two or four cells");
constexpr int DIR_BAND = 32 * NC;       // columns per warp band
constexpr int DIR_BOXW = DIR_BAND + 8;  // 4 apron + band + 4 apron floats
constexpr int DIR_WARPS = OFL_DIR_WARPS;    // warps per CTA
constexpr int DIR_STAGE_FLOATS = DIR_RB * DIR_BOXW;
constexpr uint32_t DIR_STAGE_BYTES = DIR_STAGE_FLOATS * 4;
constexpr size_t DIR_SMEM_BYTES = size_t(DIR_WARPS) * DIR_STAGES * DIR_STAGE_BYTES + DIR_WARPS * DIR_STAGES * 8;

struct DirParams {
  uint8_t* out;
  int64_t ld_out;
  int H, W;        // output rows / cols
  int y_off;       // input row of output row y is y + y_off
  int in_rows;     // rows of the input tensor
  float nd;        // float32 nodata value, NaN when no float32 can equal the band nodata
  float fillv;     // what a cell outside the input array reads as (already nodata-transformed)
  float fill_raw;  // same, before the nodata transform (for the exact path)
  int n_bands, n_chunks, chunk_rows;
  int* next_item;  // work counter: warps take (band, chunk) items in order as they become free
};

// The reference's scan, literally, over the eight float32 differences (centre - neighbour) of one cell in
// scan order E,NE,N,NW,W,SW,S,SE, none of them +inf (flow_direction.py:49-67, :94-96): diagonals divided by
// sqrt(2) in float64, first strict maximum wins, no positive slope -> undefined.
__device__ __noinline__ uint32_t d8_slopes(float d0, float d1, float d2, float d3, float d4, float d5, float d6, float d7) {
  const float d[8] = {d0, d1, d2, d3, d4, d5, d6, d7};
  double best = -INFINITY;
  int bi = -1;
  bool any_pos = false;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const double s = (i & 1) ? __ddiv_rn((double)d[i], 1.4142135623730951) : (double)d[i];
    if (s > best) {
      best = s;
      bi = i;
    }
    if (s > 0.0) any_pos = true;
  }
  return any_pos ? (uint32_t)bi : (uint32_t)OFL_DIR_UNDEFINED;
}

// One cell by the reference's rules: a NODATA neighbour is slope +inf, and the first +inf in scan order wins
// (it is the first strict maximum).  A cell without one whose differences are all finite is decided in
// float32 whenever the fast path's own argument applies (class maxima, then the sign of u outside the
// guard band); only what is left -- non-finite data, or u inside the band -- needs the float64 scan.
__device__ __forceinline__ uint32_t d8_exact(float z, float nE, float nNE, float nN, float nNW, float nW, float nSW,
                                             float nS, float nSE, float nd) {
  if (z == nd) return OFL_DIR_NODATA;
  const float n[8] = {nE, nNE, nN, nNW, nW, nSW, nS, nSE};
  float d[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) d[i] = (n[i] == nd) ? INFINITY : __fsub_rn(z, n[i]);
  uint32_t first = 8;
#pragma unroll
  for (int i = 7; i >= 0; --i) first = (d[i] == INFINITY) ? (uint32_t)i : first;
  if (first < 8) return first;
  float finite = 0.f;  // stays 0 iff every difference is finite
#pragma unroll
  for (int i = 0; i < 8; ++i) finite = __fmaf_rn(d[i], 0.f, finite);
  if (finite == 0.f) {
    const float c = fmaxf(fmaxf(d[0], d[2]), fmaxf(d[4], d[6]));
    const float dg = fmaxf(fmaxf(d[1], d[3]), fmaxf(d[5], d[7]));
    if (!(fmaxf(c, dg) > 0.f)) return OFL_DIR_UNDEFINED;
    const float u = __fmaf_rn(dg, 0.70710678118654752f, -c);
    if (fabsf(u) > __fmul_rn(fabsf(c), 1.9073486328125e-06f)) {
      if (u > 0.f) return d[1] == dg ? 1u : d[3] == dg ? 3u : d[5] == dg ? 5u : 7u;
      return d[0] == c ? 0u : d[2] == c ? 2u : d[4] == c ? 4u : 6u;
    }
  }
  return d8_slopes(d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7]);
}

// 1.0f / 0.0f comparison results (SASS FSET.BF): they feed FMA-pipe arithmetic, which keeps the
// index selection off the half-rate ALU pipe that the compares and max operations already saturate.
__device__ __forceinline__ float f_ne(float a, float b) {  // a != b or unordered
  float r;
  asm("set.neu.f32.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ float f_gt(float a, float b) {
  float r;
  asm("set.gt.f32.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ float f_leu(float a, float b) {  // !(a > b): a <= b or unordered
  float r;
  asm("set.leu.f32.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}

// Fast path for one cell.  Differences are (centre - neighbour) in float32.  Returns the code as a small
// float (0..8); `special` accumulates a non-zero value when the exact path must decide instead.
__device__ __forceinline__ float d8_fast(float dE, float dNE, float dN, float dNW, float dW, float dSW, float dS,
                                         float dSE, float& special) {
  // fmaxf ignores NaN operands, like the reference's `slope > max_slope` scan
  const float c = fmaxf(fmaxf(dE, dN), fmaxf(dW, dS));
  const float d = fmaxf(fmaxf(dNE, dNW), fmaxf(dSW, dSE));
  // first index attaining the class maximum: E,N,W,S -> 0,2,4,6 and NE,NW,SW,SE -> 1,3,5,7
  const float ic = f_ne(dE, c) * __fmaf_rn(f_ne(dN, c), __fmaf_rn(f_ne(dW, c), 2.f, 2.f), 2.f);
  const float id = __fmaf_rn(f_ne(dNE, d), __fmaf_rn(f_ne(dNW, d), __fmaf_rn(f_ne(dSW, d), 2.f, 2.f), 2.f), 1.f);
  const float m = fmaxf(c, d);
  const float u = __fmaf_rn(d, 0.70710678118654752f, -c);               // > 0: the diagonal is steeper
  // guard band: the sign of u is certain when |u| > 2^-19 |c|.  (|d| >= 4|c| makes |u| >= 0.45 |d|; otherwise
  // 2^-19 |c| > 2^-21 |d|, eight times the evaluation error of u.)  An infinite c makes the band infinite.
  const float thr = __fmul_rn(fabsf(c), 1.9073486328125e-06f);
  const float pos = f_gt(m, 0.f);
  float code = __fmaf_rn(f_gt(u, 0.f), __fsub_rn(id, ic), ic);
  code = __fmaf_rn(pos, __fsub_rn(code, 8.f), 8.f);
  // exact path: a positive maximum whose class is not certain (this includes a NaN u: +inf in both classes,
  // or a +inf centre).  A NODATA / -inf centre is caught per row by the caller.
  special = __fmaf_rn(pos, f_leu(fabsf(u), thr), special);
  return code;
}

// One input row as a lane sees it: its 4 cells plus one cell either side (nodata already -inf), and the
// float32 differences between the row above and this row, formed when this row arrived.
struct DirRow {
  float v[NC + 2];    // columns xl-1 .. xl+NC
  float uS[NC];       // above[j+1] - v[j+1]   (cell j of the row above -> its S neighbour)
  float uSE[NC + 1];  // above[j]   - v[j+1]   (cell j-1 of the row above -> its SE neighbour)
  float uSW[NC + 1];  // above[j+1] - v[j]     (cell j of the row above -> its SW neighbour)
};

// a lane's NC cells of one row plus one cell either side, from the row's slice of the TMA box (q: the lane's first
// cell minus the 4-float apron)
__device__ __forceinline__ void dir_load_cells(const float* q, float* v) {
  v[0] = q[3];
  if (NC == 4) {
    const float4 m = *reinterpret_cast<const float4*>(q + 4);
    v[1] = m.x;
    v[2] = m.y;
    v[3] = m.z;
    v[NC] = m.w;
  } else {
    const float2 m = *reinterpret_cast<const float2*>(q + 4);
    v[1] = m.x;
    v[2] = m.y;
  }
  v[NC + 1] = q[4 + NC];
}

__device__ __forceinline__ void dir_store_codes(uint8_t* o, uint32_t packed, bool all_inside, int xl, int W) {
  if (all_inside) {
    if (NC == 4)
      *reinterpret_cast<uint32_t*>(o) = packed;
    else
      *reinterpret_cast<uint16_t*>(o) = (uint16_t)packed;
  } else {
#pragma unroll
    for (int j = 0; j < NC; ++j)
      if (xl + j < W) o[j] = (uint8_t)(packed >> (8 * j));
  }
}

struct DirWarp {
  float* tiles;     // this warp's ring of stages
  uint64_t* bars;   // one mbarrier per stage
  uint32_t g0;      // boxes consumed so far: stage = g % STAGES, parity = (g / STAGES) & 1
  int lane;
};

// One (band, chunk) work item of one warp.  EDGE: the band touches the raster's left or right edge, so
// columns outside the raster must be patched; interior bands skip those checks entirely.
template <bool EDGE>
__device__ __forceinline__ void direction_item(const CUtensorMap* tm, const DirParams& p, DirWarp& wp, int x0, int y0,
                                               int y1) {
  static_assert(DIR_RB % 2 == 0, "rows alternate between two register sets per box");
  const int lane = wp.lane;
  const float nd = p.nd;
  const int iy0 = y0 + p.y_off - 1;  // first input row this item reads
  const int n_in = (y1 - y0) + 2;
  const int nblk = (n_in + DIR_RB - 1) / DIR_RB;
  const int xl = x0 + NC * lane;  // first of this lane's NC columns
  float* const tiles = wp.tiles;
  uint64_t* const bars = wp.bars;
  const uint32_t g0 = wp.g0;

  auto issue = [&](int k) {
    const uint32_t s = (g0 + k) % DIR_STAGES;
    mbar_arrive_expect_tx(&bars[s], DIR_STAGE_BYTES);
    tma_load_2d(tiles + s * DIR_STAGE_FLOATS, tm, x0 - 4, iy0 + k * DIR_RB, &bars[s]);
  };
  // A box may be refilled only after the NEXT box has been consumed (the exact path re-reads up to two
  // rows back), so STAGES-1 boxes are in flight.
  if (lane == 0) {
    const int pre = min(DIR_STAGES - 1, nblk);
    for (int k = 0; k < pre; ++k) issue(k);
  }

  // raw row for the exact path (no NODATA transform): columns xl-1 .. xl+4 of the row `rel` rows below iy0,
  // still in its pipeline stage; positions outside the input array read as the fill value
  auto raw_row = [&](int rel, float* v) {
    const int iy = iy0 + rel;
    const uint32_t s = (g0 + rel / DIR_RB) % DIR_STAGES;
    const float* q = tiles + s * DIR_STAGE_FLOATS + (rel % DIR_RB) * DIR_BOXW + NC * lane;
    dir_load_cells(q, v);
    const bool row_out = iy < 0 || iy >= p.in_rows;
#pragma unroll
    for (int j = 0; j < NC + 2; ++j) {
      const int cx = xl - 1 + j;
      if (row_out || (EDGE && (cx < 0 || cx >= p.W))) v[j] = p.fill_raw;
    }
  };

  // row rr of the box at `t` into r.v; GUARD adds the out-of-array row check (first / last box only)
  auto load_row = [&](const float* t, int rr, int i, DirRow& r, bool guard) {
    dir_load_cells(t + rr * DIR_BOXW, r.v);
    if (guard && (iy0 + i < 0 || iy0 + i >= p.in_rows)) {
#pragma unroll
      for (int j = 0; j < NC + 2; ++j) r.v[j] = p.fillv;
    } else if (EDGE) {
#pragma unroll
      for (int j = 0; j < NC + 2; ++j) {
        const int cx = xl - 1 + j;
        if (cx < 0 || cx >= p.W) r.v[j] = p.fillv;
      }
    }
    bool any_nd = false;
#pragma unroll
    for (int j = 0; j < NC + 2; ++j) any_nd |= (r.v[j] == nd);
    if (any_nd) {
#pragma unroll
      for (int j = 0; j < NC + 2; ++j) r.v[j] = (r.v[j] == nd) ? -INFINITY : r.v[j];
    }
  };

  uint8_t* orow = p.out + (int64_t)y0 * p.ld_out + xl;  // next output row of this lane
  const bool full_store = xl + NC - 1 < p.W;

  // exact codes of the lane's four cells of input row i - 1 (output row y0 + i - 2), stored over the fast ones
  auto fixup = [&](int i) {
    float r0[NC + 2], r1[NC + 2], r2[NC + 2];
    raw_row(i - 2, r0);
    raw_row(i - 1, r1);
    raw_row(i, r2);
    uint32_t packed = 0;
#pragma unroll
    for (int j = 0; j < NC; ++j)
      packed |= d8_exact(r1[j + 1], /*E*/ r1[j + 2], /*NE*/ r0[j + 2], /*N*/ r0[j + 1], /*NW*/ r0[j], /*W*/ r1[j],
                         /*SW*/ r2[j], /*S*/ r2[j + 1], /*SE*/ r2[j + 2], nd)
                << (8 * j);
    dir_store_codes(p.out + (int64_t)(y0 + i - 2) * p.ld_out + xl, packed, !EDGE || full_store, xl, p.W);
  };

  // differences between row b (above) and the new row c; emits b's fast-path codes when b is an output row.
  // Returns non-zero when some cell of the row needs the exact path: the caller looks at that once per box
  // (fixup), so the rows of a box flow through without a branch on the end of each row's dependency chain.
  auto diffs_and_emit = [&](const DirRow& b, DirRow& c, bool emit) -> float {
#pragma unroll
    for (int j = 0; j < NC; ++j) c.uS[j] = __fsub_rn(b.v[j + 1], c.v[j + 1]);
#pragma unroll
    for (int j = 0; j < NC + 1; ++j) c.uSE[j] = __fsub_rn(b.v[j], c.v[j + 1]);
#pragma unroll
    for (int j = 0; j < NC + 1; ++j) c.uSW[j] = __fsub_rn(b.v[j + 1], c.v[j]);
    if (!emit) return 0.f;
    float hE[NC + 1];
#pragma unroll
    for (int j = 0; j < NC + 1; ++j) hE[j] = __fsub_rn(b.v[j], b.v[j + 1]);  // cell j-1 -> E
    float special = 0.f, code[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j)
      code[j] = d8_fast(/*E*/ hE[j + 1], /*NE*/ -b.uSW[j + 1], /*N*/ -b.uS[j], /*NW*/ -b.uSE[j], /*W*/ -hE[j],
                        /*SW*/ c.uSW[j], /*S*/ c.uS[j], /*SE*/ c.uSE[j + 1], special);
    // a centre that is NODATA (-inf by now) or not finite: one test for the lane's cells
    float csum = __fadd_rn(b.v[1], b.v[2]);
    if (NC == 4) csum = __fadd_rn(csum, __fadd_rn(b.v[3], b.v[NC]));
    special = __fadd_rn(special, f_leu(INFINITY, fabsf(csum)));
    // codes are 0..8: pack pairs exactly in float, then take the low 16 bits of (value + 2^23)
    const uint32_t lo = __float_as_uint(__fadd_rn(__fmaf_rn(code[1], 256.f, code[0]), 8388608.f));
    uint32_t packed = lo & 0xFFFFu;
    if (NC == 4) {
      const uint32_t hi = __float_as_uint(__fadd_rn(__fmaf_rn(code[NC - 1], 256.f, code[NC - 2]), 8388608.f));
      packed = __byte_perm(lo, hi, 0x5410);
    }
    dir_store_codes(orow, packed, !EDGE || full_store, xl, p.W);
    orow += p.ld_out;
    return special;
  };

  DirRow X[2];  // row i lives in X[i & 1]; indices are compile-time inside the unrolled box loop
#pragma unroll 1
  for (int k = 0; k < nblk; ++k) {
    const uint32_t s = (g0 + k) % DIR_STAGES;
    mbar_wait(&bars[s], ((g0 + k) / DIR_STAGES) & 1);
    const float* t = tiles + s * DIR_STAGE_FLOATS + NC * lane;
    const int ib = k * DIR_RB;
    float sp[DIR_RB];
    if (k > 0 && ib + DIR_RB <= n_in - 1) {
      // interior box: every row is inside the array and has a row above it that is an output row
#pragma unroll
      for (int rr = 0; rr < DIR_RB; ++rr) {
        load_row(t, rr, ib + rr, X[rr & 1], false);
        sp[rr] = diffs_and_emit(X[(rr + 1) & 1], X[rr & 1], true);
      }
    } else {
#pragma unroll
      for (int rr = 0; rr < DIR_RB; ++rr) {
        const int i = ib + rr;
        sp[rr] = 0.f;
        if (i < n_in) {
          load_row(t, rr, i, X[rr & 1], true);
          if (i >= 1) sp[rr] = diffs_and_emit(X[(rr + 1) & 1], X[rr & 1], i >= 2);
        }
      }
    }
    // special values are sums of non-negative terms: one test for the whole box, then row by row
    float sp_any = sp[0];
#pragma unroll
    for (int rr = 1; rr < DIR_RB; ++rr) sp_any = __fadd_rn(sp_any, sp[rr]);
    if (sp_any != 0.f) {
      uint32_t rows_mask = 0;
#pragma unroll
      for (int rr = 0; rr < DIR_RB; ++rr) rows_mask |= (sp[rr] != 0.f ? 1u : 0u) << rr;
#pragma unroll 1
      for (; rows_mask; rows_mask &= rows_mask - 1) fixup(ib + __ffs(rows_mask) - 1);
    }
    __syncwarp();
    // box k-1 is no longer needed by the exact path: its stage takes box k+STAGES-1
    if (lane == 0 && (k + DIR_STAGES - 1) < nblk) issue(k + DIR_STAGES - 1);
  }
  wp.g0 = g0 + nblk;
  __syncwarp();
}

__global__ void __launch_bounds__(DIR_WARPS * 32, OFL_DIR_CTAS_PER_SM) direction_kernel(const __grid_constant__ CUtensorMap tm,
                                                                    const DirParams p) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  const int warp = threadIdx.x >> 5;
  DirWarp wp;
  wp.lane = threadIdx.x & 31;
  wp.tiles = reinterpret_cast<float*>(smem_raw) + warp * (DIR_STAGES * DIR_STAGE_FLOATS);
  wp.bars = reinterpret_cast<uint64_t*>(smem_raw + size_t(DIR_WARPS) * DIR_STAGES * DIR_STAGE_BYTES) + warp * DIR_STAGES;
  wp.g0 = 0;
  if (wp.lane == 0) {
    tma_prefetch_desc(&tm);
#pragma unroll
    for (int s = 0; s < DIR_STAGES; ++s) mbar_init(&wp.bars[s], 1);
    mbar_fence_init();
  }
  __syncwarp();

  // Work items are handed out dynamically: a warp that drew cheap items (no NODATA fix-ups, faster DRAM
  // pages) simply takes more of them.  With a static round-robin the SMs were busy for only 67 % (16k^2)
  // to 83 % (64k^2) of the kernel's duration.  The next item is drawn while the current one is computed.
  const int gwarp = blockIdx.x * DIR_WARPS + warp;
  const int nwarps = gridDim.x * DIR_WARPS;
  const int n_items = p.n_bands * p.n_chunks;
  int item = gwarp;  // the first round needs no counter: it counts the items beyond the first nwarps
  while (item < n_items) {
    int next = 0;
    if (wp.lane == 0) next = nwarps + atomicAdd(p.next_item, 1);
    const int chunk = item / p.n_bands;
    const int band = item - chunk * p.n_bands;
    const int x0 = band * DIR_BAND;
    const int y0 = chunk * p.chunk_rows;
    const int y1 = min(y0 + p.chunk_rows, p.H);
    if ((x0 == 0) || (x0 + DIR_BAND + 1 > p.W))
      direction_item<true>(&tm, p, wp, x0, y0, y1);
    else
      direction_item<false>(&tm, p, wp, x0, y0, y1);
    item = __shfl_sync(0xffffffffu, next, 0);
  }
}

__global__ void fill_border_kernel(uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld, uint8_t value) {
  const int64_t n = 2 * (rows + cols);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r, c;
    if (i < cols) {
      r = 0;
      c = i;
    } else if (i < 2 * cols) {
      r = rows - 1;
      c = i - cols;
    } else if (i < 2 * cols + rows) {
      r = i - 2 * cols;
      c = 0;
    } else {
      r = i - 2 * cols - rows;
      c = cols - 1;
    }
    fdr[r * ld + c] = value;
  }
}

int launch_fill_border(uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld, int value, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return OFL_OK;
  const int64_t n = 2 * (rows + cols);
  const int blocks = (int)((n + 255) / 256 < 1024 ? (n + 255) / 256 : 1024);
  fill_border_kernel<<<blocks, 256, 0, st>>>(fdr, rows, cols, ld, (uint8_t)value);
  OFL_CHECK_LAUNCH();
  return OFL_OK;
}

// The DEMs one launch takes (in_rows >= rows): 30-bit sides, DirParams holds ints.
int direction_shape(int64_t in_rows, int64_t cols) {
  OFL_REQUIRE(in_rows < (1ll << 30) && cols < (1ll << 30), OFL_ERR_INVALID, "raster dimension too large");
  return OFL_OK;
}

// Device-pointer launcher.  `dem` has in_rows x cols floats; `fdr` has rows x cols codes;
// input row of output row y is y + y_off (0 for raster mode, 1 for a strip with halo rows).
int launch_direction(const float* dem, int64_t in_rows, int64_t cols, int64_t ld_dem, double nodata, uint8_t* fdr,
                     int64_t rows, int64_t ld_fdr, int y_off, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return OFL_OK;
  OFL_REQUIRE((reinterpret_cast<uintptr_t>(dem) & 15) == 0 && (ld_dem % 4) == 0 && ld_dem >= cols,
              OFL_ERR_ALIGNMENT, "dem must be 16-byte aligned with ld_dem %% 4 == 0 (ld_dem=%lld)", (long long)ld_dem);
  OFL_REQUIRE((reinterpret_cast<uintptr_t>(fdr) & 3) == 0 && (ld_fdr % 4) == 0 && ld_fdr >= cols, OFL_ERR_ALIGNMENT,
              "fdr must be 4-byte aligned with ld_fdr %% 4 == 0 (ld_fdr=%lld)", (long long)ld_fdr);
  CUtensorMap tm;
  int rc = make_tensor_map_2d(&tm, dem, 4, (uint64_t)cols, (uint64_t)in_rows, (uint64_t)ld_dem * 4, DIR_BOXW, DIR_RB, OFL_DIR_L2PROMO);
  if (rc != OFL_OK) return rc;

  DirParams p;
  p.out = fdr;
  p.ld_out = ld_fdr;
  p.H = (int)rows;
  p.W = (int)cols;
  p.y_off = y_off;
  p.in_rows = (int)in_rows;
  const float nd32 = (float)nodata;
  const bool representable = ((double)nd32 == nodata);  // false for NaN and for values float32 cannot hold
  p.nd = representable ? nd32 : NAN;
  p.fill_raw = nd32;  // util/raster.py:67 fills the out-of-raster halo with nodata cast to the band dtype
  p.fillv = representable ? -INFINITY : nd32;
  p.n_bands = (int)((cols + DIR_BAND - 1) / DIR_BAND);
  // rows per work item: items are drawn dynamically, so short items balance best (measured optimum 64 rows
  // at 4k..32k, 128 at 64k); longer ones only when a warp would otherwise draw hundreds of them, shorter
  // ones on rasters too small to give every warp a few
  const int sms = sm_count();
  const int64_t warps = (int64_t)sms * OFL_DIR_CTAS_PER_SM * DIR_WARPS;
  auto items_for = [&](int c) { return (int64_t)p.n_bands * ((rows + c - 1) / c); };
  int chunk_rows = 64;
  while (chunk_rows > 32 && items_for(chunk_rows) < warps * 4) chunk_rows >>= 1;
  while (chunk_rows < 512 && items_for(chunk_rows) > warps * 200) chunk_rows <<= 1;
  if (const char* e = getenv("OFL_DIR_CHUNK_ROWS")) chunk_rows = atoi(e) > 0 ? atoi(e) : chunk_rows;  // tuning
  p.chunk_rows = chunk_rows;
  p.n_chunks = (int)((rows + chunk_rows - 1) / chunk_rows);
  const int64_t n_items = (int64_t)p.n_bands * p.n_chunks;
  OFL_REQUIRE(n_items < (1ll << 31), OFL_ERR_INVALID, "too many work items");

  static std::atomic<int> attr_gen{-1};  // function attributes belong to the device they were set on
  if (attr_gen.load() != device_generation()) {
    OFL_CUDA(cudaFuncSetAttribute(direction_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DIR_SMEM_BYTES));
    attr_gen.store(device_generation());
  }
  int ctas = (int)((n_items + DIR_WARPS - 1) / DIR_WARPS);
  const int max_ctas = sms * OFL_DIR_CTAS_PER_SM;
  if (ctas > max_ctas) ctas = max_ctas;
  {
    // one work counter per launch, from a small ring (launches in flight at once are few)
    static std::atomic<unsigned> ring{0};
    void* ctr = nullptr;
    rc = scratch_get(SCRATCH_DIRCTR, 256 * sizeof(int), &ctr);
    if (rc != OFL_OK) return rc;
    p.next_item = static_cast<int*>(ctr) + (ring.fetch_add(1) % 256);
    // items 0 .. ctas * DIR_WARPS - 1 are taken by the warps' ids; the counter hands out the rest from 0
    OFL_CUDA(cudaMemsetAsync(p.next_item, 0, sizeof(int), st));
  }
  {
    PhaseScope ps(PHASE_DIRECTION, st);
    direction_kernel<<<ctas, DIR_WARPS * 32, DIR_SMEM_BYTES, st>>>(tm, p);
  }
  OFL_CHECK_LAUNCH();
  return OFL_OK;
}

}  // namespace ofl
