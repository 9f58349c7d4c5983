// accumulation.cu -- D8 flow accumulation (upstream cell counts) for sm_100a.
//
// Replaces single_tile_flow_accumulation / get_next_cell / follow_path
// (reference src/overflow/flow_accumulation.py:13-158; Barnes 2016, arXiv 1608.04431,
// Alg. 1 and 2, the paper cited at flow_accumulation.py:61,100).
//
// The reference walks a FIFO over the whole raster.  On a B200 the raster is far larger
// than on-chip memory and a global-memory queue would move >40 B/cell with atomics, so the
// sweep is organised the way the cited paper organises its tiles, with a CTA's shared memory
// as the "tile":
//
//   pass A  (acc_tile_kernel)  one CTA per 64x64 tile: TMA-load the codes plus a
//           one-cell halo, accumulate every flow path that stays inside the tile (frontier
//           propagation in shared memory: missing-upstream counts, one shared atomic per edge,
//           warp-ballot compacted frontier queues), follow the perimeter cells that can receive
//           inflow from outside the tile to where their path leaves it (Alg. 2), and emit the
//           reduced graph: the successor perimeter cell in the next tile, the locally accumulated
//           counts that cross the tile edge, and the solve's initial state.
//   solve   (pj_solve_kernel)        the reduced graph is a forest over ~2% of the cells;
//           subtree sums over it by pointer doubling: O(log depth) rounds of
//           "add my sum to my 2^j-th ancestor, then jump", integer atomics, exact; all rounds in one
//           persistent kernel (cooperative launch, grid barrier between rounds).
//   final   (acc_final_kernel)        per tile: tile-local counts (stored by pass A with the codes, 2 B/cell) plus
//           every perimeter cell's inflow from outside the tile added along its in-tile path;
//           writes the final int64 counts.
//
// HBM traffic per cell (ncu, 64k x 64k): 4.4 B in pass A (1 B codes, 2 B local counts + codes, the reduced graph),
// 1.3 B in the solve, 10.5 B in the final pass (2 + 0.5 read, 8 written; the codes come with the local counts)
// -- against 9 B/cell compulsory.  Long drainage chains cost O(log) rounds on the reduced graph instead of O(length) sweeps.
//
// Edge rule (flow_accumulation.py:116-124): u -> c is an edge iff code(u) in 0..7, c lies
// inside the raster and code(c) != 9.  Codes >= 8 have no downstream cell (the reference's
// out-of-bounds NEIGHBOR_OFFSETS read); NODATA cells end at -9998 (:119-121,129-137).
#include <atomic>
#include <cstdlib>

#include "common.cuh"
#include "tile_geometry.cuh"

namespace ofl {

constexpr int ACS_W = 96;              // code tile pitch: columns x0-16 .. x0+79 (TMA box inner = 96 B, 16-B aligned start)
constexpr int ACS_H = AT + 2;          // rows y0-1 .. y0+64
constexpr int ACS_X0 = 16;
constexpr int ACS_Y0 = 1;
constexpr uint32_t ACS_BYTES = ACS_W * ACS_H;
constexpr int ACC_THREADS = 256;
constexpr uint8_t CODE_OUTSIDE = 15;   // positions outside the raster (halo or partial tile)
constexpr uint8_t CODE_HALO_LIVE = 14; // halo cell that is a live (non-NODATA) cell of the next tile
constexpr uint8_t CODE_HALO_STRIP = 13; // halo cell that is a live cell of the neighbouring row strip (another GPU)

// node kinds, stored in link[] bits 8..9
constexpr uint16_t KIND_TERM = 0;        // path ends inside the raster (pit, or downstream is NODATA)
constexpr uint16_t KIND_TILE_EXIT = 1;   // path continues in the next tile (succ >= 0)
constexpr uint16_t KIND_RASTER_EXIT = 2; // path leaves the raster at the link cell
constexpr uint16_t KIND_STRIP_EXIT = 3;  // path continues in the neighbouring row strip (resolved by the strip exchange)

struct AccParams {
  int rows, cols;  // raster size
  int ntx, nty;    // tiles per row / column
  int32_t* succ;   // [ntiles*SLOTS] successor node or -1
  uint16_t* link;  // [ntiles*SLOTS] exit slot | kind << 8
  unsigned long long* S;  // [ntiles*SLOTS] pass A: base inflow; final pass: total inflow from outside the tile
  uint16_t* L;            // [ntiles][64*64] tile-local counts written by pass A, read by the final pass
  long long* fac;
  int64_t ld_fac;
  int* err;  // device flag: set to 1 when a cycle is detected
  // row-strip mode: the code raster has y_off halo rows above row 0 (and as many below the last row)
  // holding the neighbouring strips' rows; strip_above / strip_below say whether a strip exists there
  int y_off, strip_above, strip_below;
  int tile_base;  // first tile handled by this launch (blockIdx.x + tile_base)
  int vec_store;  // fac rows are 16-byte aligned: the final pass may use 16-byte stores
  int* wide_list;  // [0]: number of tiles the 32-bit final pass left to the 64-bit variant, [1..]: their ids
  int force_wide;  // test hook: send every tile with an inflow through the 64-bit variant
  // pass A publishes its slots straight into the solve's initial state (pointer buffers, cleared delta entries,
  // per-segment active lists); keep_succ: it also writes `succ`, from which a strip solves its forest a second time.
  // The host always sets fuse_init.  Removing it (and publish_slot's early return) changes the parameter block of
  // every kernel that takes AccParams, so that is left to the next measured change to pass A.
  int fuse_init, keep_succ;
  int trusted_codes;  // the codes come straight from direction_kernel (0..9 only): pass A skips its sanitising sweep
  int32_t *ptr_a, *ptr_b, *list0;
  unsigned long long *d0, *d1;
  int* counts0;
  int tiles_per_seg;
  long long seg;
};

// Result of Alg. 2 for one perimeter slot (all 32 lanes call; `mine`: this lane has a slot to publish).
__device__ __forceinline__ void publish_slot(const AccParams& p, int tile, bool mine, uint32_t slot, int32_t succ,
                                             uint32_t lt_mask, int lane) {
  const size_t u = (size_t)tile * SLOTS + slot;
  if (mine && p.keep_succ) p.succ[u] = succ;  // strips solve the same forest a second time, from `succ`
  if (!p.fuse_init) return;
  const bool active = mine && succ >= 0;
  if (active) {
    p.ptr_a[u] = succ;
    p.d0[u] = 0;
    p.d1[u] = 0;
  } else if (mine) {
    p.ptr_a[u] = ~(int32_t)u;
    p.ptr_b[u] = ~(int32_t)u;
  }
  const uint32_t bal = __ballot_sync(0xffffffffu, active);
  if (bal) {
    const int sidx = tile / p.tiles_per_seg;
    int base = 0;
    if (lane == 0) base = atomicAdd(&p.counts0[sidx], __popc(bal));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (active) p.list0[(size_t)sidx * p.seg + base + __popc(bal & lt_mask)] = (int32_t)u;
  }
}

// ---------------------------------------------------------------- in-tile frontier propagation
// Kahn's algorithm inside one 64x64 tile.  Every cell (plus a one-cell halo ring) owns one 32-bit word
//
//     [31 unused | 30..27 missing | 26 live | 25..24 unused | 23..20 code | 19..8 count | 7..0 downstream offset]
//
//   * offset   signed distance, in words, to the downstream cell's word (0: no downstream cell) -- a
//              step along a flow path is one sign-extension and one scaled add, no table, no code load;
//   * live     the cell is a data cell of this tile (code <= 8, inside the raster); halo and NODATA words
//              have it clear, so they absorb hand-offs but are never scheduled;
//   * missing  in-tile upstream neighbours that have not handed their count down yet;
//   * count    running sum of the upstream counts, the cell itself NOT included (tile-local counts are
//              <= 4096): the tile-local count of a finished cell is count + 1.  Twelve bits are enough for
//              every word of the tile: each cell hands down once, so what any one word absorbs is < 4096;
//   * code     the cell's direction code, only carried along: bytes 1..2 of the finished word are the
//              cell's entry in L (12-bit count, 4-bit code), which saves the final pass the code raster.
// A cell whose missing field is 0 is complete; it hands (count + 1) to its downstream cell with ONE
// shared-memory atomic add of ((count + 1) << 8) - (1 << 27): it adds the count and decrements the missing
// field at once, and the value the atomic returns tells the thread whether it was the last hand-off the
// downstream cell waited for -- and already holds that cell's offset and running sum.  Nothing is ever
// written back to the cell's own word.  No edge is ever skipped: hand-offs into the halo, into NODATA cells
// or out of the raster land in words nobody schedules.
// Frontier levels are consecutive segments of one queue of word addresses (a cell is appended at most once); level 0
// holds the sources that have a downstream cell (a source that flows nowhere needs no visit at all).  A lane whose
// hand-off completed the downstream cell goes on with that cell at once -- the atomic's return value plus what was
// added is its word -- for up to OFL_LEVEL_STEPS hand-offs per queue entry, and only what its last hand-off completes
// is queued: a "level" is three cells deep, which cuts the levels (two CTA barriers each) and the queue round trips
// by about that factor (pass A 15.8 -> 13.9 ms at 64k^2).  Halo
// words carry, in their offset byte, how a path that steps onto them continues (KIND_*).  A level never
// grows, so once it is down to TAIL_MAX cells one thread per cell simply follows its chain (it continues
// exactly when its hand-off completed the next cell): no queue, no barriers.
// (Measured in round 2 and dropped: handing the sources' constant down from the lanes that built them, without a
// queue round trip -- with the atomics' returned values to find level 1: same time on the fractal, 14 % slower on
// a tilted plane, where almost no cell is a source; as fire-and-forget reductions plus a rescan for level 1: 4 %
// slower -- ptxas wraps every predicated shared atomic in a branch, and unpredicated ones adding 0 from every
// lane cost atomic throughput.  No levels at all -- every lane walks its chain for as long as its hand-off completes
// the next cell and an idle lane draws the next source from the queue: 15 % slower on the fractal, 50 % on the tilted
// plane; the stragglers of eight warps cost more than the level loop's bookkeeping saves.  Source contraction --
// sources flagged in their code bytes, every cell pulls "upstream neighbours that are sources" with a second
// byte-parallel stencil, sources never visited, level 0 = what that completes: bit-exact, 17.1 ms against 16.25
// (17.5 with the stencil on every tile instead of tiles with >= 1200 sources): the stencil and its two barriers cost
// more than 2250 fewer visits per tile save.)
constexpr int WP = 72;                 // word-array pitch; cell x sits in column x + 4, so quads are 16-byte aligned
constexpr int WX0 = 4;
constexpr int WORDS = (AT + 2) * WP;   // rows y = -1..64
constexpr int QMAX = AT * AT;
constexpr uint32_t W_CNT_ONE = 1u << 8;
constexpr uint32_t W_LIVE = 1u << 26;
constexpr uint32_t W_MISS_ONE = 1u << 27;
constexpr uint32_t W_COUNT_MASK = 0xFFFu << 8;   // tile-local counts without the cell itself: <= 4095
constexpr uint32_t W_CODE_SHIFT = 20;            // bits 20..23: the cell's direction code, carried to the final pass
constexpr uint32_t W_HANDOFF_SELF = W_CNT_ONE - W_MISS_ONE;  // a hand-off adds (word & W_COUNT_MASK) + this: the cell itself, one upstream less
constexpr uint32_t W_MISSING_MASK = 0xFu << 27;     // the missing field: non-zero after the propagation = never completed
constexpr uint32_t W_READY_MASK = (0xFu << 27) | W_LIVE;     // hand-off result: the downstream cell is a live cell ...
constexpr uint32_t W_READY_VAL = W_MISS_ONE | W_LIVE;        // ... and this was the hand-off it was waiting for
// downstream word offsets per direction code E, NE, N, NW | W, SW, S, SE as signed bytes (PRMT lookup tables)
constexpr uint32_t W_TAB_LO = (uint32_t)(uint8_t)(1) | ((uint32_t)(uint8_t)(1 - WP) << 8) |
                              ((uint32_t)(uint8_t)(-WP) << 16) | ((uint32_t)(uint8_t)(-WP - 1) << 24);
constexpr uint32_t W_TAB_HI = (uint32_t)(uint8_t)(-1) | ((uint32_t)(uint8_t)(WP - 1) << 8) |
                              ((uint32_t)(uint8_t)(WP) << 16) | ((uint32_t)(uint8_t)(WP + 1) << 24);
#ifndef OFL_TAIL_MAX
#define OFL_TAIL_MAX 64
#endif
#ifndef OFL_WIDE_PER_LANE
#define OFL_WIDE_PER_LANE 2
#endif
#ifndef OFL_LEVEL_STEPS
// Hand-offs a lane makes per queue entry in the level loop: a lane whose hand-off completed the downstream cell goes on
// with that cell at once instead of queueing it, up to this many steps (1: every completed cell is queued).  Measured at
// 64k^2 (fractal; pass A alone): 1: 15.82 ms, 2: 14.24, 3: 14.03, 4: 13.95, 6: 14.45 -- fewer levels (two CTA barriers
// each) and fewer queue round trips against lanes idling through steps they do not take; the tilted plane is unchanged.
#define OFL_LEVEL_STEPS 3
#endif
constexpr int WIDE_PER_LANE = OFL_WIDE_PER_LANE;      // queue entries a lane visits per turn of the level loop
constexpr int TAIL_MAX = OFL_TAIL_MAX;  // switch to chain walking once a level has at most this many cells (with three steps per entry: 64: 13.92 ms, 128: 14.03, 256: 14.13)

// Shared memory (27.2 KB, eight CTAs per SM): the code tile is only read until the words are built, so the
// frontier queue takes over its bytes afterwards.
struct TileSmem {
  static constexpr int CS = 0;                 // codes + halo (TMA destination) ...
  static constexpr int Q = 0;                  // ... then the frontier queue
  static constexpr int WORD = QMAX * 2;        // 8192
  static constexpr int TAIL = WORD + WORDS * 4;  // [0] number of sources, [1] cells appended by the level loop, [2] paths to follow
  static constexpr int BAR = TAIL + 16;
  static constexpr int LIST = BAR + 16;        // perimeter slots whose path has to be followed (u8 each)
  static constexpr int BYTES = LIST + SLOTS;
};
static_assert(ACS_BYTES <= QMAX * 2, "code tile does not fit the slot it shares with the queue");
static_assert((WORDS * 4) % 16 == 0 && (WP * 4) % 16 == 0, "word rows must be whole uint4s");
static_assert(WORDS * 4 < 65536, "queue entries are 16-bit shared addresses of words");

__device__ __forceinline__ uint32_t lds32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t a) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ uint4 lds128(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t lds16(uint32_t a) {
  uint32_t v;
  asm volatile("{.reg .u16 t; ld.shared.u16 t, [%1]; cvt.u32.u16 %0, t;}" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t lds8(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t a, uint32_t v0, uint32_t v1, uint32_t v2, uint32_t v3) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v0), "r"(v1), "r"(v2), "r"(v3) : "memory");
}
__device__ __forceinline__ void sts16(uint32_t a, uint32_t v) {
  asm volatile("{.reg .u16 t; cvt.u16.u32 t, %1; st.shared.u16 [%0], t;}" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ void sts8(uint32_t a, uint32_t v) {
  asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t atoms_add(uint32_t a, uint32_t v) {
  uint32_t o;
  asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(o) : "r"(a), "r"(v) : "memory");
  return o;
}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}
// Shared-window base as an opaque value: the compiler keeps it in a register instead of re-deriving it
// (S2R SR_CgaCtaId + LEA) in front of every shared-memory access of the hot loops.
__device__ __forceinline__ uint32_t smem_base_opaque(const void* p) {
  uint32_t a;
  asm volatile("{ .reg .u64 t; cvta.to.shared.u64 t, %1; cvt.u32.u64 %0, t; }" : "=r"(a) : "l"(p));
  return a;
}
__device__ __forceinline__ uint32_t lanemask_lt() {
  uint32_t m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// per byte (all bytes < 16): 1 where the byte of `nb` differs from the code replicated in `pat`
__device__ __forceinline__ uint32_t bytes_differ(uint32_t nb, uint32_t pat) {
  return (((nb ^ pat) + 0x7F7F7F7Fu) >> 7) & 0x01010101u;
}

// shared address of the word the flow path steps to from the word `w` at address `aw` (w's offset byte != 0)
__device__ __forceinline__ uint32_t word_next(uint32_t aw, uint32_t w) {
  return aw + (uint32_t)((int32_t)(int8_t)(w & 0xFFu) * 4);
}

#ifndef OFL_ACC_MIN_CTAS
#define OFL_ACC_MIN_CTAS 8
#endif
__global__ void __launch_bounds__(ACC_THREADS, OFL_ACC_MIN_CTAS) acc_tile_kernel(const __grid_constant__ CUtensorMap tm,
                                                                const AccParams p) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  using SM = TileSmem;
  const uint32_t sb = smem_base_opaque(smem_raw);
  const uint32_t a_cs = sb + SM::CS;      // codes + halo (TMA destination), pitch ACS_W bytes
  const uint32_t a_word = sb + SM::WORD;  // per-cell words, halo-padded, pitch WP words
  const uint32_t a_q = sb + SM::Q;        // frontier queue: shared addresses of words, u16
  const uint32_t a_tail = sb + SM::TAIL;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + SM::BAR);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tile = blockIdx.x + p.tile_base;
  int y0, x0, h, w;
  tile_rect(tile, p.ntx, p.rows, p.cols, y0, x0, h, w);

  if (sb + SM::BYTES > 0x10000u) {  // the frontier queue holds shared addresses as 16-bit values
    if (tid == 0) atomicExch(p.err, 3);
    return;
  }
  if (tid == 0) {
    mbar_init(bar, 1);
    mbar_fence_init();
    mbar_arrive_expect_tx(bar, ACS_BYTES);
    tma_load_2d(smem_raw + SM::CS, &tm, x0 - ACS_X0, y0 - ACS_Y0 + p.y_off, bar);
    sts128(a_tail, 0, 0, 0, 0);
  }
  __syncthreads();
  mbar_wait(bar, 0);

  // ---- phase 0: invalid codes (>= 10) -> 8; halo ring: codes -> {9 nodata, 14 live} so it can never look
  //      like an in-tile upstream, words -> how a path stepping there continues; then in-tile positions
  //      outside the raster (TMA zero fill) -> CODE_OUTSIDE
  const int qx = lane & 15, rp = lane >> 4;
  constexpr int RWB = ACS_W;  // code row pitch in bytes
#pragma unroll
  for (int i = 0; i < 4 && !p.trusted_codes; ++i) {
    const int y = 8 * warp + 2 * i + rp;
    const uint32_t a = a_cs + (y + ACS_Y0) * RWB + ACS_X0 + 4 * qx;
    const uint32_t v = lds32(a);
    if ((v + 0x06060606u) & 0xF0F0F0F0u) {  // some byte >= 10: invalid input, behaves like "no downstream"
      uint32_t f = 0;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        uint32_t c = (v >> (8 * b)) & 0xFF;
        if (c >= 10) c = OFL_DIR_UNDEFINED;
        f |= c << (8 * b);
      }
      sts32(a, f);
    }
  }
  {
    // thread t < 256: side t >> 6 (top, bottom, left, right), position t & 63; the four threads with
    // position 0 also take one corner each
    const int side = tid >> AT_SHIFT, k = tid & (AT - 1);
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      int hy, hx;  // halo position in tile coordinates (-1..64)
      if (pass == 0) {
        hy = side == 0 ? -1 : side == 1 ? AT : k;
        hx = side == 2 ? -1 : side == 3 ? AT : k;
      } else {
        if (k != 0) break;
        hy = (side & 1) ? AT : -1;
        hx = (side & 2) ? AT : -1;
      }
      const uint32_t a = a_cs + (hy + ACS_Y0) * RWB + hx + ACS_X0;
      const int gy = y0 + hy, gx = x0 + hx;
      const bool nodata = lds8(a) == OFL_DIR_NODATA;
      uint32_t c, kind;
      if (gx < 0 || gx >= p.cols) {
        c = CODE_OUTSIDE;
        kind = KIND_RASTER_EXIT;
      } else if (gy < 0 || gy >= p.rows) {
        const bool strip = gy < 0 ? p.strip_above : p.strip_below;
        c = strip ? (nodata ? (uint32_t)OFL_DIR_NODATA : (uint32_t)CODE_HALO_STRIP) : (uint32_t)CODE_OUTSIDE;
        kind = strip ? (nodata ? KIND_TERM : KIND_STRIP_EXIT) : KIND_RASTER_EXIT;
      } else {
        c = nodata ? (uint32_t)OFL_DIR_NODATA : (uint32_t)CODE_HALO_LIVE;
        kind = nodata ? KIND_TERM : KIND_TILE_EXIT;
      }
      // the halo word (not live: absorbs hand-offs, never scheduled) keeps, in its offset byte, how a path
      // stepping onto it continues and which way the cell there flows (8: nowhere / not a cell)
      const uint32_t raw = lds8(a);
      const uint32_t hcode = (kind == KIND_RASTER_EXIT || raw > 8) ? 8u : raw;
      sts8(a, c);
      sts32(a_word + ((hy + 1) * WP + hx + WX0) * 4, kind | (hcode << 2));
    }
  }
  if (h < AT || w < AT) {
    // partial tile at the raster's bottom / right edge: in-tile positions beyond the raster
    __syncthreads();  // the word-wise sanitise above must not race with these byte stores
    for (int idx = tid; idx < AT * AT; idx += ACC_THREADS) {
      const int yy = idx >> AT_SHIFT, xx = idx & (AT - 1);
      if (yy >= h || xx >= w) sts8(a_cs + (yy + ACS_Y0) * RWB + xx + ACS_X0, CODE_OUTSIDE);
    }
  }
  __syncthreads();

  const uint32_t lt_mask = lanemask_lt();
  // the queue tail's address through a lane-dependent zero: ptxas then leaves the hand-aggregated queue
  // atomics alone instead of wrapping each in its own warp-aggregation sequence
  const uint32_t a_tail_v = a_tail + (lt_mask >> 31);
  const uint32_t a_word0 = a_word + (WP + WX0) * 4;       // word of cell (0,0)

  // ---- phase 1: missing-counts for four cells at a time (byte-parallel) and the four words.
  //      Lane owns the quads of columns 4*qx..4*qx+3 in rows 8*warp + 4*rp + i, i = 0..3.
  uint32_t srcs[4];
  // the lane's four quads sit below one another (rows 8 * warp + 4 * rp + i): a quad's middle and lower code rows
  // are the next quad's upper and middle ones, so a quad costs three loads instead of nine (quads two rows apart,
  // nine loads each: 16.03 ms against 15.82 at 64k^2)
  constexpr uint32_t AW_STEP = WP * 4;
  const uint32_t aw_lane = a_word0 + ((8 * warp + 4 * rp) * WP + 4 * qx) * 4;
  const uint32_t a_lane = a_cs + (8 * warp + 4 * rp + ACS_Y0) * RWB + ACS_X0 + 4 * qx;
  uint32_t L0 = lds32(a_lane - RWB - 4), C0 = lds32(a_lane - RWB), R0 = lds32(a_lane - RWB + 4);
  uint32_t L1 = lds32(a_lane - 4), C1 = lds32(a_lane), R1 = lds32(a_lane + 4);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t a = a_lane + i * RWB;
    const uint32_t L2 = lds32(a + RWB - 4), C2 = lds32(a + RWB), R2 = lds32(a + RWB + 4);
    // a neighbour flows into the cell iff its code is the direction pointing back at it
    uint32_t nm = bytes_differ(__funnelshift_r(C1, R1, 8), 0x04040404u);  // E neighbour flowing W
    nm += bytes_differ(__funnelshift_r(C0, R0, 8), 0x05050505u);          // NE neighbour flowing SW
    nm += bytes_differ(C0, 0x06060606u);                                  // N neighbour flowing S
    nm += bytes_differ(__funnelshift_r(L0, C0, 24), 0x07070707u);         // NW neighbour flowing SE
    nm += bytes_differ(__funnelshift_r(L1, C1, 24), 0x00000000u);         // W neighbour flowing E
    nm += bytes_differ(__funnelshift_r(L2, C2, 24), 0x01010101u);         // SW neighbour flowing NE
    nm += bytes_differ(C2, 0x02020202u);                                  // S neighbour flowing N
    nm += bytes_differ(__funnelshift_r(C2, R2, 8), 0x03030303u);          // SE neighbour flowing NW
    const uint32_t cnt4 = 0x08080808u - nm;  // missing upstream neighbours per cell
    const uint32_t dead = C1 + 0x77777777u;  // bit 7 of a byte set: code >= 9, not a data cell
    // source with a downstream cell: missing == 0 and own code <= 7 (a source that flows nowhere, or out of
    // nothing, needs no visit at all: nothing is ever written back to a finished cell)
    srcs[i] = ~((cnt4 + 0x7F7F7F7Fu) | (C1 + 0x78787878u)) & 0x80808080u;
    // the four words: offsets by a byte-wise table lookup on the codes (codes >= 8 select in PRMT's
    // sign-replicate mode: code 8 -> sign of +1 -> 0 = no downstream; code >= 9 -> garbage in a word that
    // is never scheduled), top bytes [missing << 3 | live << 2]; one PRMT assembles each word
    const uint32_t nib = C1 | (C1 >> 4);
    const uint32_t off4 = prmt(W_TAB_LO, W_TAB_HI, prmt(nib, 0u, 0x4420u));
    const uint32_t hi4 = (cnt4 << 3) | ((~dead >> 5) & 0x04040404u);
    // bytes 2 of the words: the code in the upper nibble (the count's lower 12 bits end below it and never carry:
    // every cell hands down once, so no word -- not even a NODATA cell's, which absorbs hand-offs -- sums past 4095)
    const uint32_t mid4 = (C1 << 4) & 0xF0F0F0F0u;
    const uint32_t hmA = prmt(mid4, hi4, 0x5140u), hmB = prmt(mid4, hi4, 0x7362u);  // [mid0 hi0 mid1 hi1], [mid2 hi2 mid3 hi3]
    sts128(aw_lane + i * AW_STEP, prmt(off4, hmA, 0x54D0u), prmt(off4, hmA, 0x76F1u), prmt(off4, hmB, 0x54D2u),
           prmt(off4, hmB, 0x76F3u));
    L0 = L1, C0 = C1, R0 = R1;
    L1 = L2, C1 = C2, R1 = R2;
  }
  __syncthreads();  // every word is built; the code tile is dead from here and the queue takes its place

  // ---- sources into the queue: one exclusive scan of the per-lane source counts, one queue atomic per warp
  {
    const uint32_t mine = __popc(srcs[0]) + __popc(srcs[1]) + __popc(srcs[2]) + __popc(srcs[3]);
    uint32_t incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    uint32_t base = 0;
    if (lane == 31) base = atoms_add(a_tail_v, incl);
    base = __shfl_sync(0xffffffffu, base, 31);
    uint32_t aq = a_q + 2 * (base + incl - mine);
    const uint32_t qv = aw_lane;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        if (srcs[i] & (0x80u << (8 * b))) {
          sts16(aq, qv + i * AW_STEP + 4 * b);
          aq += 2;
        }
      }
    }
  }
  // ---- Alg. 2, part 1 (words are static from here on in everything it reads).  Thread = perimeter slot.
  //      A perimeter cell's path only has to be followed when something can arrive at the cell from outside
  //      the tile -- a neighbouring tile's (or strip's) cell flows into it -- or when the cell lies on the
  //      raster's (strip's) edge, whose links the callers ask for.  Those slots are compacted into a list;
  //      every other slot gets its final "no successor" entry right away.
  int32_t own_target = -1;
  uint32_t a_own;
  {
    const int side = tid >> AT_SHIFT, k = tid & (AT - 1);
    const int py = side == 0 ? 0 : side == 1 ? h - 1 : k;
    const int px = side == 2 ? 0 : side == 3 ? w - 1 : k;
    const bool valid = side < 2 ? (k < w && (side == 0 || h > 1)) : (k > 0 && k < h - 1 && (side == 2 || w > 1));
    a_own = a_word0 + (py * WP + px) * 4;
    const uint32_t w_own = lds32(a_own);
    const bool live = valid && (w_own & W_LIVE);
    // Does a cell outside the tile flow into this one?  The three candidates of a side sit next to each
    // other on the halo row / column facing it: word hb + {+1, 0, -1} * step, and the codes that point back
    // at this cell are three consecutive ones.  (On the cut sides of a partial tile this looks at halo
    // words beyond the raster, which flow nowhere; those cells are raster-edge cells anyway.)
    const int hb = side == 0 ? WX0 + k : side == 1 ? (AT + 1) * WP + WX0 + k : (k + 1) * WP + (side == 2 ? WX0 - 1 : WX0 + AT);
    const int step = ((side == 0 || side == 3) ? 1 : -1) * (side < 2 ? 1 : WP);
    const uint32_t back0 = (0x3715u >> (4 * side)) & 7u;  // sides top, bottom, left, right: SW, NE, SE, NW first
    const uint32_t ah = a_word + hb * 4;
    bool target = (lds8(ah + step * 4) >> 2) == back0;
    target |= (lds8(ah) >> 2) == ((back0 + 1) & 7u);
    target |= (lds8(ah - step * 4) >> 2) == ((back0 + 2) & 7u);
    if (side < 2 && (k == 0 || k == w - 1)) {  // corner: the two directions of the adjoining side
      auto inflow = [&](int d) -> bool {
        const int ny = py + dir_dy(d), nx = px + dir_dx(d);
        if ((uint32_t)ny < (uint32_t)AT && (uint32_t)nx < (uint32_t)AT) return false;
        return (lds8(a_word + ((ny + 1) * WP + nx + WX0) * 4) >> 2) == (uint32_t)((d + 4) & 7);
      };
      const int e = k == 0 ? 4 : 0;
      target |= inflow(e) | inflow(k == 0 ? (side == 0 ? 5 : 3) : (side == 0 ? 7 : 1));
    }
    const int gy = y0 + py, gx = x0 + px;
    const bool edge = gy == 0 || gy == p.rows - 1 || gx == 0 || gx == p.cols - 1;
    // the cell's own edge across the tile boundary carries its local count to the next tile
    if (live && (w_own & 0xFFu)) {
      const uint32_t an = word_next(a_own, w_own);
      const uint32_t wn = lds32(an);
      const int jn = (int)(an - a_word) >> 2;
      const int ny = jn / WP - 1, nx = jn - (ny + 1) * WP - WX0;
      if (!((uint32_t)ny < (uint32_t)AT && (uint32_t)nx < (uint32_t)AT) && (wn & 3u) == KIND_TILE_EXIT)
        own_target = node_of_cell(y0 + ny, x0 + nx, p.rows, p.cols, p.ntx);
    }
    const bool follow = live && (target || edge);
    const uint32_t bal = __ballot_sync(0xffffffffu, follow);
    uint32_t lb = 0;
    if (lane == 0 && bal) lb = atoms_add(a_tail_v + 8, __popc(bal));
    lb = __shfl_sync(0xffffffffu, lb, 0);
    if (follow) {
      sts8(sb + SM::LIST + lb + __popc(bal & lt_mask), tid);
    } else {
      p.link[(size_t)tile * SLOTS + tid] = (uint16_t)((valid ? tid : 0) | (KIND_TERM << 8));
    }
    publish_slot(p, tile, !follow, tid, -1, lt_mask, lane);
  }
  __syncthreads();

  // ---- wide levels: level k is q[lo, hi); processing it appends level k+1 right after it.  A warp takes
  //      WIDE_PER_LANE * 32 entries per turn and reserves queue slots for everything they complete with
  //      one atomic.  Queue entries are the 16-bit shared addresses of the words themselves.
  const uint32_t n_src = lds32(a_tail);  // level 1; final: the level loop appends through the second counter
  uint32_t lo = 0, hi = n_src;
  // the complete cell whose word sits at `aw` hands its count down; returns the hand-off's result (0: there
  // was none) and the address of the downstream word
  uint32_t add_[WIDE_PER_LANE];
  auto visit = [&](uint32_t aw, uint32_t& an, uint32_t& add) -> uint32_t {
    const uint32_t wv = lds32(aw);
    if (!(wv & 0xFFu)) return 0;
    an = word_next(aw, wv);
    add = (wv & W_COUNT_MASK) + W_HANDOFF_SELF;
    return atoms_add(an, add);
  };
  while (hi - lo > TAIL_MAX) {
    for (uint32_t base = lo + 32 * WIDE_PER_LANE * warp; base < hi; base += WIDE_PER_LANE * ACC_THREADS) {
      uint32_t old[WIDE_PER_LANE], an[WIDE_PER_LANE];
      if (base + 32 * WIDE_PER_LANE <= hi) {  // a full turn: no per-entry bounds checks
#pragma unroll
        for (int e = 0; e < WIDE_PER_LANE; ++e) {
          an[e] = 0;
          old[e] = visit(lds16(a_q + 2 * (base + 32 * e + lane)), an[e], add_[e]);
        }
      } else {
#pragma unroll
        for (int e = 0; e < WIDE_PER_LANE; ++e) {
          const uint32_t i = base + 32 * e + lane;
          old[e] = 0;  // reads as "nothing completed"
          an[e] = 0;
          if (i < hi) old[e] = visit(lds16(a_q + 2 * i), an[e], add_[e]);
        }
      }
      // a lane whose hand-off completed the downstream cell goes on with that cell at once (the atomic's return
      // value plus what was added IS its word) for up to OFL_LEVEL_STEPS - 1 more steps; only what the last step
      // completes is appended.  A completed cell without a downstream cell needs no visit and is not appended.
#pragma unroll
      for (int s = 1; s < OFL_LEVEL_STEPS; ++s) {
#pragma unroll
        for (int e = 0; e < WIDE_PER_LANE; ++e) {
          if ((old[e] & W_READY_MASK) == W_READY_VAL) {
            const uint32_t wv = old[e] + add_[e];
            old[e] = 0;
            if (wv & 0xFFu) {
              an[e] = word_next(an[e], wv);
              add_[e] = (wv & W_COUNT_MASK) + W_HANDOFF_SELF;
              old[e] = atoms_add(an[e], add_[e]);
            }
          }
        }
      }
      uint32_t bal[WIDE_PER_LANE], total = 0;
#pragma unroll
      for (int e = 0; e < WIDE_PER_LANE; ++e) {
        bal[e] = __ballot_sync(0xffffffffu, (old[e] & W_READY_MASK) == W_READY_VAL);
        total += __popc(bal[e]);
      }
      if (total) {
        uint32_t qb = 0;
        if (lane == 0) qb = atoms_add(a_tail_v + 4, total);
        qb = n_src + __shfl_sync(0xffffffffu, qb, 0);
#pragma unroll
        for (int e = 0; e < WIDE_PER_LANE; ++e) {
          if (bal[e] & (1u << lane)) sts16(a_q + 2 * (qb + __popc(bal[e] & lt_mask)), an[e]);
          qb += __popc(bal[e]);
        }
      }
    }
    __syncthreads();
    const uint32_t nh = n_src + lds32(a_tail + 4);
    __syncthreads();  // nobody appends to the next level before everyone has read where this one ends
    lo = hi;
    hi = nh;
  }
  // ---- narrow tail (a level never grows): one thread per frontier cell follows its chain for as long
  //      as its hand-off is the one that completes the next cell; no queue, no barriers.  The atomic's
  //      return value already is the next cell's word, so a step is one atomic.
  for (uint32_t i = lo + tid; i < hi; i += ACC_THREADS) {
    uint32_t aw = lds16(a_q + 2 * i);
    uint32_t wv = lds32(aw);
    for (;;) {
      if (!(wv & 0xFFu)) break;
      aw = word_next(aw, wv);
      const uint32_t add = (wv & W_COUNT_MASK) + W_HANDOFF_SELF;
      const uint32_t old = atoms_add(aw, add);
      if ((old & W_READY_MASK) != W_READY_VAL) break;
      wv = old + add;
    }
  }

  // ---- Alg. 2, part 2: follow the listed paths to where they leave the tile, one thread per path, taken
  //      from the high thread ids (the chain walking above keeps the low ones busy).  Only offset bytes and
  //      live bits are read, which never change, so this runs while other warps still finish their chains.
  {
    const uint32_t t = ACC_THREADS - 1 - tid;
    const bool walker = t < lds32(a_tail + 8);
    uint32_t slot = 0, aw = 0, an = 0, wn = 0;
    bool exited = false;
    int steps = 0;
    if (walker) {
      slot = lds8(sb + SM::LIST + t);
      const int side = slot >> AT_SHIFT, k = slot & (AT - 1);
      const int py = side == 0 ? 0 : side == 1 ? h - 1 : k;
      const int px = side == 2 ? 0 : side == 3 ? w - 1 : k;
      aw = a_word0 + (py * WP + px) * 4;
      uint32_t wv = lds32(aw);
      while (wv & 0xFFu) {
        an = word_next(aw, wv);
        wn = lds32(an);
        if (!(wn & W_LIVE)) {
          exited = true;
          break;
        }
        if (++steps > AT * AT) {
          atomicExch(p.err, 2);  // ran out of steps: cycle inside the tile
          break;
        }
        aw = an;
        wv = wn;
      }
    }
    __syncwarp();  // classify once per warp, not once per exit path
    int32_t succ = -1;
    if (walker) {
      // aw: the last live in-tile cell of the path; an / wn: the word it steps to when the path leaves
      const int j = (int)(aw - a_word) >> 2;
      const int cy = j / WP - 1, cx = j - (cy + 1) * WP - WX0;
      uint32_t kind = KIND_TERM;
      if (exited) {
        const int jn = (int)(an - a_word) >> 2;
        const int ny = jn / WP - 1, nx = jn - (ny + 1) * WP - WX0;
        if ((uint32_t)ny < (uint32_t)AT && (uint32_t)nx < (uint32_t)AT) {
          // a dead in-tile cell: NODATA (the path ends in front of it) or beyond the raster's edge
          kind = (ny < h && nx < w) ? KIND_TERM : KIND_RASTER_EXIT;
        } else {
          kind = wn & 3u;  // the halo word says how the path continues
          if (kind == KIND_TILE_EXIT) succ = node_of_cell(y0 + ny, x0 + nx, p.rows, p.cols, p.ntx);
        }
      }
      const int ls = slot_of(cy, cx, h, w);
      p.link[(size_t)tile * SLOTS + slot] = (uint16_t)((ls < 0 ? 0 : ls) | (kind << 8));
    }
    publish_slot(p, tile, walker, slot, succ, lt_mask, lane);
  }
  __syncthreads();  // all chains are finished: counts are final

  if (own_target >= 0) atomicAdd(&p.S[own_target], (unsigned long long)(((lds32(a_own) >> 8) & 0xFFFu) + 1u));
  // tile-local counts (<= 4096, fit 16 bits) for the final pass: tile-major, a warp stores 256 contiguous bytes
  uint2* Lt = reinterpret_cast<uint2*>(p.L + (size_t)tile * (AT * AT));
  uint32_t pending = 0;
#pragma unroll
  for (int g = tid; g < AT * AT / 4; g += ACC_THREADS) {
    const uint4 v = lds128(a_word0 + ((g >> 4) * WP + (g & 15) * 4) * 4);
    // A word of the tile that still misses a hand-off.  Looking at the live words alone is not necessary: a word
    // that is not live (NODATA, beyond the raster) counts the live cells of the tile that flow into it, all of
    // which hand down to it once they are complete, so its field is zero as well unless one of THEM never
    // completed -- and that cell's own field is then non-zero too.  Two ORs per four words instead of a table
    // look-up per word.
    pending |= v.x | v.y;
    pending |= v.z | v.w;
    // bytes 1..2 of a word: the running sum (12 bits, the cell itself not included) and the cell's code above it
    Lt[g] = make_uint2(prmt(v.x, v.y, 0x6521u), prmt(v.z, v.w, 0x6521u));
  }
  if (pending & W_MISSING_MASK) atomicExch(p.err, 1);  // a cell never completed: the raster holds a cycle
}

// ---------------------------------------------------------------- final pass
// fac(v) = L(v) + sum of the inflows I(e) of the perimeter cells e whose in-tile path runs through v.
// Pass A left L (tile-local counts) in HBM and the solve left I(e) in S, so the final pass only has to
// add every non-zero inflow along its path and write the tile out as int64 (10.5 B/cell of HBM traffic).  The
// codes come with L (4 bits on top of each 12-bit count), so the code raster is not read a second time.
//   * the perimeter slots with a non-zero inflow are compacted onto whole warps; a step of a path is one
//     shared atomic on the cell's count, one byte load of the next cell's code and two PRMT table lookups;
//   * the code tile is the exact 64 x 64 box (4 KB, unpacked from L); a step that would leave the tile (or the raster, on a
//     partial tile) is caught by the column and the cell index going out of range;
//   * counts are accumulated in 32 bits (23 KB of shared memory, eight CTAs per SM).  A tile in which an
//     inflow or a sum does not fit 32 bits -- possible only on rasters of more than 2^32 cells' worth of
//     drainage -- is put on a list instead of being written, and redone by the WIDE variant (64-bit).
struct FinalSmem {
  static constexpr int CS = 0;                       // codes (unpacked from L), pitch AT
  static constexpr int LO = AT * AT;                 // low words of the counts, pitch AT
  static constexpr int SEED = LO + AT * AT * 4;      // 64-bit inflow of every listed path
  static constexpr int LIST = SEED + SLOTS * 8;      // slots of the listed paths (u8)
  static constexpr int CNT = LIST + SLOTS;           // number of listed paths
  static constexpr int BAR = CNT + 16;
  static constexpr int HI = BAR + 16;                // high words (WIDE only)
  static constexpr int BYTES_FAST = HI;
  static constexpr int BYTES_WIDE = HI + AT * AT * 4;
};
// per direction code E, NE, N, NW | W, SW, S, SE: cell-index offset (dy * 64 + dx) and column offset
constexpr uint32_t F_TABI_LO = (uint32_t)(uint8_t)(1) | ((uint32_t)(uint8_t)(1 - AT) << 8) |
                               ((uint32_t)(uint8_t)(-AT) << 16) | ((uint32_t)(uint8_t)(-AT - 1) << 24);
constexpr uint32_t F_TABI_HI = (uint32_t)(uint8_t)(-1) | ((uint32_t)(uint8_t)(AT - 1) << 8) |
                               ((uint32_t)(uint8_t)(AT) << 16) | ((uint32_t)(uint8_t)(AT + 1) << 24);
constexpr uint32_t F_TABX_LO = 0xFF000101u;  // dx of E, NE, N, NW = +1, +1, 0, -1
constexpr uint32_t F_TABX_HI = 0x0100FFFFu;  // dx of W, SW, S, SE = -1, -1, 0, +1

// One tile.  Returns true (fast variant only) when the tile needs the 64-bit variant; nothing has been
// written to fac in that case.
template <bool WIDE>
__device__ __forceinline__ bool final_tile(const AccParams& p, int tile, uint32_t sb) {
  using SM = FinalSmem;
  const uint32_t a_cs0 = sb + SM::CS, a_lo = sb + SM::LO, a_hi = sb + SM::HI;  // a_cs0: code of cell (0,0), pitch AT
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  int y0, x0, h, w;
  tile_rect(tile, p.ntx, p.rows, p.cols, y0, x0, h, w);

  if (tid == 0) sts32(sb + SM::CNT, 0);
  // tile-local counts with the codes on top (pass A: 12 + 4 bits per cell) and this thread's perimeter inflow
  const uint4* Lt = reinterpret_cast<const uint4*>(p.L + (size_t)tile * (AT * AT));
  const uint4 q0 = Lt[tid], q1 = Lt[tid + ACC_THREADS];
  const int side = tid >> AT_SHIFT, k = tid & (AT - 1);
  const bool valid = side < 2 ? (k < w && (side == 0 || h > 1)) : (k > 0 && k < h - 1 && (side == 2 || w > 1));
  unsigned long long seed = 0;
  if (valid) seed = p.S[(size_t)tile * SLOTS + tid];
  __syncthreads();

#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const uint4 q = r ? q1 : q0;
    const uint32_t o = (tid + r * ACC_THREADS) * 32;
    sts128(a_lo + o, (q.x & 0xFFFu) + 1u, ((q.x >> 16) & 0xFFFu) + 1u, (q.y & 0xFFFu) + 1u, ((q.y >> 16) & 0xFFFu) + 1u);
    sts128(a_lo + o + 16, (q.z & 0xFFFu) + 1u, ((q.z >> 16) & 0xFFFu) + 1u, (q.w & 0xFFFu) + 1u, ((q.w >> 16) & 0xFFFu) + 1u);
    // the eight codes as bytes (the path walk and the NODATA test below read them from the code tile)
    const uint32_t c01 = (q.x >> 12) & 0x000F000Fu, c23 = (q.y >> 12) & 0x000F000Fu;
    const uint32_t c45 = (q.z >> 12) & 0x000F000Fu, c67 = (q.w >> 12) & 0x000F000Fu;
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a_cs0 + (tid + r * ACC_THREADS) * 8), "r"(prmt(c01, c23, 0x6420u)),
                 "r"(prmt(c45, c67, 0x6420u))
                 : "memory");
    if (WIDE) {
      sts128(a_hi + o, 0, 0, 0, 0);
      sts128(a_hi + o + 16, 0, 0, 0, 0);
    }
  }
  bool wide_needed = false;
  {
    // compact the slots with a non-zero inflow
    const bool has = seed != 0;
    const uint32_t bal = __ballot_sync(0xffffffffu, has);
    uint32_t lb = 0;
    if (lane == 0 && bal) lb = atoms_add(sb + SM::CNT + (lanemask_lt() >> 31), __popc(bal));
    lb = __shfl_sync(0xffffffffu, lb, 0);
    if (has) {
      const uint32_t pos = lb + __popc(bal & lanemask_lt());
      sts8(sb + SM::LIST + pos, tid);
      asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(sb + SM::SEED + 8 * pos), "r"((uint32_t)seed),
                   "r"((uint32_t)(seed >> 32))
                   : "memory");
      if (!WIDE && ((seed >> 32) || p.force_wide)) wide_needed = true;
    }
  }
  __syncthreads();

  {
    // one thread per listed path, from the high thread ids down
    const uint32_t t = ACC_THREADS - 1 - tid;
    if (t < lds32(sb + SM::CNT)) {
      const uint32_t slot = lds8(sb + SM::LIST + t);
      const uint2 sd = lds64(sb + SM::SEED + 8 * t);
      const int ss = slot >> AT_SHIFT, sk = slot & (AT - 1);
      const int y = ss == 0 ? 0 : ss == 1 ? h - 1 : sk;
      int x = ss == 2 ? 0 : ss == 3 ? w - 1 : sk;
      uint32_t idx = y * AT + x;  // cell index: code at a_cs0 + idx, count at a_lo + 4 * idx
      uint32_t code = lds8(a_cs0 + idx);
      if (WIDE || (sd.y == 0 && !p.force_wide)) {
        for (int steps = 0; steps <= AT * AT; ++steps) {
          const uint32_t old = atoms_add(a_lo + 4 * idx, sd.x);
          const bool carry = (old + sd.x) < old;
          if (WIDE) {
            const uint32_t hadd = sd.y + (carry ? 1u : 0u);
            if (hadd) atoms_add(a_hi + 4 * idx, hadd);
          } else {
            wide_needed |= carry;
          }
          if (code >= 8) break;  // pit / flat / invalid: no downstream cell
          const uint32_t sel = code * 0x1111u + 0x8880u;  // byte 0: table entry, bytes 1..3: its sign
          x += (int)prmt(F_TABX_LO, F_TABX_HI, sel);
          idx += prmt(F_TABI_LO, F_TABI_HI, sel);
          if ((uint32_t)x >= (uint32_t)w || idx >= (uint32_t)(h * AT)) break;  // leaves the tile (or the raster)
          code = lds8(a_cs0 + idx);
          if (code == OFL_DIR_NODATA) break;  // no edge into a NODATA cell
        }
      }
    }
  }
  if (__syncthreads_or(wide_needed) && !WIDE) return true;

  // final counts: each lane writes two adjacent cells as one 16-byte store, a warp one 512-byte row per
  // instruction; NODATA cells get -9998
  const uint32_t xx = 2 * lane;
  long long* orow = p.fac + (int64_t)(y0 + 8 * warp) * p.ld_fac + x0 + xx;
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int yy = 8 * warp + r;
    if (yy < h && (int)xx < w) {
      const uint32_t oo = (yy * AT + xx) * 4;
      const uint2 lo2 = lds64(a_lo + oo);
      uint2 hi2 = make_uint2(0, 0);
      if (WIDE) hi2 = lds64(a_hi + oo);
      const uint32_t c2 = lds16(a_cs0 + yy * AT + xx);
      long long v0 = (long long)(((unsigned long long)hi2.x << 32) | lo2.x);
      long long v1 = (long long)(((unsigned long long)hi2.y << 32) | lo2.y);
      if ((c2 & 0xFF) == OFL_DIR_NODATA) v0 = OFL_FAC_NODATA_EMITTED;
      if ((c2 >> 8) == OFL_DIR_NODATA) v1 = OFL_FAC_NODATA_EMITTED;
      if ((int)xx + 1 < w && p.vec_store) {
        *reinterpret_cast<longlong2*>(orow) = make_longlong2(v0, v1);
      } else {
        orow[0] = v0;
        if ((int)xx + 1 < w) orow[1] = v1;
      }
    }
    orow += p.ld_fac;
  }
  return false;
}

__global__ void __launch_bounds__(ACC_THREADS) acc_final_kernel(const AccParams p) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  const uint32_t sb = smem_base_opaque(smem_raw);
  const int tile = blockIdx.x + p.tile_base;
  if (final_tile<false>(p, tile, sb) && threadIdx.x == 0) p.wide_list[1 + atomicAdd(p.wide_list, 1)] = tile;
}

// The tiles the 32-bit variant gave up on (normally none): a small persistent grid walks the list.
__global__ void __launch_bounds__(ACC_THREADS) acc_final_wide_kernel(const AccParams p) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  const uint32_t sb = smem_base_opaque(smem_raw);
  const int n = p.wide_list[0];
  for (int i = blockIdx.x; i < n; i += gridDim.x) {
    final_tile<true>(p, p.wide_list[1 + i], sb);
    __syncthreads();  // the next tile overwrites the codes and counts this tile's output rows still read
  }
}

// ---------------------------------------------------------------- reduced-graph solve
// Subtree sums over the perimeter forest by pointer doubling, restricted to the nodes that still have
// an ancestor to jump to.  ptr[u] >= 0: u's 2^j-th ancestor.  ptr[u] < 0: ~root(u), chain exhausted.
// Round j, for every ACTIVE node w: S_j[w] is added to its 2^j-th ancestor a (through alternating delta
// buffers d0/d1 while a is itself still jumping, so a node only ever forwards sums that were complete
// before the round; directly into S[a] once a's chain is exhausted), then w jumps to a's pointer.  A
// node whose jump finds an exhausted chain retires: it is dropped from the active list and, one round
// later, its root is copied into the other ping-pong buffer and its last deltas are flushed into S.
// The node array is cut into one segment per CTA; each CTA keeps the active nodes of its segment
// compacted at the front of the segment (retirees at the back) of a ping-pong list, so compaction needs
// only shared-memory atomics and the work per round is proportional to the active nodes, which shrink
// geometrically on real terrain.
struct PjSeg {
  int64_t n;        // nodes
  int64_t seg;      // nodes per CTA segment (multiple of 32)
  int blocks;       // CTAs == segments
};

__device__ __forceinline__ void block_append(int32_t* seg_list, int* s_counter, bool pred, int32_t value, bool from_back,
                                             int64_t seg_len) {
  const uint32_t bal = __ballot_sync(0xffffffffu, pred);
  if (!bal) return;
  const int lane = threadIdx.x & 31, leader = __ffs(bal) - 1;
  int base = 0;
  if (lane == leader) base = atomicAdd(s_counter, __popc(bal));
  base = __shfl_sync(0xffffffffu, base, leader);
  if (pred) {
    const int64_t pos = base + __popc(bal & ((1u << lane) - 1));
    seg_list[from_back ? seg_len - 1 - pos : pos] = value;
  }
}

// One persistent kernel runs every round (cooperative launch: all CTAs are resident, one per segment); a
// grid-wide barrier separates the rounds and carries the number of nodes still active or just retired, so the
// kernel ends after the round that finds none -- O(log depth) rounds instead of the O(log n) a fixed
// sequence of launches has to provide for, and no launch latency between them (on a strip of an 8-GPU run
// a round is a few microseconds of work).  Everything other CTAs write between barriers is read with
// ld.global.cg (L2), never through L1.
struct PjArgs {
  const int32_t* succ;   // with_init: the forest (succ[u] = parent or -1)
  int32_t *ptr_a, *ptr_b;
  int32_t* lists;        // 2 ping-pong lists of blocks * seg entries
  const int* counts0;    // !with_init: [blocks] active nodes per segment, published by pass A
  unsigned long long *S, *d0, *d1;
  unsigned* sync;        // [0..1] grid barrier, [2 + j] nodes left after round j; zeroed before the launch
  int* leftover;         // set when max_rounds did not suffice: the forest has a cycle
  const int* run_flag;   // nullable: the whole solve is skipped (by every CTA alike) when this device word is 0
  PjSeg g;
  int with_init, max_rounds;
};

__global__ void __launch_bounds__(256, 8) pj_solve_kernel(const PjArgs a) {
  __shared__ int s_keep, s_ret;
  if (a.run_flag && *a.run_flag == 0) return;  // written by an earlier kernel: every CTA sees the same value
  const PjSeg g = a.g;
  const int64_t base = (int64_t)blockIdx.x * g.seg;
  int32_t* const list0 = a.lists + base;
  int32_t* const list1 = a.lists + (int64_t)g.blocks * g.seg + base;
  unsigned generation = 0;
  int n_active, n_retired = 0;
  if (threadIdx.x == 0) {
    s_keep = 0;
    s_ret = 0;
  }
  __syncthreads();
  if (a.with_init) {
    // the active nodes of this segment, their pointers, and cleared delta entries: deltas are only ever
    // written for a node that still has a pointer to jump along, i.e. one that starts out active
    const int64_t len = min(g.seg, g.n - base);
    for (int64_t i = threadIdx.x; i < g.seg; i += blockDim.x) {  // whole warps stay together for the ballots
      bool active = false;
      const int64_t u = base + i;
      if (i < len) {
        const int32_t sc = a.succ[u];
        active = sc >= 0;
        if (active) {
          a.ptr_a[u] = sc;
          a.d0[u] = 0;
          a.d1[u] = 0;
        } else {
          a.ptr_a[u] = ~(int32_t)u;
          a.ptr_b[u] = ~(int32_t)u;
        }
      }
      block_append(list0, &s_keep, active, (int32_t)u, false, g.seg);
    }
    grid_barrier(a.sync, generation);  // round 0 reads other segments' pointers
    n_active = s_keep;
  } else {
    n_active = a.counts0[blockIdx.x];
  }
  for (int j = 0;; ++j) {
    const int32_t* in = (j & 1) ? list1 : list0;
    int32_t* out = (j & 1) ? list0 : list1;
    const int32_t* ptr_in = (j & 1) ? a.ptr_b : a.ptr_a;
    int32_t* ptr_out = (j & 1) ? a.ptr_a : a.ptr_b;
    unsigned long long* d_prev = (j & 1) ? a.d1 : a.d0;
    unsigned long long* d_next = (j & 1) ? a.d0 : a.d1;
    __syncthreads();
    if (threadIdx.x == 0) {
      s_keep = 0;
      s_ret = 0;
    }
    __syncthreads();
    // nodes retired by the previous round: make their root visible in this round's output buffer too
    for (int i = threadIdx.x; i < n_retired; i += blockDim.x) {
      const int32_t w = __ldcg(&in[g.seg - 1 - i]);
      ptr_out[w] = __ldcg(&ptr_in[w]);
      const unsigned long long dp = __ldcg(&d_prev[w]);  // what it received during the round it retired in
      if (dp) {
        atomicAdd(&a.S[w], dp);
        d_prev[w] = 0;
      }
    }
    const int n_up = (n_active + 31) / 32 * 32;
    for (int i = threadIdx.x; i < n_up; i += blockDim.x) {
      bool keep = false, retire = false;
      int32_t w = 0;
      if (i < n_active) {
        w = __ldcg(&in[i]);
        unsigned long long sum = __ldcg(&a.S[w]);
        const unsigned long long dp = __ldcg(&d_prev[w]);
        if (dp) {
          sum += dp;
          a.S[w] = sum;
          d_prev[w] = 0;
        }
        const int32_t anc = __ldcg(&ptr_in[w]);
        const int32_t q = __ldcg(&ptr_in[anc]);
        // an ancestor that still jumps forwards what it receives next round (delta buffer); one whose
        // chain is exhausted never forwards again, so its sum takes the contribution directly
        if (sum) atomicAdd(q >= 0 ? &d_next[anc] : &a.S[anc], sum);
        ptr_out[w] = q;
        keep = q >= 0;
        retire = !keep;
      }
      block_append(out, &s_keep, keep, w, false, g.seg);
      block_append(out, &s_ret, retire, w, true, g.seg);
    }
    __syncthreads();
    n_active = s_keep;
    n_retired = s_ret;
    if (threadIdx.x == 0 && n_active + n_retired) atomicAdd(&a.sync[2 + j], (unsigned)(n_active + n_retired));
    grid_barrier(a.sync, generation);
    const unsigned left = *reinterpret_cast<volatile unsigned*>(&a.sync[2 + j]);
    if (left == 0) break;  // nothing active and the last retirees' roots and deltas are in place
    if (j + 1 >= a.max_rounds) {
      if (threadIdx.x == 0 && n_active) *a.leftover = 1;
      break;
    }
  }
}

// ---------------------------------------------------------------- links for the raster perimeter
// Cell (r, c) at position k of perimeter_indices order (flow_accumulation.py:40-51): every row's left then right
// cell, then for columns 1..C-2 the top then the bottom cell.
__device__ __forceinline__ void perimeter_cell(int64_t k, int rows, int cols, int& r, int& c) {
  if (k < 2 * (int64_t)rows) {
    r = (int)(k >> 1);
    c = (k & 1) ? cols - 1 : 0;
  } else {
    const int64_t kk = k - 2 * (int64_t)rows;
    c = 1 + (int)(kk >> 1);
    r = (kk & 1) ? rows - 1 : 0;
  }
}

// Raster cell (row, column) where the in-tile path of perimeter node `root` ends: the exit slot of its link `lk`.
__device__ __forceinline__ int2 link_exit_cell(int root, uint16_t lk, const AccParams& p) {
  int y0, x0, h, w, y, x;
  tile_rect(root / SLOTS, p.ntx, p.rows, p.cols, y0, x0, h, w);
  cell_of_slot(lk & 0xFF, h, w, y, x);
  return make_int2(y0 + y, x0 + x);
}

__global__ void links_kernel(const uint8_t* __restrict__ fdr, int64_t ld_fdr, const int32_t* __restrict__ root_ptr,
                             const uint16_t* __restrict__ link, AccParams p, long long* __restrict__ out, int64_t n) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    int r, c;
    perimeter_cell(k, p.rows, p.cols, r, c);
    long long lr, lc;
    const int code = fdr[(int64_t)r * ld_fdr + c];
    if (code >= 8) {
      // reference quirk: the out-of-bounds offset read sends codes 8/9 "outside" on the first step
      lr = lc = OFL_LINK_EXTERNAL;
    } else {
      const int u = node_of_cell(r, c, p.rows, p.cols, p.ntx);
      const int32_t pr = root_ptr[u];
      const int root = pr < 0 ? ~pr : u;
      const uint16_t lk = link[root];
      const int kind = lk >> 8;
      if (kind == KIND_RASTER_EXIT) {
        const int2 e = link_exit_cell(root, lk, p);
        const int er = e.x, ec = e.y;
        if (er == r && ec == c) {
          lr = lc = OFL_LINK_EXTERNAL;
        } else {
          lr = er;
          lc = ec;
        }
      } else {
        lr = lc = OFL_LINK_TERMINATES;
      }
    }
    out[2 * k] = lr;
    out[2 * k + 1] = lc;
  }
}

// Inflow from outside the raster into its perimeter cells (k in perimeter_indices order, like links_kernel):
// the raster is one rectangular tile of a larger, tiled raster (Barnes 2016, the consumer's second pass), and
// inflow[k] is what the other tiles send into perimeter cell k.  It joins the base inflow of the cell's
// perimeter node, so the solve and the final pass carry it down the cell's path like any inflow between
// 64 x 64 tiles.  A cell listed twice (one-row / one-column rasters) must carry its inflow once.
__global__ void perim_seed_kernel(const long long* __restrict__ inflow, AccParams p, unsigned long long* __restrict__ S,
                                  int64_t n) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    const long long v = inflow[k];
    if (v == 0) continue;
    int r, c;
    perimeter_cell(k, p.rows, p.cols, r, c);
    atomicAdd(&S[node_of_cell(r, c, p.rows, p.cols, p.ntx)], (unsigned long long)v);
  }
}

// ---------------------------------------------------------------- recurrence checker
// Row-strip form: the code raster carries y_off halo rows above row 0 (and below the last row) and the counts
// of the rows just outside the strip come as separate rows (null: the raster ends there).
__global__ void check_kernel(const uint8_t* __restrict__ fdr, int64_t ld_fdr, const long long* __restrict__ fac,
                             int64_t ld_fac, int rows, int cols, int y_off, const long long* __restrict__ fac_above,
                             const long long* __restrict__ fac_below, unsigned long long* __restrict__ n_bad) {
  const int64_t n = (int64_t)rows * cols;
  unsigned long long bad = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i - (int64_t)r * cols);
    const int code = fdr[(int64_t)(r + y_off) * ld_fdr + c];
    long long want;
    if (code == OFL_DIR_NODATA) {
      want = OFL_FAC_NODATA_EMITTED;
    } else {
      want = 1;
#pragma unroll
      for (int d = 0; d < 8; ++d) {
        const int ur = r + dir_dy(d), uc = c + dir_dx(d);
        if (uc < 0 || uc >= cols) continue;
        const long long* urow;
        if (ur < 0) {
          if (!fac_above) continue;
          urow = fac_above;
        } else if (ur >= rows) {
          if (!fac_below) continue;
          urow = fac_below;
        } else {
          urow = fac + (int64_t)ur * ld_fac;
        }
        if (fdr[(int64_t)(ur + y_off) * ld_fdr + uc] == ((d + 4) & 7)) want += urow[uc];
      }
    }
    bad += (fac[(int64_t)r * ld_fac + c] != want);
  }
  for (int o = 16; o > 0; o >>= 1) bad += __shfl_down_sync(0xffffffffu, bad, o);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(n_bad, bad);
}

// ---------------------------------------------------------------- host orchestration (device pointers)
int64_t perimeter_count(int64_t rows, int64_t cols) {
  if (rows <= 0 || cols <= 0) return 0;
  const int64_t inner = cols - 2 > 0 ? cols - 2 : 0;
  return 2 * rows + 2 * inner;
}

constexpr int PJ_MAX_ROUNDS = 40;

static int ensure_tile_attrs() {
  static std::atomic<int> attr_gen{-1};  // function attributes belong to the device they were set on
  if (attr_gen.load() != device_generation()) {
    OFL_CUDA(cudaFuncSetAttribute(acc_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  TileSmem::BYTES));
    OFL_CUDA(cudaFuncSetAttribute(acc_final_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FinalSmem::BYTES_FAST));
    OFL_CUDA(cudaFuncSetAttribute(acc_final_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  FinalSmem::BYTES_WIDE));
    attr_gen.store(device_generation());
  }
  return OFL_OK;
}

static int pj_rounds_for(int64_t n) {
  int r = 2;
  while ((1ll << (r - 1)) < n && r < PJ_MAX_ROUNDS) ++r;
  return r + 1;  // one more round copies the last retirees' roots into both pointer buffers
}

constexpr int PJ_MAX_BLOCKS = 8 * 256;  // counts0 holds this many segments (8 CTAs on each of up to 256 SMs)

static PjSeg pj_segments(int64_t n) {
  PjSeg g;
  g.n = n;
  int64_t blocks = (n + 2047) / 2048;  // at least 2048 nodes per segment
  // the solve is launched cooperatively with one CTA per segment: every segment's CTA must be resident
  int64_t cap = resident_ctas(reinterpret_cast<const void*>(pj_solve_kernel), 256, 8);
  if (cap > PJ_MAX_BLOCKS) cap = PJ_MAX_BLOCKS;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  g.seg = ((n + blocks - 1) / blocks + SLOTS - 1) / SLOTS * SLOTS;  // whole tiles (pass A appends to the lists per tile)
  g.blocks = (int)((n + g.seg - 1) / g.seg);
  return g;
}

// Words of a perimeter graph's flag block, cleared with its sums.  The tile flag (pass A saw a cycle, or a window its
// queue cannot address) and the solve flag (a solve did not converge: a cycle) are the errors a call reports; they are
// read as one pair.  The seed-route word is not an error: it says which route a strip's inflow from other strips
// takes (strip_accum_final).
enum GraphFlag { FLAG_TILE = 0, FLAG_SOLVE = 1, FLAG_SEED_ROUTE = 8, GRAPH_FLAG_WORDS = 16 };
static_assert(FLAG_SOLVE == FLAG_TILE + 1, "the two error flags are copied as one pair");

constexpr int PJ_SYNC_WORDS = PJ_MAX_ROUNDS + 4;  // the solve's grid barrier and nodes left after each round

// A whole raster's graph, a row strip's (it solves the same forest a second time, into S2), or the strips' boundary
// graph (no tiles: no pass A, and the solve builds its own initial state).
enum class GraphKind { RASTER, STRIP, BOUNDARY };

// The workspace of one perimeter graph with n nodes.
struct Graph {
  GraphKind kind;
  int64_t n;
  int32_t *succ, *ptr_a, *ptr_b;
  int32_t* lists;                        // 2 ping-pong lists of blocks * seg >= n entries
  unsigned long long *S, *S2, *d0, *d1;  // S2 is S except on a strip
  uint16_t* link;
  int* counts;     // [2 * PJ_MAX_BLOCKS]: the per-segment active nodes pass A publishes for round 0
  unsigned* sync;  // [PJ_SYNC_WORDS], zeroed by each solve
  int* flags;      // [GRAPH_FLAG_WORDS], see GraphFlag
  uint16_t* L;     // tile-local counts of pass A (empty on the boundary graph)
  int* wide;       // tiles the final pass leaves to its 64-bit variant (empty on the boundary graph)
  size_t bytes;    // size of the workspace
};

// Cuts the graph's buffers out of the workspace at `base`, each 256-byte aligned.  With a null base only `bytes` is
// meaningful.
static Graph carve_graph(void* base, int64_t n, GraphKind kind) {
  Graph g;
  g.kind = kind;
  g.n = n;
  Carver w(base);
  const size_t nodes = (size_t)n;
  const bool tiled = kind != GraphKind::BOUNDARY;
  w.take(g.succ, nodes * 4);
  w.take(g.ptr_a, nodes * 4);
  w.take(g.ptr_b, nodes * 4);
  w.take(g.lists, (nodes + 64 * (size_t)PJ_MAX_BLOCKS) * 8);
  w.take(g.S, nodes * 8);
  g.S2 = g.S;
  if (kind == GraphKind::STRIP) w.take(g.S2, nodes * 8);
  w.take(g.d0, nodes * 8);
  w.take(g.d1, nodes * 8);
  w.take(g.link, nodes * 2);
  w.take(g.counts, 2 * (size_t)PJ_MAX_BLOCKS * sizeof(int));
  w.take(g.sync, PJ_SYNC_WORDS * sizeof(unsigned));
  w.take(g.flags, GRAPH_FLAG_WORDS * sizeof(int));
  w.take(g.L, tiled ? nodes / SLOTS * AT * AT * sizeof(uint16_t) : 0);
  w.take(g.wide, tiled ? (nodes / SLOTS + 1) * sizeof(int) : 0);
  g.bytes = w.bytes;
  return g;
}

// Zero what a call that starts on the graph accumulates into: the sums S and S2 (together before d0; the solve clears
// what it uses of the delta buffers itself), the flag words and, where pass A publishes the solve's initial state, the
// per-segment counts it adds to.
static int clear_graph(const Graph& g, cudaStream_t st) {
  OFL_CUDA(cudaMemsetAsync(g.S, 0, reinterpret_cast<uint8_t*>(g.d0) - reinterpret_cast<uint8_t*>(g.S), st));
  OFL_CUDA(cudaMemsetAsync(g.flags, 0, GRAPH_FLAG_WORDS * sizeof(int), st));
  if (g.kind != GraphKind::BOUNDARY) OFL_CUDA(cudaMemsetAsync(g.counts, 0, 2 * (size_t)PJ_MAX_BLOCKS * sizeof(int), st));
  return OFL_OK;
}

// Subtree sums over the graph's forest: on return (stream order) S[u] (S is the graph's S or S2) holds the sum of the
// initial S over u's subtree and both pointer buffers hold ~root(u) for every node.  with_init: the solve starts from
// `succ`, which it preserves; otherwise from the state pass A published.  run_flag (nullable): a device word; the
// solve is skipped when it is 0.  Does not synchronise: the solve flag is set when the forest did not converge (a
// cycle).
static int pj_solve(const Graph& graph, unsigned long long* S, cudaStream_t st, bool with_init,
                    const int* run_flag = nullptr) {
  PjArgs a;
  a.run_flag = run_flag;
  a.succ = graph.succ;
  a.ptr_a = graph.ptr_a;
  a.ptr_b = graph.ptr_b;
  a.lists = graph.lists;
  a.counts0 = graph.counts;
  a.S = S;
  a.d0 = graph.d0;
  a.d1 = graph.d1;
  a.sync = graph.sync;
  a.leftover = graph.flags + FLAG_SOLVE;
  a.g = pj_segments(graph.n);
  a.with_init = with_init ? 1 : 0;
  a.max_rounds = pj_rounds_for(graph.n);
  OFL_CUDA(cudaMemsetAsync(a.sync, 0, PJ_SYNC_WORDS * sizeof(unsigned), st));
  void* args[] = {&a};
  OFL_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(pj_solve_kernel), dim3((unsigned)a.g.blocks), dim3(256),
                                       args, 0, st));
  OFL_CHECK_LAUNCH();
  return OFL_OK;
}

// One synchronisation at the end of a call.
static int check_flags(const Graph& g, cudaStream_t st) {
  int h[2] = {0, 0};  // tile flag, solve flag
  OFL_CUDA(cudaMemcpyAsync(h, g.flags + FLAG_TILE, sizeof(h), cudaMemcpyDeviceToHost, st));
  OFL_CUDA(cudaStreamSynchronize(st));
  OFL_REQUIRE(h[0] != 3, OFL_ERR_INVALID, "shared-memory window above 64 KB: the tile kernel's 16-bit queue does not apply");
  OFL_REQUIRE(h[0] == 0, OFL_ERR_CYCLE, "flow-direction raster contains a cycle (tile flag %d)", h[0]);
  OFL_REQUIRE(h[1] == 0, OFL_ERR_CYCLE, "flow-direction raster contains a cycle (perimeter graph)");
  return OFL_OK;
}

static inline int64_t node_count(int64_t rows, int64_t cols) {
  return tiles_along(rows) * tiles_along(cols) * SLOTS;
}

size_t accumulation_workspace_bytes(int64_t rows, int64_t cols) {
  if (rows <= 0 || cols <= 0) return 256;
  return carve_graph(nullptr, node_count(rows, cols), GraphKind::RASTER).bytes;
}

size_t strip_workspace_bytes(int64_t rows, int64_t cols) {
  if (rows <= 0 || cols <= 0) return 256;
  return carve_graph(nullptr, node_count(rows, cols), GraphKind::STRIP).bytes;
}

// The rasters one accumulation call takes: 30-bit sides (AccParams holds ints) and 32-bit perimeter node ids.
int accumulation_shape(int64_t rows, int64_t cols) {
  OFL_REQUIRE(rows >= 1 && cols >= 1 && rows < (1ll << 30) && cols < (1ll << 30), OFL_ERR_INVALID, "bad raster size");
  OFL_REQUIRE(node_count(rows, cols) < (1ll << 31), OFL_ERR_INVALID, "raster too large for 32-bit perimeter node ids");
  return OFL_OK;
}

// Everything one raster (or strip) needs to launch its kernels.
struct AccCtx {
  AccParams p;
  CUtensorMap tm;  // codes + halo box for pass A
  Graph graph;
  int64_t ntiles;
};

static int acc_setup(AccCtx& C, const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, int y_off, int has_above,
                     int has_below, long long* fac, int64_t ld_fac, void* workspace, bool strip) {
  OFL_REQUIRE((reinterpret_cast<uintptr_t>(fdr) & 15) == 0 && (ld_fdr % 16) == 0 && ld_fdr >= cols, OFL_ERR_ALIGNMENT,
              "fdr must be 16-byte aligned with ld_fdr %% 16 == 0 (ld_fdr=%lld)", (long long)ld_fdr);
  OFL_REQUIRE((reinterpret_cast<uintptr_t>(fac) & 7) == 0 && ld_fac >= cols, OFL_ERR_ALIGNMENT, "fac must be 8-byte aligned");
  const int64_t n = node_count(rows, cols);
  C.graph = carve_graph(workspace, n, strip ? GraphKind::STRIP : GraphKind::RASTER);
  const Graph& g = C.graph;
  AccParams& p = C.p;
  p.rows = (int)rows;
  p.cols = (int)cols;
  p.nty = (int)tiles_along(rows);
  p.ntx = (int)tiles_along(cols);
  p.succ = g.succ;
  p.link = g.link;
  p.S = g.S;
  p.fac = fac;
  p.ld_fac = ld_fac;
  p.err = g.flags + FLAG_TILE;
  p.L = g.L;
  p.wide_list = g.wide;
  p.force_wide = getenv("OFL_FORCE_WIDE_FINAL") ? 1 : 0;
  p.trusted_codes = 0;
  p.fuse_init = 1;
  p.keep_succ = strip ? 1 : 0;
  p.ptr_a = g.ptr_a;
  p.ptr_b = g.ptr_b;
  p.list0 = g.lists;
  p.d0 = g.d0;
  p.d1 = g.d1;
  p.counts0 = g.counts;
  const PjSeg seg = pj_segments(n);
  p.tiles_per_seg = (int)(seg.seg / SLOTS);
  p.seg = seg.seg;
  p.y_off = y_off;
  p.strip_above = has_above ? 1 : 0;
  p.strip_below = has_below ? 1 : 0;
  p.tile_base = 0;
  p.vec_store = ((reinterpret_cast<uintptr_t>(fac) & 15) == 0 && (ld_fac % 2) == 0) ? 1 : 0;
  C.ntiles = (int64_t)p.nty * p.ntx;
  int rc = make_tensor_map_2d(&C.tm, fdr, 1, (uint64_t)cols, (uint64_t)(rows + 2 * y_off), (uint64_t)ld_fdr, ACS_W, ACS_H);
  if (rc != OFL_OK) return rc;
  return ensure_tile_attrs();
}

// Final pass over `grid` tiles starting at p.tile_base: the 32-bit kernel, then the 64-bit one on whatever it listed.
static int launch_final(const AccParams& p, unsigned grid, cudaStream_t st) {
  OFL_CUDA(cudaMemsetAsync(p.wide_list, 0, sizeof(int), st));
  acc_final_kernel<<<grid, ACC_THREADS, FinalSmem::BYTES_FAST, st>>>(p);
  OFL_CHECK_LAUNCH();
  const unsigned wide_grid = grid < (unsigned)sm_count() * 2 ? grid : (unsigned)sm_count() * 2;
  acc_final_wide_kernel<<<wide_grid, ACC_THREADS, FinalSmem::BYTES_WIDE, st>>>(p);
  OFL_CHECK_LAUNCH();
  return OFL_OK;
}

// The phases the whole-raster and strip calls share, each timed as one phase.
static int pass_a(const AccCtx& C, cudaStream_t st) {
  {
    PhaseScope ps(PHASE_ACC_TILE_A, st);
    acc_tile_kernel<<<(unsigned)C.ntiles, ACC_THREADS, TileSmem::BYTES, st>>>(C.tm, C.p);
  }
  OFL_CHECK_LAUNCH();
  return OFL_OK;
}

static int solve_published(const AccCtx& C, cudaStream_t st) {  // from the initial state pass A published
  PhaseScope ps(PHASE_ACC_SOLVE, st);
  return pj_solve(C.graph, C.graph.S, st, false);
}

static int final_pass(const AccCtx& C, cudaStream_t st) {  // over every tile
  PhaseScope ps(PHASE_ACC_TILE_B, st);
  return launch_final(C.p, (unsigned)C.ntiles, st);
}

// The part of a whole-raster accumulation that does not depend on the codes: clear_graph.  A caller that produces the
// codes on the same device (ofl_flow_routing_f32) runs it on a second stream next to the direction kernel and passes
// prepared = true below.
int accumulation_prepare(int64_t rows, int64_t cols, void* workspace, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return OFL_OK;
  return clear_graph(carve_graph(workspace, node_count(rows, cols), GraphKind::RASTER), st);
}

int launch_accumulation(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, long long* fac,
                        int64_t ld_fac, long long* perim_links_dev, void* workspace, cudaStream_t st, bool prepared,
                        bool trusted_codes, const long long* perim_inflow_dev) {
  if (rows <= 0 || cols <= 0) return OFL_OK;
  AccCtx C;
  int rc = acc_setup(C, fdr, rows, cols, ld_fdr, 0, 0, 0, fac, ld_fac, workspace, false);
  if (rc != OFL_OK) return rc;
  C.p.trusted_codes = trusted_codes ? 1 : 0;
  if (!prepared) {
    rc = clear_graph(C.graph, st);
    if (rc != OFL_OK) return rc;
  }
  rc = pass_a(C, st);
  if (rc != OFL_OK) return rc;
  const int64_t n_perim = perimeter_count(rows, cols);
  if (perim_inflow_dev) {
    perim_seed_kernel<<<grid_for(n_perim, 16), 256, 0, st>>>(perim_inflow_dev, C.p, C.p.S, n_perim);
    OFL_CHECK_LAUNCH();
  }
  rc = solve_published(C, st);
  if (rc != OFL_OK) return rc;
  rc = final_pass(C, st);
  if (rc != OFL_OK) return rc;
  if (perim_links_dev) {
    {
      PhaseScope ps(PHASE_ACC_LINKS, st);
      links_kernel<<<grid_for(n_perim, 16), 256, 0, st>>>(fdr, ld_fdr, C.p.ptr_a, C.p.link, C.p, perim_links_dev, n_perim);
    }
    OFL_CHECK_LAUNCH();
  }
  return check_flags(C.graph, st);
}

// ================================================================ row strips (multi-GPU)
// Barnes 2016 at the strip level.  Each GPU owns a row strip [r0, r1) whose boundaries are multiples of
// the tile side, and holds the codes of the neighbouring strips' adjacent rows as halo rows.
//   local     pass A + solve with cross-strip edges as roots; pass B on the first and last tile row only
//             gives the strip-local counts of the boundary rows; emit for every boundary-row cell its
//             local count, its code and the boundary cell where its in-strip path leaves the strip
//   exchange  all-gather of those 13 B/cell boundary records (done by the caller, NCCL)
//   solve     the same pointer-doubling solve on the boundary forest (2 rows x cols x strips nodes),
//             replicated on every GPU: inflow from other strips into every boundary cell
//   final     push the strip's inflows down its own perimeter graph (second solve on seeds only, by
//             linearity), then pass B over all tiles
// boundary record of cell (t ? last row : first row, c): strip-local count, code, and where its in-strip
// path leaves the strip: (exit row selector << 30) | exit column, or -1 when it does not leave.
// A strip's records travel as ONE block of bytes (one all-gather): [2 x cols] int64 counts, then [2 x cols]
// int32 exit links, then [2 x cols] codes, padded to a multiple of 256 bytes.
size_t strip_record_bytes(int64_t cols) {
  if (cols <= 0) return 256;
  return align_up((size_t)cols * 2 * (8 + 4 + 1), 256);
}
struct RecView {  // the record blocks of n strips, `stride` bytes apart
  const uint8_t* base;
  int64_t stride, cols;
  __device__ __forceinline__ long long floc(int s, int64_t k) const {
    return reinterpret_cast<const long long*>(base + s * stride)[k];
  }
  __device__ __forceinline__ int32_t slink(int s, int64_t k) const {
    return reinterpret_cast<const int32_t*>(base + s * stride + cols * 16)[k];
  }
  __device__ __forceinline__ uint8_t code(int s, int64_t k) const { return (base + s * stride + cols * 24)[k]; }
};

__global__ void strip_boundary_extract_kernel(const uint8_t* __restrict__ fdr, int64_t ld_fdr,
                                              const long long* __restrict__ fac, int64_t ld_fac,
                                              const int32_t* __restrict__ root_ptr, const uint16_t* __restrict__ link,
                                              AccParams p, uint8_t* __restrict__ record) {
  const int64_t n = 2 * (int64_t)p.cols;
  long long* floc = reinterpret_cast<long long*>(record);
  int32_t* slink = reinterpret_cast<int32_t*>(record + (int64_t)p.cols * 16);
  uint8_t* bcode = record + (int64_t)p.cols * 24;
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    const int t = (int)(k / p.cols), c = (int)(k - (int64_t)t * p.cols);
    const int r = t ? p.rows - 1 : 0;
    const uint8_t code = fdr[(int64_t)(r + p.y_off) * ld_fdr + c];
    bcode[k] = code;
    floc[k] = fac[(int64_t)r * ld_fac + c];
    int32_t sl = -1;
    if (code < 8) {
      const int u = node_of_cell(r, c, p.rows, p.cols, p.ntx);
      const int32_t pr = root_ptr[u];
      const int root = pr < 0 ? ~pr : u;
      const uint16_t lk = link[root];
      if ((lk >> 8) == KIND_STRIP_EXIT) {
        const int2 e = link_exit_cell(root, lk, p);
        const int er = e.x, ec = e.y;
        sl = ((er == 0 ? 0 : 1) << 30) | ec;
      }
    }
    slink[k] = sl;
  }
}

// node id of boundary cell (strip s, row selector t, column c)
__device__ __forceinline__ int64_t bnode(int s, int t, int64_t c, int64_t cols) { return ((int64_t)s * 2 + t) * cols + c; }

// where does boundary cell (s, t, c) with code `code` send its water?  -1 when not across a strip boundary
__device__ __forceinline__ int64_t bnode_target(int s, int t, int64_t c, int code, int n_strips, const RecView& rec) {
  if (code >= 8) return -1;
  const int dy = dir_dy(code);
  if ((t == 0 && dy != -1) || (t == 1 && dy != 1)) return -1;
  const int s2 = s + dy;
  const int64_t c2 = c + dir_dx(code);
  if (s2 < 0 || s2 >= n_strips || c2 < 0 || c2 >= rec.cols) return -1;
  const int t2 = dy < 0 ? 1 : 0;
  return rec.code(s2, t2 * rec.cols + c2) == OFL_DIR_NODATA ? -1 : bnode(s2, t2, c2, rec.cols);
}

__global__ void strip_graph_build_kernel(const RecView rec, int n_strips, int32_t* __restrict__ succ,
                                         unsigned long long* __restrict__ base) {
  const int64_t cols = rec.cols;
  const int64_t n = (int64_t)n_strips * 2 * cols;
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(k / (2 * cols));
    const int64_t kk = k - (int64_t)s * 2 * cols;  // index inside the strip's record
    const int t = (int)(kk / cols);
    const int64_t c = kk - (int64_t)t * cols;
    // this cell's own edge across the boundary carries its strip-local count into the next strip
    const int64_t d = bnode_target(s, t, c, rec.code(s, kk), n_strips, rec);
    if (d >= 0) atomicAdd(&base[d], (unsigned long long)rec.floc(s, kk));
    // parent in the boundary forest: the entry cell fed by the cell where this cell's path leaves the strip
    int32_t parent = -1;
    const int32_t sl = rec.slink(s, kk);
    if (sl >= 0) {
      const int te = sl >> 30;
      const int64_t ce = sl & ((1 << 30) - 1);
      const int64_t dd = bnode_target(s, te, ce, rec.code(s, te * cols + ce), n_strips, rec);
      if (dd >= 0) parent = (int32_t)dd;
    }
    succ[k] = parent;
  }
}

// The inflow from other strips enters at the boundary rows and has to reach every perimeter node downstream of its
// entry cell.  On terrain those paths are short (a handful of tiles) and the entries few, so one thread per entry
// cell simply walks the preserved forest and adds its inflow to every node on the way -- after a dry walk by all of
// them has shown that no path is longer than SEED_CHASE_MAX nodes.  If one is (a long channel, a tilted plane), a
// device flag sends the step through the general route instead: subtree sums of the seeds by pointer doubling over
// the whole forest, added to S.  Both routes give the same sums (integer adds); the choice is made on the device.
constexpr int SEED_CHASE_MAX = 256;

template <bool DRY>
__global__ void strip_seed_chase_kernel(const long long* __restrict__ J, AccParams p, const int32_t* __restrict__ succ,
                                        unsigned long long* __restrict__ S, int* __restrict__ too_long) {
  if (!DRY && *too_long) return;
  const int64_t n = 2 * (int64_t)p.cols;
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    const long long j = J[k];
    if (j == 0) continue;
    const int t = (int)(k / p.cols), c = (int)(k - (int64_t)t * p.cols);
    int u = node_of_cell(t ? p.rows - 1 : 0, c, p.rows, p.cols, p.ntx);
    if (DRY) {
      int steps = 0;
      while ((u = succ[u]) >= 0)
        if (++steps > SEED_CHASE_MAX) {
          *too_long = 1;
          break;
        }
    } else {
      do {
        atomicAdd(&S[u], (unsigned long long)j);
        u = succ[u];
      } while (u >= 0);
    }
  }
}

__global__ void strip_seed_kernel_if(const long long* __restrict__ J, AccParams p, unsigned long long* __restrict__ S2,
                                     int64_t n_nodes, const int* __restrict__ run_flag) {
  if (*run_flag == 0) return;
  // the general route: S2 = 0 everywhere, then the seeds (one launch: the seeds' nodes are zeroed by their own threads)
  for (int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; u < n_nodes; u += (int64_t)gridDim.x * blockDim.x) S2[u] = 0;
}

__global__ void strip_seed_set_kernel_if(const long long* __restrict__ J, AccParams p, unsigned long long* __restrict__ S2,
                                         const int* __restrict__ run_flag) {
  if (*run_flag == 0) return;
  const int64_t n = 2 * (int64_t)p.cols;
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    const int t = (int)(k / p.cols), c = (int)(k - (int64_t)t * p.cols);
    const long long j = J[k];
    if (j != 0) S2[node_of_cell(t ? p.rows - 1 : 0, c, p.rows, p.cols, p.ntx)] = (unsigned long long)j;
  }
}

__global__ void pj_add_kernel_if(unsigned long long* __restrict__ S, const unsigned long long* __restrict__ S2, int64_t n,
                                 const int* __restrict__ run_flag) {
  if (*run_flag == 0) return;
  for (int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; u < n; u += (int64_t)gridDim.x * blockDim.x) {
    const unsigned long long d = S2[u];
    if (d) S[u] += d;
  }
}

int strip_shape(int64_t rows, int64_t cols, int has_below) {
  OFL_REQUIRE(rows >= 2, OFL_ERR_INVALID, "a strip needs at least 2 rows");
  OFL_REQUIRE(!has_below || rows % AT == 0, OFL_ERR_INVALID,
              "a strip with a strip below it must have a multiple of %d rows (got %lld)", AT, (long long)rows);
  return accumulation_shape(rows, cols);
}

// The three strip calls below only enqueue work; strip_collect_flags hands out their error flags.
int strip_accum_local(const uint8_t* fdr_halo, int64_t rows, int64_t cols, int64_t ld_fdr, int has_above, int has_below,
                      long long* fac, int64_t ld_fac, void* workspace, void* record, cudaStream_t st) {
  AccCtx C;
  int rc = acc_setup(C, fdr_halo, rows, cols, ld_fdr, 1, has_above, has_below, fac, ld_fac, workspace, true);
  if (rc != OFL_OK) return rc;
  rc = clear_graph(C.graph, st);
  if (rc != OFL_OK) return rc;
  rc = pass_a(C, st);
  if (rc != OFL_OK) return rc;
  rc = solve_published(C, st);
  if (rc != OFL_OK) return rc;
  // strip-local counts of the first and last tile row (their cells include both boundary rows)
  {
    PhaseScope ps(PHASE_STRIP_EDGE, st);
    AccParams pb = C.p;
    rc = launch_final(pb, (unsigned)pb.ntx, st);
    if (rc == OFL_OK && pb.nty > 1) {
      pb.tile_base = (pb.nty - 1) * pb.ntx;
      rc = launch_final(pb, (unsigned)pb.ntx, st);
    }
  }
  if (rc != OFL_OK) return rc;
  strip_boundary_extract_kernel<<<grid_for(2 * cols, 8), 256, 0, st>>>(fdr_halo, ld_fdr, fac, ld_fac, C.p.ptr_a, C.p.link, C.p,
                                                                       static_cast<uint8_t*>(record));
  OFL_CHECK_LAUNCH();
  return OFL_OK;
}

size_t strip_boundary_workspace_bytes(int64_t n_strips, int64_t cols) {
  return carve_graph(nullptr, (int64_t)n_strips * 2 * cols, GraphKind::BOUNDARY).bytes;
}

int boundary_shape(int64_t n_strips, int64_t cols) {
  OFL_REQUIRE(n_strips >= 1 && cols >= 1, OFL_ERR_INVALID, "bad boundary graph size");
  OFL_REQUIRE(n_strips * 2 * cols < (1ll << 31), OFL_ERR_INVALID, "boundary graph too large");
  return OFL_OK;
}

int strip_boundary_solve(const void* records_all, int n_strips, int64_t cols, long long* J_all, void* workspace,
                         cudaStream_t st) {
  const int64_t n = (int64_t)n_strips * 2 * cols;
  const Graph g = carve_graph(workspace, n, GraphKind::BOUNDARY);
  int rc = clear_graph(g, st);
  if (rc != OFL_OK) return rc;
  RecView rec;
  rec.base = static_cast<const uint8_t*>(records_all);
  rec.stride = (int64_t)strip_record_bytes(cols);
  rec.cols = cols;
  strip_graph_build_kernel<<<grid_for(n, 8), 256, 0, st>>>(rec, n_strips, g.succ, g.S);
  OFL_CHECK_LAUNCH();
  {
    PhaseScope ps(PHASE_ACC_SOLVE, st);
    rc = pj_solve(g, g.S, st, true);
  }
  if (rc != OFL_OK) return rc;
  OFL_CUDA(cudaMemcpyAsync(J_all, g.S, (size_t)n * 8, cudaMemcpyDeviceToDevice, st));
  return OFL_OK;
}

// Error flags of a strip's calls since its last strip_accum_local, and of the boundary solve, as four ints in
// device memory: [0] tile flag, [1] strip solve, [2..3] the same for the boundary workspace (zero when null).
// Stream-ordered; the caller reads them (after reducing them over the ranks, if there are several).
int strip_collect_flags(const void* strip_workspace, int64_t rows, int64_t cols, const void* boundary_workspace,
                        int n_strips, int32_t* flags_dev, cudaStream_t st) {
  OFL_CUDA(cudaMemsetAsync(flags_dev, 0, 4 * sizeof(int32_t), st));
  if (strip_workspace) {
    const Graph g = carve_graph(const_cast<void*>(strip_workspace), node_count(rows, cols), GraphKind::STRIP);
    OFL_CUDA(cudaMemcpyAsync(flags_dev, g.flags + FLAG_TILE, 2 * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  }
  if (boundary_workspace) {
    const Graph g = carve_graph(const_cast<void*>(boundary_workspace), (int64_t)n_strips * 2 * cols, GraphKind::BOUNDARY);
    OFL_CUDA(cudaMemcpyAsync(flags_dev + 2, g.flags + FLAG_TILE, 2 * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  }
  return OFL_OK;
}

int strip_accum_final(const uint8_t* fdr_halo, int64_t rows, int64_t cols, int64_t ld_fdr, int has_above, int has_below,
                      const long long* J_mine, void* workspace, long long* fac, int64_t ld_fac, cudaStream_t st) {
  AccCtx C;
  int rc = acc_setup(C, fdr_halo, rows, cols, ld_fdr, 1, has_above, has_below, fac, ld_fac, workspace, true);
  if (rc != OFL_OK) return rc;
  const Graph& g = C.graph;
  // inflow from other strips: walked down the forest from its entry cells when every such path is short, else
  // (device flag) subtree sums of the seeds over the whole forest -- see strip_seed_chase_kernel
  int* too_long = g.flags + FLAG_SEED_ROUTE;
  const bool force_general = getenv("OFL_SEED_GENERAL") != nullptr;  // test hook: always the general route
  OFL_CUDA(cudaMemsetAsync(too_long, force_general ? 1 : 0, sizeof(int), st));
  {
    PhaseScope ps(PHASE_ACC_SOLVE, st);
    const int gs = grid_for(2 * cols, 8);
    strip_seed_chase_kernel<true><<<gs, 256, 0, st>>>(J_mine, C.p, g.succ, g.S, too_long);
    OFL_CHECK_LAUNCH();
    strip_seed_chase_kernel<false><<<gs, 256, 0, st>>>(J_mine, C.p, g.succ, g.S, too_long);
    OFL_CHECK_LAUNCH();
    strip_seed_kernel_if<<<grid_for(g.n, 8), 256, 0, st>>>(J_mine, C.p, g.S2, g.n, too_long);
    OFL_CHECK_LAUNCH();
    strip_seed_set_kernel_if<<<gs, 256, 0, st>>>(J_mine, C.p, g.S2, too_long);
    OFL_CHECK_LAUNCH();
    rc = pj_solve(g, g.S2, st, true, too_long);
    if (rc != OFL_OK) return rc;
    pj_add_kernel_if<<<grid_for(g.n, 8), 256, 0, st>>>(g.S, g.S2, g.n, too_long);  // S += S2
    OFL_CHECK_LAUNCH();
  }
  return final_pass(C, st);
}

int launch_check(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, const long long* fac, int64_t ld_fac,
                 unsigned long long* n_bad_dev, cudaStream_t st, int y_off, const long long* fac_above,
                 const long long* fac_below) {
  OFL_CUDA(cudaMemsetAsync(n_bad_dev, 0, sizeof(unsigned long long), st));
  if (rows <= 0 || cols <= 0) return OFL_OK;
  check_kernel<<<grid_for(rows * cols, 16), 256, 0, st>>>(fdr, ld_fdr, fac, ld_fac, (int)rows, (int)cols, y_off, fac_above,
                                                          fac_below, n_bad_dev);
  OFL_CHECK_LAUNCH();
  return OFL_OK;
}

}  // namespace ofl
