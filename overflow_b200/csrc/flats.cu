// flats.cu -- flat resolution (Barnes, Lehman & Mulla 2014) on the device: the reference's
// src/overflow/fix_flats.py (flat_edges :13-62, label_flats :65-108, away_from_higher :111-161,
// towards_lower :164-224, resolve_flats :227-288, d8_masked_flow_dirs :291-339).
//
// The reference is a chain of sequential scans and FIFO sweeps.  What it computes is order-free, and that is
// what runs here:
//   * flat_edges is a 3x3 stencil (a cell is a low edge iff it has a direction and an equally high
//     neighbour without one; a high edge iff it has none and a higher neighbour that is not NODATA).
//   * label_flats floods cells of equal elevation, 8-connected, whatever their direction code; labels are
//     handed out in the order the row-major low-edge list meets unlabelled cells.  Here: union-find over
//     "equal elevation" links (atomicMin hooking, path halving), the smallest low-edge index of every
//     component by atomicMin, and label = 1 + rank of that index among all components' smallest low edges
//     (a prefix sum over the raster).  Components without a low edge keep label 0.
//   * away_from_higher / towards_lower are breadth-first sweeps with a level marker: a cell's value is its
//     BFS level from the seed edges through same-label cells without a direction.  Here: relaxation of 32 x 32
//     tiles in shared memory to the same (unique) fixpoint, the passes over the queued tiles inside one
//     persistent kernel; flat_height[label] = max level by atomicMax (the reference's "last write" is the
//     largest level because levels only grow).
//   * d8_masked_flow_dirs is a 3x3 stencil over flat_mask and labels, slopes in float64 as in the reference.
// Everything is integer work except the two float compares (==, <) on elevations and the float64 slope
// division, so results are compared bit for bit with the reference's.
#include <limits.h>
#include <stdio.h>
#include <stdlib.h>

#include <math_constants.h>

#include "common.cuh"

namespace ofl {

namespace {

constexpr int FL_UNDEF = OFL_DIR_UNDEFINED, FL_NODATA = OFL_DIR_NODATA;
constexpr unsigned FL_NONE = 0xFFFFFFFFu;  // minlow: the component has no low edge (see flat_lowroot_kernel for cell 2^32 - 1)
constexpr int FL_THREADS = 256;
constexpr int FL_SCAN_THREADS = 1024;

// counters (uint32) kept in device memory
enum {
  CNT_LOW = 0, CNT_HIGH, CNT_LABELS, CNT_SEEDS,
  CNT_TCOUNT0, CNT_TCOUNT1, CNT_TCOUNT2,  // tiles queued for pass k in slot k % 3
  CNT_TTAKE0, CNT_TTAKE1, CNT_TTAKE2,     // tiles of pass k handed out so far
  CNT_BAR, CNT_RELEASE,                   // grid barrier of the sweep kernel
  CNT_PASSES, CNT_MAXLEVEL,
  CNT_VISITS, CNT_ROUNDS,                 // statistics of the sweep (OFL_FLATS_DEBUG)
  CNT_MAXROUNDS,                          // most rounds in one visit
  CNT_LASTLOW, CNT_LASTROOT,              // cell 2^32 - 1 is a low edge / its root (a raster of exactly 2^32 cells)
  CNT_CYC_LOAD, CNT_CYC_ROUNDS, CNT_CYC_STORE,  // clock cycles / 64 spent in the three parts of a tile visit (sums)
  CNT_PASSTIME0,                          // start of pass k in ns (low word), 40 slots
  CNT_SLOTS = 64
};

__constant__ int c_dy[8] = {0, -1, -1, -1, 0, 1, 1, 1};  // E NE N NW W SW S SE: constants.py:29-40
__constant__ int c_dx[8] = {1, 1, 0, -1, -1, -1, 0, 1};

// ---------------------------------------------------------------- flat_edges (fix_flats.py:13-62)
// Also initialises the union-find forest and the per-component "smallest low edge" slot.  The forest starts with
// every horizontal run of equal elevation already hanging off its first cell as far as one warp sees it (a ballot
// and a count-leading-zeros, no atomics), which is most of the linking on a plateau.
__global__ void __launch_bounds__(FL_THREADS)
flat_edges_kernel(const float* __restrict__ dem, const uint8_t* __restrict__ fdr, int rows, int cols, uint8_t* edges,
                  unsigned* parent, unsigned* minlow, unsigned* cnt) {
  // cell indices are 32-bit unsigned (a raster holds at most 2^32 cells); only the bound needs 64 bits
  const int64_t n = (int64_t)rows * cols;
  const unsigned i = blockIdx.x * FL_THREADS + threadIdx.x;
  const bool inside = (int64_t)blockIdx.x * FL_THREADS + threadIdx.x < n;
  int flag = 0;
  bool left_eq = false;
  if (inside) {
    const int r = (int)(i / (unsigned)cols), c = (int)(i - (unsigned)r * (unsigned)cols);
    const int cur = fdr[i];
    const float z = dem[i];
    left_eq = c > 0 && dem[i - 1] == z;
    // The two kinds exclude each other, so each cell runs one loop only, and the result does not depend on the
    // order the neighbours are visited in.  A cell with a direction reads a neighbour's elevation only where
    // that neighbour has none (rare outside flats); cells off the raster's ring skip the bounds checks.
    const bool inner = r > 0 && r + 1 < rows && c > 0 && c + 1 < cols;
    if (cur != FL_UNDEF) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int nr = r + c_dy[k], nc = c + c_dx[k];
        if (!inner && (nr < 0 || nr >= rows || nc < 0 || nc >= cols)) continue;
        const unsigned j = (unsigned)nr * (unsigned)cols + (unsigned)nc;
        if (fdr[j] == FL_UNDEF && dem[j] == z) flag = 1;  // :45-53
      }
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int nr = r + c_dy[k], nc = c + c_dx[k];
        if (!inner && (nr < 0 || nr >= rows || nc < 0 || nc >= cols)) continue;
        const unsigned j = (unsigned)nr * (unsigned)cols + (unsigned)nc;
        if (z < dem[j] && fdr[j] != FL_NODATA) flag = 2;  // :41-43, :54-60
      }
    }
    edges[i] = (uint8_t)flag;
  }
  if (parent) {
    const int lane = threadIdx.x & 31;
    const unsigned em = __ballot_sync(0xffffffffu, left_eq);
    const unsigned starts = (~em & ((2u << lane) - 1u)) | 1u;  // lanes <= mine that begin a run (lane 0 always does)
    if (inside) {
      parent[i] = i - (unsigned)(lane - (31 - __clz(starts)));
      minlow[i] = FL_NONE;
    }
  }
  const int lo = __syncthreads_count(flag == 1), hi = __syncthreads_count(flag == 2);
  if (threadIdx.x == 0) {
    if (lo) atomicAdd(&cnt[CNT_LOW], (unsigned)lo);
    if (hi) atomicAdd(&cnt[CNT_HIGH], (unsigned)hi);
  }
}

// The same for rasters whose width is a multiple of 32 (dense, so every row starts 16-byte aligned): a thread owns
// four adjacent cells of one row -- three float4 + six scalar elevation loads and three word + six byte code loads
// instead of 72 scalar ones -- and the neighbours' tests share their column work: "some neighbour without NODATA is
// higher" is one maximum over per-column maxima, "some neighbour without a direction is equally high" compares against
// values that are NaN wherever the neighbour has a direction.  A warp covers 128 consecutive cells of a row; the
// forest starts with every run hanging off its first cell as far as those 128 cells go (runs continue across the
// 128-cell seams through flat_merge_kernel's hand-over at every 32nd cell, which includes the seams).
__global__ void __launch_bounds__(FL_THREADS)
flat_edges4_kernel(const float* __restrict__ dem, const uint8_t* __restrict__ fdr, int rows, int cols, uint8_t* edges,
                   unsigned* parent, unsigned* minlow, unsigned* cnt) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int r = blockIdx.y * (FL_THREADS / 32) + w;
  const int c = (blockIdx.x * 32 + lane) * 4;
  const bool inside = r < rows && c < cols;  // cols % 4 == 0: the four cells are inside together
  unsigned flags = 0, eq = 0;                // eq bit j: cell c + j continues the run of the cell to its left
  if (inside) {
    float v[3][6];
    unsigned f[3][6];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int rr = r + k - 1;
      if (rr < 0 || rr >= rows) {
#pragma unroll
        for (int x = 0; x < 6; ++x) {
          v[k][x] = 0.f;
          f[k][x] = FL_NODATA;  // fails both tests below, like a cell that is not there
        }
      } else {
        const size_t o = (size_t)rr * (size_t)cols + (size_t)c;
        const float4 m = *reinterpret_cast<const float4*>(dem + o);
        const unsigned fw = *reinterpret_cast<const unsigned*>(fdr + o);
        v[k][1] = m.x;
        v[k][2] = m.y;
        v[k][3] = m.z;
        v[k][4] = m.w;
        f[k][1] = fw & 0xFFu;
        f[k][2] = (fw >> 8) & 0xFFu;
        f[k][3] = (fw >> 16) & 0xFFu;
        f[k][4] = fw >> 24;
        v[k][0] = c > 0 ? dem[o - 1] : 0.f;
        f[k][0] = c > 0 ? fdr[o - 1] : (unsigned)FL_NODATA;
        v[k][5] = c + 4 < cols ? dem[o + 4] : 0.f;
        f[k][5] = c + 4 < cols ? fdr[o + 4] : (unsigned)FL_NODATA;
      }
    }
    // hi[k][x]: the elevation where a higher neighbour counts (not NODATA), else -inf; per column the maximum of the
    // rows above and below (m02) and of all three (m3).  fmaxf skips NaN like "z < NaN" is false.
    float m02[6], m3[6];
#pragma unroll
    for (int x = 0; x < 6; ++x) {
      const float a = f[0][x] != (unsigned)FL_NODATA ? v[0][x] : -CUDART_INF_F;
      const float b = f[1][x] != (unsigned)FL_NODATA ? v[1][x] : -CUDART_INF_F;
      const float d = f[2][x] != (unsigned)FL_NODATA ? v[2][x] : -CUDART_INF_F;
      m02[x] = fmaxf(a, d);
      m3[x] = fmaxf(m02[x], b);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float z = v[1][j + 1];
      unsigned flag = 0;
      if (f[1][j + 1] != (unsigned)FL_UNDEF) {
        bool low = false;  // :45-53: an equally high neighbour without a direction
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
          for (int x = j; x <= j + 2; ++x)
            if (!(k == 1 && x == j + 1)) low |= f[k][x] == (unsigned)FL_UNDEF && v[k][x] == z;
        flag = low ? 1u : 0u;
      } else {
        flag = fmaxf(fmaxf(m3[j], m3[j + 2]), m02[j + 1]) > z ? 2u : 0u;  // :41-43, :54-60
      }
      flags |= flag << (8 * j);
      if (v[1][j] == z && c + j > 0) eq |= 1u << j;
    }
    *reinterpret_cast<unsigned*>(edges + (size_t)r * (size_t)cols + (size_t)c) = flags;
  }
  if (parent) {
    // run starts: a lane's last cell that does not continue a run (or none); a cell with no start at or before it in
    // its own lane hangs off the start of the nearest lane to the left that has one (lane 0's first cell is one)
    const int last_start = eq == 0xFu ? (lane == 0 ? 0 : -1) : 31 - __clz((~eq & 0xFu) | (lane == 0 ? 1u : 0u));
    const unsigned has = __ballot_sync(0xffffffffu, last_start >= 0);
    const unsigned left = has & ((1u << lane) - 1u);
    const int src = left ? 31 - __clz(left) : 0;
    const int src_start = __shfl_sync(0xffffffffu, last_start, src);
    if (inside) {
      const unsigned base = (unsigned)r * (unsigned)cols + (unsigned)(c - 4 * lane);  // first cell of the warp's span
      unsigned from_left = base + 4u * (unsigned)src + (unsigned)src_start;
      if (lane == 0) from_left = base;
      unsigned p4[4];
      unsigned run = from_left;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (!((eq >> j) & 1u) || (lane == 0 && j == 0)) run = base + 4u * (unsigned)lane + (unsigned)j;
        p4[j] = run;
      }
      const size_t i = (size_t)r * (size_t)cols + (size_t)c;
      *reinterpret_cast<uint4*>(parent + i) = make_uint4(p4[0], p4[1], p4[2], p4[3]);
      *reinterpret_cast<uint4*>(minlow + i) = make_uint4(FL_NONE, FL_NONE, FL_NONE, FL_NONE);
    }
  }
  // one pair of counter atomics per CTA (1024 cells): every CTA of the raster adds to the same two words
  __shared__ unsigned s_lo, s_hi;
  if (threadIdx.x == 0) s_lo = s_hi = 0;
  __syncthreads();
  const unsigned lo = __reduce_add_sync(0xffffffffu, (unsigned)__popc(flags & 0x01010101u));
  const unsigned hi = __reduce_add_sync(0xffffffffu, (unsigned)__popc(flags & 0x02020202u));
  if (lane == 0) {
    if (lo) atomicAdd(&s_lo, lo);
    if (hi) atomicAdd(&s_hi, hi);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s_lo) atomicAdd(&cnt[CNT_LOW], s_lo);
    if (s_hi) atomicAdd(&cnt[CNT_HIGH], s_hi);
  }
}

// ---------------------------------------------------------------- equal-elevation components
__device__ __forceinline__ unsigned uf_find(unsigned* p, unsigned i) {
  unsigned cur = __ldcg(p + i);
  while (cur != i) {
    const unsigned nxt = __ldcg(p + cur);
    if (nxt != cur) p[i] = nxt;  // path halving; any ancestor is a valid parent
    i = cur;
    cur = nxt;
  }
  return i;
}

// read-only walk to the root (used once the forest is final: concurrent halving could overwrite a flattened entry)
__device__ __forceinline__ unsigned uf_find_ro(const unsigned* p, unsigned i) {
  unsigned cur = __ldcg(p + i);
  while (cur != i) {
    i = cur;
    cur = __ldcg(p + cur);
  }
  return i;
}

__device__ __forceinline__ void uf_unite(unsigned* p, unsigned a, unsigned b) {
  for (;;) {
    a = uf_find(p, a);
    b = uf_find(p, b);
    if (a == b) return;
    if (a < b) {
      const unsigned t = a;
      a = b;
      b = t;
    }
    const unsigned old = atomicMin(p + a, b);  // hook the larger root under the smaller one
    if (old == a) return;
    a = old;  // a was no longer a root: carry on from what it pointed to
  }
}

// Unions between runs.  Inside a row only the hand-over between warps is left (lane 31 -> lane 0).  Between rows a
// vertical pair needs a union only where one of the two runs begins (further right the pair to the left is the same
// two runs), and a diagonal pair only when neither the cell below nor the cell beside it continues a run that the
// vertical rule already ties in.
__global__ void __launch_bounds__(FL_THREADS)
flat_merge_kernel(const float* __restrict__ dem, int rows, int cols, unsigned* parent) {
  const unsigned i = blockIdx.x * FL_THREADS + threadIdx.x;
  if ((int64_t)blockIdx.x * FL_THREADS + threadIdx.x >= (int64_t)rows * cols) return;
  const int r = (int)(i / (unsigned)cols), c = (int)(i - (unsigned)r * (unsigned)cols);
  const float z = dem[i];
  const bool left_eq = c > 0 && dem[i - 1] == z;
  const bool right_eq = c + 1 < cols && dem[i + 1] == z;
  if (right_eq && (threadIdx.x & 31) == 31) uf_unite(parent, i, i + 1u);
  if (r + 1 < rows) {
    const unsigned j = i + (unsigned)cols;
    if (dem[j] == z) {
      if (!left_eq || !(dem[j - 1] == z)) uf_unite(parent, i, j);  // c == 0 implies !left_eq
    } else {
      if (c > 0 && !left_eq && dem[j - 1] == z) uf_unite(parent, i, j - 1u);
      if (c + 1 < cols && !right_eq && dem[j + 1] == z) uf_unite(parent, i, j + 1u);
    }
  }
}

// The same unions, four adjacent cells of a row per thread (width a multiple of 32): two float4 + four scalar loads
// instead of up to six per cell, and a sixteenth of the CTAs.  The hand-over inside a row stays at every 32nd cell,
// which covers both forest initialisations (32-cell groups, 128-cell spans).
__global__ void __launch_bounds__(FL_THREADS)
flat_merge4_kernel(const float* __restrict__ dem, int rows, int cols, unsigned* parent) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int r = blockIdx.y * (FL_THREADS / 32) + w;
  const int c = (blockIdx.x * 32 + lane) * 4;
  if (r >= rows || c >= cols) return;
  const size_t o = (size_t)r * (size_t)cols + (size_t)c;
  const float none = __int_as_float(0x7fc00000);  // NaN: equals nothing, like a cell that is not there
  float a[6], b[6];
  {
    const float4 m = *reinterpret_cast<const float4*>(dem + o);
    a[0] = c > 0 ? dem[o - 1] : none;
    a[1] = m.x;
    a[2] = m.y;
    a[3] = m.z;
    a[4] = m.w;
    a[5] = c + 4 < cols ? dem[o + 4] : none;
  }
  const bool below = r + 1 < rows;
  if (below) {
    const size_t o1 = o + (size_t)cols;
    const float4 m = *reinterpret_cast<const float4*>(dem + o1);
    b[0] = c > 0 ? dem[o1 - 1] : none;
    b[1] = m.x;
    b[2] = m.y;
    b[3] = m.z;
    b[4] = m.w;
    b[5] = c + 4 < cols ? dem[o1 + 4] : none;
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float z = a[j + 1];
    const unsigned i = (unsigned)o + (unsigned)j;
    const bool left_eq = a[j] == z, right_eq = a[j + 2] == z;
    if (right_eq && ((c + j) & 31) == 31) uf_unite(parent, i, i + 1u);
    if (below) {
      const unsigned jn = i + (unsigned)cols;
      if (b[j + 1] == z) {
        if (!left_eq || !(b[j] == z)) uf_unite(parent, i, jn);
      } else {
        if (!left_eq && b[j] == z) uf_unite(parent, i, jn - 1u);
        if (!right_eq && b[j + 2] == z) uf_unite(parent, i, jn + 1u);
      }
    }
  }
}

// The passes below only care about the flagged few cells: a thread reads four flag bytes as one word and a
// 1024-thread CTA covers 4096 cells (one thread per byte spent its time scheduling CTAs, not moving data).
constexpr int FL_CELLS_PER_CTA = 4 * FL_SCAN_THREADS;

__device__ __forceinline__ unsigned flag_word(const uint8_t* bytes, int64_t n, int64_t i0, bool aligned) {
  if (i0 >= n) return 0u;
  if (aligned && i0 + 4 <= n) return *reinterpret_cast<const unsigned*>(bytes + i0);
  unsigned w = 0;
  for (int k = 0; k < 4; ++k)
    if (i0 + k < n) w |= (unsigned)bytes[i0 + k] << (8 * k);
  return w;
}

// exclusive prefix of a per-thread count over the CTA (1024 threads); returns the CTA total through *total
__device__ __forceinline__ unsigned cta_exclusive(unsigned c, unsigned* total) {
  __shared__ unsigned warp_sum[FL_SCAN_THREADS / 32];
  __shared__ unsigned cta_total;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  unsigned inc = c;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const unsigned t = __shfl_up_sync(0xffffffffu, inc, off);
    if (lane >= off) inc += t;
  }
  if (lane == 31) warp_sum[w] = inc;
  __syncthreads();
  if (w == 0) {
    const unsigned v = warp_sum[lane];
    unsigned ws = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const unsigned t = __shfl_up_sync(0xffffffffu, ws, off);
      if (lane >= off) ws += t;
    }
    warp_sum[lane] = ws - v;
    if (lane == 31) cta_total = ws;
  }
  __syncthreads();
  *total = cta_total;
  return warp_sum[w] + inc - c;
}

// low edges look their root up (making their own pointer direct) and post their index to the root's slot
__global__ void __launch_bounds__(FL_SCAN_THREADS)
flat_lowroot_kernel(int64_t n, unsigned* parent, const uint8_t* __restrict__ edges, unsigned* minlow, unsigned* cnt) {
  const int64_t i0 = 4 * ((int64_t)blockIdx.x * FL_SCAN_THREADS + threadIdx.x);
  const unsigned w = flag_word(edges, n, i0, true) & 0x01010101u;
  if (w == 0) return;
  for (int k = 0; k < 4; ++k)
    if ((w >> (8 * k)) & 1u) {
      const unsigned i = (unsigned)(i0 + k);
      const unsigned root = uf_find_ro(parent, i);
      parent[i] = root;  // own entry only, and a root is a valid parent for any reader walking by
      if (__ldcg(minlow + root) > i) atomicMin(minlow + root, i);  // a plain look first: most low edges lose to an earlier one
      // cell 2^32 - 1 (the last cell of a raster of exactly 2^32 cells) looks like FL_NONE in minlow: when it is
      // its component's only low edge the slot says "none", and the labelling asks these two words instead
      if (i == FL_NONE) {
        cnt[CNT_LASTROOT] = root;
        cnt[CNT_LASTLOW] = 1u;
      }
    }
}

// a seed is the first low edge (row-major) of its component; bit k of the result: cell i0 + k is one
__device__ __forceinline__ unsigned seed_bits(int64_t n, int64_t i0, const unsigned* parent, const uint8_t* edges,
                                              const unsigned* minlow) {
  const unsigned w = flag_word(edges, n, i0, true) & 0x01010101u;
  unsigned bits = 0;
  if (w)
    for (int k = 0; k < 4; ++k)
      if (((w >> (8 * k)) & 1u) && minlow[parent[i0 + k]] == (unsigned)(i0 + k)) bits |= 1u << k;
  return bits;
}

__global__ void __launch_bounds__(FL_SCAN_THREADS)
flat_seed_count_kernel(int64_t n, const unsigned* parent, const uint8_t* __restrict__ edges, const unsigned* minlow,
                       int* blockcnt) {
  const int64_t i0 = 4 * ((int64_t)blockIdx.x * FL_SCAN_THREADS + threadIdx.x);
  unsigned total;
  cta_exclusive(__popc(seed_bits(n, i0, parent, edges, minlow)), &total);
  if (threadIdx.x == 0) blockcnt[blockIdx.x] = (int)total;
}

// exclusive scan of blockcnt[nb] in place (one CTA), total -> cnt[CNT_LABELS]
__global__ void __launch_bounds__(FL_SCAN_THREADS) flat_seed_scan_kernel(int nb, int* blockcnt, unsigned* cnt) {
  __shared__ int part[FL_SCAN_THREADS];
  const int t = threadIdx.x;
  const int per = (nb + FL_SCAN_THREADS - 1) / FL_SCAN_THREADS;
  const int lo = t * per, hi = min(nb, lo + per);
  int s = 0;
  for (int k = lo; k < hi; ++k) s += blockcnt[k];
  part[t] = s;
  __syncthreads();
  for (int off = 1; off < FL_SCAN_THREADS; off <<= 1) {  // Hillis-Steele inclusive scan
    const int v = t >= off ? part[t - off] : 0;
    __syncthreads();
    part[t] += v;
    __syncthreads();
  }
  int run = part[t] - s;
  for (int k = lo; k < hi; ++k) {
    const int v = blockcnt[k];
    blockcnt[k] = run;
    run += v;
  }
  if (t == FL_SCAN_THREADS - 1) cnt[CNT_LABELS] = (unsigned)part[t];
}

// seedlabel[i] = 1 + rank of seed i (row-major)
__global__ void __launch_bounds__(FL_SCAN_THREADS)
flat_seed_rank_kernel(int64_t n, const unsigned* parent, const uint8_t* __restrict__ edges, const unsigned* minlow,
                      const int* __restrict__ blockoff, int* seedlabel) {
  const int64_t i0 = 4 * ((int64_t)blockIdx.x * FL_SCAN_THREADS + threadIdx.x);
  const unsigned bits = seed_bits(n, i0, parent, edges, minlow);
  unsigned total;
  unsigned before = cta_exclusive(__popc(bits), &total) + (unsigned)blockoff[blockIdx.x];
  for (int k = 0; k < 4; ++k)
    if ((bits >> k) & 1u) seedlabel[i0 + k] = (int)(++before);
}

// Every cell takes the label of its component: root -> the component's smallest low edge -> that seed's label
// (0 when the component has no low edge).  The walk to the root is read-only (low edges already point at it).
// open[i] is the sweeps' one-word view of a cell: 0 = never a candidate (it has a direction), otherwise
// (label + 1) << 2 (the two low bits are the tile kernel's own flags in shared memory).
__device__ __forceinline__ unsigned flat_state(int lab) { return (unsigned)(lab + 1) << 2; }

__global__ void __launch_bounds__(FL_THREADS)
flat_spread_label_kernel(int64_t n, const unsigned* __restrict__ parent, const unsigned* __restrict__ minlow,
                         const int* __restrict__ seedlabel, int* labels, const uint8_t* __restrict__ fdr, unsigned* open,
                         const unsigned* __restrict__ cnt) {
  const int64_t i = (int64_t)blockIdx.x * FL_THREADS + threadIdx.x;
  if (i >= n) return;
  const unsigned root = uf_find_ro(parent, (unsigned)i);
  const unsigned m = minlow[root];
  int lab = 0;
  if (m != FL_NONE || (cnt[CNT_LASTLOW] && cnt[CNT_LASTROOT] == root)) lab = seedlabel[m];
  labels[i] = lab;
  open[i] = (fdr[i] == FL_UNDEF) ? flat_state(lab) : 0u;
}

// four cells per thread (cell count a multiple of 4, 16-byte aligned rasters): cells of one run share their parent, so
// the walk to the root and the two look-ups behind it are done once per run piece, not once per cell
__global__ void __launch_bounds__(FL_THREADS)
flat_spread_label4_kernel(int64_t n4, const unsigned* __restrict__ parent, const unsigned* __restrict__ minlow,
                          const int* __restrict__ seedlabel, int4* labels, const unsigned* __restrict__ fdr4, uint4* open,
                          const unsigned* __restrict__ cnt) {
  const int64_t q = (int64_t)blockIdx.x * FL_THREADS + threadIdx.x;
  if (q >= n4) return;
  const uint4 pv = reinterpret_cast<const uint4*>(parent)[q];
  const unsigned p[4] = {pv.x, pv.y, pv.z, pv.w};
  const unsigned codes = fdr4[q];
  int lab[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (j > 0 && p[j] == p[j - 1]) {
      lab[j] = lab[j - 1];
      continue;
    }
    const unsigned self = (unsigned)(4 * q + j);
    const unsigned root = p[j] == self ? self : uf_find_ro(parent, p[j]);
    const unsigned m = minlow[root];
    lab[j] = 0;
    if (m != FL_NONE || (cnt[CNT_LASTLOW] && cnt[CNT_LASTROOT] == root)) lab[j] = seedlabel[m];
  }
  labels[q] = make_int4(lab[0], lab[1], lab[2], lab[3]);
  unsigned o[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) o[j] = ((codes >> (8 * j)) & 0xFFu) == (unsigned)FL_UNDEF ? flat_state(lab[j]) : 0u;
  open[q] = make_uint4(o[0], o[1], o[2], o[3]);
}

// ---------------------------------------------------------------- gradients (away_from_higher / towards_lower)
// edge cells -> seed list, in no particular order (the sweeps are order-free); one queue atomic per CTA
__global__ void __launch_bounds__(FL_SCAN_THREADS)
flat_collect_kernel(int64_t n, const uint8_t* __restrict__ edges, unsigned bit, const int* __restrict__ labels,
                    unsigned* seeds, unsigned* cnt) {
  __shared__ unsigned cta_base;
  const int64_t i0 = 4 * ((int64_t)blockIdx.x * FL_SCAN_THREADS + threadIdx.x);
  const unsigned w = flag_word(edges, n, i0, true) & (bit * 0x01010101u);
  unsigned bits = 0;
  if (w)
    for (int k = 0; k < 4; ++k)  // fix_flats.py:273-274: high edges outside labelled flats drop out (low edges never do)
      if ((w >> (8 * k)) & 0xffu && labels[i0 + k] != 0) bits |= 1u << k;
  unsigned total;
  unsigned at = cta_exclusive(__popc(bits), &total);
  if (total == 0) return;
  if (threadIdx.x == 0) cta_base = atomicAdd(&cnt[CNT_SEEDS], total);
  __syncthreads();
  at += cta_base;
  for (int k = 0; k < 4; ++k)
    if ((bits >> k) & 1u) seeds[at++] = (unsigned)(i0 + k);
}

// Sweep modes: 0 away_from_higher; 1 towards_lower on a mask that was negated first (the standalone entry point,
// any caller-supplied mask); 2 towards_lower straight on the away sweep's mask (resolve_flats: every cell the away
// sweep valued is reached again, so the reference's negation never shows in the result and is not materialised).
enum { SWEEP_AWAY = 0, SWEEP_TOWARDS_NEGATED = 1, SWEEP_TOWARDS = 2 };

// standalone sweeps: towards_lower negates the mask (fix_flats.py:200); candidates are armed from the mask
__global__ void __launch_bounds__(FL_THREADS)
flat_prepare_kernel(int64_t n, int mode, int* flat_mask, const int* __restrict__ labels, const uint8_t* __restrict__ fdr,
                    unsigned* open) {
  const int64_t i = (int64_t)blockIdx.x * FL_THREADS + threadIdx.x;
  if (i >= n) return;
  int fm = flat_mask[i];
  if (mode != SWEEP_AWAY) {
    fm = -fm;
    flat_mask[i] = fm;
  }
  open[i] = (fdr[i] == FL_UNDEF && fm <= 0) ? flat_state(labels[i]) : 0u;
}

// The sweeps as tile relaxation.  A cell's value is its breadth-first level from the seed cells through candidate
// cells of the same label: the least fixpoint of  D(q) = 1 + min{ D(p) : p a neighbour of q with q's label },
// D(seed) = 1, which any relaxation order reaches.  The level-synchronous form of round 1 paid one kernel launch
// (13-27 us, a chain of dependent loads) per level, hundreds of levels per sweep.  Here the unit of scheduling is a
// tile of FT x FT cells: a CTA loads the tile's D and candidate words with a one-cell ring into shared memory,
// relaxes it to its own fixpoint with a frontier queue in shared memory (a level costs one CTA barrier, not a
// launch), writes the cells that improved back, and queues the neighbouring tiles whose ring it changed for the next
// pass.  One persistent kernel runs the passes with a grid barrier in between, so a sweep needs about
// (flat diameter / FT) passes and no host round trip.  A tile writes its own cells only; a ring read that is stale
// is still an upper bound, and whoever lowers it afterwards queues the reader again.
#ifndef OFL_FL_TILE
#define OFL_FL_TILE 32
#endif
constexpr int FT = OFL_FL_TILE;       // tile edge
constexpr int FTW = FT + 2;           // with the ring
constexpr int FT_CELLS = FTW * FTW;
#ifndef OFL_FL_QCAP
#define OFL_FL_QCAP (OFL_FL_TILE * OFL_FL_TILE + 256)
#endif
constexpr int FT_QCAP = OFL_FL_QCAP;  // entries of one in-tile frontier queue; beyond that the tile falls back to dense sweeps
#ifndef OFL_FL_SWEEP_THREADS
#define OFL_FL_SWEEP_THREADS 128
#endif
constexpr int FS_THREADS = OFL_FL_SWEEP_THREADS;  // threads of the CTA that relaxes a tile
static_assert(FS_THREADS >= 64 && FS_THREADS % 32 == 0, "whole warps, at least two");
constexpr int FL_INF = 0x7f7f7f7f;    // "not reached": what cudaMemsetAsync(0x7f) leaves

struct SweepArgs {
  int rows, cols, tiles_x, tiles_y, n_tiles;
  int* D;                // level per cell, FL_INF where the sweep has not come
  const unsigned* open;  // candidate words: 0 = cannot take a value, else (label + 1) << 2
  const int* labels;
  int* lists;            // three tile lists of n_tiles entries: pass k reads list k % 3 and fills list (k + 1) % 3
  int* stamp;            // per tile: 1 + the last pass it has been queued for
  int* seen;             // per tile: visited before
  unsigned* cnt;
};

__device__ __forceinline__ void tile_activate(const SweepArgs& a, int tile, int pass) {
  if (atomicMax(a.stamp + tile, pass + 1) < pass + 1)
    a.lists[(size_t)(pass % 3) * a.n_tiles + atomicAdd(&a.cnt[CNT_TCOUNT0 + pass % 3], 1u)] = tile;
}

// level 1: the seed cells (:146-148 / :202-204).  A seed that is not a candidate (a low edge: it has a direction)
// counts only while its mask is not positive (:150-151 / :207-208), like every cell the reference pops.
__global__ void __launch_bounds__(FL_THREADS)
flat_tile_seed_kernel(const unsigned* __restrict__ seeds, const int* __restrict__ flat_mask, SweepArgs a) {
  const int64_t n_seed = a.cnt[CNT_SEEDS];
  for (int64_t idx = (int64_t)blockIdx.x * FL_THREADS + threadIdx.x; idx < n_seed; idx += (int64_t)gridDim.x * FL_THREADS) {
    const unsigned p = seeds[idx];
    if (a.open[p] == 0u && flat_mask[p] > 0) continue;
    a.D[p] = 1;
    // its own tile, and the tiles that see it in their ring
    const int r = (int)(p / (unsigned)a.cols), c = (int)(p - (unsigned)r * (unsigned)a.cols);
    const int ty = r / FT, tx = c / FT, lr = r - ty * FT, lc = c - tx * FT;
    const int vr = lr == 0 ? -1 : (lr == FT - 1 ? 1 : 0), vc = lc == 0 ? -1 : (lc == FT - 1 ? 1 : 0);
    for (int dy = -1; dy <= 1; ++dy)
      for (int dx = -1; dx <= 1; ++dx) {
        if ((dy != 0 && dy != vr) || (dx != 0 && dx != vc)) continue;
        const int nty = ty + dy, ntx = tx + dx;
        if (nty < 0 || nty >= a.tiles_y || ntx < 0 || ntx >= a.tiles_x) continue;
        const int tile = nty * a.tiles_x + ntx;
        if (__ldcg(a.stamp + tile) == 0) tile_activate(a, tile, 0);
      }
  }
}

// Shared-memory image of a tile: FT x FT cells, the ring around them and one more guard ring that is never a
// candidate, so that any neighbour of a tile or ring cell is a valid index and needs no bounds check.
constexpr int FTS = FT + 4;  // row stride
constexpr int FT_IMG = FTS * FTS;
static_assert(FT_IMG < 65536, "queue entries are 16-bit image indices");
static_assert(FT_QCAP >= FT_CELLS, "the first round queues every valued cell of the tile and its ring");

struct TileSmem {
  int D[FT_IMG];
  // (label + 1) << 2 | flags.  A cell of the tile: 1 = candidate (may take a value), 2 = improved on this visit.
  // A cell of the ring: 2 = candidate (of its own tile; it never takes a value here).  Guard cells: 0.
  unsigned S[FT_IMG];
  uint16_t q[2][FT_QCAP];  // image indices (< 2^16)
  unsigned qn[3];    // round j reads qn[j % 3], fills qn[(j + 1) % 3] and clears qn[(j + 2) % 3]
  unsigned act;      // neighbouring tiles to queue, bit (dty + 1) * 3 + (dtx + 1)
  int overflow, changed;
  unsigned take, n_act;
};

// __syncthreads() is an aligned barrier: the warp has to arrive as one.  The loops below leave lanes at different
// points (a lane with no cell skips the body), so the warp is gathered explicitly first.
__device__ __forceinline__ void cta_sync() {
  __syncwarp();
  __syncthreads();
}

// image index of cell (lr, lc) of the tile-with-ring, 0 <= lr, lc < FTW
__device__ __forceinline__ int tile_img(int lr, int lc) { return (lr + 1) * FTS + lc + 1; }

// e-th cell of the square frame with corners (lo, lo) and (hi, hi): top row, bottom row, left column, right
// column, 4 * (hi - lo) cells in all
__device__ __forceinline__ void frame_cell(int e, int lo, int hi, int* lr, int* lc) {
  const int len = hi - lo, side = e / len, t = e - side * len;
  *lr = side == 0 ? lo : side == 1 ? hi : side == 2 ? lo + 1 + t : lo + t;
  *lc = side == 0 ? lo + t : side == 1 ? lo + 1 + t : side == 2 ? lo : hi;
}

// image offset of neighbour k (E NE N NW W SW S SE)
__device__ __forceinline__ int tile_off(int k) {
  const int dy = (k >= 1 && k <= 3) ? -1 : (k >= 5 ? 1 : 0);
  const int dx = (k == 0 || k == 1 || k == 7) ? 1 : ((k >= 3 && k <= 5) ? -1 : 0);
  return dy * FTS + dx;
}

// a cell with state s offers level d1 (its own + 1) to the cell at image index nidx; true when that cell improved
__device__ __forceinline__ bool tile_relax(TileSmem& sm, int nidx, int d1, unsigned s) {
  const unsigned ns = sm.S[nidx];
  if (!(ns & 1u) || ((ns ^ s) & ~3u) != 0u || sm.D[nidx] <= d1) return false;
  if (atomicMin(&sm.D[nidx], d1) <= d1) return false;
  if (!(ns & 2u)) sm.S[nidx] = ns | 2u;  // every writer stores the same word
  return true;
}

__device__ __forceinline__ void tile_push(TileSmem& sm, int which, uint16_t* q, int idx) {
  const unsigned at = atomicAdd(&sm.qn[which], 1u);
  if (at < FT_QCAP)
    q[at] = (uint16_t)idx;
  else
    sm.overflow = 1;
}

__device__ void tile_process(const SweepArgs& a, TileSmem& sm, int tile, int pass) {
  const int ty = tile / a.tiles_x, tx = tile - ty * a.tiles_x;
  const int r0 = ty * FT - 1, c0 = tx * FT - 1;
  if (threadIdx.x == 0) {
    sm.qn[0] = sm.qn[1] = sm.qn[2] = 0;
    sm.act = 0;
#ifdef OFL_FL_FORCE_DENSE
    sm.overflow = 1;  // test build: every tile takes the dense fallback
#else
    sm.overflow = 0;
#endif
  }
  const long long t0 = clock64();
  // the first visit finds seeds anywhere in the tile; later the tile's own cells are at their fixpoint and
  // only the ring brings news
  const bool first = __ldcg(a.seen + tile) == 0;
  for (int base = 0; base < FT_CELLS; base += FS_THREADS) {
    const int e = base + (int)threadIdx.x;
    if (e >= FT_CELLS) continue;
    const int lr = e / FTW, lc = e - lr * FTW;
    const int r = r0 + lr, c = c0 + lc;
    int d = FL_INF;
    unsigned s = 0;
    if (r >= 0 && r < a.rows && c >= 0 && c < a.cols) {
      const int64_t g = (int64_t)r * a.cols + c;
      d = __ldcg(a.D + g);
      const unsigned o = a.open[g];
      if (o)
        s = (o & ~3u) | ((lr >= 1 && lr <= FT && lc >= 1 && lc <= FT) ? 1u : 2u);
      else if (d < FL_INF)
        s = flat_state(a.labels[g]);  // a seed with a direction: gives, never takes
    }
    sm.D[tile_img(lr, lc)] = d;
    sm.S[tile_img(lr, lc)] = s;
  }
  cta_sync();
  // round 0: the valued cells (on later visits: of the ring only) are the first frontier
  {
    const int n_src = first ? FT_CELLS : 4 * (FT + 1);
    for (int base = 0; base < n_src; base += FS_THREADS) {
      const int e = base + (int)threadIdx.x;
      if (e >= n_src) continue;
      int lr, lc;
      if (first) {
        lr = e / FTW;
        lc = e - lr * FTW;
      } else {
        frame_cell(e, 0, FTW - 1, &lr, &lc);
      }
      const int idx = tile_img(lr, lc);
      if (sm.D[idx] < FL_INF) tile_push(sm, 0, sm.q[0], idx);
    }
  }
  // frontier rounds: a lane takes a queued cell and offers its level to the eight neighbours (the flags keep
  // ring and guard cells from taking it); the improved ones are appended warp by warp
  const long long t1 = clock64();
  int rounds = 0;
  for (int slot = 0;; ++rounds) {
    cta_sync();
    const unsigned n = min(sm.qn[slot], (unsigned)FT_QCAP);
    if (n == 0 || sm.overflow) break;
    const int next = slot == 2 ? 0 : slot + 1;
    if (threadIdx.x == 0) sm.qn[next == 2 ? 0 : next + 1] = 0;
    const uint16_t* qin = sm.q[rounds & 1];
    uint16_t* qout = sm.q[(rounds & 1) ^ 1];
    for (unsigned i0 = (threadIdx.x & ~31u); i0 < n; i0 += FS_THREADS) {  // warp-uniform bounds
      const unsigned i = i0 + (threadIdx.x & 31u);
      unsigned won = 0;
      int idx = 0;
      if (i < n) {
        idx = qin[i];
        const int d1 = sm.D[idx] + 1;
        const unsigned s = sm.S[idx];
        // four neighbours at a time: their words and levels are read before any of them is judged, so the
        // loads overlap (one after the other, a round was a chain of some thirty dependent accesses)
#pragma unroll
        for (int h = 0; h < 8; h += 4) {
          unsigned ns[4];
          int nd[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) ns[k] = sm.S[idx + tile_off(h + k)];
#pragma unroll
          for (int k = 0; k < 4; ++k) nd[k] = sm.D[idx + tile_off(h + k)];
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if ((ns[k] & 1u) && ((ns[k] ^ s) & ~3u) == 0u && nd[k] > d1 &&
                atomicMin(&sm.D[idx + tile_off(h + k)], d1) > d1) {
              if (!(ns[k] & 2u)) sm.S[idx + tile_off(h + k)] = ns[k] | 2u;
              won |= 1u << (h + k);
            }
        }
      }
      if (!__any_sync(0xffffffffu, won != 0u)) continue;
      const int lane = threadIdx.x & 31;
      int inc = __popc(won);  // inclusive prefix over the warp
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
      }
      unsigned at = 0;
      if (lane == 31) at = atomicAdd(&sm.qn[next], (unsigned)inc);
      at = __shfl_sync(0xffffffffu, at, 31) + (unsigned)(inc - __popc(won));
      for (; won; won &= won - 1u, ++at) {
        if (at < FT_QCAP)
          qout[at] = (uint16_t)(idx + tile_off(__ffs(won) - 1));
        else
          sm.overflow = 1;
      }
    }
    slot = next;
  }
  if (sm.overflow) {
    // a queue ran over (cells improved several times per round): dense sweeps to the same fixpoint
    for (;;) {
      cta_sync();
      if (threadIdx.x == 0) sm.changed = 0;
      cta_sync();
      bool any = false;
      for (int base = 0; base < FT_CELLS; base += FS_THREADS) {
        const int e = base + (int)threadIdx.x;
        if (e >= FT_CELLS) continue;
        const int lr = e / FTW, idx = tile_img(lr, e - lr * FTW);
        const int d = sm.D[idx];
        if (d >= FL_INF) continue;
        const unsigned s = sm.S[idx];
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) any |= tile_relax(sm, idx + tile_off(kk), d + 1, s);
      }
      if (any) sm.changed = 1;
      cta_sync();
      if (!sm.changed) break;
    }
  }
  cta_sync();
  const long long t2 = clock64();
  // improved cells go back
  for (int base = 0; base < FT * FT; base += FS_THREADS) {
    const int e = base + (int)threadIdx.x;
    if (e >= FT * FT) continue;
    const int lr = e / FT + 1, lc = e - (lr - 1) * FT + 1;
    const int idx = tile_img(lr, lc);
    if (sm.S[idx] & 2u) a.D[(int64_t)(r0 + lr) * a.cols + (c0 + lc)] = sm.D[idx];
  }
  // an improved cell on the tile's rim wakes a neighbouring tile if a cell of that tile (its value as of this
  // visit's load, an upper bound of what it holds now) could take a lower level from it
  for (int base = 0; base < 4 * (FT - 1); base += FS_THREADS) {
    const int e = base + (int)threadIdx.x;
    if (e >= 4 * (FT - 1)) continue;
    int lr, lc;
    frame_cell(e, 1, FT, &lr, &lc);
    const int idx = tile_img(lr, lc);
    const unsigned s = sm.S[idx];
    if (!(s & 2u)) continue;
    const int d1 = sm.D[idx] + 1;
    unsigned bits = 0;
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {
      const int nidx = idx + tile_off(kk);
      const unsigned ns = sm.S[nidx];
      if ((ns & 3u) == 2u && ((ns ^ s) & ~3u) == 0u && sm.D[nidx] > d1) {  // (ns & 3) == 2: a candidate on the ring
        const int nr = lr + c_dy[kk], nc = lc + c_dx[kk];
        bits |= 1u << (((nr < 1 ? -1 : nr > FT ? 1 : 0) + 1) * 3 + (nc < 1 ? -1 : nc > FT ? 1 : 0) + 1);
      }
    }
    if (bits) atomicOr(&sm.act, bits);
  }
  cta_sync();
  if (threadIdx.x == 32) {
    if (first) a.seen[tile] = 1;
    atomicAdd(&a.cnt[CNT_VISITS], 1u);
    atomicAdd(&a.cnt[CNT_ROUNDS], (unsigned)rounds);
    if (__ldcg(&a.cnt[CNT_MAXROUNDS]) < (unsigned)rounds) atomicMax(&a.cnt[CNT_MAXROUNDS], (unsigned)rounds);
    const long long t3 = clock64();
    atomicAdd(&a.cnt[CNT_CYC_LOAD], (unsigned)((t1 - t0) >> 6));
    atomicAdd(&a.cnt[CNT_CYC_ROUNDS], (unsigned)((t2 - t1) >> 6));
    atomicAdd(&a.cnt[CNT_CYC_STORE], (unsigned)((t3 - t2) >> 6));
  }
  if (threadIdx.x < 9 && ((sm.act >> threadIdx.x) & 1u)) {
    const int nty = ty + (int)threadIdx.x / 3 - 1, ntx = tx + (int)threadIdx.x % 3 - 1;
    if (nty >= 0 && nty < a.tiles_y && ntx >= 0 && ntx < a.tiles_x) tile_activate(a, nty * a.tiles_x + ntx, pass + 1);
  }
}

// The passes of one sweep: cooperative launch, every CTA resident.  Tiles of a pass are drawn from a counter.
#ifndef OFL_FL_SWEEP_CTAS
#define OFL_FL_SWEEP_CTAS 14  // 128 threads, 36 registers, 15.5 KB of shared memory (16-bit queue entries): 10 / 12 / 14 / 16 measured
#endif
__global__ void __launch_bounds__(FS_THREADS, OFL_FL_SWEEP_CTAS) flat_tile_sweep_kernel(SweepArgs a) {
  __shared__ TileSmem sm;
  unsigned generation = 0;
  for (int i = threadIdx.x; i < FT_IMG; i += FS_THREADS) {  // the guard ring stays like this
    sm.D[i] = FL_INF;
    sm.S[i] = 0u;
  }
  for (int pass = 0;; ++pass) {
    if (threadIdx.x == 0) sm.n_act = __ldcg(&a.cnt[CNT_TCOUNT0 + pass % 3]);
    if (blockIdx.x == 0 && threadIdx.x == 0) {  // the slots of pass + 2: last read in pass - 1
      a.cnt[CNT_TCOUNT0 + (pass + 2) % 3] = 0;
      a.cnt[CNT_TTAKE0 + (pass + 2) % 3] = 0;
      a.cnt[CNT_PASSES] = (unsigned)pass;
      if (pass < 40) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        a.cnt[CNT_PASSTIME0 + pass] = (unsigned)t;
      }
    }
    __syncthreads();
    const unsigned n_act = sm.n_act;
    if (n_act == 0) break;
    // thread 0 draws the CTA's next ticket while the current tile is processed (the atomic's round trip is hidden);
    // the tickets drawn past the end of the list are simply not used
    unsigned ticket = 0;
    if (threadIdx.x == 0) ticket = atomicAdd(&a.cnt[CNT_TTAKE0 + pass % 3], 1u);
    for (;;) {
      __syncthreads();
      if (threadIdx.x == 0) sm.take = ticket;
      __syncthreads();
      const unsigned t = sm.take;
      if (t >= n_act) break;
      if (threadIdx.x == 0) ticket = atomicAdd(&a.cnt[CNT_TTAKE0 + pass % 3], 1u);
      tile_process(a, sm, __ldcg(a.lists + (size_t)(pass % 3) * a.n_tiles + t), pass);
    }
    grid_barrier(&a.cnt[CNT_BAR], generation);
  }
}

// The sweep's levels become mask values (:153-154 / :209-214) and, for the away sweep, flat heights (the largest
// level of a flat; the reference's last write is the largest because levels only grow).  Neighbouring cells mostly
// share a label: a warp reduces per label before it touches flat_height.
__global__ void __launch_bounds__(FL_THREADS)
flat_tile_assign_kernel(int64_t n, int mode, const int* __restrict__ D, const unsigned* __restrict__ open,
                        const int* __restrict__ labels, int* flat_mask, const int* fh_read, int* fh_acc, unsigned* cnt) {
  const int64_t i = (int64_t)blockIdx.x * FL_THREADS + threadIdx.x;
  int d = 0, lab = 0;
  if (i < n) {
    d = D[i];
    if (d >= FL_INF) d = 0;
  }
  if (d > 0) {
    const unsigned o = open[i];
    lab = o ? (int)(o >> 2) - 1 : labels[i];
    if (mode == SWEEP_AWAY) {
      flat_mask[i] = d;
    } else {
      const int fm = flat_mask[i];
      int away = 0;  // flat_height - (increments away from higher terrain), 0 where the away sweep never came
      if (lab > 0) {
        if (mode == SWEEP_TOWARDS_NEGATED && fm < 0) away = fm + fh_read[lab - 1];
        if (mode == SWEEP_TOWARDS && fm > 0) away = fh_read[lab - 1] - fm;
      }
      flat_mask[i] = away + 2 * d;
    }
  }
  const int top = __reduce_max_sync(0xffffffffu, d);
  if (top == 0) return;  // warp-uniform
  if ((threadIdx.x & 31) == 0 && __ldcg(cnt + CNT_MAXLEVEL) < (unsigned)top) atomicMax(cnt + CNT_MAXLEVEL, (unsigned)top);
  if (mode != SWEEP_AWAY) return;
  const int key = d > 0 ? lab : 0;
  const unsigned grp = __match_any_sync(0xffffffffu, key);
  const int m = __reduce_max_sync(grp, d);
  if (key > 0 && (threadIdx.x & 31) == __ffs(grp) - 1 && __ldcg(fh_acc + key - 1) < m) atomicMax(fh_acc + key - 1, m);
}

// flat_height[k] takes the sweep's value where the sweep reached label k+1 (standalone away_from_higher)
__global__ void __launch_bounds__(FL_THREADS) flat_height_merge_kernel(int64_t n, const int* __restrict__ acc, int* fh) {
  const int64_t i = (int64_t)blockIdx.x * FL_THREADS + threadIdx.x;
  if (i < n && acc[i] > 0) fh[i] = acc[i];
}

// ---------------------------------------------------------------- d8_masked_flow_dirs (fix_flats.py:291-339)
// Slopes in float64 with the reference's division (:335-340).  (An exact integer comparison, b^2 against 2 a^2,
// was measured: it needs all eight differences in registers at once and ran 18 % slower; the kernel waits on its
// sixteen neighbour loads, not on the divisions.)
__device__ __forceinline__ int masked_dir_of(int64_t i, const int* __restrict__ flat_mask, const int* __restrict__ labels,
                                             int rows, int cols) {
  const int r = (int)(i / cols), c = (int)(i - (int64_t)r * cols);
  const int lab = labels[i];
  const double fm = (double)flat_mask[i];
  int nmin = FL_UNDEF;
  double min_slope = CUDART_INF;
  const bool inner = r > 0 && r + 1 < rows && c > 0 && c + 1 < cols;  // off the raster's ring: no bounds checks
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int nr = r + c_dy[k], nc = c + c_dx[k];
    if (!inner && (nr < 0 || nr >= rows || nc < 0 || nc >= cols)) continue;
    const int64_t j = (int64_t)nr * cols + nc;
    if (labels[j] != lab) continue;
    const double dz = (double)flat_mask[j] - fm;
    const double slope = (k & 1) ? __ddiv_rn(dz, 1.4142135623730951) : dz;  // odd codes are the diagonals
    if (slope < min_slope) {
      min_slope = slope;
      nmin = k;
    }
  }
  return nmin;
}

// a thread looks at four codes at once; only cells without a direction cost anything
__global__ void __launch_bounds__(FL_THREADS)
flat_masked_dirs_kernel(const int* __restrict__ flat_mask, const int* __restrict__ labels, uint8_t* fdr, int rows,
                        int cols, int aligned) {
  const int64_t n = (int64_t)rows * cols;
  const int64_t i0 = 4 * ((int64_t)blockIdx.x * FL_THREADS + threadIdx.x);
  const unsigned w = flag_word(fdr, n, i0, aligned != 0);
  for (int k = 0; k < 4; ++k)
    if (i0 + k < n && ((w >> (8 * k)) & 0xffu) == (unsigned)FL_UNDEF)
      fdr[i0 + k] = (uint8_t)masked_dir_of(i0 + k, flat_mask, labels, rows, cols);
}

// The same with the sixteen neighbour values of a cell shared between the four cells of a thread (width a multiple
// of 4, 16-byte aligned rasters): the kernel waits on its loads, and these are three int4 + six scalar loads per raster
// for four cells instead of sixteen scalar loads per cell.  Threads whose four cells all have a direction load nothing.
__global__ void __launch_bounds__(FL_THREADS)
flat_masked_dirs4_kernel(const int* __restrict__ flat_mask, const int* __restrict__ labels, uint8_t* fdr, int rows, int cols) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int r = blockIdx.y * (FL_THREADS / 32) + w;
  const int c = (blockIdx.x * 32 + lane) * 4;
  if (r >= rows || c >= cols) return;
  const size_t o = (size_t)r * (size_t)cols + (size_t)c;
  unsigned codes = *reinterpret_cast<const unsigned*>(fdr + o);
  // bytes equal to FL_UNDEF (8): x ^ 0x08 == 0
  const unsigned x8 = codes ^ 0x08080808u;
  const unsigned undef = ~(((x8 & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x8) & 0x80808080u;
  if (!undef) return;
  int fm[3][6], lb[3][6];
  bool row_ok[3];
  const bool left_ok = c > 0, right_ok = c + 4 < cols;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int rr = r + k - 1;
    row_ok[k] = rr >= 0 && rr < rows;
    if (!row_ok[k]) {
#pragma unroll
      for (int x = 0; x < 6; ++x) fm[k][x] = lb[k][x] = 0;
    } else {
      const size_t ok = (size_t)rr * (size_t)cols + (size_t)c;
      const int4 m = *reinterpret_cast<const int4*>(flat_mask + ok);
      const int4 l = *reinterpret_cast<const int4*>(labels + ok);
      fm[k][1] = m.x, fm[k][2] = m.y, fm[k][3] = m.z, fm[k][4] = m.w;
      lb[k][1] = l.x, lb[k][2] = l.y, lb[k][3] = l.z, lb[k][4] = l.w;
      fm[k][0] = left_ok ? flat_mask[ok - 1] : 0;
      lb[k][0] = left_ok ? labels[ok - 1] : 0;
      fm[k][5] = right_ok ? flat_mask[ok + 4] : 0;
      lb[k][5] = right_ok ? labels[ok + 4] : 0;
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (!((undef >> (8 * j + 7)) & 1u)) continue;
    const int lab = lb[1][j + 1];
    const double f0 = (double)fm[1][j + 1];
    int nmin = FL_UNDEF;
    double min_slope = CUDART_INF;
#pragma unroll
    for (int k = 0; k < 8; ++k) {  // E NE N NW W SW S SE
      const int dy = (k >= 1 && k <= 3) ? -1 : (k >= 5 ? 1 : 0);
      const int dx = (k == 0 || k == 1 || k == 7) ? 1 : ((k >= 3 && k <= 5) ? -1 : 0);
      const int x = j + 1 + dx;
      if (!row_ok[1 + dy] || (x == 0 && !left_ok) || (x == 5 && !right_ok)) continue;  // off the raster
      if (lb[1 + dy][x] != lab) continue;
      const double dz = (double)fm[1 + dy][x] - f0;
      const double slope = (k & 1) ? __ddiv_rn(dz, 1.4142135623730951) : dz;
      if (slope < min_slope) {
        min_slope = slope;
        nmin = k;
      }
    }
    codes = (codes & ~(0xFFu << (8 * j))) | ((unsigned)nmin << (8 * j));
  }
  *reinterpret_cast<unsigned*>(fdr + o) = codes;
}

inline unsigned blocks_for(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

// the row-wise kernels (a warp = 128 consecutive cells of a row, a CTA = eight rows): usable when the width is a
// multiple of `mult` and the row count fits gridDim.y
bool rows_vector_ok(int64_t rows, int64_t cols, int mult) {
  return cols % mult == 0 && (rows + FL_THREADS / 32 - 1) / (FL_THREADS / 32) <= 65535 && !getenv("OFL_FLATS_SCALAR");
}
dim3 rows_grid(int64_t rows, int64_t cols) {
  return dim3((unsigned)((cols / 4 + 31) / 32), (unsigned)((rows + FL_THREADS / 32 - 1) / (FL_THREADS / 32)));
}

// flat_edges over the raster: the four-cells-per-thread form where the layout allows it
int launch_edges_kernel(const float* dem, const uint8_t* fdr, int64_t rows, int64_t cols, uint8_t* edges, unsigned* parent,
                        unsigned* minlow, unsigned* cnt, cudaStream_t st) {
  const bool vec = rows_vector_ok(rows, cols, 32) && (reinterpret_cast<uintptr_t>(dem) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(fdr) & 3) == 0 && (reinterpret_cast<uintptr_t>(edges) & 3) == 0;
  if (vec) {
    flat_edges4_kernel<<<rows_grid(rows, cols), FL_THREADS, 0, st>>>(dem, fdr, (int)rows, (int)cols, edges, parent, minlow, cnt);
  } else {
    flat_edges_kernel<<<blocks_for(rows * cols, FL_THREADS), FL_THREADS, 0, st>>>(dem, fdr, (int)rows, (int)cols, edges, parent,
                                                                               minlow, cnt);
  }
  OFL_CHECK_LAUNCH();
  return OFL_OK;
}

// The same, four cells per thread (cell count a multiple of 4, 16-byte aligned rasters): int4 loads and stores, and
// quads the sweep never reached cost one load.
__global__ void __launch_bounds__(FL_THREADS)
flat_tile_assign4_kernel(int64_t n4, int mode, const int4* __restrict__ D, const uint4* __restrict__ open,
                         const int* __restrict__ labels, int4* flat_mask, const int* fh_read, int* fh_acc, unsigned* cnt) {
  const int64_t q = (int64_t)blockIdx.x * FL_THREADS + threadIdx.x;
  int top = 0, key = 0, kmax = 0;  // key / kmax: the label of the thread's last valued cell and the largest level seen for it
  if (q < n4) {
    const int4 dv = D[q];
    int d[4] = {dv.x, dv.y, dv.z, dv.w};
    if (d[0] < FL_INF || d[1] < FL_INF || d[2] < FL_INF || d[3] < FL_INF) {
      const uint4 ov = open[q];
      const unsigned o[4] = {ov.x, ov.y, ov.z, ov.w};
      int4 mv = make_int4(0, 0, 0, 0);
      if (mode != SWEEP_AWAY) mv = flat_mask[q];
      int m[4] = {mv.x, mv.y, mv.z, mv.w};
      bool any = false;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (d[j] >= FL_INF) continue;
        any = true;
        const int lab = o[j] ? (int)(o[j] >> 2) - 1 : labels[4 * q + j];
        if (mode == SWEEP_AWAY) {
          m[j] = d[j];
          if (lab > 0) {
            if (lab != key && key > 0 && __ldcg(fh_acc + key - 1) < kmax) atomicMax(fh_acc + key - 1, kmax);
            kmax = lab == key ? max(kmax, d[j]) : d[j];
            key = lab;
          }
        } else {
          int away = 0;  // flat_height - (increments away from higher terrain), 0 where the away sweep never came
          if (lab > 0) {
            if (mode == SWEEP_TOWARDS_NEGATED && m[j] < 0) away = m[j] + fh_read[lab - 1];
            if (mode == SWEEP_TOWARDS && m[j] > 0) away = fh_read[lab - 1] - m[j];
          }
          m[j] = away + 2 * d[j];
        }
        top = max(top, d[j]);
      }
      if (any) {
        if (mode == SWEEP_AWAY) {
          // cells the sweep did not reach keep their mask: write only the valued ones' lanes of the quad
          int* out = reinterpret_cast<int*>(flat_mask + q);
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (d[j] < FL_INF) out[j] = m[j];
        } else {
          flat_mask[q] = make_int4(m[0], m[1], m[2], m[3]);
        }
      }
    }
  }
  const int wtop = __reduce_max_sync(0xffffffffu, top);
  if (wtop == 0) return;  // warp-uniform
  if ((threadIdx.x & 31) == 0 && __ldcg(cnt + CNT_MAXLEVEL) < (unsigned)wtop) atomicMax(cnt + CNT_MAXLEVEL, (unsigned)wtop);
  if (mode != SWEEP_AWAY) return;
  const unsigned grp = __match_any_sync(0xffffffffu, key);
  const int gm = __reduce_max_sync(grp, kmax);
  if (key > 0 && (threadIdx.x & 31) == __ffs(grp) - 1 && __ldcg(fh_acc + key - 1) < gm) atomicMax(fh_acc + key - 1, gm);
}

struct FlatsWork {
  unsigned* parent;  // union-find forest, later flat_height
  int* q0;           // block counts of the label scan, later the sweeps' level per cell
  unsigned* q1;      // smallest low edge per component, later the seed list
  unsigned* open;  // the sweeps' candidate words
  uint8_t* edges;
  unsigned* cnt;
  int* tiles;   // three tile lists and the tile stamps of the sweeps
  size_t bytes;  // size of the workspace
};

int64_t sweep_tiles(int64_t rows, int64_t cols) { return ((rows + FT - 1) / FT) * ((cols + FT - 1) / FT); }

// Cuts the workspace at `base` into its buffers; with a null base only `bytes` is meaningful.
FlatsWork flats_layout(void* base, int64_t rows, int64_t cols) {
  const size_t n = (size_t)(rows * cols);
  FlatsWork w;
  Carver c(base);
  c.take(w.parent, n * sizeof(int));
  c.take(w.q0, n * sizeof(int));
  c.take(w.q1, n * sizeof(int));
  c.take(w.open, n * sizeof(int));
  c.take(w.edges, n);
  c.take(w.cnt, CNT_SLOTS * sizeof(unsigned));
  c.take(w.tiles, (size_t)sweep_tiles(rows, cols) * 5 * sizeof(int));
  w.bytes = c.bytes;
  return w;
}

// One sweep from the seed list in w.q1 (count in cnt[CNT_SEEDS]): levels by tile relaxation, then mask values.
// Asynchronous unless the caller wants the level count.
int run_gradient(int rows, int cols, const int* labels, const uint8_t* fdr, int mode, bool open_ready, int* flat_mask,
                 const int* fh_read, int* fh_acc, const FlatsWork& w, int64_t* levels_out, cudaStream_t st) {
  // open_ready: w.open already describes the candidates (resolve_flats: armed by the labelling, the same for both
  // sweeps); otherwise they are armed from the mask, negated first for towards_lower
  const int64_t n = (int64_t)rows * cols;
  SweepArgs a;
  a.rows = rows;
  a.cols = cols;
  a.tiles_x = (cols + FT - 1) / FT;
  a.tiles_y = (rows + FT - 1) / FT;
  a.n_tiles = a.tiles_x * a.tiles_y;
  a.D = w.q0;
  a.open = w.open;
  a.labels = labels;
  a.lists = w.tiles;
  a.stamp = w.tiles + (size_t)3 * a.n_tiles;
  a.seen = w.tiles + (size_t)4 * a.n_tiles;
  a.cnt = w.cnt;
  OFL_CUDA(cudaMemsetAsync(w.cnt + CNT_TCOUNT0, 0, (CNT_SLOTS - CNT_TCOUNT0) * sizeof(unsigned), st));
  OFL_CUDA(cudaMemsetAsync(a.stamp, 0, (size_t)2 * a.n_tiles * sizeof(int), st));  // stamps and seen flags
  OFL_CUDA(cudaMemsetAsync(a.D, 0x7f, (size_t)n * sizeof(int), st));
  if (!open_ready) {
    flat_prepare_kernel<<<blocks_for(n, FL_THREADS), FL_THREADS, 0, st>>>(n, mode, flat_mask, labels, fdr, w.open);
    OFL_CHECK_LAUNCH();
  }
  flat_tile_seed_kernel<<<(unsigned)(sm_count() * 8), FL_THREADS, 0, st>>>(w.q1, flat_mask, a);
  OFL_CHECK_LAUNCH();
  {
    // persistent: as many CTAs as are resident at once (the grid barrier needs them all)
    const void* sweep = reinterpret_cast<const void*>(flat_tile_sweep_kernel);
    void* args[] = {&a};
    OFL_CUDA(cudaLaunchCooperativeKernel(sweep, dim3((unsigned)resident_ctas(sweep, FS_THREADS)), dim3(FS_THREADS), args, 0, st));
  }
  if (n % 4 == 0 && (reinterpret_cast<uintptr_t>(flat_mask) & 15) == 0 && !getenv("OFL_FLATS_SCALAR"))
    flat_tile_assign4_kernel<<<blocks_for(n / 4, FL_THREADS), FL_THREADS, 0, st>>>(
        n / 4, mode, reinterpret_cast<const int4*>(a.D), reinterpret_cast<const uint4*>(w.open), labels,
        reinterpret_cast<int4*>(flat_mask), fh_read, fh_acc, w.cnt);
  else
    flat_tile_assign_kernel<<<blocks_for(n, FL_THREADS), FL_THREADS, 0, st>>>(n, mode, a.D, w.open, labels, flat_mask, fh_read,
                                                                              fh_acc, w.cnt);
  OFL_CHECK_LAUNCH();
  if (levels_out) {
    unsigned* h_cnt = nullptr;
    int rc = pinned_get(256, reinterpret_cast<void**>(&h_cnt));
    if (rc != OFL_OK) return rc;
    OFL_CUDA(cudaMemcpyAsync(h_cnt, w.cnt + CNT_PASSES, (CNT_SLOTS - CNT_PASSES) * sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    OFL_CUDA(cudaStreamSynchronize(st));
    *levels_out = h_cnt[CNT_MAXLEVEL - CNT_PASSES];
    if (getenv("OFL_FLATS_DEBUG"))
      fprintf(stderr, "[flats sweep mode %d] tiles %d passes %u tile visits %u in-tile rounds %u levels %u\n", mode, a.n_tiles,
              h_cnt[0], h_cnt[CNT_VISITS - CNT_PASSES], h_cnt[CNT_ROUNDS - CNT_PASSES], h_cnt[CNT_MAXLEVEL - CNT_PASSES]);
    if (getenv("OFL_FLATS_DEBUG")) {
      fprintf(stderr, "  most rounds in a visit %u; pass durations (us):", h_cnt[CNT_MAXROUNDS - CNT_PASSES]);
      for (unsigned k = 0; k + 1 <= h_cnt[0] && k + 1 < 40; ++k)
        fprintf(stderr, " %.0f", (h_cnt[CNT_PASSTIME0 - CNT_PASSES + k + 1] - h_cnt[CNT_PASSTIME0 - CNT_PASSES + k]) * 1e-3);
      fprintf(stderr, "\n  cycles per visit: load %.0f, rounds %.0f (%.0f per round), store + wake %.0f\n",
              64.0 * h_cnt[CNT_CYC_LOAD - CNT_PASSES] / h_cnt[CNT_VISITS - CNT_PASSES],
              64.0 * h_cnt[CNT_CYC_ROUNDS - CNT_PASSES] / h_cnt[CNT_VISITS - CNT_PASSES],
              64.0 * h_cnt[CNT_CYC_ROUNDS - CNT_PASSES] / (h_cnt[CNT_ROUNDS - CNT_PASSES] + h_cnt[CNT_VISITS - CNT_PASSES]),
              64.0 * h_cnt[CNT_CYC_STORE - CNT_PASSES] / h_cnt[CNT_VISITS - CNT_PASSES]);
    }
  }
  return OFL_OK;
}

}  // namespace

size_t flats_workspace_bytes(int64_t rows, int64_t cols) { return flats_layout(nullptr, rows, cols).bytes; }

// One tile of at most 2^32 cells: cell indices are unsigned 32-bit on the device.
int flats_shape(int64_t rows, int64_t cols) {
  OFL_REQUIRE(rows > 0 && cols > 0 && rows < (1ll << 31) && cols < (1ll << 31) && rows * cols <= (1ll << 32), OFL_ERR_INVALID,
              "flat resolution works on one tile of at most 2^32 cells (got %lld x %lld)", (long long)rows,
              (long long)cols);
  return OFL_OK;
}

// edges[i]: bit 0 low edge, bit 1 high edge; counts -> host.  Dense rasters (ld == cols), device pointers.
int launch_flat_edges(const float* dem, const uint8_t* fdr, int64_t rows, int64_t cols, uint8_t* edges, int64_t* n_low,
                      int64_t* n_high, unsigned* cnt_dev, cudaStream_t st) {
  PhaseScope ps(PHASE_FLATS, st);
  OFL_CUDA(cudaMemsetAsync(cnt_dev, 0, CNT_SLOTS * sizeof(unsigned), st));
  int rc = launch_edges_kernel(dem, fdr, rows, cols, edges, nullptr, nullptr, cnt_dev, st);
  if (rc != OFL_OK) return rc;
  unsigned* h = nullptr;
  rc = pinned_get(256, reinterpret_cast<void**>(&h));
  if (rc != OFL_OK) return rc;
  OFL_CUDA(cudaMemcpyAsync(h, cnt_dev, 2 * sizeof(unsigned), cudaMemcpyDeviceToHost, st));
  OFL_CUDA(cudaStreamSynchronize(st));
  if (n_low) *n_low = h[CNT_LOW];
  if (n_high) *n_high = h[CNT_HIGH];
  return OFL_OK;
}

// resolve_flats (fix_flats.py:227-288).  All pointers device, dense.  info (host, nullable) receives
// {low edges, high edges, labels, levels of the away sweep, levels of the towards sweep}.
int launch_resolve_flats(const float* dem, const uint8_t* fdr, int64_t rows, int64_t cols, int* flat_mask, int* labels,
                         int64_t* info, void* workspace, cudaStream_t st) {
  const int64_t n = rows * cols;
  const FlatsWork w = flats_layout(workspace, rows, cols);
  const unsigned nb = blocks_for(n, FL_THREADS), nbc = blocks_for(n, FL_CELLS_PER_CTA);
  OFL_CUDA(cudaMemsetAsync(w.cnt, 0, CNT_SLOTS * sizeof(unsigned), st));
  int* flat_height = reinterpret_cast<int*>(w.parent);  // lives where the forest was once the labels are known
  unsigned* minlow = w.q1;      // per-component smallest low edge, until the labels are known
  int* seedlabel = flat_mask;   // label of each component's first low edge, until the labels are known
  unsigned* h = nullptr;
  int rc = pinned_get(256, reinterpret_cast<void**>(&h));
  if (rc != OFL_OK) return rc;
  int64_t lv_away = 0, lv_low = 0;
  {
    PhaseScope ps(PHASE_FLATS_LABEL, st);
    rc = launch_edges_kernel(dem, fdr, rows, cols, w.edges, w.parent, minlow, w.cnt, st);
    if (rc != OFL_OK) return rc;
    if (rows_vector_ok(rows, cols, 32) && (reinterpret_cast<uintptr_t>(dem) & 15) == 0)
      flat_merge4_kernel<<<rows_grid(rows, cols), FL_THREADS, 0, st>>>(dem, (int)rows, (int)cols, w.parent);
    else
      flat_merge_kernel<<<nb, FL_THREADS, 0, st>>>(dem, (int)rows, (int)cols, w.parent);
    OFL_CHECK_LAUNCH();
    flat_lowroot_kernel<<<nbc, FL_SCAN_THREADS, 0, st>>>(n, w.parent, w.edges, minlow, w.cnt);
    OFL_CHECK_LAUNCH();
    flat_seed_count_kernel<<<nbc, FL_SCAN_THREADS, 0, st>>>(n, w.parent, w.edges, minlow, w.q0);
    OFL_CHECK_LAUNCH();
    flat_seed_scan_kernel<<<1, FL_SCAN_THREADS, 0, st>>>((int)nbc, w.q0, w.cnt);
    OFL_CHECK_LAUNCH();
    flat_seed_rank_kernel<<<nbc, FL_SCAN_THREADS, 0, st>>>(n, w.parent, w.edges, minlow, w.q0, seedlabel);
    OFL_CHECK_LAUNCH();
    // one look at the counts: nothing to do without low edges (fix_flats.py:258-264), and flat_height needs
    // only as many cleared entries as there are labels
    OFL_CUDA(cudaMemcpyAsync(h, w.cnt, 3 * sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    OFL_CUDA(cudaStreamSynchronize(st));
    const unsigned n_low = h[CNT_LOW], n_high = h[CNT_HIGH], n_labels = h[CNT_LABELS];
    if (info) {
      info[0] = n_low;
      info[1] = n_high;
      info[2] = n_labels;
    }
    OFL_REQUIRE(n_labels < (1u << 29), OFL_ERR_INVALID, "more than 2^29 flats in one tile");
    if (n_labels == 0) {
      OFL_CUDA(cudaMemsetAsync(labels, 0, (size_t)n * sizeof(int), st));
      OFL_CUDA(cudaMemsetAsync(flat_mask, 0, (size_t)n * sizeof(int), st));
      return OFL_OK;
    }
    if (n % 4 == 0 && (reinterpret_cast<uintptr_t>(labels) & 15) == 0 && (reinterpret_cast<uintptr_t>(fdr) & 3) == 0 &&
        !getenv("OFL_FLATS_SCALAR"))
      flat_spread_label4_kernel<<<blocks_for(n / 4, FL_THREADS), FL_THREADS, 0, st>>>(
          n / 4, w.parent, minlow, seedlabel, reinterpret_cast<int4*>(labels), reinterpret_cast<const unsigned*>(fdr),
          reinterpret_cast<uint4*>(w.open), w.cnt);
    else
      flat_spread_label_kernel<<<nb, FL_THREADS, 0, st>>>(n, w.parent, minlow, seedlabel, labels, fdr, w.open, w.cnt);
    OFL_CHECK_LAUNCH();
    OFL_CUDA(cudaMemsetAsync(flat_mask, 0, (size_t)n * sizeof(int), st));
    OFL_CUDA(cudaMemsetAsync(flat_height, 0, ((size_t)n_labels + 1) * sizeof(int), st));
  }
  PhaseScope ps(PHASE_FLATS_SWEEP, st);
  flat_collect_kernel<<<nbc, FL_SCAN_THREADS, 0, st>>>(n, w.edges, 2u, labels, w.q1, w.cnt);
  OFL_CHECK_LAUNCH();
  rc = run_gradient((int)rows, (int)cols, labels, fdr, SWEEP_AWAY, true, flat_mask, flat_height, flat_height, w, info ? &lv_away : nullptr, st);
  if (rc != OFL_OK) return rc;
  OFL_CUDA(cudaMemsetAsync(w.cnt + CNT_SEEDS, 0, sizeof(unsigned), st));
  flat_collect_kernel<<<nbc, FL_SCAN_THREADS, 0, st>>>(n, w.edges, 1u, labels, w.q1, w.cnt);
  OFL_CHECK_LAUNCH();
  rc = run_gradient((int)rows, (int)cols, labels, fdr, SWEEP_TOWARDS, true, flat_mask, flat_height, flat_height, w, info ? &lv_low : nullptr, st);
  if (rc != OFL_OK) return rc;
  if (info) {
    info[3] = lv_away;
    info[4] = lv_low;
  }
  return OFL_OK;
}

// Standalone away_from_higher (towards == 0) / towards_lower (towards == 1) from a caller-supplied seed list
// (cell indices, device).  flat_height has n_heights entries (device).
int launch_flat_gradient(const int* labels, const uint8_t* fdr, int64_t rows, int64_t cols, const int* seeds,
                         int64_t n_seeds, int towards, int* flat_mask, int* flat_height, int64_t n_heights,
                         void* workspace, cudaStream_t st) {
  const int64_t n = rows * cols;
  const FlatsWork w = flats_layout(workspace, rows, cols);
  PhaseScope ps(PHASE_FLATS, st);
  OFL_CUDA(cudaMemsetAsync(w.cnt, 0, CNT_SLOTS * sizeof(unsigned), st));
  const unsigned ns = (unsigned)n_seeds;
  OFL_CUDA(cudaMemcpyAsync(w.cnt + CNT_SEEDS, &ns, sizeof(unsigned), cudaMemcpyHostToDevice, st));
  OFL_CUDA(cudaStreamSynchronize(st));  // `ns` is a stack variable
  if (n_seeds) OFL_CUDA(cudaMemcpyAsync(w.q1, seeds, (size_t)n_seeds * sizeof(int), cudaMemcpyDeviceToDevice, st));
  int* acc = reinterpret_cast<int*>(w.parent);  // the sweep's own maxima; merged below so untouched labels keep the caller's value
  OFL_CUDA(cudaMemsetAsync(acc, 0, (size_t)n * sizeof(int), st));
  const int rc = run_gradient((int)rows, (int)cols, labels, fdr, towards ? SWEEP_TOWARDS_NEGATED : SWEEP_AWAY, false, flat_mask,
                    flat_height, acc, w, nullptr, st);
  if (rc != OFL_OK) return rc;
  if (!towards && n_heights) {
    flat_height_merge_kernel<<<blocks_for(n_heights, FL_THREADS), FL_THREADS, 0, st>>>(n_heights, acc, flat_height);
    OFL_CHECK_LAUNCH();
  }
  return OFL_OK;
}

int launch_masked_flow_dirs(const int* flat_mask, const int* labels, uint8_t* fdr, int64_t rows, int64_t cols,
                            cudaStream_t st) {
  PhaseScope ps(PHASE_FLATS, st);
  const int aligned = (reinterpret_cast<uintptr_t>(fdr) & 3u) == 0;
  if (rows_vector_ok(rows, cols, 4) && aligned && (reinterpret_cast<uintptr_t>(flat_mask) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(labels) & 15) == 0)
    flat_masked_dirs4_kernel<<<rows_grid(rows, cols), FL_THREADS, 0, st>>>(flat_mask, labels, fdr, (int)rows, (int)cols);
  else
    flat_masked_dirs_kernel<<<blocks_for((rows * cols + 3) / 4, FL_THREADS), FL_THREADS, 0, st>>>(flat_mask, labels, fdr,
                                                                                                    (int)rows, (int)cols, aligned);
  OFL_CHECK_LAUNCH();
  return OFL_OK;
}

}  // namespace ofl
