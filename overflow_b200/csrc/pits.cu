// pits.cu -- single-cell pit breaching on the device: the reference's
// src/overflow/breach_single_cell_pits.py:9-63 (breach_single_cell_pits_in_chunk).
//
// The reference finds the pits of the incoming chunk in a parallel pass (a cell whose eight neighbours are all
// strictly higher and none of them NODATA), then visits them ONE BY ONE in row-major order: a pit looks at the
// sixteen cells two steps away and, for each that is not higher (or is NODATA), writes the mean of the two
// elevations into the cell between them.  That second pass is order dependent -- a pit may read a cell an
// earlier pit has lowered, and two pits may write the same cell, the later one winning -- but only locally: a
// pit writes within one cell of itself and reads within two, so two pits interact only when they are at most
// three cells apart (chessboard distance).  Here the pits are collected into a list and breached in rounds: a
// pit is ready when no EARLIER pit within distance three is still waiting; the ready pits of a round are more
// than three cells apart from each other, so they run concurrently on disjoint cells and every pit sees exactly
// the chunk the reference's sequential loop would show it.  The earliest waiting pit is always ready, so the
// rounds end; on terrain they number a handful.
//
// Arithmetic as numba types it for a float32 chunk: float32 sum, float64 division by two, float32 store; the
// NODATA test compares in float64.  Bit-exact against the reference (tests/golden/breach_pits.npz).
#include <math_constants.h>

#include <cstdlib>

#include "common.cuh"

namespace ofl {
namespace {

constexpr int PT = 256;
enum { PC_PITS = 0, PC_ROUNDS, PC_UNSOLVED, PC_BARRIER, PC_RELEASE, PC_NEXT0, PC_NEXT1, PC_SLOTS = 16 };

__constant__ int p_dx[8] = {1, 1, 1, 0, -1, -1, -1, 0};  // breach_single_cell_pits.py:27-31
__constant__ int p_dy[8] = {-1, 0, 1, 1, 1, 0, -1, -1};
__constant__ int p_dx2[16] = {2, 2, 2, 2, 2, 1, 0, -1, -2, -2, -2, -2, -2, -1, 0, 1};
__constant__ int p_dy2[16] = {-2, -1, 0, 1, 2, 2, 2, 2, 2, 1, 0, -1, -2, -2, -2, -2};
__constant__ int p_breach[16] = {0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 0};

// pass 1 (:38-50): pits of the chunk as it came in -> unsolved = waiting = 1, index appended to the list
__global__ void __launch_bounds__(PT)
pits_detect_kernel(const float* __restrict__ chunk, int rows, int cols, int64_t ld, float nd_f, bool nd_exact,
                   int8_t* unsolved, uint8_t* waiting, unsigned* list, unsigned* cnt) {
  __shared__ unsigned warp_off[PT / 32];
  __shared__ unsigned cta_base;
  const unsigned long long n = (unsigned long long)rows * (unsigned long long)cols;  // up to 2^32: indices fit 32 bits
  const unsigned i = blockIdx.x * PT + threadIdx.x;
  bool pit = false;
  if ((unsigned long long)i < n) {
    const int r = (int)(i / (unsigned)cols), c = (int)(i - (unsigned)r * (unsigned)cols);
    if (r >= 2 && r < rows - 2 && c >= 2 && c < cols - 2) {
      const float* at = chunk + (int64_t)r * ld + c;
      const float z = *at;
      // Branch-free form of :40-50.  (double)x == nodata <=> x == (float)nodata when float32 holds nodata exactly,
      // and never otherwise.  fminf skips NaN neighbours exactly as "zn <= z" is false for them; starting from NaN
      // and testing "not (lowest <= z)" keeps the reference's answer when z or every neighbour is NaN.
      float lowest = CUDART_NAN_F;
      bool nodata_seen = false;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float zn = at[(int64_t)p_dy[k] * ld + p_dx[k]];
        lowest = fminf(lowest, zn);
        nodata_seen = nodata_seen || zn == nd_f;
      }
      pit = !(nd_exact && (nodata_seen || z == nd_f)) && !(lowest <= z);
    }
    unsolved[i] = pit ? 1 : 0;
    waiting[i] = pit ? 1 : 0;
  }
  // one list atomic per CTA
  const unsigned m = __ballot_sync(0xffffffffu, pit);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) warp_off[w] = __popc(m);
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned run = 0;
    for (int k = 0; k < PT / 32; ++k) {
      const unsigned v = warp_off[k];
      warp_off[k] = run;
      run += v;
    }
    cta_base = run ? atomicAdd(&cnt[PC_PITS], run) : 0u;
  }
  __syncthreads();
  if (pit) list[cta_base + warp_off[w] + __popc(m & ((1u << lane) - 1u))] = i;
}

// pass 1, vector form (dense pitch and columns that are multiples of four, 16-byte aligned rows): a thread owns four
// adjacent cells of one row -- three float4 loads and six scalars instead of 36 loads, the flags of its cells leave as
// one 32-bit store each; a CTA covers 128 columns x 8 rows and makes one list reservation.
__global__ void __launch_bounds__(PT)
pits_detect4_kernel(const float* __restrict__ chunk, int rows, int cols, int64_t ld, float nd_f, bool nd_exact,
                    int8_t* unsolved, uint8_t* waiting, unsigned* list, unsigned* cnt) {
  __shared__ unsigned warp_off[PT / 32];
  __shared__ unsigned cta_base;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int r = blockIdx.y * (PT / 32) + w;
  const int c = (blockIdx.x * 32 + lane) * 4;
  uint32_t pits = 0;  // bit j: cell c + j is a pit
  const bool in_raster = r < rows && c < cols;
  if (in_raster && r >= 2 && r < rows - 2) {
    const float* row = chunk + (int64_t)r * ld + c;
    float v[3][6];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float* q = row + (int64_t)(k - 1) * ld;
      const float4 m = *reinterpret_cast<const float4*>(q);
      v[k][0] = c > 0 ? q[-1] : 0.f;
      v[k][1] = m.x;
      v[k][2] = m.y;
      v[k][3] = m.z;
      v[k][4] = m.w;
      v[k][5] = c + 4 < cols ? q[4] : 0.f;
    }
    // the four cells share their neighbours: per column the minimum of the rows above and below (m), of all three
    // rows (m3), and whether any of the three is NODATA (nd3) -- 20 minima and 18 compares for four cells, not 32 + 36
    float m[6], m3[6];
    bool nd3[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      m[k] = fminf(v[0][k], v[2][k]);
      m3[k] = fminf(m[k], v[1][k]);
      nd3[k] = v[0][k] == nd_f || v[1][k] == nd_f || v[2][k] == nd_f;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int cc = c + j;
      if (cc < 2 || cc >= cols - 2) continue;
      const float z = v[1][j + 1];
      // the branch-free form of :40-50, as in pits_detect_kernel: fminf skips NaN neighbours exactly as "zn <= z" is
      // false for them, and "not (lowest <= z)" keeps the reference's answer when z or every neighbour is NaN
      const float lowest = fminf(fminf(m3[j], m3[j + 2]), m[j + 1]);
      const bool nodata_seen = nd3[j] || nd3[j + 1] || nd3[j + 2];  // a neighbour or the cell itself
      if (!(nd_exact && nodata_seen) && !(lowest <= z)) pits |= 1u << j;
    }
  }
  if (in_raster) {
    const uint32_t flags = ((pits & 1u) ? 0x01u : 0u) | ((pits & 2u) ? 0x0100u : 0u) | ((pits & 4u) ? 0x010000u : 0u) |
                           ((pits & 8u) ? 0x01000000u : 0u);
    const size_t i = (size_t)r * (size_t)cols + (size_t)c;
    *reinterpret_cast<uint32_t*>(unsolved + i) = flags;
    *reinterpret_cast<uint32_t*>(waiting + i) = flags;
  }
  // one list reservation per CTA: exclusive scan of the per-thread counts
  const unsigned mine = __popc(pits);
  unsigned incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) warp_off[w] = incl;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned run = 0;
    for (int k = 0; k < PT / 32; ++k) {
      const unsigned v2 = warp_off[k];
      warp_off[k] = run;
      run += v2;
    }
    cta_base = run ? atomicAdd(&cnt[PC_PITS], run) : 0u;
  }
  __syncthreads();
  unsigned pos = cta_base + warp_off[w] + incl - mine;
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (pits & (1u << j)) list[pos++] = (unsigned)r * (unsigned)cols + (unsigned)(c + j);
}

// pass 2 (:52-63) in dependency-ordered rounds, ONE persistent kernel (cooperative launch, grid barriers).
// Round: (a) a waiting pit is READY when no earlier (row-major) pit within chessboard distance 3 is still waiting;
// (b) the ready pits -- more than three cells apart, hence on disjoint cells -- are breached exactly as the
// reference's sequential loop would breach them, the others go to the next round's list.  The earliest waiting pit is
// always ready, so the rounds end.  Everything other CTAs wrote in earlier rounds is read past L1 (ld.global.cg).
struct PitsArgs {
  unsigned *list_a, *list_b;
  uint8_t *waiting, *ready;
  float* chunk;
  int rows, cols;
  int64_t ld;
  double nodata;
  int8_t* unsolved;
  unsigned* cnt;
};

// (a) of a round, for the pits cur[t], t = tid, tid + nthr, .. < n_cur
__device__ __forceinline__ void pits_ready_phase(const PitsArgs& a, const unsigned* cur, unsigned n_cur, unsigned tid,
                                                 unsigned nthr) {
  const int cols = a.cols;
  for (unsigned t = tid; t < n_cur; t += nthr) {
    const unsigned i = __ldcg(&cur[t]);
    const int r = (int)(i / (unsigned)cols), c = (int)(i - (unsigned)r * (unsigned)cols);
    // all 27 flags are loaded before any is looked at: independent loads, not a chain of them with early exits
    unsigned any = 0;
#pragma unroll
    for (int dr = -3; dr <= 0; ++dr) {
      const int rr = r + dr;
#pragma unroll
      for (int dc = -3; dc <= 3; ++dc) {
        if (dr == 0 && dc >= 0) continue;  // the pit's own row: only cells before it
        const int cc = c + dc;
        if (rr >= 0 && cc >= 0 && cc < cols) any |= __ldcg(&a.waiting[(size_t)rr * cols + cc]);
      }
    }
    a.ready[t] = any == 0 ? 1 : 0;
  }
}

// (b) of a round: the ready pits are breached, the others appended to nxt (count in *n_next)
__device__ __forceinline__ void pits_breach_phase(const PitsArgs& a, const unsigned* cur, unsigned* nxt, unsigned n_cur,
                                                  unsigned* n_next, unsigned tid, unsigned nthr) {
  const int cols = a.cols;
  const unsigned lane = threadIdx.x & 31u;
  unsigned n_unsolved = 0;
  for (unsigned t = tid; t < n_cur; t += nthr) {
    const unsigned i = __ldcg(&cur[t]);
    if (!a.ready[t]) {  // written by this thread in phase (a)
      // one counter update for the lanes of the warp that are here together
      const unsigned m = __activemask();
      const int leader = __ffs(m) - 1;
      unsigned base = 0;
      if ((int)lane == leader) base = atomicAdd(n_next, (unsigned)__popc(m));
      base = __shfl_sync(m, base, leader);
      nxt[base + __popc(m & ((1u << lane) - 1u))] = i;
      continue;
    }
    const int r = (int)(i / (unsigned)cols), c = (int)(i - (unsigned)r * (unsigned)cols);
    float* at = a.chunk + (int64_t)r * a.ld + c;
    const float z = __ldcg(at);
    // the sixteen cells two steps away are read first (the pit writes only within one step of itself), then
    // breached in order: two k share a breach cell and the later one wins
    float zn[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) zn[k] = __ldcg(&at[(int64_t)p_dy2[k] * a.ld + p_dx2[k]]);
    bool solved = false;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      if (zn[k] <= z || (double)zn[k] == a.nodata) {
        solved = true;
        const int b = p_breach[k];
        at[(int64_t)p_dy[b] * a.ld + p_dx[b]] = __double2float_rn((double)__fadd_rn(z, zn[k]) / 2.0);
      }
    }
    if (solved)
      a.unsolved[i] = 0;
    else
      ++n_unsolved;
    a.waiting[i] = 0;
  }
  // every thread of the grid gets here: one counter update per warp
  n_unsolved = __reduce_add_sync(0xffffffffu, n_unsolved);
  if (lane == 0 && n_unsolved) atomicAdd(&a.cnt[PC_UNSOLVED], n_unsolved);
}

// Round 1 holds most of the pits (on terrain four in five are ready at once): two ordinary launches over the
// whole list, the grid sized for it.  (The same thread handles pit t in both: ready[t] needs no fence.)
__global__ void __launch_bounds__(PT) pits_first_ready_kernel(const PitsArgs a) {
  pits_ready_phase(a, a.list_a, a.cnt[PC_PITS], blockIdx.x * PT + threadIdx.x, gridDim.x * PT);
}
__global__ void __launch_bounds__(PT) pits_first_breach_kernel(const PitsArgs a) {
  pits_breach_phase(a, a.list_a, a.list_b, a.cnt[PC_PITS], &a.cnt[PC_NEXT1], blockIdx.x * PT + threadIdx.x, gridDim.x * PT);
}

// The later rounds -- few pits each, many of them -- in ONE persistent kernel on a small grid (cooperative launch,
// a grid barrier between the two phases and between rounds; everything other CTAs wrote is read past L1).
__global__ void __launch_bounds__(PT) pits_rounds_kernel(const PitsArgs a) {
  unsigned generation = 0;
  const unsigned tid = blockIdx.x * PT + threadIdx.x, nthr = gridDim.x * PT;
  unsigned rounds = 1;  // round 1 ran as two ordinary launches: its survivors are list_b, counted in PC_NEXT1
  unsigned n_cur = *reinterpret_cast<volatile unsigned*>(&a.cnt[PC_NEXT1]);
  unsigned* cur = a.list_b;
  unsigned* nxt = a.list_a;
  if (*reinterpret_cast<volatile unsigned*>(&a.cnt[PC_PITS]) == 0) rounds = 0;
  while (n_cur) {
    unsigned* n_next = &a.cnt[PC_NEXT0 + ((rounds + 1) & 1)];
    pits_ready_phase(a, cur, n_cur, tid, nthr);
    grid_barrier(&a.cnt[PC_BARRIER], generation);
    pits_breach_phase(a, cur, nxt, n_cur, n_next, tid, nthr);
    grid_barrier(&a.cnt[PC_BARRIER], generation);
    n_cur = *reinterpret_cast<volatile unsigned*>(n_next);
    ++rounds;
    if (tid == 0) a.cnt[PC_NEXT0 + ((rounds + 1) & 1)] = 0;  // next round's counter: not touched before the next barrier
    unsigned* t2 = cur;
    cur = nxt;
    nxt = t2;
  }
  if (tid == 0) a.cnt[PC_ROUNDS] = rounds;
}

// Cuts the workspace at `base` into a's pit lists, flags and counters and returns its size; with a null base only the
// size is meaningful.
size_t pits_layout(void* base, int64_t rows, int64_t cols, PitsArgs& a) {
  const size_t n = (size_t)rows * (size_t)cols;
  Carver c(base);
  // pits are never adjacent, so there are at most n / 4 of them: two lists fit the n ints
  c.take(a.list_a, n * sizeof(int));
  a.list_b = a.list_a + (n + 1) / 2;
  c.take(a.waiting, n);
  c.take(a.ready, n);
  c.take(a.cnt, PC_SLOTS * sizeof(unsigned));
  return c.bytes;
}

}  // namespace

size_t pits_workspace_bytes(int64_t rows, int64_t cols) {
  PitsArgs a;
  return pits_layout(nullptr, rows, cols, a);
}

// One chunk of at most 2^32 cells: cell indices are unsigned 32-bit on the device.
int pits_shape(int64_t rows, int64_t cols) {
  OFL_REQUIRE(rows > 0 && cols > 0 && rows < (1ll << 31) && cols < (1ll << 31) && rows * cols <= (1ll << 32), OFL_ERR_INVALID,
              "pit breaching works on one chunk of at most 2^32 cells (got %lld x %lld)", (long long)rows, (long long)cols);
  return OFL_OK;
}

// chunk: device, rows x cols with leading dimension ld, breached in place.  unsolved: device int8, dense.
// info (host, nullable): {pits found, pits left unsolved, rounds}.  Synchronises the stream (once, at the end).
int launch_breach_pits(float* chunk, int64_t rows, int64_t cols, int64_t ld, double nodata, int8_t* unsolved,
                       int64_t* info, void* workspace, cudaStream_t st) {
  PitsArgs a;
  pits_layout(workspace, rows, cols, a);
  a.chunk = chunk;
  a.rows = (int)rows;
  a.cols = (int)cols;
  a.ld = ld;
  a.nodata = nodata;
  a.unsolved = unsolved;
  const size_t n = (size_t)rows * (size_t)cols;
  PhaseScope ps(PHASE_PITS, st);
  OFL_CUDA(cudaMemsetAsync(a.cnt, 0, PC_SLOTS * sizeof(unsigned), st));
  const float nd_f = (float)nodata;
  const bool nd_exact = (double)nd_f == nodata;  // false for NaN and for values float32 cannot hold: nothing matches then
  // the vector path's grid has a row of CTAs per PT / 32 chunk rows, at most 65535 of them
  const dim3 grid((unsigned)((cols / 4 + 31) / 32), (unsigned)((rows + PT / 32 - 1) / (PT / 32)));
  const bool vec = cols % 4 == 0 && ld % 4 == 0 && (reinterpret_cast<uintptr_t>(chunk) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(unsolved) & 3) == 0 && grid.y <= 65535u && !getenv("OFL_PITS_SCALAR");
  if (vec) {
    pits_detect4_kernel<<<grid, PT, 0, st>>>(chunk, (int)rows, (int)cols, ld, nd_f, nd_exact, unsolved, a.waiting, a.list_a,
                                             a.cnt);
  } else {
    const unsigned nb = (unsigned)((n + PT - 1) / PT);
    pits_detect_kernel<<<nb, PT, 0, st>>>(chunk, (int)rows, (int)cols, ld, nd_f, nd_exact, unsolved, a.waiting, a.list_a,
                                          a.cnt);
  }
  OFL_CHECK_LAUNCH();
  {
    // round 1 over the whole list (its length is only known on the device: the grid covers the worst case a
    // strided loop needs, one pit per thread and 16 turns)
    const unsigned g1 = (unsigned)(sm_count() * 8);
    pits_first_ready_kernel<<<g1, PT, 0, st>>>(a);
    OFL_CHECK_LAUNCH();
    pits_first_breach_kernel<<<g1, PT, 0, st>>>(a);
    OFL_CHECK_LAUNCH();
    void* args[] = {&a};
    OFL_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(pits_rounds_kernel), dim3((unsigned)sm_count()),
                                         dim3(PT), args, 0, st));
    OFL_CHECK_LAUNCH();
  }
  unsigned* h = nullptr;
  int rc = pinned_get(64, reinterpret_cast<void**>(&h));
  if (rc != OFL_OK) return rc;
  OFL_CUDA(cudaMemcpyAsync(h, a.cnt, 3 * sizeof(unsigned), cudaMemcpyDeviceToHost, st));
  OFL_CUDA(cudaStreamSynchronize(st));
  if (info) {
    info[0] = h[PC_PITS];
    info[1] = h[PC_UNSOLVED];
    info[2] = h[PC_ROUNDS];
  }
  return OFL_OK;
}

}  // namespace ofl
