// basins.cu -- drainage basins: the outlet every cell's D8 path reaches (sm_100a).
//
// Edge rule of the accumulation (accumulation.cu header): succ(c) exists iff code(c) in 0..7, the downstream
// cell d lies inside the raster and code(d) != 9.  A data cell without succ is an OUTLET; outlet (r, c) has the
// label r * cols + c + 1, every data cell gets the label of the outlet its path ends at, NODATA cells get 0.
// With pour points, a pour point is a root with its own label (its outgoing edge is cut), natural outlets get 0.
//
// The accumulation's structure, with a label copied down the forest instead of a count summed up it:
//   tile pass  (basins_tile_kernel)  one CTA per 64 x 64 tile: codes + a one-cell halo into shared memory, every
//              cell resolved to its in-tile terminal by pointer jumping over 16-bit in-tile pointers (at most
//              13 rounds, early exit).  A terminal is a root (outlet or pour point) or a perimeter cell whose step
//              leaves the tile.  Writes each cell's terminal (2 B/cell) and one 8-byte record per perimeter node:
//              the resolved label, or the id of the node its path enters in the neighbouring tile.
//   solve      (basins_solve_kernel)  pointer jumping over the perimeter nodes (~6 % of the cells), in place,
//              one launch per round; round 0 scans every node, later rounds only the nodes still unresolved
//              (compacted lists).  Host-driven with a fixed round count: no read-back between rounds.
//   final      (basins_final_kernel)  per tile: the terminal of each cell becomes its label -- the root's own
//              label, or the resolved record of the exit node.
// The final pass reads the terminals the tile pass stored (2 B/cell each way) instead of recomputing them from the
// codes: recomputing repeats the pointer jumping, which is what bounds the tile pass.
//
// HBM traffic per cell: tile pass 1 B codes + 2 B terminals, final pass 2 B terminals + 8 B labels, the solve
// ~0.5 B; against 9 B/cell compulsory (codes in, labels out).
#include <cstdlib>

#include "common.cuh"
#include "tile_geometry.cuh"

namespace ofl {
namespace {

constexpr int B_THREADS = 256;
constexpr int B_PER_THREAD = AT * AT / B_THREADS;   // 16 cells: rows (tid >> 6) + 4k, column tid & 63
constexpr int CS_W = AT + 4;                        // code tile pitch: columns -1 .. 64 at 1 .. 66
constexpr int CS_H = AT + 2;                        // rows -1 .. 64
constexpr int TILE_ROUNDS = 2 * AT_SHIFT + 1;       // ceil(log2(AT * AT)) + 1
constexpr uint16_t P_TERM = 0x8000;                 // pointer flag: the cell pointed at is a terminal
constexpr uint16_t T_ZERO = 0xFFFF;                 // stored terminal: the cell's label is 0
constexpr unsigned long long R_RESOLVED = 1ull << 63;  // node record: the low bits are the final label

// terminal kinds (shared memory, one byte per cell)
constexpr uint8_t K_PATH = 0;   // the cell has an in-tile successor
constexpr uint8_t K_ROOT = 1;   // labelled root: an outlet, or a pour point
constexpr uint8_t K_ZERO = 2;   // label 0: NODATA, outside the raster, or a natural outlet when pour points are given
constexpr uint8_t K_EXIT = 3;   // the cell's step leaves the tile into a data cell of the neighbouring tile

// Workspace flag words.
enum { BF_TILE = 0, BF_POUR = 1, BF_WORDS = 4 };
constexpr int MAX_ROUNDS = 40;

static_assert(B_PER_THREAD * B_THREADS == AT * AT, "the threads of a CTA cover its tile");
static_assert(B_PER_THREAD == 16, "the tile pass loads one 16-byte piece of codes per thread");
static_assert(B_THREADS == SLOTS, "one thread per perimeter slot writes and reads the node records");
static_assert(AT * AT <= 0x8000, "an in-tile pointer holds a cell in 15 bits, P_TERM in bit 15");

struct BasinParams {
  const uint8_t* fdr;
  int64_t ld_fdr;
  long long* labels;
  int64_t ld_labels;
  int rows, cols;
  int ntx, nty;
  unsigned long long* rec;  // [ntiles * SLOTS] perimeter node records
  uint16_t* term;           // [ntiles][64 * 64] in-tile terminal of each cell (T_ZERO: label 0)
  const uint32_t* pour;     // pour-point bit per cell (raster order), null without pour points
  int* flags;               // [BF_WORDS]
  int vec_store;            // labels rows are 16-byte aligned: the final pass stores two labels at once
};

__device__ __forceinline__ bool pour_bit(const uint32_t* pour, int64_t i) { return (pour[i >> 5] >> (i & 31)) & 1u; }

__global__ void __launch_bounds__(B_THREADS) basins_tile_kernel(const BasinParams p) {
  __shared__ __align__(16) uint8_t codes[CS_H * CS_W];  // cell (y, x) at (y + 1) * CS_W + x + 1; 9 outside the raster
  __shared__ uint16_t ptr[AT * AT];
  __shared__ uint8_t kind[AT * AT];
  const int tid = threadIdx.x;
  const int tile = blockIdx.x;
  int ty0, tx0, h, w;
  tile_rect(tile, p.ntx, p.rows, p.cols, ty0, tx0, h, w);

  // codes: the 64 x 64 body in 16-byte pieces (a piece never runs past the row pitch: ld_fdr % 16 == 0), the ring
  // byte by byte
  {
    const int y = tid >> 2, x = (tid & 3) * 16;
    uint4 v = make_uint4(0x09090909u, 0x09090909u, 0x09090909u, 0x09090909u);
    if (y < h && x < w) v = *reinterpret_cast<const uint4*>(p.fdr + (int64_t)(ty0 + y) * p.ld_fdr + tx0 + x);
    uint8_t b[16];
    *reinterpret_cast<uint4*>(b) = v;
#pragma unroll
    for (int i = 0; i < 16; ++i) codes[(y + 1) * CS_W + x + 1 + i] = (x + i < w) ? b[i] : (uint8_t)OFL_DIR_NODATA;
  }
  for (int i = tid; i < 4 * (AT + 2); i += B_THREADS) {
    const int side = i / (AT + 2), k = i % (AT + 2) - 1;  // k = -1 .. 64
    const int y = side == 0 ? -1 : side == 1 ? AT : k, x = side < 2 ? k : (side == 2 ? -1 : AT);
    if (side >= 2 && (k < 0 || k >= AT)) continue;  // the corners come with the top and bottom rows
    const int gy = ty0 + y, gx = tx0 + x;
    const bool in = gy >= 0 && gy < p.rows && gx >= 0 && gx < p.cols;
    codes[(y + 1) * CS_W + x + 1] = in ? p.fdr[(int64_t)gy * p.ld_fdr + gx] : (uint8_t)OFL_DIR_NODATA;
  }
  __syncthreads();

  // successors and terminal kinds
  uint16_t nxt[B_PER_THREAD];
#pragma unroll
  for (int k = 0; k < B_PER_THREAD; ++k) {
    const int c = tid + k * B_THREADS, y = c >> AT_SHIFT, x = c & (AT - 1);
    const int code = codes[(y + 1) * CS_W + x + 1];
    uint8_t kd;
    nxt[k] = (uint16_t)c;
    if (code == OFL_DIR_NODATA) {
      kd = K_ZERO;
    } else if (p.pour && pour_bit(p.pour, (int64_t)(ty0 + y) * p.cols + tx0 + x)) {
      kd = K_ROOT;
    } else if (code > 7) {
      kd = p.pour ? K_ZERO : K_ROOT;
    } else {
      const int ny = y + dir_dy(code), nx = x + dir_dx(code);
      if (codes[(ny + 1) * CS_W + nx + 1] == OFL_DIR_NODATA) {  // NODATA or outside the raster
        kd = p.pour ? K_ZERO : K_ROOT;
      } else if (ny < 0 || ny >= AT || nx < 0 || nx >= AT) {
        kd = K_EXIT;
      } else {
        kd = K_PATH;
        nxt[k] = (uint16_t)((ny << AT_SHIFT) | nx);
      }
    }
    kind[c] = kd;
  }
  __syncthreads();
  uint32_t pending = 0;
#pragma unroll
  for (int k = 0; k < B_PER_THREAD; ++k) {
    const int c = tid + k * B_THREADS;
    if (nxt[k] == c) {
      nxt[k] |= P_TERM;
    } else if (kind[nxt[k]] != K_PATH) {
      nxt[k] |= P_TERM;
    } else {
      pending |= 1u << k;
    }
    ptr[c] = nxt[k];
  }

  // pointer jumping: values only move further down the same path, so updates in place are safe
  for (int round = 0;; ++round) {
    if (!__syncthreads_or(pending != 0)) break;
    if (round == TILE_ROUNDS) {  // a path longer than the tile has cells: a cycle
      if (pending) atomicOr(&p.flags[BF_TILE], 1);
      break;
    }
#pragma unroll
    for (int k = 0; k < B_PER_THREAD; ++k) {
      if (pending & (1u << k)) {
        const uint16_t q = ptr[nxt[k]];
        nxt[k] = q;
        ptr[tid + k * B_THREADS] = q;
        if (q & P_TERM) pending &= ~(1u << k);
      }
    }
  }

  // terminals of the cells
  uint16_t* term = p.term + (size_t)tile * (AT * AT);
#pragma unroll
  for (int k = 0; k < B_PER_THREAD; ++k) {
    const int t = nxt[k] & (AT * AT - 1);
    term[tid + k * B_THREADS] = kind[t] == K_ZERO ? T_ZERO : (uint16_t)t;
  }

  // perimeter node records (the pointer array is final after the last barrier of the loop)
  {
    const int s = tid;
    int y, x;
    unsigned long long r = R_RESOLVED;
    if (cell_of_slot(s, h, w, y, x)) {
      const int t = ptr[(y << AT_SHIFT) | x] & (AT * AT - 1);
      const int tyy = t >> AT_SHIFT, txx = t & (AT - 1);
      const uint8_t kd = kind[t];
      if (kd == K_ROOT) {
        r = R_RESOLVED | (unsigned long long)((int64_t)(ty0 + tyy) * p.cols + tx0 + txx + 1);
      } else if (kd == K_EXIT) {
        const int code = codes[(tyy + 1) * CS_W + txx + 1];
        r = (unsigned long long)node_of_cell(ty0 + tyy + dir_dy(code), tx0 + txx + dir_dx(code), p.rows, p.cols, p.ntx);
      }
    }
    p.rec[(size_t)tile * SLOTS + s] = r;
  }
}

// Scatter the pour points into the cell bitmask; an index outside the raster sets the pour flag.
__global__ void basins_pour_kernel(const long long* __restrict__ pour, int64_t n_pour, int64_t n_cells,
                                   uint32_t* __restrict__ mask, int* __restrict__ flags) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n_pour; k += (int64_t)gridDim.x * blockDim.x) {
    const long long i = pour[k];
    if (i < 0 || i >= n_cells) {
      atomicOr(&flags[BF_POUR], 1);
      continue;
    }
    atomicOr(&mask[i >> 5], 1u << (i & 31));
  }
}

// One round of pointer jumping over the unresolved nodes: the nodes of list_in (all nodes when cnt_in is null);
// those still unresolved afterwards are appended to list_out.
__global__ void __launch_bounds__(256) basins_solve_kernel(unsigned long long* __restrict__ rec, int64_t n_nodes,
                                                           const int32_t* __restrict__ list_in,
                                                           const int* __restrict__ cnt_in, int32_t* __restrict__ list_out,
                                                           int* __restrict__ cnt_out) {
  const int64_t n = cnt_in ? (int64_t)*cnt_in : n_nodes;
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  // whole warps iterate together so that the append below can use the warp's ballot
  for (int64_t k0 = blockIdx.x * (int64_t)blockDim.x + (threadIdx.x & ~31); k0 < n; k0 += stride) {
    const int64_t k = k0 + lane;
    bool keep = false;
    int32_t u = 0;
    if (k < n) {
      u = list_in ? list_in[k] : (int32_t)k;
      const unsigned long long v = __ldcg(&rec[u]);
      if (!(v & R_RESOLVED)) {
        const unsigned long long w2 = __ldcg(&rec[v]);
        __stcg(&rec[u], w2);
        keep = !(w2 & R_RESOLVED);
      }
    }
    const uint32_t bal = __ballot_sync(0xffffffffu, keep);
    if (bal) {
      int base = 0;
      if (lane == 0) base = atomicAdd(cnt_out, __popc(bal));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (keep) list_out[base + __popc(bal & ((1u << lane) - 1))] = u;
    }
  }
}

__global__ void __launch_bounds__(B_THREADS) basins_final_kernel(const BasinParams p) {
  __shared__ long long srec[SLOTS];
  const int tid = threadIdx.x;
  const int tile = blockIdx.x;
  int ty0, tx0, h, w;
  tile_rect(tile, p.ntx, p.rows, p.cols, ty0, tx0, h, w);
  srec[tid] = (long long)(__ldcg(&p.rec[(size_t)tile * SLOTS + tid]) & ~R_RESOLVED);
  __syncthreads();
  const uint32_t* term = reinterpret_cast<const uint32_t*>(p.term + (size_t)tile * (AT * AT));
#pragma unroll 4
  for (int k = 0; k < AT * AT / 2 / B_THREADS; ++k) {
    const int pair = tid + k * B_THREADS;
    const int y = pair >> (AT_SHIFT - 1), x = (pair & (AT / 2 - 1)) * 2;
    if (y >= h || x >= w) continue;
    const uint32_t tt = __ldcs(&term[pair]);
    long long lab[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const uint32_t t = (tt >> (16 * j)) & 0xFFFFu;
      if (t == T_ZERO) {
        lab[j] = 0;
      } else {
        const int yy = (int)(t >> AT_SHIFT), xx = (int)(t & (AT - 1));
        const int s = slot_of(yy, xx, h, w);
        lab[j] = s >= 0 ? srec[s] : (long long)(ty0 + yy) * p.cols + tx0 + xx + 1;
      }
    }
    long long* out = p.labels + (int64_t)(ty0 + y) * p.ld_labels + tx0 + x;
    if (x + 1 < w && p.vec_store) {
      __stcs(reinterpret_cast<longlong2*>(out), make_longlong2(lab[0], lab[1]));
    } else {
      __stcs(out, lab[0]);
      if (x + 1 < w) __stcs(out + 1, lab[1]);
    }
  }
}

// Counts the cells that break the labelling rule: a NODATA cell has label 0; a cell with a successor that is not a
// pour point has its successor's label; a root has its own index + 1, or 0 for a natural outlet when pour points
// are given.  Zero violations on an acyclic raster prove the labels exact (by induction along each path).
__global__ void basins_check_kernel(const uint8_t* __restrict__ fdr, int64_t ld_fdr, const long long* __restrict__ labels,
                                    int64_t ld_labels, int rows, int cols, const uint32_t* __restrict__ pour,
                                    unsigned long long* __restrict__ n_bad) {
  const int64_t n = (int64_t)rows * cols;
  unsigned long long bad = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i - (int64_t)r * cols);
    const int code = fdr[(int64_t)r * ld_fdr + c];
    const long long got = labels[(int64_t)r * ld_labels + c];
    long long want;
    if (code == OFL_DIR_NODATA) {
      want = 0;
    } else {
      const bool is_pour = pour && pour_bit(pour, i);
      bool has_succ = false;
      int nr = 0, nc = 0;
      if (code <= 7) {
        nr = r + dir_dy(code);
        nc = c + dir_dx(code);
        has_succ = nr >= 0 && nr < rows && nc >= 0 && nc < cols && fdr[(int64_t)nr * ld_fdr + nc] != OFL_DIR_NODATA;
      }
      if (has_succ && !is_pour) {
        want = labels[(int64_t)nr * ld_labels + nc];
      } else {
        want = (is_pour || !pour) ? i + 1 : 0;
      }
    }
    bad += (got != want);
  }
  for (int o = 16; o > 0; o >>= 1) bad += __shfl_down_sync(0xffffffffu, bad, o);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(n_bad, bad);
}

// ---------------------------------------------------------------- host orchestration (device pointers)
struct BasinLayout {
  unsigned long long* rec;
  uint16_t* term;
  int32_t *list_a, *list_b;
  int* counts;  // [MAX_ROUNDS] nodes left after each solve round
  int* flags;   // [BF_WORDS], right after the counts: both are cleared by one memset
  uint32_t* pour;
  size_t bytes;
};

BasinLayout carve(void* base, int64_t rows, int64_t cols) {
  BasinLayout L;
  const size_t ntiles = (size_t)tiles_along(rows) * (size_t)tiles_along(cols);
  const size_t nodes = ntiles * SLOTS;
  Carver w(base);
  w.take(L.rec, nodes * 8);
  w.take(L.term, ntiles * (AT * AT) * 2);
  w.take(L.list_a, nodes * 4);
  w.take(L.list_b, nodes * 4);
  w.take(L.counts, (MAX_ROUNDS + BF_WORDS) * sizeof(int));
  L.flags = L.counts + MAX_ROUNDS;
  w.take(L.pour, ((size_t)rows * (size_t)cols + 31) / 32 * 4);
  L.bytes = w.bytes;
  return L;
}

// ceil(log2 nodes) + 2 rounds: a longer chain of perimeter nodes than there are nodes is a cycle
int solve_rounds(int64_t nodes) {
  int r = 0;
  while ((1ll << r) < nodes) ++r;
  return r + 2 < MAX_ROUNDS ? r + 2 : MAX_ROUNDS;
}

// Clear the pour mask and scatter the pour points into it (n_pour > 0).
int scatter_pour(const long long* pour, int64_t n_pour, int64_t n_cells, uint32_t* mask, int* flags, cudaStream_t st) {
  OFL_CUDA(cudaMemsetAsync(mask, 0, (size_t)(n_cells + 31) / 32 * 4, st));
  basins_pour_kernel<<<grid_for(n_pour, 4), 256, 0, st>>>(pour, n_pour, n_cells, mask, flags);
  OFL_CHECK_LAUNCH();
  return OFL_OK;
}

}  // namespace

size_t basins_workspace_bytes(int64_t rows, int64_t cols) {
  if (rows <= 0 || cols <= 0) return 256;
  return carve(nullptr, rows, cols).bytes;
}

// 30-bit sides (BasinParams holds ints) and 32-bit perimeter node ids.
int basins_shape(int64_t rows, int64_t cols) {
  OFL_REQUIRE(rows < (1ll << 30) && cols < (1ll << 30), OFL_ERR_INVALID, "bad raster size");
  OFL_REQUIRE(tiles_along(rows) * tiles_along(cols) * SLOTS < (1ll << 31), OFL_ERR_INVALID,
              "raster too large for 32-bit perimeter node ids");
  return OFL_OK;
}

int launch_basins(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, const long long* pour, int64_t n_pour,
                  long long* labels, int64_t ld_labels, void* workspace, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return OFL_OK;
  OFL_REQUIRE((reinterpret_cast<uintptr_t>(fdr) & 15) == 0 && (ld_fdr % 16) == 0 && ld_fdr >= cols, OFL_ERR_ALIGNMENT,
              "fdr must be 16-byte aligned with ld_fdr %% 16 == 0 (ld_fdr=%lld)", (long long)ld_fdr);
  OFL_REQUIRE((reinterpret_cast<uintptr_t>(labels) & 7) == 0 && ld_labels >= cols, OFL_ERR_ALIGNMENT,
              "labels must be 8-byte aligned");
  const int ntx = (int)tiles_along(cols), nty = (int)tiles_along(rows);
  const int64_t ntiles = (int64_t)ntx * nty, nodes = ntiles * SLOTS;
  const BasinLayout L = carve(workspace, rows, cols);
  BasinParams p;
  p.fdr = fdr;
  p.ld_fdr = ld_fdr;
  p.labels = labels;
  p.ld_labels = ld_labels;
  p.rows = (int)rows;
  p.cols = (int)cols;
  p.ntx = ntx;
  p.nty = nty;
  p.rec = L.rec;
  p.term = L.term;
  p.pour = n_pour > 0 ? L.pour : nullptr;
  p.flags = L.flags;
  p.vec_store = ((reinterpret_cast<uintptr_t>(labels) & 15) == 0 && (ld_labels % 2) == 0) ? 1 : 0;
  OFL_CUDA(cudaMemsetAsync(L.counts, 0, (MAX_ROUNDS + BF_WORDS) * sizeof(int), st));
  const int rounds = solve_rounds(nodes);
  {
    PhaseScope ps(PHASE_BASINS_TILE, st);
    if (n_pour > 0) {
      const int rc = scatter_pour(pour, n_pour, rows * cols, L.pour, L.flags, st);
      if (rc != OFL_OK) return rc;
    }
    basins_tile_kernel<<<(unsigned)ntiles, B_THREADS, 0, st>>>(p);
    OFL_CHECK_LAUNCH();
  }
  {
    PhaseScope ps(PHASE_BASINS_SOLVE, st);
    const int grid = grid_for(nodes, 8);
    for (int r = 0; r < rounds; ++r) {
      int32_t* lists[2] = {L.list_a, L.list_b};
      basins_solve_kernel<<<grid, 256, 0, st>>>(L.rec, nodes, r ? lists[(r - 1) & 1] : nullptr,
                                                r ? L.counts + r - 1 : nullptr, lists[r & 1], L.counts + r);
      OFL_CHECK_LAUNCH();
    }
  }
  {
    PhaseScope ps(PHASE_BASINS_FINAL, st);
    basins_final_kernel<<<(unsigned)ntiles, B_THREADS, 0, st>>>(p);
    OFL_CHECK_LAUNCH();
  }
  int h[3] = {0, 0, 0};  // tile flag, pour flag, nodes left after the last round
  OFL_CUDA(cudaMemcpyAsync(h, L.flags, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
  OFL_CUDA(cudaMemcpyAsync(h + 2, L.counts + rounds - 1, sizeof(int), cudaMemcpyDeviceToHost, st));
  OFL_CUDA(cudaStreamSynchronize(st));
  OFL_REQUIRE(h[1] == 0, OFL_ERR_INVALID, "pour point outside the raster");
  OFL_REQUIRE(h[0] == 0, OFL_ERR_CYCLE, "flow-direction raster contains a cycle (tile pass)");
  OFL_REQUIRE(h[2] == 0, OFL_ERR_CYCLE, "flow-direction raster contains a cycle (perimeter graph)");
  return OFL_OK;
}

// Pour-point mask in SCRATCH_WORK, violation counter and flags in SCRATCH_MISC.  Synchronises the stream.
int check_basins(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, const long long* pour, int64_t n_pour,
                 const long long* labels, int64_t ld_labels, int64_t* n_bad, cudaStream_t st) {
  *n_bad = 0;
  if (rows <= 0 || cols <= 0) return OFL_OK;
  void* misc = nullptr;
  int rc = scratch_get(SCRATCH_MISC, 256, &misc);
  if (rc != OFL_OK) return rc;
  unsigned long long* d_bad = static_cast<unsigned long long*>(misc);
  int* flags = reinterpret_cast<int*>(d_bad + 2);
  OFL_CUDA(cudaMemsetAsync(misc, 0, 16 + BF_WORDS * sizeof(int), st));
  uint32_t* mask = nullptr;
  if (n_pour > 0) {
    rc = scratch_get(SCRATCH_WORK, ((size_t)rows * (size_t)cols + 31) / 32 * 4, reinterpret_cast<void**>(&mask));
    if (rc == OFL_OK) rc = scatter_pour(pour, n_pour, rows * cols, mask, flags, st);
    if (rc != OFL_OK) return rc;
  }
  basins_check_kernel<<<grid_for(rows * cols, 16), 256, 0, st>>>(fdr, ld_fdr, labels, ld_labels, (int)rows, (int)cols,
                                                                  mask, d_bad);
  OFL_CHECK_LAUNCH();
  struct {
    unsigned long long bad, unused;
    int flags[BF_WORDS];
  } h = {};
  static_assert(sizeof(h) == 16 + BF_WORDS * sizeof(int), "read-back layout");
  OFL_CUDA(cudaMemcpyAsync(&h, misc, sizeof(h), cudaMemcpyDeviceToHost, st));
  OFL_CUDA(cudaStreamSynchronize(st));
  OFL_REQUIRE(h.flags[BF_POUR] == 0, OFL_ERR_INVALID, "pour point outside the raster");
  *n_bad = (int64_t)h.bad;
  return OFL_OK;
}

}  // namespace ofl
