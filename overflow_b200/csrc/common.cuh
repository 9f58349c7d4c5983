// common.cuh -- shared host/device helpers for liboverflow_b200 (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <limits.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/overflow_b200.h"

namespace ofl {

// ---------------------------------------------------------------- error handling
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);
void count_launch(int n = 1);
bool debug_sync();  // OFL_DEBUG_SYNC=1: synchronise after every launch so faults name their kernel

#define OFL_CUDA(expr)                                                        \
  do {                                                                        \
    cudaError_t _e = (expr);                                                  \
    if (_e != cudaSuccess) return ::ofl::cuda_fail(_e, #expr, __FILE__, __LINE__); \
  } while (0)

#define OFL_CHECK_LAUNCH()                                                    \
  do {                                                                        \
    ::ofl::count_launch();                                                    \
    cudaError_t _e = cudaGetLastError();                                      \
    if (_e == cudaSuccess && ::ofl::debug_sync()) _e = cudaDeviceSynchronize(); \
    if (_e != cudaSuccess) return ::ofl::cuda_fail(_e, "kernel launch", __FILE__, __LINE__); \
  } while (0)

#define OFL_REQUIRE(cond, code, ...)  \
  do {                                \
    if (!(cond)) {                    \
      ::ofl::set_error(__VA_ARGS__);  \
      return (code);                  \
    }                                 \
  } while (0)

// ---------------------------------------------------------------- per-phase CUDA-event timing
// When enabled (ofl_phase_timing_enable), every phase is bracketed by cudaEventRecord on the
// launching stream; ofl_phase_timing_read drains the pairs into per-phase sums.
enum Phase { PHASE_DIRECTION = 0, PHASE_ACC_TILE_A, PHASE_ACC_SOLVE, PHASE_ACC_TILE_B, PHASE_ACC_LINKS, PHASE_STRIP_EDGE, PHASE_FLATS, PHASE_FLATS_LABEL, PHASE_FLATS_SWEEP, PHASE_PITS, PHASE_BASINS_TILE, PHASE_BASINS_SOLVE, PHASE_BASINS_FINAL, PHASE_COUNT };
struct PhaseScope {
  int phase;
  cudaStream_t st;
  cudaEvent_t start;
  PhaseScope(int phase, cudaStream_t st);
  ~PhaseScope();
};

// ---------------------------------------------------------------- device properties / scratch
int sm_count();
// Bumped whenever the library moves to another device (ofl_init) or shuts down: everything created on "the
// current device" -- streams, events, per-function attributes -- is keyed on it and re-made when it changes.
int device_generation();
// Called, with the OLD device still current, before the library leaves a device (ofl_init to another device,
// ofl_shutdown): destroy what was created there.
void register_device_cleanup(void (*fn)());

// Library-owned device scratch, grown on demand and kept until ofl_shutdown (slot-indexed).  A host-memory call
// stages its argument i in slot SCRATCH_STAGE0 + i (api.cu).
constexpr int SCRATCH_STAGE_SLOTS = 5;
enum ScratchSlot { SCRATCH_STAGE0 = 0, SCRATCH_WORK = SCRATCH_STAGE0 + SCRATCH_STAGE_SLOTS, SCRATCH_MISC, SCRATCH_DIRCTR, SCRATCH_SLOTS };
int scratch_get(int slot, size_t bytes, void** out);
// Pinned host scratch (slot-indexed) for small read-backs.
int pinned_get(size_t bytes, void** out);

// ---------------------------------------------------------------- launch sizes and workspace layout (host)
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Grid of a grid-stride kernel with 256 threads per CTA over n items: a CTA per 256 items, at most per_sm CTAs per SM.
inline int grid_for(int64_t n, int per_sm) {
  const int64_t want = (n + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * per_sm;
  return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

// CTAs of a cooperatively launched kernel (`threads` per CTA, no dynamic shared memory) that are resident at once on
// the current device, at most max_per_sm on each SM.  Cached per kernel and device_generation().
int resident_ctas(const void* kernel, int threads, int max_per_sm = INT_MAX);

// Cuts a workspace at `base` into buffers, in the order they are taken, each 256-byte aligned.  With a null base only
// `bytes`, the size of the workspace, is meaningful.
struct Carver {
  uintptr_t base;
  size_t bytes = 0;
  explicit Carver(void* base_) : base(reinterpret_cast<uintptr_t>(base_)) {}
  template <class T>
  void take(T*& ptr, size_t n_bytes) {
    ptr = reinterpret_cast<T*>(base + bytes);
    bytes = align_up(bytes + n_bytes, 256);
  }
};

// ---------------------------------------------------------------- TMA tensor maps (host)
// 2-D row-major tensor, element size `esz`, `cols` x `rows`, row pitch in bytes, box_w x box_h tile.
int make_tensor_map_2d(CUtensorMap* tm, const void* base, int esz, uint64_t cols, uint64_t rows,
                       uint64_t pitch_bytes, uint32_t box_w, uint32_t box_h, int l2_promotion_bytes = 128);

// ---------------------------------------------------------------- device-side helpers and PTX wrappers
#ifdef __CUDACC__
// Step of D8 code 0..7 (E, NE, N, NW, W, SW, S, SE).
__device__ __forceinline__ int dir_dy(int code) { return ((0xA901 >> (2 * code)) & 3) - 1; }  // dy+1 = 1,0,0,0,1,2,2,2
__device__ __forceinline__ int dir_dx(int code) { return ((0x901A >> (2 * code)) & 3) - 1; }  // dx+1 = 2,2,1,0,0,0,1,2

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t addr = smem_u32(bar);
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(addr),
      "r"(parity)
      : "memory");
}
// TMA 2-D tile load global -> shared, completion signalled on an mbarrier (tx bytes).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tm, int x, int y, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::
          "r"(smem_u32(smem_dst)),
      "l"(tm), "r"(x), "r"(y), "r"(smem_u32(bar))
      : "memory");
}
// Grid-wide barrier of a cooperatively launched kernel (every CTA resident).  `bar` points at two device words
// zeroed before the launch: bar[0] counts arrivals (monotonic), bar[1] is the generation released so far;
// `generation` is a per-thread count of the barriers passed.  The last CTA to arrive releases the others, which
// poll the release word -- not the word the arrivals are added to -- with a short sleep between polls: a thousand
// CTAs spinning on the arrival counter itself made a barrier cost ~10 us.  Writes made before the barrier are
// visible after it to loads that do not go through L1 (ld.global.cg / volatile).
__device__ __forceinline__ void grid_barrier(unsigned* bar, unsigned& generation) {
  __syncthreads();
  if (threadIdx.x == 0) {
    ++generation;
    __threadfence();
    const unsigned arrived = atomicAdd(&bar[0], 1u) + 1u;
    if (arrived == generation * gridDim.x) {
      atomicExch(&bar[1], generation);
    } else {
      while (*reinterpret_cast<volatile unsigned*>(&bar[1]) < generation) __nanosleep(32);
    }
    __threadfence();
  }
  __syncthreads();
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory");
}
#endif  // __CUDACC__

}  // namespace ofl
