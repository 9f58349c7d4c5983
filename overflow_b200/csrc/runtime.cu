// runtime.cu -- library state: error strings, device scratch, tensor-map encoding.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace ofl {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

const char* last_error() { return g_err; }

int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  set_error("CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
  return e == cudaErrorMemoryAllocation ? OFL_ERR_NOMEM : OFL_ERR_CUDA;
}

bool debug_sync() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("OFL_DEBUG_SYNC");
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
int64_t launch_count() { return g_launches.load(); }
void launch_count_reset() { g_launches.store(0); }

// ---------------------------------------------------------------- phase timing
struct PendingPhase {
  int phase;
  cudaEvent_t start, stop;
};
static bool g_timing = false;
static std::vector<PendingPhase> g_pending;
static std::vector<cudaEvent_t> g_event_pool;
static double g_phase_ms[PHASE_COUNT] = {};
static int64_t g_phase_n[PHASE_COUNT] = {};
static std::mutex g_timing_mu;

static cudaEvent_t event_get() {
  if (!g_event_pool.empty()) {
    cudaEvent_t e = g_event_pool.back();
    g_event_pool.pop_back();
    return e;
  }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}

PhaseScope::PhaseScope(int phase_, cudaStream_t st_) : phase(phase_), st(st_), start(nullptr) {
  if (!g_timing) return;
  std::lock_guard<std::mutex> lk(g_timing_mu);
  start = event_get();
  if (start) cudaEventRecord(start, st);
}

PhaseScope::~PhaseScope() {
  if (!start) return;
  std::lock_guard<std::mutex> lk(g_timing_mu);
  cudaEvent_t stop = event_get();
  if (stop) cudaEventRecord(stop, st);
  g_pending.push_back({phase, start, stop});
}

void phase_timing_enable(int on) {
  std::lock_guard<std::mutex> lk(g_timing_mu);
  g_timing = on != 0;
}

int phase_timing_read(double* ms, int64_t* counts, int n, int reset) {
  std::lock_guard<std::mutex> lk(g_timing_mu);
  for (auto& pp : g_pending) {
    if (pp.start && pp.stop) {
      float t = 0.f;
      if (cudaEventSynchronize(pp.stop) == cudaSuccess && cudaEventElapsedTime(&t, pp.start, pp.stop) == cudaSuccess) {
        g_phase_ms[pp.phase] += t;
        g_phase_n[pp.phase] += 1;
      }
    }
    if (pp.start) g_event_pool.push_back(pp.start);
    if (pp.stop) g_event_pool.push_back(pp.stop);
  }
  g_pending.clear();
  for (int i = 0; i < n && i < PHASE_COUNT; ++i) {
    if (ms) ms[i] = g_phase_ms[i];
    if (counts) counts[i] = g_phase_n[i];
  }
  if (reset)
    for (int i = 0; i < PHASE_COUNT; ++i) {
      g_phase_ms[i] = 0;
      g_phase_n[i] = 0;
    }
  return PHASE_COUNT;
}

// ---------------------------------------------------------------- device state
struct State {
  int device = -1;
  int sms = 0;
  void* scratch[SCRATCH_SLOTS] = {};
  size_t scratch_bytes[SCRATCH_SLOTS] = {};
  void* pinned = nullptr;
  size_t pinned_bytes = 0;
};
static State g_state;
static std::mutex g_mu;
static std::atomic<int> g_generation{0};
static std::vector<void (*)()> g_cleanups;

int device_generation() { return g_generation.load(); }

void register_device_cleanup(void (*fn)()) {
  std::lock_guard<std::mutex> lk(g_mu);
  for (auto f : g_cleanups)
    if (f == fn) return;
  g_cleanups.push_back(fn);
}

// g_mu held; the device being left is current
static void leave_device() {
  if (g_state.device < 0) return;
  cudaDeviceSynchronize();
  for (auto f : g_cleanups) f();
  {
    std::lock_guard<std::mutex> lk(g_timing_mu);
    for (auto& pp : g_pending) {
      if (pp.start) cudaEventDestroy(pp.start);
      if (pp.stop) cudaEventDestroy(pp.stop);
    }
    g_pending.clear();
    for (auto e : g_event_pool) cudaEventDestroy(e);
    g_event_pool.clear();
  }
  for (int i = 0; i < SCRATCH_SLOTS; ++i) {
    if (g_state.scratch[i]) cudaFree(g_state.scratch[i]);
    g_state.scratch[i] = nullptr;
    g_state.scratch_bytes[i] = 0;
  }
  g_generation.fetch_add(1);
}

int init_device(int device) {
  std::lock_guard<std::mutex> lk(g_mu);
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    set_error("no usable CUDA device (%s); liboverflow_b200 has no CPU fallback",
              e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    return OFL_ERR_CUDA;
  }
  OFL_REQUIRE(device >= 0 && device < n, OFL_ERR_INVALID, "device %d out of range (have %d)", device, n);
  if (g_state.device != device) {
    cudaDeviceProp prop;
    OFL_CUDA(cudaGetDeviceProperties(&prop, device));
    OFL_REQUIRE(prop.major >= 10, OFL_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                prop.major, prop.minor);
    // one device at a time: everything the library created on the device it leaves (scratch, streams, events,
    // kernel attributes) is released there first
    if (g_state.device >= 0 && cudaSetDevice(g_state.device) == cudaSuccess) leave_device();
    g_state.device = device;
    g_state.sms = prop.multiProcessorCount;
  }
  OFL_CUDA(cudaSetDevice(device));
  return OFL_OK;
}

int ensure_init() {
  if (g_state.device >= 0) return OFL_OK;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) dev = 0;
  return init_device(dev);
}

int shutdown() {
  std::lock_guard<std::mutex> lk(g_mu);
  if (g_state.device >= 0 && cudaSetDevice(g_state.device) == cudaSuccess) leave_device();
  g_state.device = -1;
  if (g_state.pinned) cudaFreeHost(g_state.pinned);
  g_state.pinned = nullptr;
  g_state.pinned_bytes = 0;
  return OFL_OK;
}

int sm_count() { return g_state.sms > 0 ? g_state.sms : 148; }

int resident_ctas(const void* kernel, int threads, int max_per_sm) {
  struct Entry {
    const void* kernel;
    int generation, ctas;
  };
  static std::mutex mu;
  static std::vector<Entry> cache;
  std::lock_guard<std::mutex> lk(mu);
  Entry* e = nullptr;
  for (Entry& c : cache)
    if (c.kernel == kernel) e = &c;
  if (!e) {
    cache.push_back({kernel, -1, 0});
    e = &cache.back();
  }
  if (e->generation != device_generation()) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
    e->ctas = (per_sm < max_per_sm ? per_sm : max_per_sm) * sm_count();
    e->generation = device_generation();
  }
  return e->ctas;
}

int scratch_get(int slot, size_t bytes, void** out) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (bytes == 0) bytes = 256;
  if (g_state.scratch_bytes[slot] < bytes) {
    if (g_state.scratch[slot]) cudaFree(g_state.scratch[slot]);
    g_state.scratch[slot] = nullptr;
    g_state.scratch_bytes[slot] = 0;
    cudaError_t e = cudaMalloc(&g_state.scratch[slot], bytes);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(scratch)", __FILE__, __LINE__);
    g_state.scratch_bytes[slot] = bytes;
  }
  *out = g_state.scratch[slot];
  return OFL_OK;
}

int pinned_get(size_t bytes, void** out) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (g_state.pinned_bytes < bytes) {
    if (g_state.pinned) cudaFreeHost(g_state.pinned);
    g_state.pinned = nullptr;
    g_state.pinned_bytes = 0;
    cudaError_t e = cudaMallocHost(&g_state.pinned, bytes);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMallocHost", __FILE__, __LINE__);
    g_state.pinned_bytes = bytes;
  }
  *out = g_state.pinned;
  return OFL_OK;
}

// ---------------------------------------------------------------- tensor maps
// cuTensorMapEncodeTiled is a driver API; it is resolved through the runtime so the library
// needs no link-time dependency on libcuda.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

int make_tensor_map_2d(CUtensorMap* tm, const void* base, int esz, uint64_t cols, uint64_t rows, uint64_t pitch_bytes,
                       uint32_t box_w, uint32_t box_h, int l2_promotion_bytes) {
  EncodeTiledFn fn = get_encode_fn();
  OFL_REQUIRE(fn != nullptr, OFL_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  CUtensorMapDataType dt;
  switch (esz) {
    case 1: dt = CU_TENSOR_MAP_DATA_TYPE_UINT8; break;
    case 4: dt = CU_TENSOR_MAP_DATA_TYPE_FLOAT32; break;
    case 8: dt = CU_TENSOR_MAP_DATA_TYPE_UINT64; break;
    default: set_error("unsupported tensor-map element size %d", esz); return OFL_ERR_INVALID;
  }
  // L2 promotion widens every fetch to that granularity: boxes whose rows are far apart in memory (wide
  // rasters) and not aligned to it would drag in neighbouring bytes they never use
  const CUtensorMapL2promotion promo = l2_promotion_bytes >= 256   ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B
                                       : l2_promotion_bytes >= 128 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B
                                       : l2_promotion_bytes >= 64  ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B
                                                                   : CU_TENSOR_MAP_L2_PROMOTION_NONE;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {pitch_bytes};
  cuuint32_t box[2] = {box_w, box_h};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  OFL_REQUIRE(r == CUDA_SUCCESS, OFL_ERR_CUDA,
              "cuTensorMapEncodeTiled failed (%d) for %llux%llu esz=%d pitch=%llu box=%ux%u", (int)r,
              (unsigned long long)cols, (unsigned long long)rows, esz, (unsigned long long)pitch_bytes, box_w, box_h);
  return OFL_OK;
}

}  // namespace ofl
