// api.cu -- the extern "C" surface declared in include/overflow_b200.h.
// Host-pointer calls stage through library-owned device buffers; device-pointer calls launch directly.
#include <cstdlib>
#include <initializer_list>

#include "common.cuh"

namespace ofl {
const char* last_error();
int init_device(int device);
int ensure_init();
int shutdown();
int64_t launch_count();
void launch_count_reset();
void phase_timing_enable(int on);
int phase_timing_read(double* ms, int64_t* counts, int n, int reset);

int direction_shape(int64_t in_rows, int64_t cols);
int launch_direction(const float* dem, int64_t in_rows, int64_t cols, int64_t ld_dem, double nodata, uint8_t* fdr,
                     int64_t rows, int64_t ld_fdr, int y_off, cudaStream_t st);
int launch_direction_generic(const void* dem, int kind, int64_t in_rows, int64_t cols, int64_t ld_dem, double nodata,
                             uint8_t* fdr, int64_t rows, int64_t ld_fdr, int y_off, cudaStream_t st);
int launch_fill_border(uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld, int value, cudaStream_t st);
int64_t perimeter_count(int64_t rows, int64_t cols);
size_t accumulation_workspace_bytes(int64_t rows, int64_t cols);
int accumulation_shape(int64_t rows, int64_t cols);
int launch_accumulation(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, long long* fac, int64_t ld_fac,
                        long long* perim_links_dev, void* workspace, cudaStream_t st, bool prepared = false,
                        bool trusted_codes = false, const long long* perim_inflow_dev = nullptr);
int accumulation_prepare(int64_t rows, int64_t cols, void* workspace, cudaStream_t st);
size_t strip_workspace_bytes(int64_t rows, int64_t cols);
size_t strip_boundary_workspace_bytes(int64_t n_strips, int64_t cols);
size_t strip_record_bytes(int64_t cols);
int strip_shape(int64_t rows, int64_t cols, int has_below);
int strip_accum_local(const uint8_t* fdr_halo, int64_t rows, int64_t cols, int64_t ld_fdr, int has_above, int has_below,
                      long long* fac, int64_t ld_fac, void* workspace, void* record, cudaStream_t st);
int boundary_shape(int64_t n_strips, int64_t cols);
int strip_boundary_solve(const void* records_all, int n_strips, int64_t cols, long long* J_all, void* workspace,
                         cudaStream_t st);
int strip_collect_flags(const void* strip_workspace, int64_t rows, int64_t cols, const void* boundary_workspace,
                        int n_strips, int32_t* flags_dev, cudaStream_t st);
int strip_accum_final(const uint8_t* fdr_halo, int64_t rows, int64_t cols, int64_t ld_fdr, int has_above, int has_below,
                      const long long* J_mine, void* workspace, long long* fac, int64_t ld_fac, cudaStream_t st);
int launch_check(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, const long long* fac, int64_t ld_fac,
                 unsigned long long* n_bad_dev, cudaStream_t st, int y_off = 0, const long long* fac_above = nullptr,
                 const long long* fac_below = nullptr);
size_t flats_workspace_bytes(int64_t rows, int64_t cols);
int flats_shape(int64_t rows, int64_t cols);
int launch_flat_edges(const float* dem, const uint8_t* fdr, int64_t rows, int64_t cols, uint8_t* edges, int64_t* n_low,
                      int64_t* n_high, unsigned* cnt_dev, cudaStream_t st);
int launch_resolve_flats(const float* dem, const uint8_t* fdr, int64_t rows, int64_t cols, int* flat_mask, int* labels,
                         int64_t* info, void* workspace, cudaStream_t st);
int launch_flat_gradient(const int* labels, const uint8_t* fdr, int64_t rows, int64_t cols, const int* seeds,
                         int64_t n_seeds, int towards, int* flat_mask, int* flat_height, int64_t n_heights,
                         void* workspace, cudaStream_t st);
int launch_masked_flow_dirs(const int* flat_mask, const int* labels, uint8_t* fdr, int64_t rows, int64_t cols,
                            cudaStream_t st);
size_t pits_workspace_bytes(int64_t rows, int64_t cols);
int pits_shape(int64_t rows, int64_t cols);
int launch_breach_pits(float* chunk, int64_t rows, int64_t cols, int64_t ld, double nodata, int8_t* unsolved,
                       int64_t* info, void* workspace, cudaStream_t st);
size_t basins_workspace_bytes(int64_t rows, int64_t cols);
int basins_shape(int64_t rows, int64_t cols);
int launch_basins(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, const long long* pour, int64_t n_pour,
                  long long* labels, int64_t ld_labels, void* workspace, cudaStream_t st);
int check_basins(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, const long long* pour, int64_t n_pour,
                 const long long* labels, int64_t ld_labels, int64_t* n_bad, cudaStream_t st);
int launch_synth(float* dem, int64_t rows, int64_t cols, int64_t ld, int64_t row0, int64_t total_rows, uint64_t seed,
                 int kind, float relief, int holes_permille, float nodata, cudaStream_t st);
}  // namespace ofl

using namespace ofl;

// ---------------------------------------------------------------- host rasters: banded pipeline
// A host DEM goes to the device in row bands on its own stream; the stencil of band b runs as soon as
// the first row of band b+1 has arrived, and its codes return to the host on a third stream, so the
// upload, the kernel and the download overlap (PCIe is full duplex).  The staging buffers hold the whole
// raster: accumulation needs every code before it can finish a single count.
namespace {
// Streams and events of the host pipeline belong to the device they were created on: they are keyed on the
// library's device generation and destroyed (by the cleanup hook, on their own device) when it moves on.
struct HostPipe {
  cudaStream_t h2d = nullptr, d2h = nullptr;
  cudaEvent_t ev_in = nullptr, ev_prep = nullptr;
  cudaEvent_t pool[2 * 256] = {};  // band events of direction_from_host, created on demand, reused by every call
  int n_pool = 0;
  int gen = -1;
};
HostPipe g_pipe;

void pipe_cleanup() {
  if (g_pipe.h2d) cudaStreamDestroy(g_pipe.h2d);
  if (g_pipe.d2h) cudaStreamDestroy(g_pipe.d2h);
  if (g_pipe.ev_in) cudaEventDestroy(g_pipe.ev_in);
  if (g_pipe.ev_prep) cudaEventDestroy(g_pipe.ev_prep);
  for (int i = 0; i < g_pipe.n_pool; ++i) cudaEventDestroy(g_pipe.pool[i]);
  g_pipe = HostPipe();
}

int pipe_streams() {
  if (g_pipe.gen == device_generation() && g_pipe.h2d) return OFL_OK;
  g_pipe = HostPipe();  // whatever an older generation held was destroyed by pipe_cleanup on its own device
  register_device_cleanup(pipe_cleanup);
  OFL_CUDA(cudaStreamCreateWithFlags(&g_pipe.h2d, cudaStreamNonBlocking));
  OFL_CUDA(cudaStreamCreateWithFlags(&g_pipe.d2h, cudaStreamNonBlocking));
  OFL_CUDA(cudaEventCreateWithFlags(&g_pipe.ev_in, cudaEventDisableTiming));
  OFL_CUDA(cudaEventCreateWithFlags(&g_pipe.ev_prep, cudaEventDisableTiming));
  g_pipe.gen = device_generation();
  return OFL_OK;
}

constexpr int64_t PIPE_BAND_BYTES = 512ll << 20;  // ~0.5 GiB of DEM per band
constexpr int PIPE_MAX_BANDS = 256;

int pipe_events(int n) {
  while (g_pipe.n_pool < n) {
    OFL_CUDA(cudaEventCreateWithFlags(&g_pipe.pool[g_pipe.n_pool], cudaEventDisableTiming));
    ++g_pipe.n_pool;
  }
  return OFL_OK;
}

// dem: host, in_rows x cols.  d_dem / d_fdr: device staging (pitches ldd / ldo).  fdr_host may be null.
// Output row y reads input rows y + y_off - 1 .. y + y_off + 1.  Enqueues the whole banded pipeline and returns
// at the first error; finish_call drains the streams.
int direction_from_host(const float* dem, int64_t in_rows, int64_t rows, int64_t cols, int64_t ld_dem, double nodata,
                        int y_off, float* d_dem, int64_t ldd, uint8_t* d_fdr, int64_t ldo, uint8_t* fdr_host,
                        int64_t ld_fdr, cudaStream_t st) {
  int rc = pipe_streams();
  if (rc != OFL_OK) return rc;
  int64_t band_bytes = PIPE_BAND_BYTES;
  if (const char* e = getenv("OFL_PIPE_BAND_BYTES")) band_bytes = atoll(e) > 0 ? atoll(e) : band_bytes;  // tests: many small bands
  int64_t band = band_bytes / (cols * (int64_t)sizeof(float));
  band = band < 64 ? 64 : band / 64 * 64;
  if ((in_rows + band - 1) / band > PIPE_MAX_BANDS) band = ((in_rows + PIPE_MAX_BANDS - 1) / PIPE_MAX_BANDS + 63) / 64 * 64;
  const int n_in = (int)((in_rows + band - 1) / band), n_out = (int)((rows + band - 1) / band);
  rc = pipe_events(n_in + n_out);
  if (rc != OFL_OK) return rc;
  cudaEvent_t* ev_up = g_pipe.pool;
  cudaEvent_t* ev_dir = g_pipe.pool + n_in;
  for (int b = 0; b < n_in; ++b) {
    const int64_t r0 = b * band, r1 = (r0 + band < in_rows) ? r0 + band : in_rows;
    OFL_CUDA(cudaMemcpy2DAsync(d_dem + r0 * ldd, ldd * sizeof(float), dem + r0 * ld_dem, ld_dem * sizeof(float),
                               cols * sizeof(float), r1 - r0, cudaMemcpyHostToDevice, g_pipe.h2d));
    OFL_CUDA(cudaEventRecord(ev_up[b], g_pipe.h2d));
  }
  for (int b = 0; b < n_out; ++b) {
    const int64_t r0 = b * band, r1 = (r0 + band < rows) ? r0 + band : rows;
    int64_t in_lo = r0 + y_off - 1, in_hi = r1 + y_off + 1;  // input rows [in_lo, in_hi)
    if (in_lo < 0) in_lo = 0;
    if (in_hi > in_rows) in_hi = in_rows;
    OFL_CUDA(cudaStreamWaitEvent(st, ev_up[(in_hi - 1) / band], 0));  // uploads complete in order
    rc = launch_direction(d_dem + in_lo * ldd, in_hi - in_lo, cols, ldd, nodata, d_fdr + r0 * ldo, r1 - r0, ldo,
                          (int)(r0 + y_off - in_lo), st);
    if (rc != OFL_OK) return rc;
    if (fdr_host) {
      OFL_CUDA(cudaEventRecord(ev_dir[b], st));
      OFL_CUDA(cudaStreamWaitEvent(g_pipe.d2h, ev_dir[b], 0));
      OFL_CUDA(cudaMemcpy2DAsync(fdr_host + r0 * ld_fdr, ld_fdr, d_fdr + r0 * ldo, ldo, cols, r1 - r0,
                                 cudaMemcpyDeviceToHost, g_pipe.d2h));
    }
  }
  return OFL_OK;
}

// ---------------------------------------------------------------- staging of host-memory calls
// Every entry point runs one body against device pointers.  Under OFL_MEM_DEVICE those are the caller's; under
// OFL_MEM_HOST stage_in gives argument i scratch slot SCRATCH_STAGE0 + i and uploads it, and finish_call downloads
// the results and returns only once nothing the call started is still copying, whether it succeeded or not.
// Calls list their rasters widest element first, then their vectors, so that different calls share slots of
// like size.
enum { COPY_NONE = 0, COPY_IN = 1, COPY_OUT = 2 };

struct CallArg {                      // one raster or vector (one row) argument of a call
  const void* caller;                 // the caller's buffer; a nullable host argument may be null (staging only)
  int64_t rows, row_bytes, pitch;     // its layout in bytes
  int copy;                           // what a host call moves between `caller` and its slot (COPY_*)
  int64_t align;                      // a slot row is row_bytes rounded up to this; 1: packed rows, copied in one piece
  bool nullable;                      // the call accepts a null `caller`
  void* dev;                          // set by stage_in: what the body reads and writes
  int64_t dev_pitch;
  template <class T> T* d() const { return static_cast<T*>(dev); }
  int64_t ld(int64_t elem_bytes) const { return dev_pitch / elem_bytes; }
};

// A pitched raster goes as a 2-D copy even when its rows happen to be contiguous: on a B200 (1000 W), one
// cudaMemcpyAsync of the 34 GB counts of a 65536^2 raster took ~2 ms longer than the 2-D copy.
cudaError_t copy_rows(bool packed, void* dst, int64_t dpitch, const void* src, int64_t spitch, int64_t width,
                      int64_t rows, cudaMemcpyKind kind, cudaStream_t st) {
  if (packed) return cudaMemcpyAsync(dst, src, (size_t)(width * rows), kind, st);
  return cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, rows, kind, st);
}

template <int N>
int stage_in(CallArg (&a)[N], int mem_kind, cudaStream_t st) {
  static_assert(N <= SCRATCH_STAGE_SLOTS, "more arguments than staging slots");
  for (int i = 0; i < N; ++i) {
    CallArg& x = a[i];
    if (mem_kind == OFL_MEM_DEVICE) {
      x.dev = const_cast<void*>(x.caller);
      x.dev_pitch = x.pitch;
      continue;
    }
    x.dev_pitch = align_up(x.row_bytes, x.align);
    int rc = scratch_get(SCRATCH_STAGE0 + i, (size_t)(x.rows * x.dev_pitch), &x.dev);
    if (rc != OFL_OK) return rc;
    if ((x.copy & COPY_IN) && x.caller && x.rows * x.row_bytes > 0)
      OFL_CUDA(copy_rows(x.align == 1, x.dev, x.dev_pitch, x.caller, x.pitch, x.row_bytes, x.rows,
                         cudaMemcpyHostToDevice, st));
  }
  return OFL_OK;
}

// Host calls: after a successful body, download every COPY_OUT argument; then, in every case, wait for `st` and
// the band pipeline.  Returns rc, or the first copy error if rc was OFL_OK.  Device calls: returns rc.
template <int N>
int finish_call(int rc, const CallArg (&a)[N], int mem_kind, cudaStream_t st) {
  if (mem_kind == OFL_MEM_DEVICE) return rc;
  cudaError_t e = cudaSuccess;
  for (int i = 0; i < N && rc == OFL_OK && e == cudaSuccess; ++i) {
    const CallArg& x = a[i];
    if ((x.copy & COPY_OUT) && x.caller && x.rows * x.row_bytes > 0)
      e = copy_rows(x.align == 1, const_cast<void*>(x.caller), x.pitch, x.dev, x.dev_pitch, x.row_bytes, x.rows,
                    cudaMemcpyDeviceToHost, st);
  }
  cudaStream_t streams[3] = {st, g_pipe.h2d, g_pipe.d2h};  // the pipeline's exist once a call has used it
  for (int i = 0; i < (g_pipe.h2d ? 3 : 1); ++i) {
    const cudaError_t s = cudaStreamSynchronize(streams[i]);
    if (e == cudaSuccess) e = s;
  }
  if (rc == OFL_OK && e != cudaSuccess) rc = cuda_fail(e, "host staging copy", __FILE__, __LINE__);
  return rc;
}

// Reads a device counter back; returns once it is in *out.
int read_counter(int64_t* out, const void* d_cnt, cudaStream_t st) {
  unsigned long long h = 0;
  OFL_CUDA(cudaMemcpyAsync(&h, d_cnt, sizeof(h), cudaMemcpyDeviceToHost, st));
  OFL_CUDA(cudaStreamSynchronize(st));
  *out = (int64_t)h;
  return OFL_OK;
}

// ---------------------------------------------------------------- argument checks
// Every compute entry point lists its CallArgs and runs through run_call; checks that need more than its raster's
// shape (enums, counts, a strip's rows) come before it.  So an argument error is reported before the call touches
// the device, and a host call is refused only before its first copy.  After that a call fails only on the data it
// reads (a cycle, a pour point outside the raster, more than 2^29 flats in one tile) or on CUDA.
struct Result {  // a scalar result in host memory: zeroed first, so that a refused call leaves zeros behind
  int64_t* p;
  int n;
  bool nullable;
};

struct Workspace {  // a device workspace: the caller's, which must hold need(rows, cols) bytes, or else the library's
  void** ptr;
  size_t* bytes;
  size_t (*need)(int64_t, int64_t);
  const char* what;
};

inline int no_limit(int64_t, int64_t) { return OFL_OK; }
constexpr int EMPTY_RASTER = 1;

template <int N, class Limit>
int check_call(const CallArg (&a)[N], int64_t rows, int64_t cols, int mem_kind, std::initializer_list<Result> results,
               Limit shape_limit, const Workspace& w) {
  for (const Result& r : results) {
    OFL_REQUIRE(r.p || r.nullable, OFL_ERR_INVALID, "null result pointer");
    for (int k = 0; r.p && k < r.n; ++k) r.p[k] = 0;
  }
  OFL_REQUIRE(rows >= 0 && cols >= 0, OFL_ERR_INVALID, "negative raster size");
  OFL_REQUIRE(mem_kind == OFL_MEM_HOST || mem_kind == OFL_MEM_DEVICE, OFL_ERR_INVALID, "unknown mem_kind %d", mem_kind);
  if (rows == 0 || cols == 0) return EMPTY_RASTER;
  for (const CallArg& x : a) {
    OFL_REQUIRE(x.caller || x.nullable, OFL_ERR_INVALID, "null raster pointer");
    OFL_REQUIRE(!x.caller || x.pitch >= x.row_bytes, OFL_ERR_INVALID, "leading dimension smaller than cols");
  }
  int rc = shape_limit(rows, cols);
  if (rc != OFL_OK) return rc;
  const size_t need = w.ptr ? w.need(rows, cols) : 0;
  OFL_REQUIRE(!w.ptr || !*w.ptr || *w.bytes >= need, OFL_ERR_WORKSPACE, "%s workspace too small: need %zu bytes, have %zu",
              w.what, need, w.ptr ? *w.bytes : 0);
  rc = ensure_init();
  if (rc != OFL_OK || !w.ptr || *w.ptr) return rc;
  *w.bytes = need;
  return scratch_get(SCRATCH_WORK, need, w.ptr);
}

// Runs one compute entry point: zeroes the results; checks the sizes, mem_kind, and for a non-empty raster every
// argument's pointer and pitch, the shape limit of the kernels and the workspace; brings the device up, takes the
// library's workspace if the caller gave none, stages the arguments, runs body(stream) and finishes the call.  An
// empty raster returns OFL_OK once the sizes are checked.
template <int N, class Limit, class Body>
int run_call(CallArg (&a)[N], int64_t rows, int64_t cols, int mem_kind, void* stream,
             std::initializer_list<Result> results, Limit shape_limit, Workspace w, Body body) {
  int rc = check_call(a, rows, cols, mem_kind, results, shape_limit, w);
  if (rc != OFL_OK) return rc == EMPTY_RASTER ? OFL_OK : rc;
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = stage_in(a, mem_kind, st);
  if (rc == OFL_OK) rc = body(st);
  return finish_call(rc, a, mem_kind, st);
}
}  // namespace

extern "C" {

const char* ofl_last_error(void) { return last_error(); }
int ofl_abi_version(void) { return OFL_ABI_VERSION; }
int ofl_init(int device) { return init_device(device); }
int ofl_shutdown(void) { return shutdown(); }
int64_t ofl_launch_count(void) { return launch_count(); }
void ofl_launch_count_reset(void) { launch_count_reset(); }
void ofl_phase_timing_enable(int on) { phase_timing_enable(on); }
int ofl_phase_timing_read(double* ms, int64_t* counts, int n, int reset) { return phase_timing_read(ms, counts, n, reset); }
int64_t ofl_perimeter_count(int64_t rows, int64_t cols) { return perimeter_count(rows, cols); }
size_t ofl_accumulation_workspace_bytes(int64_t rows, int64_t cols) { return accumulation_workspace_bytes(rows, cols); }

int ofl_flow_direction_f32(const float* dem, int64_t rows, int64_t cols, int64_t ld_dem, double nodata, uint8_t* fdr,
                           int64_t ld_fdr, int mode, int mem_kind, void* stream) {
  OFL_REQUIRE(mode == OFL_DIR_MODE_TILE || mode == OFL_DIR_MODE_RASTER || mode == OFL_DIR_MODE_STRIP, OFL_ERR_INVALID,
              "unknown direction mode %d", mode);
  const int y_off = (mode == OFL_DIR_MODE_STRIP) ? 1 : 0;
  const int64_t in_rows = rows + 2 * y_off;
  const bool tile = mode == OFL_DIR_MODE_TILE;
  // host: the DEM goes up in bands; the codes come back band by band, or in TILE mode in one copy after the ring fill
  CallArg a[] = {{dem, in_rows, cols * 4, ld_dem * 4, COPY_NONE, 16},
                 {fdr, rows, cols, ld_fdr, tile ? COPY_OUT : COPY_NONE, 16}};
  const auto limit = [&](int64_t, int64_t) {  // a host DEM reaches the kernel in row bands
    return direction_shape(mem_kind == OFL_MEM_DEVICE ? in_rows : 0, cols);
  };
  return run_call(a, rows, cols, mem_kind, stream, {}, limit, {}, [&](cudaStream_t st) {
    int rc = mem_kind == OFL_MEM_HOST
                 ? direction_from_host(dem, in_rows, rows, cols, ld_dem, nodata, y_off, a[0].d<float>(), a[0].ld(4),
                                       a[1].d<uint8_t>(), a[1].ld(1), tile ? nullptr : fdr, ld_fdr, st)
                 : launch_direction(dem, in_rows, cols, ld_dem, nodata, fdr, rows, ld_fdr, y_off, st);
    if (rc == OFL_OK && tile) rc = launch_fill_border(a[1].d<uint8_t>(), rows, cols, a[1].ld(1), OFL_DIR_NODATA, st);
    return rc;
  });
}

int ofl_flow_direction_x64(const void* dem, int elem_kind, int64_t rows, int64_t cols, int64_t ld_dem, double nodata,
                           uint8_t* fdr, int64_t ld_fdr, int mode, int mem_kind, void* stream) {
  OFL_REQUIRE(elem_kind == OFL_ELEM_F64 || elem_kind == OFL_ELEM_I64 || elem_kind == OFL_ELEM_U64, OFL_ERR_INVALID,
              "unknown element kind %d", elem_kind);
  OFL_REQUIRE(mode == OFL_DIR_MODE_TILE || mode == OFL_DIR_MODE_RASTER || mode == OFL_DIR_MODE_STRIP, OFL_ERR_INVALID,
              "unknown direction mode %d", mode);
  const int y_off = (mode == OFL_DIR_MODE_STRIP) ? 1 : 0;
  const int64_t in_rows = rows + 2 * y_off;
  CallArg a[] = {{dem, in_rows, cols * 8, ld_dem * 8, COPY_IN, 8}, {fdr, rows, cols, ld_fdr, COPY_OUT, 16}};
  return run_call(a, rows, cols, mem_kind, stream, {}, no_limit, {}, [&](cudaStream_t st) {
    int rc = launch_direction_generic(a[0].dev, elem_kind, in_rows, cols, a[0].ld(8), nodata, a[1].d<uint8_t>(), rows,
                                      a[1].ld(1), y_off, st);
    if (rc == OFL_OK && mode == OFL_DIR_MODE_TILE)
      rc = launch_fill_border(a[1].d<uint8_t>(), rows, cols, a[1].ld(1), OFL_DIR_NODATA, st);
    return rc;
  });
}

int ofl_fill_border_u8(uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, int value, void* stream) {
  CallArg a[] = {{fdr, rows, cols, ld_fdr}};
  return run_call(a, rows, cols, OFL_MEM_DEVICE, stream, {}, no_limit, {},
                  [&](cudaStream_t st) { return launch_fill_border(fdr, rows, cols, ld_fdr, value, st); });
}

// shared by ofl_flow_accumulation_u8 and ofl_flow_accumulation_seeded_u8
static int accumulation_entry(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, int64_t* fac, int64_t ld_fac,
                              const int64_t* perim_inflow, int64_t* perim_links, void* workspace, size_t workspace_bytes,
                              int mem_kind, void* stream) {
  const int64_t n_perim = perimeter_count(rows, cols);
  CallArg a[] = {{fac, rows, cols * 8, ld_fac * 8, COPY_OUT, 16},
                 {fdr, rows, cols, ld_fdr, COPY_IN, 16},
                 {perim_links, 1, n_perim * 16, n_perim * 16, COPY_OUT, 1, true},
                 {perim_inflow, 1, n_perim * 8, n_perim * 8, COPY_IN, 1, true}};
  return run_call(a, rows, cols, mem_kind, stream, {}, accumulation_shape,
                  {&workspace, &workspace_bytes, accumulation_workspace_bytes, "accumulation"}, [&](cudaStream_t st) {
                    return launch_accumulation(a[1].d<const uint8_t>(), rows, cols, a[1].ld(1), a[0].d<long long>(),
                                               a[0].ld(8), perim_links ? a[2].d<long long>() : nullptr, workspace, st,
                                               false, false, perim_inflow ? a[3].d<const long long>() : nullptr);
                  });
}

int ofl_flow_accumulation_u8(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, int64_t* fac,
                             int64_t ld_fac, int64_t* perim_links, void* workspace, size_t workspace_bytes,
                             int mem_kind, void* stream) {
  return accumulation_entry(fdr, rows, cols, ld_fdr, fac, ld_fac, nullptr, perim_links, workspace, workspace_bytes,
                            mem_kind, stream);
}

int ofl_flow_accumulation_seeded_u8(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, int64_t* fac,
                                    int64_t ld_fac, const int64_t* perim_inflow, int64_t* perim_links, void* workspace,
                                    size_t workspace_bytes, int mem_kind, void* stream) {
  return accumulation_entry(fdr, rows, cols, ld_fdr, fac, ld_fac, perim_inflow, perim_links, workspace, workspace_bytes,
                            mem_kind, stream);
}

// Device rasters: the workspace is cleared on a second stream while the stencil runs.  Host rasters: the DEM goes up
// and the codes come back in bands, overlapping; the counts follow the accumulation.
static int routing_on_device(const float* dem, int64_t rows, int64_t cols, int64_t ld_dem, double nodata, uint8_t* fdr,
                             int64_t ld_fdr, int64_t* fac, int64_t ld_fac, int64_t* perim_links, void* work,
                             cudaStream_t st) {
  int rc = pipe_streams();
  if (rc != OFL_OK) return rc;
  OFL_CUDA(cudaEventRecord(g_pipe.ev_in, st));
  OFL_CUDA(cudaStreamWaitEvent(g_pipe.h2d, g_pipe.ev_in, 0));
  rc = accumulation_prepare(rows, cols, work, g_pipe.h2d);
  if (rc != OFL_OK) return rc;
  OFL_CUDA(cudaEventRecord(g_pipe.ev_prep, g_pipe.h2d));
  rc = launch_direction(dem, rows, cols, ld_dem, nodata, fdr, rows, ld_fdr, 0, st);
  if (rc != OFL_OK) return rc;
  OFL_CUDA(cudaStreamWaitEvent(st, g_pipe.ev_prep, 0));
  return launch_accumulation(fdr, rows, cols, ld_fdr, reinterpret_cast<long long*>(fac), ld_fac,
                             reinterpret_cast<long long*>(perim_links), work, st, true, true);
}

int ofl_flow_routing_f32(const float* dem, int64_t rows, int64_t cols, int64_t ld_dem, double nodata, uint8_t* fdr,
                         int64_t ld_fdr, int64_t* fac, int64_t ld_fac, int64_t* perim_links, int mem_kind, void* stream) {
  const int64_t n_perim = perimeter_count(rows, cols);
  CallArg a[] = {{fac, rows, cols * 8, ld_fac * 8, COPY_OUT, 16},
                 {dem, rows, cols * 4, ld_dem * 4, COPY_NONE, 16},
                 {fdr, rows, cols, ld_fdr, COPY_NONE, 16, mem_kind == OFL_MEM_HOST},
                 {perim_links, 1, n_perim * 16, n_perim * 16, COPY_OUT, 1, true}};
  void* work = nullptr;
  size_t need = 0;
  return run_call(a, rows, cols, mem_kind, stream, {}, accumulation_shape,
                  {&work, &need, accumulation_workspace_bytes, "accumulation"}, [&](cudaStream_t st) {
                    if (mem_kind == OFL_MEM_DEVICE)
                      return routing_on_device(dem, rows, cols, ld_dem, nodata, fdr, ld_fdr, fac, ld_fac, perim_links,
                                               work, st);
                    int rc = direction_from_host(dem, rows, rows, cols, ld_dem, nodata, 0, a[1].d<float>(), a[1].ld(4),
                                                 a[2].d<uint8_t>(), a[2].ld(1), fdr, ld_fdr, st);
                    if (rc != OFL_OK) return rc;
                    return launch_accumulation(a[2].d<const uint8_t>(), rows, cols, a[2].ld(1), a[0].d<long long>(),
                                               a[0].ld(8), perim_links ? a[3].d<long long>() : nullptr, work, st,
                                               false, true);
                  });
}

// The checkers count violations in SCRATCH_MISC.
int ofl_check_accumulation_u8(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, const int64_t* fac,
                              int64_t ld_fac, int64_t* n_bad, int mem_kind, void* stream) {
  CallArg a[] = {{fac, rows, cols * 8, ld_fac * 8, COPY_IN, 8}, {fdr, rows, cols, ld_fdr, COPY_IN, 16}};
  return run_call(a, rows, cols, mem_kind, stream, {{n_bad, 1, false}}, no_limit, {}, [&](cudaStream_t st) {
    void* d_cnt = nullptr;
    int rc = scratch_get(SCRATCH_MISC, 256, &d_cnt);
    if (rc == OFL_OK)
      rc = launch_check(a[1].d<const uint8_t>(), rows, cols, a[1].ld(1), a[0].d<const long long>(), a[0].ld(8),
                        static_cast<unsigned long long*>(d_cnt), st);
    return rc == OFL_OK ? read_counter(n_bad, d_cnt, st) : rc;
  });
}

int ofl_strip_check_accumulation_u8(const uint8_t* fdr_halo, int64_t rows, int64_t cols, int64_t ld_fdr,
                                    const int64_t* fac, int64_t ld_fac, const int64_t* fac_above,
                                    const int64_t* fac_below, int64_t* n_bad, void* stream) {
  CallArg a[] = {{fdr_halo, rows + 2, cols, ld_fdr}, {fac, rows, cols * 8, ld_fac * 8}};
  return run_call(a, rows, cols, OFL_MEM_DEVICE, stream, {{n_bad, 1, false}}, no_limit, {}, [&](cudaStream_t st) {
    void* d_cnt = nullptr;
    int rc = scratch_get(SCRATCH_MISC, 256, &d_cnt);
    if (rc == OFL_OK)
      rc = launch_check(fdr_halo, rows, cols, ld_fdr, reinterpret_cast<const long long*>(fac), ld_fac,
                        static_cast<unsigned long long*>(d_cnt), st, 1, reinterpret_cast<const long long*>(fac_above),
                        reinterpret_cast<const long long*>(fac_below));
    return rc == OFL_OK ? read_counter(n_bad, d_cnt, st) : rc;
  });
}

// ---------------------------------------------------------------- flat resolution (csrc/flats.cu)
size_t ofl_flats_workspace_bytes(int64_t rows, int64_t cols) {
  return (rows > 0 && cols > 0) ? flats_workspace_bytes(rows, cols) : 0;
}

int ofl_flat_edges_f32(const float* dem, const uint8_t* fdr, int64_t rows, int64_t cols, uint8_t* edges, int64_t* n_low,
                       int64_t* n_high, int mem_kind, void* stream) {
  CallArg a[] = {{dem, rows, cols * 4, cols * 4, COPY_IN, 1},
                 {fdr, rows, cols, cols, COPY_IN, 1},
                 {edges, rows, cols, cols, COPY_OUT, 1}};
  return run_call(a, rows, cols, mem_kind, stream, {{n_low, 1, true}, {n_high, 1, true}}, flats_shape, {},
                  [&](cudaStream_t st) {
                    void* d_cnt = nullptr;
                    const int rc = scratch_get(SCRATCH_MISC, 256, &d_cnt);
                    if (rc != OFL_OK) return rc;
                    return launch_flat_edges(a[0].d<const float>(), a[1].d<const uint8_t>(), rows, cols,
                                             a[2].d<uint8_t>(), n_low, n_high, static_cast<unsigned*>(d_cnt), st);
                  });
}

// resolve (+ with `fix`, rewrite the codes in place): shared by ofl_resolve_flats_f32 and ofl_fix_flats_f32
static int flats_entry(const float* dem, const uint8_t* fdr, bool fix, int64_t rows, int64_t cols, int32_t* flat_mask,
                       int32_t* labels, int64_t* info, void* workspace, size_t workspace_bytes, int mem_kind,
                       void* stream) {
  const bool staged_only = fix && mem_kind == OFL_MEM_HOST;  // a host fix_flats caller need not see mask and labels
  CallArg a[] = {{dem, rows, cols * 4, cols * 4, COPY_IN, 1},
                 {flat_mask, rows, cols * 4, cols * 4, COPY_OUT, 1, staged_only},
                 {labels, rows, cols * 4, cols * 4, COPY_OUT, 1, staged_only},
                 {fdr, rows, cols, cols, fix ? COPY_IN | COPY_OUT : COPY_IN, 1}};
  return run_call(a, rows, cols, mem_kind, stream, {{info, 5, true}}, flats_shape,
                  {&workspace, &workspace_bytes, flats_workspace_bytes, "flats"}, [&](cudaStream_t st) {
                    int rc = launch_resolve_flats(a[0].d<const float>(), a[3].d<const uint8_t>(), rows, cols,
                                                  a[1].d<int>(), a[2].d<int>(), info, workspace, st);
                    if (rc == OFL_OK && fix)
                      rc = launch_masked_flow_dirs(a[1].d<int>(), a[2].d<int>(), a[3].d<uint8_t>(), rows, cols, st);
                    return rc;
                  });
}

int ofl_resolve_flats_f32(const float* dem, const uint8_t* fdr, int64_t rows, int64_t cols, int32_t* flat_mask,
                          int32_t* labels, int64_t* info, void* workspace, size_t workspace_bytes, int mem_kind,
                          void* stream) {
  return flats_entry(dem, fdr, false, rows, cols, flat_mask, labels, info, workspace, workspace_bytes, mem_kind, stream);
}

int ofl_fix_flats_f32(const float* dem, uint8_t* fdr, int64_t rows, int64_t cols, int32_t* flat_mask, int32_t* labels,
                      int64_t* info, void* workspace, size_t workspace_bytes, int mem_kind, void* stream) {
  return flats_entry(dem, fdr, true, rows, cols, flat_mask, labels, info, workspace, workspace_bytes, mem_kind, stream);
}

int ofl_d8_masked_flow_dirs_i32(const int32_t* flat_mask, const int32_t* labels, uint8_t* fdr, int64_t rows, int64_t cols,
                                int mem_kind, void* stream) {
  CallArg a[] = {{flat_mask, rows, cols * 4, cols * 4, COPY_IN, 1},
                 {labels, rows, cols * 4, cols * 4, COPY_IN, 1},
                 {fdr, rows, cols, cols, COPY_IN | COPY_OUT, 1}};
  return run_call(a, rows, cols, mem_kind, stream, {}, flats_shape, {}, [&](cudaStream_t st) {
    return launch_masked_flow_dirs(a[0].d<const int>(), a[1].d<const int>(), a[2].d<uint8_t>(), rows, cols, st);
  });
}

int ofl_flat_gradient_i32(const int32_t* labels, const uint8_t* fdr, int64_t rows, int64_t cols, const int32_t* seeds,
                          int64_t n_seeds, int towards, int32_t* flat_mask, int32_t* flat_height, int64_t n_heights,
                          void* workspace, size_t workspace_bytes, int mem_kind, void* stream) {
  CallArg a[] = {{labels, rows, cols * 4, cols * 4, COPY_IN, 1},
                 {flat_mask, rows, cols * 4, cols * 4, COPY_IN | COPY_OUT, 1},
                 {fdr, rows, cols, cols, COPY_IN, 1},
                 {seeds, 1, n_seeds * 4, n_seeds * 4, COPY_IN, 1, n_seeds == 0},
                 {flat_height, 1, n_heights * 4, n_heights * 4, COPY_IN | COPY_OUT, 1, n_heights == 0}};
  const auto limit = [&](int64_t r, int64_t c) -> int {
    OFL_REQUIRE(n_seeds >= 0 && n_seeds <= r * c && n_seeds < (1ll << 32) && n_heights >= 0 && n_heights <= r * c,
                OFL_ERR_INVALID, "seed / flat_height count out of range");
    return flats_shape(r, c);
  };
  return run_call(a, rows, cols, mem_kind, stream, {}, limit,
                  {&workspace, &workspace_bytes, flats_workspace_bytes, "flats"}, [&](cudaStream_t st) {
                    return launch_flat_gradient(a[0].d<const int>(), a[2].d<const uint8_t>(), rows, cols,
                                                a[3].d<const int>(), n_seeds, towards, a[1].d<int>(), a[4].d<int>(),
                                                n_heights, workspace, st);
                  });
}

// ---------------------------------------------------------------- single-cell pit breaching (csrc/pits.cu)
size_t ofl_pits_workspace_bytes(int64_t rows, int64_t cols) {
  return (rows > 0 && cols > 0) ? pits_workspace_bytes(rows, cols) : 0;
}

int ofl_breach_single_cell_pits_f32(float* chunk, int64_t rows, int64_t cols, int64_t ld_chunk, double nodata,
                                    int8_t* unsolved, int64_t* info, void* workspace, size_t workspace_bytes, int mem_kind,
                                    void* stream) {
  CallArg a[] = {{chunk, rows, cols * 4, ld_chunk * 4, COPY_IN | COPY_OUT, 4},
                 {unsolved, rows, cols, cols, COPY_OUT, 1}};
  return run_call(a, rows, cols, mem_kind, stream, {{info, 3, true}}, pits_shape,
                  {&workspace, &workspace_bytes, pits_workspace_bytes, "pits"}, [&](cudaStream_t st) {
                    return launch_breach_pits(a[0].d<float>(), rows, cols, a[0].ld(4), nodata, a[1].d<int8_t>(), info,
                                              workspace, st);
                  });
}

// ---------------------------------------------------------------- row strips (csrc/accumulation.cu), device pointers
size_t ofl_strip_workspace_bytes(int64_t rows, int64_t cols) { return strip_workspace_bytes(rows, cols); }
size_t ofl_strip_boundary_workspace_bytes(int n_strips, int64_t cols) {
  return strip_boundary_workspace_bytes(n_strips, cols);
}

size_t ofl_strip_record_bytes(int64_t cols) { return strip_record_bytes(cols); }

// A strip is never empty, so its shape is checked first.  Device buffers the strip calls only pass on are listed with
// an empty row: run_call checks their pointers.
int ofl_strip_accum_local(const uint8_t* fdr_halo, int64_t rows, int64_t cols, int64_t ld_fdr, int has_above,
                          int has_below, int64_t* fac, int64_t ld_fac, void* workspace, size_t workspace_bytes,
                          void* record, void* stream) {
  CallArg a[] = {{fdr_halo, rows + 2, cols, ld_fdr}, {fac, rows, cols * 8, ld_fac * 8}, {workspace}, {record}};
  const int rc = strip_shape(rows, cols, has_below);
  if (rc != OFL_OK) return rc;
  return run_call(a, rows, cols, OFL_MEM_DEVICE, stream, {}, no_limit,
                  {&workspace, &workspace_bytes, strip_workspace_bytes, "strip"}, [&](cudaStream_t st) {
                    return strip_accum_local(fdr_halo, rows, cols, ld_fdr, has_above, has_below,
                                             reinterpret_cast<long long*>(fac), ld_fac, workspace, record, st);
                  });
}

int ofl_strip_boundary_solve(const void* records_all, int n_strips, int64_t cols, int64_t* J_all, void* workspace,
                             size_t workspace_bytes, void* stream) {
  CallArg a[] = {{records_all}, {J_all}, {workspace}};
  const int rc = boundary_shape(n_strips, cols);
  if (rc != OFL_OK) return rc;
  return run_call(a, n_strips, cols, OFL_MEM_DEVICE, stream, {}, no_limit,
                  {&workspace, &workspace_bytes, strip_boundary_workspace_bytes, "boundary"}, [&](cudaStream_t st) {
                    return strip_boundary_solve(records_all, n_strips, cols, reinterpret_cast<long long*>(J_all),
                                                workspace, st);
                  });
}

int ofl_strip_collect_flags(const void* strip_workspace, int64_t rows, int64_t cols, const void* boundary_workspace,
                            int n_strips, int32_t* flags, void* stream) {
  OFL_REQUIRE(flags != nullptr, OFL_ERR_INVALID, "null pointer");
  OFL_REQUIRE(strip_workspace == nullptr || (rows >= 1 && cols >= 1), OFL_ERR_INVALID, "bad strip size");
  OFL_REQUIRE(boundary_workspace == nullptr || (n_strips >= 1 && cols >= 1), OFL_ERR_INVALID, "bad boundary graph size");
  int rc = ensure_init();
  if (rc != OFL_OK) return rc;
  return strip_collect_flags(strip_workspace, rows, cols, boundary_workspace, n_strips, flags,
                             static_cast<cudaStream_t>(stream));
}

int ofl_strip_accum_final(const uint8_t* fdr_halo, int64_t rows, int64_t cols, int64_t ld_fdr, int has_above,
                          int has_below, const int64_t* J_mine, void* workspace, size_t workspace_bytes, int64_t* fac,
                          int64_t ld_fac, void* stream) {
  CallArg a[] = {{fdr_halo, rows + 2, cols, ld_fdr}, {fac, rows, cols * 8, ld_fac * 8}, {workspace}, {J_mine}};
  const int rc = strip_shape(rows, cols, has_below);
  if (rc != OFL_OK) return rc;
  return run_call(a, rows, cols, OFL_MEM_DEVICE, stream, {}, no_limit,
                  {&workspace, &workspace_bytes, strip_workspace_bytes, "strip"}, [&](cudaStream_t st) {
                    return strip_accum_final(fdr_halo, rows, cols, ld_fdr, has_above, has_below,
                                             reinterpret_cast<const long long*>(J_mine), workspace,
                                             reinterpret_cast<long long*>(fac), ld_fac, st);
                  });
}

// ---------------------------------------------------------------- drainage basins (csrc/basins.cu)
size_t ofl_basins_workspace_bytes(int64_t rows, int64_t cols) { return basins_workspace_bytes(rows, cols); }

int ofl_label_basins_u8(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, const int64_t* pour_points,
                        int64_t n_pour, int64_t* labels, int64_t ld_labels, void* workspace, size_t workspace_bytes,
                        int mem_kind, void* stream) {
  OFL_REQUIRE(n_pour >= 0, OFL_ERR_INVALID, "negative pour-point count");
  CallArg a[] = {{labels, rows, cols * 8, ld_labels * 8, COPY_OUT, 16},
                 {fdr, rows, cols, ld_fdr, COPY_IN, 16},
                 {pour_points, 1, n_pour * 8, n_pour * 8, COPY_IN, 1, n_pour == 0}};
  return run_call(a, rows, cols, mem_kind, stream, {}, basins_shape,
                  {&workspace, &workspace_bytes, basins_workspace_bytes, "basins"}, [&](cudaStream_t st) {
                    return launch_basins(a[1].d<const uint8_t>(), rows, cols, a[1].ld(1), a[2].d<const long long>(),
                                         n_pour, a[0].d<long long>(), a[0].ld(8), workspace, st);
                  });
}

int ofl_check_basins_u8(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, const int64_t* pour_points,
                        int64_t n_pour, const int64_t* labels, int64_t ld_labels, int64_t* n_bad, int mem_kind,
                        void* stream) {
  OFL_REQUIRE(n_pour >= 0, OFL_ERR_INVALID, "negative pour-point count");
  CallArg a[] = {{labels, rows, cols * 8, ld_labels * 8, COPY_IN, 8},
                 {fdr, rows, cols, ld_fdr, COPY_IN, 16},
                 {pour_points, 1, n_pour * 8, n_pour * 8, COPY_IN, 1, n_pour == 0}};
  return run_call(a, rows, cols, mem_kind, stream, {{n_bad, 1, false}}, no_limit, {}, [&](cudaStream_t st) {
    return check_basins(a[1].d<const uint8_t>(), rows, cols, a[1].ld(1), a[2].d<const long long>(), n_pour,
                        a[0].d<const long long>(), a[0].ld(8), n_bad, st);
  });
}

int ofl_synth_dem_f32(float* dem, int64_t rows, int64_t cols, int64_t ld_dem, int64_t row0, int64_t total_rows,
                      uint64_t seed, int kind, float relief, int holes_permille, float nodata, void* stream) {
  OFL_REQUIRE(ld_dem >= cols, OFL_ERR_INVALID, "leading dimension smaller than cols");  // empty rasters included
  OFL_REQUIRE(kind >= 0 && kind <= 4, OFL_ERR_INVALID, "unknown synthetic DEM kind %d", kind);
  OFL_REQUIRE((kind != 3 && kind != 4) || total_rows / 2 * cols < 0xFD000000ll, OFL_ERR_INVALID,
              "serpentine DEM: the chain would run out of finite float32 values");
  CallArg a[] = {{dem, rows, cols * 4, ld_dem * 4}};
  return run_call(a, rows, cols, OFL_MEM_DEVICE, stream, {}, no_limit, {}, [&](cudaStream_t st) {
    return launch_synth(dem, rows, cols, ld_dem, row0, total_rows, seed, kind, relief, holes_permille, nodata, st);
  });
}

}  // extern "C"
