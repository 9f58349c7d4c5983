// direction_generic.cu -- D8 flow direction for DEMs that are not float32: float64 and the integer types.
//
// The reference's stencil (src/overflow/flow_direction.py:14-96) is dtype-generic under numba: the
// elevation difference is taken in the ARRAY's arithmetic -- float64 for float64, int64 for the signed
// integer types, and uint64 for the unsigned ones, where an uphill neighbour wraps around to a huge
// positive difference -- and only then widened to float64 and divided by 1 or sqrt(2) (:94-96).  The
// nodata test compares the cell, widened to float64, with the band's nodata value (:49, :91).  These
// element kinds are rare next to float32, so this kernel restates the algorithm literally, one thread per
// cell with the 3x3 window read through L1/L2; float32 (and the 8/16-bit signed integers, whose
// differences float32 holds exactly) take the TMA kernel in direction.cu.
#include <math.h>

#include "common.cuh"

namespace ofl {

template <int KIND>
struct ElemOf;
template <>
struct ElemOf<OFL_ELEM_F64> {
  typedef double type;
  static __device__ __forceinline__ double widen(double v) { return v; }
  static __device__ __forceinline__ double diff(double z, double n) { return __dsub_rn(z, n); }
};
template <>
struct ElemOf<OFL_ELEM_I64> {
  typedef long long type;
  static __device__ __forceinline__ double widen(long long v) { return __ll2double_rn(v); }
  static __device__ __forceinline__ double diff(long long z, long long n) {
    return __ll2double_rn((long long)((unsigned long long)z - (unsigned long long)n));  // wraps like int64
  }
};
template <>
struct ElemOf<OFL_ELEM_U64> {
  typedef unsigned long long type;
  static __device__ __forceinline__ double widen(unsigned long long v) { return __ull2double_rn(v); }
  static __device__ __forceinline__ double diff(unsigned long long z, unsigned long long n) {
    return __ull2double_rn(z - n);  // an uphill neighbour wraps to ~2^64, exactly as in the reference
  }
};

struct GenParams {
  const void* dem;
  int64_t ld_dem;
  int64_t in_rows, cols;  // input array
  uint8_t* out;
  int64_t ld_out;
  int64_t rows;  // output rows; output row y reads input rows y + y_off - 1 .. y + y_off + 1
  int y_off;
  double nodata;
  unsigned long long fill_bits;  // what a position outside the input array reads as (nodata cast to the element type)
};

template <int KIND>
__global__ void direction_generic_kernel(const GenParams p) {
  typedef typename ElemOf<KIND>::type T;
  const T* dem = static_cast<const T*>(p.dem);
  T fill;
  memcpy(&fill, &p.fill_bits, sizeof(T));
  const int64_t n = p.rows * p.cols;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t y = i / p.cols, x = i - y * p.cols;
    const int64_t iy = y + p.y_off;
    auto at = [&](int64_t r, int64_t c) -> T {
      return (r < 0 || r >= p.in_rows || c < 0 || c >= p.cols) ? fill : dem[r * p.ld_dem + c];
    };
    const T z = at(iy, x);
    uint32_t code;
    if (ElemOf<KIND>::widen(z) == p.nodata) {
      code = OFL_DIR_NODATA;
    } else {
      // scan order E, NE, N, NW, W, SW, S, SE (constants.py:29-40); first strict maximum wins
      double best = -INFINITY;
      int bi = -1;
      bool any_pos = false;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int dy = dir_dy(k), dx = dir_dx(k);
        const T v = at(iy + dy, x + dx);
        double s;
        if (ElemOf<KIND>::widen(v) == p.nodata)
          s = INFINITY;
        else
          s = (k & 1) ? __ddiv_rn(ElemOf<KIND>::diff(z, v), 1.4142135623730951) : ElemOf<KIND>::diff(z, v);
        if (s > best) {
          best = s;
          bi = k;
        }
        if (s > 0.0) any_pos = true;
      }
      code = any_pos ? (uint32_t)bi : (uint32_t)OFL_DIR_UNDEFINED;
    }
    p.out[y * p.ld_out + x] = (uint8_t)code;
  }
}

// Device-pointer launcher (same row convention as launch_direction in direction.cu).
int launch_direction_generic(const void* dem, int kind, int64_t in_rows, int64_t cols, int64_t ld_dem, double nodata,
                             uint8_t* fdr, int64_t rows, int64_t ld_fdr, int y_off, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return OFL_OK;
  OFL_REQUIRE((reinterpret_cast<uintptr_t>(dem) & 7) == 0, OFL_ERR_ALIGNMENT, "dem must be 8-byte aligned");
  GenParams p;
  p.dem = dem;
  p.ld_dem = ld_dem;
  p.in_rows = in_rows;
  p.cols = cols;
  p.out = fdr;
  p.ld_out = ld_fdr;
  p.rows = rows;
  p.y_off = y_off;
  p.nodata = nodata;
  // util/raster.py:67 fills the out-of-raster halo with the nodata value cast to the band's dtype
  p.fill_bits = 0;
  if (kind == OFL_ELEM_F64) {
    memcpy(&p.fill_bits, &nodata, sizeof(double));
  } else if (kind == OFL_ELEM_I64) {
    const long long v = (nodata >= -9.2e18 && nodata <= 9.2e18) ? (long long)nodata : 0;
    memcpy(&p.fill_bits, &v, sizeof(v));
  } else {
    const unsigned long long v = (nodata >= 0.0 && nodata <= 1.8e19) ? (unsigned long long)nodata : 0;
    memcpy(&p.fill_bits, &v, sizeof(v));
  }
  const int64_t n = rows * cols;
  const int64_t want = (n + 255) / 256;
  const int blocks = (int)(want < (int64_t)sm_count() * 16 ? want : (int64_t)sm_count() * 16);
  {
    PhaseScope ps(PHASE_DIRECTION, st);
    if (kind == OFL_ELEM_F64)
      direction_generic_kernel<OFL_ELEM_F64><<<blocks, 256, 0, st>>>(p);
    else if (kind == OFL_ELEM_I64)
      direction_generic_kernel<OFL_ELEM_I64><<<blocks, 256, 0, st>>>(p);
    else
      direction_generic_kernel<OFL_ELEM_U64><<<blocks, 256, 0, st>>>(p);
  }
  OFL_CHECK_LAUNCH();
  return OFL_OK;
}

}  // namespace ofl
