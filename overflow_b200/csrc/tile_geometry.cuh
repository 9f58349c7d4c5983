// tile_geometry.cuh -- the 64 x 64 work tile of the accumulation and the basins, and the numbering of its perimeter.
//
// A raster is cut into AT x AT tiles, row-major, ntx tiles per row; the tiles at the bottom and right edges may be
// partial.  Each tile has SLOTS perimeter slots, and perimeter-graph node tile * SLOTS + slot stands for the tile
// cell in that slot.
#pragma once
#include "common.cuh"

namespace ofl {

constexpr int AT = 64;                 // tile side (cells)
constexpr int AT_SHIFT = 6;
constexpr int SLOTS = 4 * AT;          // perimeter slots per tile (top, bottom, left, right)
static_assert(AT == 1 << AT_SHIFT, "the tile side is 2^AT_SHIFT");

// Tiles along a raster side of n cells.
inline int64_t tiles_along(int64_t n) { return (n + AT - 1) / AT; }

// Tile `tile` of a rows x cols raster: its first cell (y0, x0) and its extent h x w.
__device__ __forceinline__ void tile_rect(int tile, int ntx, int rows, int cols, int& y0, int& x0, int& h, int& w) {
  const int ty = tile / ntx, tx = tile - ty * ntx;
  y0 = ty << AT_SHIFT;
  x0 = tx << AT_SHIFT;
  h = min(AT, rows - y0);
  w = min(AT, cols - x0);
}

// Perimeter slot of tile cell (y, x) in an h x w tile, -1 inside.
__device__ __forceinline__ int slot_of(int y, int x, int h, int w) {
  if (y == 0) return x;
  if (y == h - 1) return AT + x;
  if (x == 0) return 2 * AT + y;
  if (x == w - 1) return 3 * AT + y;
  return -1;
}

// Tile cell of slot s; false when the slot names no cell of an h x w tile.
__device__ __forceinline__ bool cell_of_slot(int s, int h, int w, int& y, int& x) {
  const int side = s >> AT_SHIFT, k = s & (AT - 1);
  if (side == 0) {
    y = 0;
    x = k;
    return k < w;
  }
  if (side == 1) {
    y = h - 1;
    x = k;
    return k < w && h > 1;
  }
  if (side == 2) {
    y = k;
    x = 0;
    return k > 0 && k < h - 1;
  }
  y = k;
  x = w - 1;
  return k > 0 && k < h - 1 && w > 1;
}

// Perimeter node of raster cell (gy, gx), which lies on its tile's perimeter.
__device__ __forceinline__ int node_of_cell(int gy, int gx, int rows, int cols, int ntx) {
  const int ty = gy >> AT_SHIFT, tx = gx >> AT_SHIFT;
  const int h = min(AT, rows - (ty << AT_SHIFT)), w = min(AT, cols - (tx << AT_SHIFT));
  return (ty * ntx + tx) * SLOTS + slot_of(gy & (AT - 1), gx & (AT - 1), h, w);
}

}  // namespace ofl
