/*
 * overflow_b200.h -- C ABI of liboverflow_b200.so: the D8 flow-routing hot path of
 * Denver-Automation-Analytics/overflow, hand-written CUDA for NVIDIA B200 (sm_100a).
 *
 * The reference has no FFI: its replaceable seam is two numba-jitted Python functions.
 * Each entry point below names the reference interface it stands in for (paths relative
 * to the reference tree):
 *
 *   ofl_flow_direction_f32        src/overflow/flow_direction.py:14-69   flow_direction_for_tile
 *                                 (+ calculate_slope :72-96; driver loop :121-124)
 *   ofl_flow_accumulation_u8      src/overflow/flow_accumulation.py:95-158 single_tile_flow_accumulation
 *                                 (get_next_cell :13-37, perimeter_indices :40-51, follow_path :54-92)
 *   ofl_flow_accumulation_seeded_u8  the same for one rectangular tile of a tiled raster, with the inflow the other
 *                                 tiles send into its perimeter cells (Barnes 2016: the consumer's second pass)
 *   ofl_check_accumulation_u8     no reference counterpart: exactness check of the accumulation recurrence
 *   ofl_strip_check_accumulation_u8  the same check on one row strip (halo codes, neighbour strips' boundary counts)
 *   ofl_strip_*                   no reference counterpart: row-strip (multi-GPU) decomposition in the
 *                                 structure of Barnes 2016 (arXiv 1608.04431), the paper cited at
 *                                 src/overflow/flow_accumulation.py:61,100
 *   ofl_flat_edges_f32            src/overflow/fix_flats.py:13-62    flat_edges
 *   ofl_resolve_flats_f32         src/overflow/fix_flats.py:227-288  resolve_flats (label_flats :65-108,
 *                                 away_from_higher :111-161, towards_lower :164-224)
 *   ofl_flat_gradient_i32         src/overflow/fix_flats.py:111-224  away_from_higher / towards_lower on their own
 *   ofl_d8_masked_flow_dirs_i32   src/overflow/fix_flats.py:291-339  d8_masked_flow_dirs
 *   ofl_fix_flats_f32             resolve_flats followed by d8_masked_flow_dirs, codes rewritten in place
 *   ofl_breach_single_cell_pits_f32  src/overflow/breach_single_cell_pits.py:9-63  breach_single_cell_pits_in_chunk
 *   ofl_label_basins_u8           no reference counterpart: drainage basins -- the outlet (or pour point) each cell's
 *                                 D8 path reaches, over the accumulation's edge rule
 *   ofl_check_basins_u8           no reference counterpart: exactness check of a basin labelling
 *   ofl_synth_dem_f32             no reference counterpart: seeded synthetic DEM for benchmarks
 *
 * Conventions
 *   - plain pointers and sizes only; rasters are row-major with an explicit leading dimension in ELEMENTS
 *   - mem_kind says where the raster pointers live (OFL_MEM_HOST: the library stages through device
 *     buffers it owns and copies results back; OFL_MEM_DEVICE: pointers are CUDA device pointers)
 *   - `stream` is a cudaStream_t (NULL = the legacy default stream); device-pointer calls are
 *     asynchronous on it unless stated, host-pointer calls return after the results are in host memory
 *   - a host-pointer call returns only after every copy it started has finished, whether it succeeds or
 *     fails: on return the library no longer reads or writes the caller's host buffers
 *   - every function returns OFL_OK (0) or a negative ofl_status; ofl_last_error() gives the message
 *     for the calling thread
 *   - argument errors (OFL_ERR_INVALID, and OFL_ERR_WORKSPACE for a caller workspace) are reported before the
 *     call allocates, copies or launches anything; what depends on the data read is found only by running the
 *     call: a cycle (OFL_ERR_CYCLE), a pour point outside the raster, more than 2^29 flats in one tile
 *   - there is no CPU fallback: without a usable CUDA device every compute entry point fails
 */
#ifndef OVERFLOW_B200_H
#define OVERFLOW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OFL_ABI_VERSION 2

typedef enum ofl_status {
  OFL_OK = 0,
  OFL_ERR_INVALID = -1,   /* bad argument (NULL pointer, negative size, unknown enum) */
  OFL_ERR_ALIGNMENT = -2, /* device raster violates the alignment contract below */
  OFL_ERR_CUDA = -3,      /* a CUDA call failed; message carries cudaGetErrorString */
  OFL_ERR_NOMEM = -4,     /* device or host allocation failed */
  OFL_ERR_CYCLE = -5,     /* flow-direction raster contains a cycle (never produced by flow direction) */
  OFL_ERR_WORKSPACE = -6  /* caller-provided workspace too small */
} ofl_status;

typedef enum ofl_mem_kind { OFL_MEM_HOST = 0, OFL_MEM_DEVICE = 1 } ofl_mem_kind;

/* Direction codes and sentinels: src/overflow/constants.py:15-24,57-59 */
#define OFL_DIR_EAST 0
#define OFL_DIR_NORTH_EAST 1
#define OFL_DIR_NORTH 2
#define OFL_DIR_NORTH_WEST 3
#define OFL_DIR_WEST 4
#define OFL_DIR_SOUTH_WEST 5
#define OFL_DIR_SOUTH 6
#define OFL_DIR_SOUTH_EAST 7
#define OFL_DIR_UNDEFINED 8
#define OFL_DIR_NODATA 9
#define OFL_FAC_NODATA (-9999)
/* what the reference actually leaves in NODATA cells (flow_accumulation.py:119-121,129-137) */
#define OFL_FAC_NODATA_EMITTED (-9998)
#define OFL_LINK_TERMINATES (-1)
#define OFL_LINK_EXTERNAL (-2)

/* How ofl_flow_direction_f32 treats the input array. */
typedef enum ofl_dir_mode {
  /* flow_direction_for_tile semantics: dem carries its own one-cell ring; interior cells are
   * computed, the ring of `fdr` (uninitialised in the reference) is set to OFL_DIR_NODATA. */
  OFL_DIR_MODE_TILE = 0,
  /* whole raster: every cell is computed and cells outside the array read as the band nodata
   * value cast to float32 -- what flow_direction()'s chunk loop with raster_chunker(buffer=1)
   * produces for the whole file (flow_direction.py:121-124, util/raster.py:67). */
  OFL_DIR_MODE_RASTER = 1,
  /* row strip with halo: dem has rows+2 rows (row 0 and row rows+1 are the neighbours' rows or
   * nodata at the raster top/bottom); fdr has `rows` rows; columns behave as in RASTER mode. */
  OFL_DIR_MODE_STRIP = 2
} ofl_dir_mode;

const char* ofl_last_error(void);
int ofl_abi_version(void);

/* Select the CUDA device for the calling thread's subsequent calls and create library state on it. */
int ofl_init(int device);
/* Free cached staging buffers and workspaces. */
int ofl_shutdown(void);
/* Number of kernels this library has launched since ofl_init / the last reset (bench accounting). */
int64_t ofl_launch_count(void);
void ofl_launch_count_reset(void);

/*
 * Per-phase device timing (benchmarks).  When enabled, each phase is bracketed by CUDA events on the
 * launching stream.  ofl_phase_timing_read waits for the recorded events, adds them to per-phase
 * totals and copies up to n totals (milliseconds) and launch counts out; returns the number of phases:
 *   0 direction kernel   1 accumulation tile pass A   2 perimeter-graph solve
 *   3 accumulation tile pass B   4 perimeter links   5 strip mode: pass B on the strip's first/last tile row
 *   6 flat resolution: the edge / masked-direction stencils   7 flat labelling (edges, components, label order)
 *   8 the two gradient sweeps of flat resolution   9 single-cell pit breaching
 *   10 basins tile pass (with the pour-point scatter)   11 basins perimeter-node solve   12 basins final pass
 */
#define OFL_PHASE_COUNT 13
void ofl_phase_timing_enable(int on);
int ofl_phase_timing_read(double* ms, int64_t* counts, int n, int reset);

/*
 * D8 steepest-descent flow direction.
 *   dem      float32, `rows` x `cols` (STRIP mode: rows+2 x cols), leading dimension ld_dem
 *   nodata   the band nodata value as a double; a cell is nodata iff (double)cell == nodata
 *   fdr      uint8 out, `rows` x `cols`, leading dimension ld_fdr
 * Device-pointer alignment contract: dem 16-byte aligned with ld_dem % 4 == 0;
 * fdr 4-byte aligned with ld_fdr % 4 == 0.  Host pointers have no alignment requirement.
 */
int ofl_flow_direction_f32(const float* dem, int64_t rows, int64_t cols, int64_t ld_dem, double nodata,
                           uint8_t* fdr, int64_t ld_fdr, int mode, int mem_kind, void* stream);

/*
 * The same stencil for DEMs that are not float32.  The reference's arithmetic follows the array's dtype
 * (flow_direction.py:94-96 under numba): float64 differences for float64, int64 for the signed integer
 * types, and uint64 -- with wrap-around for uphill neighbours -- for the unsigned ones; callers widen their
 * elements to one of these three 8-byte kinds (exact for every integer type).  Arguments as for
 * ofl_flow_direction_f32; device pointers need 8-byte alignment for dem, 4-byte for fdr.
 */
typedef enum ofl_elem_kind { OFL_ELEM_F64 = 0, OFL_ELEM_I64 = 1, OFL_ELEM_U64 = 2 } ofl_elem_kind;
int ofl_flow_direction_x64(const void* dem, int elem_kind, int64_t rows, int64_t cols, int64_t ld_dem, double nodata,
                           uint8_t* fdr, int64_t ld_fdr, int mode, int mem_kind, void* stream);

/* Perimeter entries of `links` in perimeter_indices order (flow_accumulation.py:40-51). */
int64_t ofl_perimeter_count(int64_t rows, int64_t cols);

/* Device workspace ofl_flow_accumulation_u8 needs for a rows x cols raster (bytes). */
size_t ofl_accumulation_workspace_bytes(int64_t rows, int64_t cols);

/*
 * Flow accumulation of a whole flow-direction raster (one "tile" in the reference's terms).
 *   fdr          uint8 codes, rows x cols, leading dimension ld_fdr; 9 = NODATA, 8 or >= 10 = no downstream
 *   fac          int64 out, rows x cols, leading dimension ld_fac; NODATA cells get -9998
 *   perim_links  nullable; int64 [ofl_perimeter_count][2] in perimeter_indices order:
 *                (-2,-2) drains straight out, (-1,-1) terminates inside, else (row,col) of the exit cell
 *   workspace    device scratch of at least ofl_accumulation_workspace_bytes (NULL: library-owned, cached)
 * Device-pointer alignment contract: fdr 16-byte aligned with ld_fdr % 16 == 0; fac 16-byte aligned
 * with ld_fac % 2 == 0; perim_links is a device pointer when mem_kind is OFL_MEM_DEVICE.
 * Synchronous with respect to the host (the pointer-jumping phase reads a device flag).
 */
int ofl_flow_accumulation_u8(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, int64_t* fac,
                             int64_t ld_fac, int64_t* perim_links, void* workspace, size_t workspace_bytes,
                             int mem_kind, void* stream);

/*
 * Both steps in one call: flow direction of a whole DEM (RASTER semantics: every cell computed,
 * out-of-raster neighbours read as nodata -- what flow_direction() writes for the file,
 * flow_direction.py:99-124 with util/raster.py:67) followed by flow accumulation of those codes.
 * Host rasters are uploaded in row bands that overlap the stencil and the download of the codes, and
 * the codes never make the round trip through the host that two separate calls need.
 *   fdr   uint8 out, nullable for host callers that only want the counts
 * Alignment contracts as for the two functions above.  Synchronous with respect to the host.
 */
int ofl_flow_routing_f32(const float* dem, int64_t rows, int64_t cols, int64_t ld_dem, double nodata, uint8_t* fdr,
                         int64_t ld_fdr, int64_t* fac, int64_t ld_fac, int64_t* perim_links, int mem_kind, void* stream);

/*
 * The same for ONE RECTANGULAR TILE of a larger, tiled raster (the consumer's second pass in Barnes 2016, the
 * paper behind src/overflow/flow_accumulation.py:61,100): perim_inflow[k] is what the other tiles send into the
 * tile's k-th perimeter cell (perimeter_indices order, the order of perim_links; int64, nullable = no inflow),
 * on any of the four sides.  It is carried down the cell's path inside the tile, so fac holds the FINAL counts of
 * the tile's cells.  A cell listed twice in perimeter_indices (one-row / one-column tiles) carries its inflow once.
 * overflow_b200/tiles.py drives the two passes and solves the graph of all tiles' perimeter cells on the host.
 */
int ofl_flow_accumulation_seeded_u8(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, int64_t* fac,
                                    int64_t ld_fac, const int64_t* perim_inflow, int64_t* perim_links, void* workspace,
                                    size_t workspace_bytes, int mem_kind, void* stream);

/*
 * Exactness check: counts cells where fac != 1 + sum(fac of upstream neighbours) (data cells) or
 * fac != -9998 (NODATA cells).  On an acyclic raster zero violations prove fac is THE answer.
 */
int ofl_check_accumulation_u8(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, const int64_t* fac,
                              int64_t ld_fac, int64_t* n_bad, int mem_kind, void* stream);

/*
 * The same check on one row strip of a partitioned raster (device pointers).  fdr_halo carries one halo row
 * above and below the strip's `rows` rows (as for ofl_strip_accum_local); fac_above / fac_below are the `cols`
 * counts of the rows just outside the strip, owned by the neighbouring strips (null: the raster ends there).
 * Zero violations on every strip prove the partitioned result exact.
 */
int ofl_strip_check_accumulation_u8(const uint8_t* fdr_halo, int64_t rows, int64_t cols, int64_t ld_fdr,
                                    const int64_t* fac, int64_t ld_fac, const int64_t* fac_above,
                                    const int64_t* fac_below, int64_t* n_bad, void* stream);

/* Set the one-cell ring of a device uint8 raster to `value` (TILE mode helper for device callers). */
int ofl_fill_border_u8(uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, int value, void* stream);

/*
 * Row strips (one per GPU).  A strip is `rows` consecutive raster rows, all columns; strips that have a
 * strip below them must have a multiple of 64 rows.  `fdr_halo` is the strip's code raster with ONE halo
 * row above and below: (rows+2) x cols, row 0 = last row of the strip above, row rows+1 = first row of
 * the strip below (contents ignored where has_above / has_below is 0: that side is the raster edge).
 * All pointers are DEVICE pointers; fdr_halo 16-byte aligned with ld_fdr % 16 == 0.
 *
 *   1. ofl_strip_accum_local     strip-local solve; writes the strip's boundary RECORD, one block of
 *                                ofl_strip_record_bytes(cols) bytes describing the strip's first (t=0) and last
 *                                (t=1) row: [2][cols] int64 strip-local counts, then [2][cols] int32 exit links
 *                                ((exit row selector << 30) | exit column of the cell where the cell's path
 *                                leaves the strip, or -1), then [2][cols] uint8 direction codes, zero padding.
 *                                `fac` (rows x cols) is used as scratch for the boundary rows.
 *   2. all-gather the record blocks of the strips in order (caller; ONE NCCL all-gather)
 *                                -> records_all, n_strips consecutive blocks
 *   3. ofl_strip_boundary_solve  same on every GPU: inflow from other strips into every boundary cell,
 *                                J_all [n_strips][2][cols] int64
 *   4. ofl_strip_accum_final     J_mine = J_all[this strip]; writes the final counts of the strip to `fac`
 *   5. ofl_strip_collect_flags   the error flags of 1-4 as int32[4] in device memory (stream-ordered):
 *                                [0] tile pass, [1] strip solve, [2..3] the same for the boundary workspace;
 *                                any non-zero value means the flow-direction raster holds a cycle
 *                                (OFL_ERR_CYCLE).  Either workspace may be NULL (its flags read 0).
 * The strip workspace must be the same buffer in steps 1, 4 and 5.  None of these calls synchronises: they
 * enqueue work on `stream`, and the caller reads the flags once per step (after a MAX all-reduce over the
 * ranks, so that every rank sees the same status).
 */
size_t ofl_strip_workspace_bytes(int64_t rows, int64_t cols);
size_t ofl_strip_boundary_workspace_bytes(int n_strips, int64_t cols);
size_t ofl_strip_record_bytes(int64_t cols);
int ofl_strip_accum_local(const uint8_t* fdr_halo, int64_t rows, int64_t cols, int64_t ld_fdr, int has_above,
                          int has_below, int64_t* fac, int64_t ld_fac, void* workspace, size_t workspace_bytes,
                          void* record, void* stream);
int ofl_strip_boundary_solve(const void* records_all, int n_strips, int64_t cols, int64_t* J_all, void* workspace,
                             size_t workspace_bytes, void* stream);
int ofl_strip_accum_final(const uint8_t* fdr_halo, int64_t rows, int64_t cols, int64_t ld_fdr, int has_above,
                          int has_below, const int64_t* J_mine, void* workspace, size_t workspace_bytes, int64_t* fac,
                          int64_t ld_fac, void* stream);
int ofl_strip_collect_flags(const void* strip_workspace, int64_t rows, int64_t cols, const void* boundary_workspace,
                            int n_strips, int32_t* flags, void* stream);

/*
 * Flat resolution (Barnes, Lehman & Mulla 2014; the reference's src/overflow/fix_flats.py).  One tile of at most
 * 2^32 cells (cell indices are 32-bit unsigned on the device); every raster is DENSE row-major (leading dimension
 * == cols).  Host-pointer calls stage through library buffers; device-pointer calls take CUDA pointers.  Calls that
 * return counts (n_low / n_high, info) synchronise the stream before they return.
 *   dem        float32 elevations (compared with == and <, as the reference does on the array's own dtype)
 *   fdr        uint8 direction codes; 8 = no direction (the flats), 9 = NODATA
 *   edges      uint8 out: bit 0 = low edge, bit 1 = high edge (the reference returns two lists, row-major)
 *   flat_mask  int32 out: increments per cell      labels  int32 out: flat labels, numbered in the order the
 *              row-major low-edge list first meets each flat (1-based; 0 = not in a drainable flat)
 *   info       nullable int64[5] out: low edges, high edges, labels, levels of the away / towards sweeps
 *   workspace  device scratch of ofl_flats_workspace_bytes (NULL: library-owned, cached)
 * ofl_flat_gradient_i32 runs one sweep from a list of seed cell indices (row * cols + col, read as uint32): towards == 0 is
 * away_from_higher, towards == 1 is towards_lower (which negates flat_mask first and reads flat_height).
 * ofl_fix_flats_f32 rewrites the code-8 cells of fdr in place; for host callers flat_mask / labels may be NULL.
 */
size_t ofl_flats_workspace_bytes(int64_t rows, int64_t cols);
int ofl_flat_edges_f32(const float* dem, const uint8_t* fdr, int64_t rows, int64_t cols, uint8_t* edges, int64_t* n_low,
                       int64_t* n_high, int mem_kind, void* stream);
int ofl_resolve_flats_f32(const float* dem, const uint8_t* fdr, int64_t rows, int64_t cols, int32_t* flat_mask,
                          int32_t* labels, int64_t* info, void* workspace, size_t workspace_bytes, int mem_kind,
                          void* stream);
int ofl_flat_gradient_i32(const int32_t* labels, const uint8_t* fdr, int64_t rows, int64_t cols, const int32_t* seeds,
                          int64_t n_seeds, int towards, int32_t* flat_mask, int32_t* flat_height, int64_t n_heights,
                          void* workspace, size_t workspace_bytes, int mem_kind, void* stream);
int ofl_d8_masked_flow_dirs_i32(const int32_t* flat_mask, const int32_t* labels, uint8_t* fdr, int64_t rows, int64_t cols,
                                int mem_kind, void* stream);
int ofl_fix_flats_f32(const float* dem, uint8_t* fdr, int64_t rows, int64_t cols, int32_t* flat_mask, int32_t* labels,
                      int64_t* info, void* workspace, size_t workspace_bytes, int mem_kind, void* stream);

/*
 * Single-cell pit breaching (the reference's breach_single_cell_pits_in_chunk): `chunk` is breached IN PLACE, as in
 * the reference; the two outermost rows and columns are the chunk's buffer and are only read.
 *   chunk     float32, rows x cols, leading dimension ld_chunk (in and out)
 *   nodata    the band nodata value as a double; a cell is nodata iff (double)cell == nodata
 *   unsolved  int8 out, dense rows x cols: 1 where a single-cell pit could not be breached (the reference's result)
 *   info      nullable int64[3] out: pits found, pits left unsolved, rounds of the dependency-ordered second pass
 *   workspace device scratch of ofl_pits_workspace_bytes (NULL: library-owned, cached)
 * One chunk of at most 2^32 cells (a 65536 x 65536 raster; cell indices are unsigned 32-bit).  Synchronises the
 * stream once, at the end.
 */
size_t ofl_pits_workspace_bytes(int64_t rows, int64_t cols);
int ofl_breach_single_cell_pits_f32(float* chunk, int64_t rows, int64_t cols, int64_t ld_chunk, double nodata,
                                    int8_t* unsolved, int64_t* info, void* workspace, size_t workspace_bytes, int mem_kind,
                                    void* stream);

/*
 * Drainage basins.  Edge rule of the accumulation: cell c drains into d iff code(c) is 0..7, d lies inside the
 * raster and code(d) != 9.  A data cell that drains nowhere is an OUTLET (code 8, codes >= 10, a step off the
 * raster or into NODATA); outlet (r, c) has the label r * cols + c + 1.
 *   fdr          uint8 codes, rows x cols, leading dimension ld_fdr
 *   pour_points  nullable; n_pour row-major cell indices r * cols + c.  With pour points, a pour point is a root
 *                (its outgoing edge is cut) and labels its cells p + 1, where p is the first pour point on the
 *                cell's path (the cell itself included); a cell whose path meets none gets 0.  A pour point on a
 *                NODATA cell has no effect; duplicates are allowed; an index outside [0, rows * cols) is
 *                OFL_ERR_INVALID.
 *   labels       int64 out, rows x cols, leading dimension ld_labels: the label of the outlet (or pour point) the
 *                cell's path ends at; NODATA cells get OFL_BASIN_NODATA
 *   workspace    device scratch of at least ofl_basins_workspace_bytes, which includes the pour-point mask
 *                (NULL: library-owned, cached)
 * Alignment contracts as for ofl_flow_accumulation_u8: fdr like its fdr, labels like its fac.  A cyclic raster
 * is OFL_ERR_CYCLE.  Synchronous with respect to the host (the cycle and pour-point checks read device flags).
 * ofl_check_basins_u8 counts the cells that break the rule: a NODATA cell has label 0, a cell that drains into a
 * cell and is not a pour point has that cell's label, a root has its own index + 1 (0 for a natural outlet when
 * pour points are given).  On an acyclic raster zero violations prove the labels exact.  Synchronises the stream.
 */
#define OFL_BASIN_NODATA 0
size_t ofl_basins_workspace_bytes(int64_t rows, int64_t cols);
int ofl_label_basins_u8(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, const int64_t* pour_points,
                        int64_t n_pour, int64_t* labels, int64_t ld_labels, void* workspace, size_t workspace_bytes,
                        int mem_kind, void* stream);
int ofl_check_basins_u8(const uint8_t* fdr, int64_t rows, int64_t cols, int64_t ld_fdr, const int64_t* pour_points,
                        int64_t n_pour, const int64_t* labels, int64_t ld_labels, int64_t* n_bad, int mem_kind,
                        void* stream);

/*
 * Seeded synthetic DEM written straight into device memory (benchmarks / large parity runs).
 * Cell (row0 + r, c) depends only on its global coordinates and the seed, so every rank of a
 * row-strip run can synthesise its own strip and halo rows.
 *   kind 0: multi-octave value-noise fractal in [0, relief]   kind 1: same, quantised to 1.0 (terraces)
 *   kind 2: tilted plane draining south-east                   holes_permille: nodata rectangles
 *   kind 3: walled serpentine, ONE channel of about rows * cols / 2 cells through the whole raster (every other
 *           row, alternating east / west, consecutive float32 values walked downwards), walls draining into it
 *   kind 4: the same channel transposed -- it runs north-south and crosses every row-strip boundary cols / 2 times
 */
int ofl_synth_dem_f32(float* dem, int64_t rows, int64_t cols, int64_t ld_dem, int64_t row0, int64_t total_rows,
                      uint64_t seed, int kind, float relief, int holes_permille, float nodata, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OVERFLOW_B200_H */
