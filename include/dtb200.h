/*
 * dtb200.h -- C ABI of libdtb200.so: descriptools' per-cell terrain-descriptor path
 * (slope, D8, flow accumulation, flow distance / river index / HAND, downslope, GFI,
 * ln(hl/H), TI / MTI) as hand-written sm_100a CUDA kernels.
 *
 * The reference (JVBSouza/descriptools) has no FFI: its boundary is a set of Python
 * module functions that move NumPy arrays to the device, launch one Numba @cuda.jit
 * kernel and copy the result back.  Each entry point below replaces one of those
 * host-wrapper + kernel pairs; the reference interface it replaces is cited as
 * file:line (paths under descriptools/ in the reference checkout).  The Python modules
 * in descriptools_b200/ keep the reference's function names and NumPy signatures and
 * call these symbols through ctypes (see INTEGRATION.md for the binding a maintainer
 * of the reference would add).
 *
 * Conventions
 *   - every array pointer is a DEVICE pointer unless its name ends in _host; buffers are
 *     caller-owned, row-major, dense (leading dimension == cols); nothing is allocated
 *     or freed by the library except through dtb_ws_* ;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); calls
 *     are asynchronous with respect to the host unless stated;
 *   - return value: 0 = DTB_OK, negative = error (dtb_error_string()); no exceptions,
 *     no CPU fallback: without a usable CUDA device every compute call fails;
 *   - nodata sentinel is -100 everywhere (slope.py:231, flowhand.py:601, gfi.py:289);
 *   - D8 codes: 1=E 2=SE 4=S 8=SW 16=W 32=NW 64=N 128=NE, 0 = nodata
 *     (flowhand.py:801-824, downslope.py:490-513);
 *   - linear cell index idx = row * cols + col over the FULL raster (flowhand.py:845).
 *
 * Row bands (multi-GPU): the *_band entry points operate on rows [row0, row0+rows) of a
 * raster with grows x cols cells; see each function.
 */
#ifndef DTB200_H
#define DTB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DTB_ABI_VERSION 1

enum {
    DTB_OK = 0,
    DTB_ERR_INVALID = -1,   /* bad argument (null pointer, negative size, bad dtype)  */
    DTB_ERR_CUDA = -2,      /* a CUDA runtime/driver call failed; see dtb_last_cuda_error */
    DTB_ERR_WORKSPACE = -3, /* workspace too small                                   */
    DTB_ERR_UNSUPPORTED = -4
};

enum { DTB_F32 = 0, DTB_I16 = 1 };  /* DEM / HAND element type            */
enum { DTB_I32 = 0, DTB_I64 = 1 };  /* index / accumulation element type  */

int dtb_abi_version(void);
const char *dtb_error_string(int code);
/* text of the last CUDA error seen by this thread's library calls ("" if none) */
const char *dtb_last_cuda_error(void);
/* number of kernels launched by the library since load / last reset (all threads) */
int64_t dtb_launch_count(void);
void dtb_reset_launch_count(void);
/* Optional per-kernel timing: while enabled, every kernel launch of the library is bracketed by CUDA
 * events on its stream.  dtb_profile_collect waits for the recorded events, writes one text line per
 * kernel name ("name total_ms launches\n", in first-launch order) into buf (NUL-terminated, truncated
 * to cap), clears the records and returns the untruncated length.  Used by bench.py for the roofline
 * of the dominant kernel; off by default. */
void dtb_profile_enable(int on);
int64_t dtb_profile_collect(char *buf, int64_t cap);

/* ---- slope + D8 (fused 3x3 stencil) -----------------------------------------------
 * Replaces slope_cpu + slope_gpu (slope.py:152-206, 209-259) and adds the D8 direction
 * the reference only consumes (flowhand.py:801-824).  `dem` holds buf_rows x cols
 * elements; rows [row_begin,row_end) are computed and written to slope/d8 starting at
 * their element 0 (i.e. out[(r-row_begin)*cols + c]).  Rows outside [0,buf_rows) are
 * off-raster.  For a band, the caller passes a buffer with one halo row above and below
 * (NaN-filled where the band touches the raster edge) and row_begin = 1.
 * slope (f32, percent) and d8 may each be NULL. */
int dtb_slope_d8(const void *dem, int dem_dtype, int64_t buf_rows, int64_t cols,
                 int64_t row_begin, int64_t row_end, double px, float *slope, uint8_t *d8,
                 void *stream);

/* ---- D8 flow accumulation ------------------------------------------------------------
 * New stage (no reference code; convention pinned by 12_fdr.tif -> 12_fac.tif and the
 * consumers gfi.py:432, topoindexes.py:252-255): acc[p] = number of cells strictly
 * upstream of p.  code-0 cells receive nodata_fill.  acc is int32 or int64 (acc_dtype).
 * Returns in *unfinalised_host (may be NULL, forces a stream sync) the number of valid
 * cells on or below D8 cycles (they keep their partial count). */
size_t dtb_flowacc_workspace_bytes(int64_t rows, int64_t cols);
int dtb_flowacc(const uint8_t *d8, int64_t rows, int64_t cols, void *acc, int acc_dtype,
                int64_t nodata_fill, void *ws, size_t ws_bytes, int64_t *unfinalised_host,
                void *stream);

/* Row-band form (multi-GPU, SURVEY.md 8e): `d8` holds the band's rows x cols codes;
 * halo_above / halo_below are the code rows adjacent to the band (NULL at the raster
 * edge); inflow_above / inflow_below give, per column of those halo rows, acc+1 of the
 * halo cell (NULL = 0; only cells that point into the band are read).  A band that has
 * a halo_below must have rows % 64 == 0 (band seams sit on tile seams).
 *   mode DTB_FA_FULL    : whole computation in one call (what dtb_flowacc does).
 *   mode DTB_FA_SUMMARY : tile pass + node sweep with zero inflow, then the band's boundary
 *       summary for its first (above) / last (below) row:
 *         exit_X[c] = band-local acc[c]+1 if the cell drains into the halo row, else 0;
 *         term_X[c] = -2 if the cell takes no flow from that halo row, else where the in-band
 *                     path that starts there leaves the band: (side << 30) | column of the band's
 *                     own first/last-row cell it leaves through (side 0 = above, 1 = below), or -1
 *                     if it ends in the band.
 *       acc receives the tile-local counts (an intermediate the FINISH call completes in place).
 *   mode DTB_FA_FINISH  : adds the resolved inflow to the node counts the SUMMARY call left in the same,
 *       untouched workspace (each seam entry pushes its inflow down its chain: the forest is not
 *       swept a second time), then the final tile pass writes acc.
 * The band driver (descriptools_b200/bands.py) solves the boundary graph between the two calls.
 * Cross-band D8 cycles are not detected (dtb_slope_d8 never produces cycles). */
enum { DTB_FA_FULL = 0, DTB_FA_SUMMARY = 1, DTB_FA_FINISH = 2 };
typedef struct dtb_flowacc_args {
    const uint8_t *d8;
    int64_t rows, cols;
    const uint8_t *halo_above, *halo_below;
    const int64_t *inflow_above, *inflow_below;
    void *acc;
    int acc_dtype;
    int64_t nodata_fill;
    int64_t *exit_above, *exit_below;
    int32_t *term_above, *term_below;
    int mode;
    int64_t *unfinalised_host;
    /* Optional fusion with the HAND stage (pass the same hand_ws in every mode of one computation): if hand_ws is a workspace of
     * dtb_hand_workspace_bytes(rows, cols) bytes, the final tile pass also performs dtb_hand's first
     * pass (entry-node walks) for the river mask acc > hand_river_threshold (example.py:52) and leaves
     * the node states there; the following dtb_hand call on the same fdr / acc / threshold / workspace
     * passes entry_done = 1 and skips that pass. */
    void *hand_ws;
    size_t hand_ws_bytes;
    int64_t hand_river_threshold;
} dtb_flowacc_args;
int dtb_flowacc_band(const dtb_flowacc_args *args, void *ws, size_t ws_bytes, void *stream);

/* The boundary graph between row bands, solved in one call (every rank runs it on the all-gathered summaries):
 * summ int64 [nbands][6][cols] = exit_above, exit_below, term_above, term_below, first and last row of D8 codes of every
 * band (the DTB_FA_SUMMARY outputs); inflow int64 [nbands][2][cols] = what the halo row above / below each band carries
 * (acc + 1), the inflow_above / inflow_below of the DTB_FA_FINISH calls.  *unresolved (device int): a cycle across seams. */
size_t dtb_flowacc_boundary_workspace_bytes(int64_t nbands, int64_t cols);
int dtb_flowacc_boundary_solve(const int64_t *summ, int64_t nbands, int64_t cols, int64_t *inflow, int *unresolved,
                               void *ws, size_t ws_bytes, void *stream);

/* Generic forest accumulation used by the band driver for the boundary graph between row bands:
 * out[i] = base[i] + sum of out[j] over all j with next[j] == i (next[j] < 0: no successor).
 * *unresolved (device int) becomes non-zero if the graph has a cycle.  ws: dtb_forest_workspace_bytes(n). */
size_t dtb_forest_workspace_bytes(int64_t n);
int dtb_forest_accumulate(const int64_t *next, const int64_t *base, int64_t n, int64_t *out,
                          int *unresolved, void *ws, size_t ws_bytes, void *stream);

/* HAND across band seams (multi-GPU driver, rank 0): summ [nbands][8][cols] holds, for the first and then the last
 * row of every band, the summary (state, river index, elevation bits, accumulation) dtb_hand(DTB_HAND_SUMMARY)
 * wrote; res [nbands][8][cols] receives the resolved path behind the halo row above and then below every band --
 * the res_* arrays of dtb_hand_seam for the DTB_HAND_FINISH call.  `rounds` launches of in-place pointer jumping
 * (each at least quadruples the seam crossings covered); *unresolved (device int) becomes non-zero if a path is
 * still crossing seams after that (a cycle across bands): it is reported as FAIL.  The reference has no counterpart
 * (flowhand.py:282-402 walks its partitions serially). */
size_t dtb_hand_boundary_workspace_bytes(int64_t nbands, int64_t cols);
int dtb_hand_boundary_solve(const int64_t *summ, int64_t nbands, int64_t cols, int rounds, int64_t *res,
                            int *unresolved, void *ws, size_t ws_bytes, void *stream);

/* ---- flow distance + river-cell index + HAND (+ optional fused GFI) -------------------
 * Replaces flow_distance_index_cpu + flow_distance_index_gpu (flowhand.py:476-562,
 * 565-846, unpartitioned: out = 0) and hand_calculator (flowhand.py:414-442); with
 * gfi != NULL also river_accumulation + geomorphic_flood_index_gpu (gfi.py:118-147,
 * 267-294) in the same epilogue.
 *   fdr u8, river i8 (0/1) or NULL with (acc, river_threshold): river = acc > threshold
 *   (example.py:52); dem f32 or i16.
 * Outputs (each may be NULL): fdist f32; idx int32/int64 (idx_dtype; -100 = unresolved);
 * hand in the DEM's dtype; gfi f32 (needs acc).  max_moves <= 0 selects the reference's
 * 20000 (flowhand.py:835). */
typedef struct dtb_hand_args {
    const uint8_t *fdr;
    const int8_t *river;      /* or NULL */
    const void *acc;          /* int32/int64 per acc_dtype; needed if river==NULL or gfi */
    int acc_dtype;
    int64_t river_threshold;
    const void *dem;          /* f32 / i16 per dem_dtype; needed for hand / gfi */
    int dem_dtype;
    int64_t rows, cols;
    double px;
    int64_t max_moves;
    float *fdist;
    void *idx;
    int idx_dtype;
    void *hand;
    float *gfi;
    double gfi_n, gfi_b, gfi_size;
    const struct dtb_hand_band *band; /* NULL: the buffers hold the whole raster */
    int entry_done;                   /* 1: the entry-node pass was done by dtb_flowacc_band (hand_ws) */
} dtb_hand_args;

/* Row-band form (multi-GPU).  One dtb_hand_seam per side of the band.
 *   mode DTB_HAND_SUMMARY: entry walks + node jumping inside the band, then per column of the band's
 *     first / last row the state of the path that starts there, for cells that take flow from the
 *     halo row (sum_state = 0 otherwise): packed [63..62 kind | 61..47 n_diag | 46..32 n_card | 31..0 ptr]
 *     with kind 1 = reaches a river cell in the band (sum_idx = its GLOBAL cell index, sum_z its
 *     elevation, sum_acc its accumulation), 2 = fails, 3 = leaves the band again
 *     (ptr = (side << 30) | column of the halo cell it lands on).  No rasters are written.
 *   mode DTB_HAND_FINISH: the tile pass + epilogue; a path that leaves the band continues with
 *     res_*[column]: the resolved path that starts AT that halo cell (kind 1 or 2, move counts,
 *     global river index, river elevation and accumulation), as solved by the band driver.
 *     Reuses the node states the SUMMARY call left in the same, untouched workspace.
 * idx outputs are global: row_offset * cols + local index.  rows % 64 == 0 if below.halo != NULL. */
enum { DTB_HAND_FULL = 0, DTB_HAND_SUMMARY = 1, DTB_HAND_FINISH = 2 };
typedef struct dtb_hand_seam {
    const uint8_t *halo;
    uint64_t *sum_state;
    int64_t *sum_idx;
    double *sum_z;
    int64_t *sum_acc;
    const uint64_t *res_state;
    const int64_t *res_idx;
    const double *res_z;
    const int64_t *res_acc;
} dtb_hand_seam;
typedef struct dtb_hand_band {
    int mode;
    int64_t row_offset;
    dtb_hand_seam above, below;
} dtb_hand_band;

size_t dtb_hand_workspace_bytes(int64_t rows, int64_t cols);
int dtb_hand(const dtb_hand_args *args, void *ws, size_t ws_bytes, void *stream);

/* hand_calculator alone (flowhand.py:414-442) on a caller-supplied index raster.  Indices other than -100 address
 * dem.flat like NumPy does (negative ones count from the end); an index outside [-n, n) -- an IndexError in the
 * reference -- is never dereferenced: the cell gets -100 and *oob (a device int32, may be NULL) is set to 1. */
int dtb_hand_from_index(const void *dem, int dem_dtype, const void *idx, int idx_dtype,
                        int64_t n, void *hand, int32_t *oob, void *stream);

/* ---- self-check of a finished chain (no reference counterpart) ---------------------------
 * Size-independent identities of D8 / accumulation / river index / HAND over rows [row0, row0 + rows) of a raster with
 * total_rows rows, counted into out[0..7] (device, zeroed by the call; csrc/verify.cu lists them): summed over all
 * bands, out[0] == out[1] and out[2..5] == 0 for a correct chain.  idx / dem / hand may be NULL (accumulation only).
 * Used by bench.py after its timed region at sizes no CPU oracle reaches; tests/ pin it against the oracle. */
int dtb_chain_check(const uint8_t *d8, const void *acc, int acc_dtype, const void *idx, int idx_dtype,
                    const float *dem, const float *hand, int64_t rows, int64_t cols, int64_t row0,
                    int64_t total_rows, int64_t river_threshold, unsigned long long *out, void *stream);

/* ---- downslope index -------------------------------------------------------------------
 * Replaces downslope_cpu + downslope_gpu (downslope.py:379-431, 434-532) AND the CPU
 * fix-up pass over the -50 flags (downslope_sequential_jit, downslope.py:160-314,
 * 373-374): one kernel produces the composite result.  max_moves <= 0 selects 5000. */
int dtb_downslope(const void *dem, int dem_dtype, const uint8_t *fdr, int64_t rows,
                  int64_t cols, double px, double delta, int64_t max_moves, float *out,
                  void *stream);
/* rows [row_begin, row_end) only (out holds those rows); the walks still see the whole buffer. */
int dtb_downslope_rows(const void *dem, int dem_dtype, const uint8_t *fdr, int64_t rows, int64_t cols,
                       int64_t row_begin, int64_t row_end, double px, double delta, int64_t max_moves,
                       float *out, void *stream);
/* Row-band form: the buffer is a window of a larger raster -- a band plus halo rows on the sides that are open
 * (open_above / open_below != 0: the first / last buffer row is not the raster's edge).  A walk that would leave the
 * window through an open side cannot be finished in it: the cell gets -50, the reference's own "redo" marker
 * (downslope.py:526-529), and *escaped (device, zeroed by the caller) counts it.  The band driver widens the halo until
 * nothing escapes: the counterpart of the reference's "GPU pass per tile + global CPU pass over the -50 flags"
 * (downslope.py:366-374), without any rank ever holding more than its band plus halo. */
int dtb_downslope_window(const void *dem, int dem_dtype, const uint8_t *fdr, int64_t rows, int64_t cols,
                         int64_t row_begin, int64_t row_end, double px, double delta, int64_t max_moves,
                         float *out, int open_above, int open_below, unsigned long long *escaped, void *stream);

/* The host glue of example.py:42-43 on the device, one in-place pass over a float32 DEM: cells equal to the file's
 * nodata value (has_nodata != 0) and NaN cells become the path's sentinel -100.  (It cannot live in the stencil's load
 * alone: HAND reads the same DEM, hand_calculator flowhand.py:431-436.) */
int dtb_nodata_to_sentinel_f32(float *dem, int64_t n, float nodata, int has_nodata, void *stream);

/* ---- pointwise indices -----------------------------------------------------------------
 * dtb_river_accumulation: gfi.py:118-147.  out has acc's dtype.  Index handling as in
 *          dtb_hand_from_index (out-of-range cells read element 0, *oob is set).
 * dtb_gfi: geomorphic_flood_index_cpu/_gpu (gfi.py:210-264, 267-294); racc is the
 *          pre-gathered river accumulation.
 * dtb_lnhlh: ln_hl_H_cpu/_gpu (gfi.py:349-400, 403-440).
 * dtb_ti_mti: topographic_index_cpu + both kernels (topoindexes.py:170-230, 233-295)
 *          in one pass; ti / mti may each be NULL. */
int dtb_river_accumulation(const void *acc, int acc_dtype, const void *idx, int idx_dtype,
                           int64_t n, void *out, int32_t *oob, void *stream);
int dtb_gfi(const void *hand, int hand_dtype, const void *racc, int acc_dtype, int64_t n,
            double expo, double scale, double size, float *out, void *stream);
int dtb_lnhlh(const void *hand, int hand_dtype, const void *acc, int acc_dtype, int64_t n,
              double expo, double scale, double size, float *out, void *stream);
int dtb_ti_mti(const void *acc, int acc_dtype, const float *slope_rad, int64_t n, double px,
               double expo, float *ti, float *mti, void *stream);
/* example.py:63-64 glue: slope in percent -> radians with nodata patched back to -100 */
int dtb_slope_to_radians(const float *slope_pct, int64_t n, float *slope_rad, void *stream);

/* ---- threshold calibration against a benchmark flood map (SURVEY.md 8 f1) ------------------------------
 * evaluation.py:5-9 (minMaxScale), :90-123 (binary_map), :126-171 (avaliacao), :12-87 (calibration is a host loop
 * over dtb_eval_counts, descriptools_b200/evaluation.py).
 * dtb_eval_counts: confusion counts (tn, fp, fn, tp) of up to 32 strictly ascending thresholds in ONE pass over
 *   the rasters.  desc f32/f64; cells equal to `nodata` (the reference uses descriptor_matrix[0,0]) or NaN are never
 *   flooded; flood int8 with avaliacao's remapping (1 -> 2, -100 -> 0); under != 0: flooded = desc <= threshold, else >=.
 *   counts_host: k x 4 int64, valid on return (the call synchronises the stream).  ws >= 4*33*8 bytes.
 * dtb_eval_class_map: binary map and / or class map (0 tn, 1 fp, 2 fn, 3 tp) for one threshold.
 * dtb_minmax_scale: (mat - mn) / (mx - mn) in f64, nodata and NaN -> NaN. */
enum { DTB_EV_F32 = 0, DTB_EV_F64 = 1, DTB_EV_I16 = 2 };
int dtb_eval_counts(const void *desc, int desc_is_f64, const int8_t *flood, int64_t n, double nodata,
                    const double *thresholds_host, int k, int under, int64_t *counts_host, void *ws,
                    size_t ws_bytes, void *stream);
int dtb_eval_class_map(const void *desc, int desc_is_f64, const int8_t *flood, int64_t n, double nodata,
                       double threshold, int under, int8_t *binary, int8_t *cls, void *stream);
int dtb_minmax_scale(const void *mat, int mat_dtype, int64_t n, double mn, double mx, double nodata,
                     double *out, void *stream);
/* dtb_eval_counts_from_hist (host only): the prefix sums that turn a histogram into the counts of dtb_eval_counts.
 *   hist_host: 4 x 33 uint64, hist[c * 33 + j] = cells of avaliacao class c (0..3, the remapped benchmark) for which
 *   exactly j of the k thresholds do not flag the cell before the first one that does (under: j = #{th < d}, over:
 *   j = #{th <= d}; never-flagged cells at j = k under, j = 0 over); counts_host: k x 4 (tn, fp, fn, tp).
 *
 * Calibration without the float64 raster of minMaxScale (a descriptor on the device, or one row band of it):
 * dtb_eval_extrema: the two ends of np.unique(desc) in one pass, no host sync.  desc f32 / i16 (DTB_EV_F32 / DTB_EV_I16);
 *   out (device, 5 doubles) = smallest and second-smallest DISTINCT non-NaN values, largest non-NaN value, number of
 *   distinct non-NaN values capped at 2 (entries past it are 0), 1 if a NaN occurs.  +0 and -0 are one value (stored as
 *   +0), +-inf are ordinary values.  ws >= dtb_eval_extrema_workspace_bytes().
 * dtb_eval_hist: the histogram above for desc f32 / i16 scaled on load: cell v becomes
 *   (v == nodata || v != v) ? NaN : (v - mn) / (mx - mn) in f64 -- exactly dtb_minmax_scale's value -- and binary_map's
 *   nodata is the scaled value of `corner`, the RAW value of the raster's cell (0, 0).  ADDS into hist (device, 4 x 33
 *   uint64, zeroed by the caller): row bands of one raster may add into one buffer.  Thresholds as for dtb_eval_counts.
 *   No host sync.
 * dtb_eval_class_scaled: the class map (int8: 0 tn, 1 fp, 2 fn, 3 tp after avaliacao's remapping of the benchmark) of
 *   one threshold with the same scaling: avaliacao(binary_map(minMaxScale(desc), threshold), flood). */
int dtb_eval_counts_from_hist(const unsigned long long *hist_host, int k, int under, int64_t *counts_host);
size_t dtb_eval_extrema_workspace_bytes(void);
int dtb_eval_extrema(const void *desc, int desc_dtype, int64_t n, double *out, void *ws, size_t ws_bytes, void *stream);
int dtb_eval_hist(const void *desc, int desc_dtype, const int8_t *flood, int64_t n, double mn, double mx, double nodata,
                  double corner, const double *thresholds_host, int k, int under, unsigned long long *hist, void *stream);
int dtb_eval_class_scaled(const void *desc, int desc_dtype, const int8_t *flood, int64_t n, double mn, double mx,
                          double nodata, double corner, double threshold, int under, int8_t *cls, void *stream);

/* ---- raster files: GeoTIFF chunks decoded on the device (SURVEY.md section 8 f3) ---------
 * Replaces the pixel decode inside rasterio's `rio.open(p).read(1)` (Example/example.py:33-39) for tiled or
 * striped single-band files that are stored, LZW-, Deflate- or PackBits-compressed (GDAL wrote 12_dem / 12_fdr / 12_fac
 * with LZW):
 * the compressed chunks are copied to the device as they lie in the file and one warp decodes each chunk
 * (LZW, Deflate or PackBits, byte order, predictor 2 / 3) into the raster.  File parsing stays on the host (include/dtb200_io.h).
 *   lay          geometry of the file (a chunk decodes to at most 1 MiB: DTB_ERR_UNSUPPORTED otherwise); chunk i covers chunk-row i / across, chunk-column i % across
 *                (across = ceil(cols / chunk_cols) for tiles, 1 for strips); tiles are stored whole, the last
 *                strip holds only the rows that exist.
 *   comp         device buffer with the compressed bytes; chunk first_chunk + i is comp[comp_off[i] ..
 *                comp_off[i] + comp_len[i]); comp_off / comp_len are DEVICE arrays; comp_len[i] == 0 = absent
 *                chunk (reads as zeros).
 *   out          device pointer to the raster (rows x cols samples of bps bytes, dense), or to the row band
 *                [lay->row_lo, lay->row_hi) of it.
 *   ws           dtb_tiff_decode_workspace_bytes(lay, n_chunks) bytes (one scratch chunk + string table per
 *                resident warp; fewer bytes = fewer warps, at least one).
 *   status       device word, zeroed by the caller: stays 0, or receives ((chunk + 1) << 3) | reason for the
 *                first chunk that failed (1 corrupt stream, 2 pre-6.0 LZW, 3 chunk decodes short).
 * dtb_selftest_tiff_decode_host runs the kernel's per-lane code on the CPU over HOST pointers; it exists for
 * the CPU test-suite (no device there) and is not called by the package. */
typedef struct dtb_tiff_layout {
    int64_t rows, cols;
    int32_t bps;         /* bytes per sample: 1, 2, 4, 8                     */
    int32_t predictor;   /* 1 none, 2 horizontal differencing, 3 floating point */
    int32_t compression; /* 1 stored, 5 LZW; decode only: 8 Deflate, 32773 PackBits */
    int32_t tiled;       /* 1 tiles, 0 strips                                 */
    int32_t chunk_rows;  /* TileLength or RowsPerStrip                        */
    int32_t chunk_cols;  /* TileWidth (ignored for strips)                    */
    int32_t big_endian;  /* samples stored most significant byte first        */
    /* a row window, both 0 = the whole raster.  Decoding: `out` holds raster rows [row_lo, row_hi) (a row band: out
     * points at row row_lo) and only those rows are stored.  Encoding: `raster` points at row row_lo and only rows
     * [row_lo, row_hi) are read; every chunk encoded must lie inside the window (the last chunk-row may end at `rows`,
     * its padding rows are replicated as usual), else DTB_ERR_INVALID before any launch.  A chunk's stream is the same
     * whichever window it was encoded from. */
    int64_t row_lo, row_hi;
} dtb_tiff_layout;
size_t dtb_tiff_decode_workspace_bytes(const dtb_tiff_layout *lay, int64_t n_chunks);
int dtb_tiff_decode_chunks(const dtb_tiff_layout *lay, const uint8_t *comp, const uint64_t *comp_off,
                           const uint64_t *comp_len, int64_t first_chunk, int64_t n_chunks, void *out, void *ws,
                           size_t ws_bytes, unsigned long long *status, void *stream);
int dtb_selftest_tiff_decode_host(const dtb_tiff_layout *lay, const uint8_t *comp_host, const uint64_t *comp_off_host,
                                  const uint64_t *comp_len_host, int64_t first_chunk, int64_t n_chunks, void *out_host,
                                  unsigned long long *status_host);

/* The way back -- replaces the pixel encode inside `rio.open(out, "w", **meta).write(...)` (example.py:216-217):
 * dtb_tiff_encode_chunks: one warp gathers chunk first_chunk + i from the raster (partial tiles padded by edge
 *   replication), applies lay->predictor and encodes it (lay->compression 5 LZW, 1 stored; little-endian only) into
 *   enc + i * dtb_tiff_encode_bound(lay); sizes[i] receives the encoded byte count (DEVICE array).  With a row window
 *   (lay->row_lo / row_hi) `raster` holds only those rows: what one rank of a row-band run holds.
 * dtb_tiff_pack_chunks: copies the n_chunks streams to blob + offsets[i] (DEVICE arrays; the caller computes the
 *   offsets from the sizes), so that one device-to-host copy and one write carry the group
 *   (dtbio_write_encoded, include/dtb200_io.h).
 * dtb_selftest_tiff_encode_host: the encode kernel's per-lane code on the CPU over HOST pointers, row window included
 *   (CPU test-suite). */
size_t dtb_tiff_encode_bound(const dtb_tiff_layout *lay);
size_t dtb_tiff_encode_workspace_bytes(const dtb_tiff_layout *lay, int64_t n_chunks);
int dtb_tiff_encode_chunks(const dtb_tiff_layout *lay, const void *raster, int64_t first_chunk, int64_t n_chunks, uint8_t *enc,
                           long long *sizes, void *ws, size_t ws_bytes, void *stream);
int dtb_tiff_pack_chunks(const uint8_t *enc, size_t bound, const long long *sizes, const long long *offsets, int64_t n_chunks,
                         uint8_t *blob, void *stream);
int dtb_selftest_tiff_encode_host(const dtb_tiff_layout *lay, const void *raster_host, int64_t first_chunk, int64_t n_chunks,
                                  uint8_t *enc_host, long long *sizes_host);

/* ---- benchmark support: synthetic DEM "dtb-synth-v1" + depression filling ---------------
 * No reference counterpart (its fixtures were conditioned by an external GIS,
 * Example/example.py:33-39).  Bit-identical to oracle/dt_condition.cpp. */
int dtb_synth_dem_f32(int64_t rows, int64_t cols, int64_t row0, uint32_t seed,
                      const float *amp10_host, float z0, float sr, float sc, float depth,
                      float *out, void *stream);
/* in-place priority-flood+epsilon fixed point; ws = rows*cols floats + 256 bytes.
 * Synchronous.  *iterations_host (may be NULL) receives the number of sweeps. */
size_t dtb_fill_workspace_bytes(int64_t rows, int64_t cols);
int dtb_fill_depressions_f32(float *dem, int64_t rows, int64_t cols, void *ws, size_t ws_bytes,
                             int *iterations_host, void *stream);

/* The same fill over row bands (block-Jacobi: the result equals dtb_fill_depressions_f32 on the
 * whole raster, bit for bit).  dem_halo is (rows + 2) x cols: row 0 and row rows + 1 are halo rows
 * holding the neighbour's row next to the seam, read only where has_above / has_below is 1 and
 * never written; rows 1 .. rows are the band, filled in place.  ws (dtb_fill_band_workspace_bytes)
 * keeps the band's elevations and seed mask from the INIT call to the SOLVE calls after it.
 *   mode DTB_FILL_INIT : halo rows = the neighbours' DEM rows (a cell next to nodata across a seam
 *                        is a seed).  Writes an upper bound of the fill into the band.
 *   mode DTB_FILL_SOLVE: halo rows = the neighbours' current seam rows of the fill.  Relaxes the
 *                        band until a pass changes nothing.  *seam_changed_host = 1 if a cell of
 *                        the band's first or last row was lowered.
 * The driver runs INIT once, then exchanges the seam rows and runs SOLVE on every band until no
 * band reports a seam change.  Synchronous.  *passes_host (may be NULL) receives the number of
 * sweeps (0 for INIT); more than 200000 sweeps in one call return DTB_ERR_UNSUPPORTED. */
enum { DTB_FILL_INIT = 0, DTB_FILL_SOLVE = 1 };
size_t dtb_fill_band_workspace_bytes(int64_t rows, int64_t cols);
int dtb_fill_band_f32(float *dem_halo, int64_t rows, int64_t cols, int has_above, int has_below, int mode,
                      void *ws, size_t ws_bytes, int *passes_host, int *seam_changed_host, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DTB200_H */
