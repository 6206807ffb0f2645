// tiffcodec.cu -- GeoTIFF chunks decoded and encoded on the device (SURVEY.md section 8 f3).
//
// The reference lets GDAL decode its rasters on one host thread (rio.open(p).read(1), example.py:33-39).  A
// 40 000 x 40 000 DEM is ~10^5 independent LZW tiles: here the compressed tiles travel over PCIe as they lie in
// the file (a fraction of the decoded bytes) and every tile is decoded by one warp -- the lanes run the serial LZW
// recurrence in lock step (lzw.cuh, the same function the host codec uses: uniform control flow, broadcast loads,
// string copies spread over the lanes) into a per-warp scratch chunk, then undo the predictor one row each and
// store the rows to the raster together.  Thousands of tiles are
// in flight at once; nothing here is bandwidth-bound, the point is to take the decode off the host cores and to
// halve the bytes crossing PCIe.
//
// The way back (example.py:216-217 writes one class map; the chain writes seven rasters) mirrors it: a warp gathers
// its tile from the raster, applies the predictor, LZW-encodes it (lzw.cuh: forgetful 2-way hash dictionary of 32-bit
// slots) into a worst-case slot; a second kernel packs the streams back to back so that one
// device-to-host copy and one file write carry a whole group of tiles.
//
// Everything a lane does is in __host__ __device__ phase functions; dtb_selftest_tiff_decode_host() /
// dtb_selftest_tiff_encode_host() run the same functions lane by lane on the CPU so the tile geometry, predictor,
// coder and store logic are tested without a device (tests/test_raster_io.py).  The package never calls them.
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "common.cuh"
#include "inflate.cuh"
#include "lzw.cuh"

namespace dtb {
namespace {

constexpr int TD_WARPS = 4;  // warps per CTA, string / hash tables in global memory
constexpr int TD_LANES = 32;
constexpr int TD_CTAS_PER_SM = 8;  // 64 registers x 128 threads: 8 CTAs fill the register file
// tables in shared memory: 32 KB per warp, 7 warps = 224 KB of the 227 KB a CTA may have, one CTA per SM.  Fewer chunks
// in flight (1 036 instead of 4 736) but a table access costs tens of cycles instead of an L2 / DRAM round trip.
constexpr int TS_WARPS = 7;
constexpr size_t TS_TABLE_BYTES = 32768;
static_assert(sizeof(LzwPackedSlot) * kLzwTableSlots == TS_TABLE_BYTES, "decoder table must be 32 KB");
static_assert(sizeof(uint32_t) * kLzwHashSlots == TS_TABLE_BYTES, "encoder table must be 32 KB");
static_assert(sizeof(InflateScratch) <= TS_TABLE_BYTES, "the Huffman tables live in the warp's table area");
constexpr int TC_LZW = 5, TC_DEFLATE = 8, TC_PACKBITS = 32773;  // TIFF compression codes (stored chunks run through the LZW instantiation)

struct ChunkGeom {
    int64_t cy, cx;        // chunk row / column
    int64_t data_rows;     // rows of the chunk inside the raster
    int64_t stored_rows;   // rows the chunk is stored with (tiles are whole)
    int64_t row_bytes;     // chunk_cols * bps
    int64_t raw_bytes;     // row_bytes * stored_rows
    int64_t x0, ncols;     // first raster column, columns inside the raster
};

__host__ __device__ inline int64_t td_across(const dtb_tiff_layout &L)
{
    return L.tiled ? (L.cols + L.chunk_cols - 1) / L.chunk_cols : 1;
}

__host__ __device__ inline ChunkGeom td_geom(const dtb_tiff_layout &L, int64_t chunk)
{
    ChunkGeom g;
    const int64_t across = td_across(L);
    const int64_t cw = L.tiled ? L.chunk_cols : L.cols;
    g.cy = chunk / across;
    g.cx = chunk % across;
    const int64_t left = L.rows - g.cy * L.chunk_rows;
    g.data_rows = left < L.chunk_rows ? left : L.chunk_rows;
    g.stored_rows = L.tiled ? L.chunk_rows : g.data_rows;
    g.row_bytes = cw * L.bps;
    g.raw_bytes = g.row_bytes * g.stored_rows;
    g.x0 = g.cx * cw;
    g.ncols = (L.cols - g.x0) < cw ? (L.cols - g.x0) : cw;
    return g;
}

__host__ __device__ inline size_t td_scratch_bytes(const dtb_tiff_layout &L)
{
    const int64_t cw = L.tiled ? L.chunk_cols : L.cols;
    const size_t raw = (size_t)cw * L.bps * (size_t)L.chunk_rows;
    return ((raw + 15) & ~(size_t)15) + sizeof(LzwPackedSlot) * kLzwTableSlots;
}

// status word: 0 = ok, else ((chunk + 1) << 3) | reason   (reason 1 corrupt, 2 old-style LZW, 3 short chunk)
__host__ __device__ inline long long td_status(int64_t chunk, int reason) { return (long long)(((chunk + 1) << 3) | reason); }

// ---- phase 1 (all lanes in lock step): compressed bytes -> scratch chunk.  Returns bytes produced or a negative
// reason, the same value in every lane.  [lane0, lane1) of nlanes: see lzw.cuh.  CODEC is a template parameter so
// that each kernel carries one decoder only. ----
template <int CODEC>
__host__ __device__ inline int64_t td_phase1(const ChunkGeom &g, const uint8_t *comp, uint64_t len, uint8_t *buf, void *tab, int lane0,
                                             int lane1)
{
    if (CODEC == TC_PACKBITS) return packbits_decode_lanes(comp, (size_t)len, buf, (size_t)g.raw_bytes, lane0, lane1, TD_LANES);
    if (CODEC == TC_DEFLATE)
        return zlib_inflate(comp, (size_t)len, buf, (size_t)g.raw_bytes, static_cast<InflateScratch *>(tab), lane0, lane1, TD_LANES);
    return lzw_decode(comp, (size_t)len, buf, (size_t)g.raw_bytes, static_cast<LzwPackedSlot *>(tab), lane0, lane1, TD_LANES);
}

// stored chunks: all lanes copy the bytes into the scratch chunk (the predictor works in place)
__host__ __device__ inline void td_copy_stored(const uint8_t *comp, uint64_t n, uint8_t *buf, int lane)
{
    for (uint64_t i = (uint64_t)lane; i < n; i += TD_LANES) buf[i] = comp[i];
}

template <typename T>
__host__ __device__ inline void td_hacc(uint8_t *row, int64_t width)
{
    T *p = reinterpret_cast<T *>(row);
    T run = p[0];
    for (int64_t i = 1; i < width; ++i) {
        run = (T)(run + p[i]);
        p[i] = run;
    }
}

__host__ __device__ inline void td_swap(uint8_t *row, int64_t width, int bps)
{
    for (int64_t i = 0; i < width; ++i) {
        uint8_t *s = row + i * bps;
        for (int a = 0, b = bps - 1; a < b; ++a, --b) {
            const uint8_t t = s[a];
            s[a] = s[b];
            s[b] = t;
        }
    }
}

// ---- phase 2 (one row per lane): byte order and predictor, in place -------------------------------------------
__host__ __device__ inline void td_phase2(const dtb_tiff_layout &L, const ChunkGeom &g, uint8_t *buf, int lane)
{
    const int64_t width = g.row_bytes / L.bps;
    for (int64_t r = lane; r < g.data_rows; r += TD_LANES) {
        uint8_t *row = buf + r * g.row_bytes;
        if (L.big_endian && L.predictor != 3 && L.bps > 1) td_swap(row, width, L.bps);
        if (L.predictor == 2) {
            switch (L.bps) {
                case 1: td_hacc<uint8_t>(row, width); break;
                case 2: td_hacc<uint16_t>(row, width); break;
                case 4: td_hacc<uint32_t>(row, width); break;
                case 8: td_hacc<unsigned long long>(row, width); break;
            }
        } else if (L.predictor == 3) {
            // floating-point predictor: byte planes, differenced byte by byte over the whole row
            uint8_t run = row[0];
            for (int64_t i = 1; i < g.row_bytes; ++i) {
                run = (uint8_t)(run + row[i]);
                row[i] = run;
            }
        }
    }
}

// ---- phase 3 (all lanes per row): scratch rows -> raster ---------------------------------------------------------
__host__ __device__ inline void td_phase3(const dtb_tiff_layout &L, const ChunkGeom &g, const uint8_t *buf, uint8_t *out, int lane)
{
    const int64_t width = g.row_bytes / L.bps;
    const int64_t bytes = g.ncols * L.bps;
    const int64_t lo = L.row_lo, hi = L.row_hi > 0 ? L.row_hi : L.rows;  // the rows `out` holds
    for (int64_t r = 0; r < g.data_rows; ++r) {
        const int64_t R = g.cy * L.chunk_rows + r;
        if (R < lo || R >= hi) continue;
        const uint8_t *row = buf + r * g.row_bytes;
        uint8_t *dst = out + ((R - lo) * L.cols + g.x0) * L.bps;
        if (L.predictor == 3) {
            // sample i, byte b (little-endian) sits in plane bps-1-b at position i
            for (int64_t i = lane; i < g.ncols; i += TD_LANES)
                for (int b = 0; b < L.bps; ++b) dst[i * L.bps + b] = row[(int64_t)(L.bps - 1 - b) * width + i];
        } else if ((((uintptr_t)dst | (uintptr_t)row | (uintptr_t)bytes) & 3u) == 0) {
            const uint32_t *s = reinterpret_cast<const uint32_t *>(row);
            uint32_t *d = reinterpret_cast<uint32_t *>(dst);
            for (int64_t i = lane; i < bytes / 4; i += TD_LANES) d[i] = s[i];
        } else {
            for (int64_t i = lane; i < bytes; i += TD_LANES) dst[i] = row[i];
        }
    }
}

// an absent chunk (offset or byte count 0: GDAL's SPARSE_OK) reads as zeros
__host__ __device__ inline void td_zero(const dtb_tiff_layout &L, const ChunkGeom &g, uint8_t *out, int lane)
{
    const int64_t bytes = g.ncols * L.bps;
    const int64_t lo = L.row_lo, hi = L.row_hi > 0 ? L.row_hi : L.rows;
    for (int64_t r = 0; r < g.data_rows; ++r) {
        const int64_t R = g.cy * L.chunk_rows + r;
        if (R < lo || R >= hi) continue;
        uint8_t *dst = out + ((R - lo) * L.cols + g.x0) * L.bps;
        for (int64_t i = lane; i < bytes; i += TD_LANES) dst[i] = 0;
    }
}

extern __shared__ __align__(16) uint8_t tc_smem[];  // TS_WARPS tables when the kernel is instantiated with SMEM

template <int WARPS, bool SMEM, int CODEC>
__global__ void __launch_bounds__(WARPS *TD_LANES)
tiff_decode_kernel(dtb_tiff_layout L, const uint8_t *__restrict__ comp, const uint64_t *__restrict__ comp_off,
                   const uint64_t *__restrict__ comp_len, int64_t first_chunk, int64_t n_chunks, uint8_t *__restrict__ out,
                   uint8_t *__restrict__ ws, int64_t n_warps, unsigned long long *__restrict__ status)
{
    const int lane = threadIdx.x % TD_LANES;
    const int64_t warp = (int64_t)blockIdx.x * WARPS + threadIdx.x / TD_LANES;
    if (warp >= n_warps) return;
    const size_t per = td_scratch_bytes(L);
    uint8_t *buf = ws + (size_t)warp * per;
    LzwPackedSlot *tab = SMEM ? reinterpret_cast<LzwPackedSlot *>(tc_smem + (threadIdx.x / TD_LANES) * TS_TABLE_BYTES)
                              : reinterpret_cast<LzwPackedSlot *>(buf + (per - sizeof(LzwPackedSlot) * kLzwTableSlots));
    for (int64_t c = warp; c < n_chunks; c += n_warps) {
        const ChunkGeom g = td_geom(L, first_chunk + c);
        const uint64_t off = comp_off[c], len = comp_len[c];
        if (len == 0) {
            td_zero(L, g, out, lane);
            continue;
        }
        long long got = 0;
        if (L.compression == 1) {
            got = (long long)(len < (uint64_t)g.raw_bytes ? len : (uint64_t)g.raw_bytes);
            td_copy_stored(comp + off, (uint64_t)got, buf, lane);
        } else {
            got = td_phase1<CODEC>(g, comp + off, len, buf, tab, lane, lane + 1);
        }
        if (got < g.row_bytes * g.data_rows) {
            if (lane == 0) atomicCAS(status, 0ull, (unsigned long long)td_status(first_chunk + c, got == -2 ? 2 : got < 0 ? 1 : 3));
            continue;  // uniform across the warp
        }
        __syncwarp();
        td_phase2(L, g, buf, lane);
        __syncwarp();
        td_phase3(L, g, buf, out, lane);
        __syncwarp();  // the scratch chunk is reused by this warp's next chunk
    }
}


// =====================================================================================================
// encoding
// =====================================================================================================
__host__ __device__ inline size_t te_raw_bytes(const dtb_tiff_layout &L)
{
    const int64_t cw = L.tiled ? L.chunk_cols : L.cols;
    return (size_t)cw * L.bps * (size_t)L.chunk_rows;
}

// bytes reserved per encoded chunk
__host__ __device__ inline size_t te_bound(const dtb_tiff_layout &L)
{
    const size_t raw = te_raw_bytes(L);
    return ((L.compression == 5 ? lzw_encode_bound(raw) : raw) + 15) & ~(size_t)15;
}

__host__ __device__ inline size_t te_scratch_bytes(const dtb_tiff_layout &L)
{
    return ((te_raw_bytes(L) + 15) & ~(size_t)15) + sizeof(uint32_t) * kLzwHashSlots;
}

// ---- phase 1 (all lanes per row): raster -> scratch chunk.  A partial tile is padded by repeating its last
// column / row (never read back, compresses well); predictor 3 lays the row out as byte planes, most significant
// byte of every sample first.  `raster` holds rows from L.row_lo on (0 for a whole raster); the geometry stays the
// raster's, so a chunk's stream does not depend on the window it was gathered from. ----
__host__ __device__ inline void te_gather(const dtb_tiff_layout &L, const ChunkGeom &g, const uint8_t *raster, uint8_t *buf, int lane)
{
    const int64_t width = g.row_bytes / L.bps;
    for (int64_t r = 0; r < g.stored_rows; ++r) {
        const int64_t rr = r < g.data_rows ? r : g.data_rows - 1;
        const uint8_t *src = raster + ((g.cy * L.chunk_rows + rr - L.row_lo) * L.cols + g.x0) * L.bps;
        uint8_t *row = buf + r * g.row_bytes;
        for (int64_t i = lane; i < width; i += TD_LANES) {
            const int64_t ii = i < g.ncols ? i : g.ncols - 1;
            for (int b = 0; b < L.bps; ++b) {
                const uint8_t v = src[ii * L.bps + b];
                if (L.predictor == 3) row[(int64_t)(L.bps - 1 - b) * width + i] = v;
                else row[i * L.bps + b] = v;
            }
        }
    }
}

template <typename T>
__host__ __device__ inline void te_hdiff(uint8_t *row, int64_t width)
{
    T *p = reinterpret_cast<T *>(row);
    for (int64_t i = width - 1; i >= 1; --i) p[i] = (T)(p[i] - p[i - 1]);
}

// ---- phase 2 (one row per lane): predictor, in place ----
__host__ __device__ inline void te_predict(const dtb_tiff_layout &L, const ChunkGeom &g, uint8_t *buf, int lane)
{
    const int64_t width = g.row_bytes / L.bps;
    for (int64_t r = lane; r < g.stored_rows; r += TD_LANES) {
        uint8_t *row = buf + r * g.row_bytes;
        if (L.predictor == 2) {
            switch (L.bps) {
                case 1: te_hdiff<uint8_t>(row, width); break;
                case 2: te_hdiff<uint16_t>(row, width); break;
                case 4: te_hdiff<uint32_t>(row, width); break;
                case 8: te_hdiff<unsigned long long>(row, width); break;
            }
        } else if (L.predictor == 3) {
            for (int64_t i = g.row_bytes - 1; i >= 1; --i) row[i] = (uint8_t)(row[i] - row[i - 1]);
        }
    }
}

// ---- phase 3: scratch chunk -> encoded slot; returns the encoded size (the same in every lane) ----
__host__ __device__ inline int64_t te_encode(const dtb_tiff_layout &L, const ChunkGeom &g, const uint8_t *buf, uint8_t *slot, size_t bound,
                                             uint64_t *tab, int lane0, int lane1)
{
    if (L.compression == 5) return lzw_encode(buf, (size_t)g.raw_bytes, slot, bound, tab, lane0, lane1, TD_LANES);
    for (int l = lane0; l < lane1; ++l)
        for (int64_t i = l; i < g.raw_bytes; i += TD_LANES) slot[i] = buf[i];
    return g.raw_bytes;
}

template <int WARPS, bool SMEM>
__global__ void __launch_bounds__(WARPS *TD_LANES)
tiff_encode_kernel(dtb_tiff_layout L, const uint8_t *__restrict__ raster, int64_t first_chunk, int64_t n_chunks,
                   uint8_t *__restrict__ enc, long long *__restrict__ sizes, uint8_t *__restrict__ ws, int64_t n_warps)
{
    const int lane = threadIdx.x % TD_LANES;
    const int64_t warp = (int64_t)blockIdx.x * WARPS + threadIdx.x / TD_LANES;
    if (warp >= n_warps) return;
    const size_t per = te_scratch_bytes(L), bound = te_bound(L);
    uint8_t *buf = ws + (size_t)warp * per;
    uint64_t *tab = SMEM ? reinterpret_cast<uint64_t *>(tc_smem + (threadIdx.x / TD_LANES) * TS_TABLE_BYTES)
                         : reinterpret_cast<uint64_t *>(buf + (per - sizeof(uint32_t) * kLzwHashSlots));
    for (int64_t c = warp; c < n_chunks; c += n_warps) {
        const ChunkGeom g = td_geom(L, first_chunk + c);
        te_gather(L, g, raster, buf, lane);
        __syncwarp();
        te_predict(L, g, buf, lane);
        __syncwarp();
        const int64_t n = te_encode(L, g, buf, enc + (size_t)c * bound, bound, tab, lane, lane + 1);
        if (lane == 0) sizes[c] = n;
        __syncwarp();  // the scratch chunk is reused by this warp's next chunk
    }
}

constexpr int TP_THREADS = 256;

// encoded slots -> one contiguous blob (chunk c at blob + offsets[c])
__global__ void __launch_bounds__(TP_THREADS)
tiff_pack_kernel(const uint8_t *__restrict__ enc, size_t bound, const long long *__restrict__ sizes,
                 const long long *__restrict__ offsets, int64_t n_chunks, uint8_t *__restrict__ blob)
{
    for (int64_t c = blockIdx.x; c < n_chunks; c += gridDim.x) {
        const uint8_t *src = enc + (size_t)c * bound;
        uint8_t *dst = blob + offsets[c];
        const long long n = sizes[c];
        for (long long i = threadIdx.x; i < n; i += TP_THREADS) dst[i] = src[i];
    }
}

// resident CTAs per SM: TD_CTAS_PER_SM, or the tuning override DTB_TIFF_CTAS_PER_SM=1..8 (fewer warps keep the string
// tables in L2, more warps hide more latency)
int64_t td_warp_cap()
{
    int ctas = TD_CTAS_PER_SM;
    if (const char *e = getenv("DTB_TIFF_CTAS_PER_SM")) {
        const int v = atoi(e);
        if (v >= 1 && v <= TD_CTAS_PER_SM) ctas = v;
    }
    return (int64_t)kNumSMs * ctas * TD_WARPS;
}

// Where the tables live.  Measured on a B200 (profiles/r1z_raster_codec_tables_16384.json): a warp with its table in
// shared memory runs ~2.4x faster, but only 1 036 of them are resident against 4 736 with the tables in global memory --
// so shared memory wins while a launch has at most two shared-memory waves of chunks.  DTB_TIFF_TABLES=shared | global
// overrides the choice.
bool tc_tables_in_smem(int64_t n_chunks)
{
    if (const char *e = getenv("DTB_TIFF_TABLES")) {
        if (strcmp(e, "shared") == 0) return true;
        if (strcmp(e, "global") == 0) return false;
    }
    return n_chunks <= 2 * (int64_t)kNumSMs * TS_WARPS;
}

// the shared-memory instantiations need the opt-in to 224 KB of dynamic shared memory, once per process
template <typename K>
cudaError_t tc_allow_smem(K kernel, bool &done)
{
    if (done) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(TS_WARPS * TS_TABLE_BYTES));
    if (e == cudaSuccess) done = true;
    return e;
}

int td_validate_common(const dtb_tiff_layout *L)
{
    if (!L || L->rows <= 0 || L->cols <= 0 || L->chunk_rows <= 0) return DTB_ERR_INVALID;
    if (L->bps != 1 && L->bps != 2 && L->bps != 4 && L->bps != 8) return DTB_ERR_INVALID;
    if (L->predictor < 1 || L->predictor > 3) return DTB_ERR_INVALID;
    if (L->tiled && L->chunk_cols <= 0) return DTB_ERR_INVALID;
    if (L->compression != 1 && L->compression != TC_LZW && L->compression != TC_DEFLATE && L->compression != TC_PACKBITS) return DTB_ERR_UNSUPPORTED;
    if ((L->compression == 1 || L->compression == TC_PACKBITS) && L->predictor != 1) return DTB_ERR_INVALID;  // the predictor belongs to LZW / Deflate
    if (L->row_lo != 0 || L->row_hi != 0)
        if (L->row_lo < 0 || L->row_lo >= L->row_hi || L->row_hi > L->rows) return DTB_ERR_INVALID;
    return DTB_OK;
}

int te_validate(const dtb_tiff_layout *L)
{
    const int v = td_validate_common(L);
    if (v != DTB_OK) return v;
    if (L->compression == TC_DEFLATE || L->compression == TC_PACKBITS) return DTB_ERR_UNSUPPORTED;  // chunks are written stored or LZW-compressed
    if (L->big_endian) return DTB_ERR_UNSUPPORTED;  // files are written little-endian
    if (L->predictor == 3 && L->bps < 4) return DTB_ERR_INVALID;
    return DTB_OK;
}

// chunks [first, first + n) of an encode call: inside the raster, and with a row window set, inside the window (a
// chunk-row that ends at the raster's last row counts as ending there, its padding rows are replicated)
int te_validate_range(const dtb_tiff_layout *L, int64_t first, int64_t n)
{
    if (first < 0 || n < 0) return DTB_ERR_INVALID;
    const int64_t across = td_across(*L);
    if (first + n > across * ((L->rows + L->chunk_rows - 1) / L->chunk_rows)) return DTB_ERR_INVALID;
    if (n == 0 || (L->row_lo == 0 && L->row_hi == 0)) return DTB_OK;
    const int64_t top = first / across * L->chunk_rows, end = ((first + n - 1) / across + 1) * L->chunk_rows;
    if (top < L->row_lo || (end < L->rows ? end : L->rows) > L->row_hi) return DTB_ERR_INVALID;
    return DTB_OK;
}

int td_validate(const dtb_tiff_layout *L)
{
    const int v = td_validate_common(L);
    if (v != DTB_OK) return v;
    const int64_t cw = L->tiled ? L->chunk_cols : L->cols;
    if ((size_t)cw * L->bps * (size_t)L->chunk_rows > LzwPackedSlot::kMaxChunkBytes) return DTB_ERR_UNSUPPORTED;  // 20-bit offsets
    return DTB_OK;
}

}  // namespace
}  // namespace dtb

using namespace dtb;

extern "C" {

size_t dtb_tiff_decode_workspace_bytes(const dtb_tiff_layout *lay, int64_t n_chunks)
{
    if (td_validate(lay) != DTB_OK || n_chunks <= 0) return 0;
    const int64_t cap = (int64_t)kNumSMs * TD_CTAS_PER_SM * TD_WARPS;  // the most any setting uses
    const int64_t warps = n_chunks < cap ? n_chunks : cap;
    return (size_t)warps * td_scratch_bytes(*lay) + 256;
}

int dtb_tiff_decode_chunks(const dtb_tiff_layout *lay, const uint8_t *comp, const uint64_t *comp_off, const uint64_t *comp_len,
                           int64_t first_chunk, int64_t n_chunks, void *out, void *ws, size_t ws_bytes,
                           unsigned long long *status, void *stream)
{
    const int v = td_validate(lay);
    if (v != DTB_OK) return v;
    if (n_chunks == 0) return DTB_OK;
    if (!comp || !comp_off || !comp_len || !out || !ws || !status || n_chunks < 0 || first_chunk < 0) return DTB_ERR_INVALID;
    const int64_t total = td_across(*lay) * ((lay->rows + lay->chunk_rows - 1) / lay->chunk_rows);
    if (first_chunk + n_chunks > total) return DTB_ERR_INVALID;
    const size_t per = td_scratch_bytes(*lay);
    if (ws_bytes < per + 256) return DTB_ERR_WORKSPACE;
    int64_t warps = (int64_t)((ws_bytes - 256) / per);
    const bool smem = tc_tables_in_smem(n_chunks);
    const int64_t cap = smem ? (int64_t)kNumSMs * TS_WARPS : td_warp_cap();
    if (warps > cap) warps = cap;
    if (warps > n_chunks) warps = n_chunks;
    // scratch chunks start 256-byte aligned
    uint8_t *base = reinterpret_cast<uint8_t *>(((uintptr_t)ws + 255) & ~(uintptr_t)255);
    cudaStream_t st = as_stream(stream);
    if (smem) {
        const unsigned blocks = (unsigned)((warps + TS_WARPS - 1) / TS_WARPS);
        if (lay->compression == TC_PACKBITS) {
            static bool allowed = false;
            DTB_CUDA(tc_allow_smem(tiff_decode_kernel<TS_WARPS, true, TC_PACKBITS>, allowed));
            DTB_KERNEL("tiff_packbits_kernel<shared>", st,
                       tiff_decode_kernel<TS_WARPS, true, TC_PACKBITS><<<blocks, TS_WARPS * TD_LANES, TS_WARPS * TS_TABLE_BYTES, st>>>(
                           *lay, comp, comp_off, comp_len, first_chunk, n_chunks, (uint8_t *)out, base, warps, status));
        } else if (lay->compression == TC_DEFLATE) {
            static bool allowed = false;
            DTB_CUDA(tc_allow_smem(tiff_decode_kernel<TS_WARPS, true, TC_DEFLATE>, allowed));
            DTB_KERNEL("tiff_inflate_kernel<shared>", st,
                       tiff_decode_kernel<TS_WARPS, true, TC_DEFLATE><<<blocks, TS_WARPS * TD_LANES, TS_WARPS * TS_TABLE_BYTES, st>>>(
                           *lay, comp, comp_off, comp_len, first_chunk, n_chunks, (uint8_t *)out, base, warps, status));
        } else {
            static bool allowed = false;
            DTB_CUDA(tc_allow_smem(tiff_decode_kernel<TS_WARPS, true, TC_LZW>, allowed));
            DTB_KERNEL("tiff_decode_kernel<shared>", st,
                       tiff_decode_kernel<TS_WARPS, true, TC_LZW><<<blocks, TS_WARPS * TD_LANES, TS_WARPS * TS_TABLE_BYTES, st>>>(
                           *lay, comp, comp_off, comp_len, first_chunk, n_chunks, (uint8_t *)out, base, warps, status));
        }
    } else {
        const unsigned blocks = (unsigned)((warps + TD_WARPS - 1) / TD_WARPS);
        if (lay->compression == TC_PACKBITS)
            DTB_KERNEL("tiff_packbits_kernel", st,
                       tiff_decode_kernel<TD_WARPS, false, TC_PACKBITS><<<blocks, TD_WARPS * TD_LANES, 0, st>>>(
                           *lay, comp, comp_off, comp_len, first_chunk, n_chunks, (uint8_t *)out, base, warps, status));
        else if (lay->compression == TC_DEFLATE)
            DTB_KERNEL("tiff_inflate_kernel", st,
                       tiff_decode_kernel<TD_WARPS, false, TC_DEFLATE><<<blocks, TD_WARPS * TD_LANES, 0, st>>>(
                           *lay, comp, comp_off, comp_len, first_chunk, n_chunks, (uint8_t *)out, base, warps, status));
        else
            DTB_KERNEL("tiff_decode_kernel", st,
                       tiff_decode_kernel<TD_WARPS, false, TC_LZW><<<blocks, TD_WARPS * TD_LANES, 0, st>>>(
                           *lay, comp, comp_off, comp_len, first_chunk, n_chunks, (uint8_t *)out, base, warps, status));
    }
    return DTB_OK;
}

int dtb_selftest_tiff_decode_host(const dtb_tiff_layout *lay, const uint8_t *comp_host, const uint64_t *comp_off_host,
                                  const uint64_t *comp_len_host, int64_t first_chunk, int64_t n_chunks, void *out_host,
                                  unsigned long long *status_host)
{
    const int v = td_validate(lay);
    if (v != DTB_OK) return v;
    if (!comp_host || !comp_off_host || !comp_len_host || !out_host || !status_host || n_chunks < 0) return DTB_ERR_INVALID;
    const dtb_tiff_layout &L = *lay;
    std::vector<uint8_t> scratch(td_scratch_bytes(L));
    uint8_t *buf = scratch.data();
    LzwPackedSlot *tab = reinterpret_cast<LzwPackedSlot *>(buf + (scratch.size() - sizeof(LzwPackedSlot) * kLzwTableSlots));
    *status_host = 0;
    for (int64_t c = 0; c < n_chunks; ++c) {
        const ChunkGeom g = td_geom(L, first_chunk + c);
        const uint64_t off = comp_off_host[c], len = comp_len_host[c];
        if (len == 0) {
            for (int lane = 0; lane < TD_LANES; ++lane) td_zero(L, g, (uint8_t *)out_host, lane);
            continue;
        }
        long long got;
        if (L.compression == 1) {
            got = (long long)(len < (uint64_t)g.raw_bytes ? len : (uint64_t)g.raw_bytes);
            for (int lane = 0; lane < TD_LANES; ++lane) td_copy_stored(comp_host + off, (uint64_t)got, buf, lane);
        } else {
            got = L.compression == TC_DEFLATE    ? td_phase1<TC_DEFLATE>(g, comp_host + off, len, buf, tab, 0, TD_LANES)
                  : L.compression == TC_PACKBITS ? td_phase1<TC_PACKBITS>(g, comp_host + off, len, buf, tab, 0, TD_LANES)
                                                 : td_phase1<TC_LZW>(g, comp_host + off, len, buf, tab, 0, TD_LANES);
        }
        if (got < g.row_bytes * g.data_rows) {
            if (*status_host == 0) *status_host = (unsigned long long)td_status(first_chunk + c, got == -2 ? 2 : got < 0 ? 1 : 3);
            continue;
        }
        for (int lane = 0; lane < TD_LANES; ++lane) td_phase2(L, g, buf, lane);
        for (int lane = 0; lane < TD_LANES; ++lane) td_phase3(L, g, buf, (uint8_t *)out_host, lane);
    }
    return DTB_OK;
}

size_t dtb_tiff_encode_bound(const dtb_tiff_layout *lay) { return te_validate(lay) == DTB_OK ? te_bound(*lay) : 0; }

size_t dtb_tiff_encode_workspace_bytes(const dtb_tiff_layout *lay, int64_t n_chunks)
{
    if (te_validate(lay) != DTB_OK || n_chunks <= 0) return 0;
    const int64_t cap = (int64_t)kNumSMs * TD_CTAS_PER_SM * TD_WARPS;
    const int64_t warps = n_chunks < cap ? n_chunks : cap;
    return (size_t)warps * te_scratch_bytes(*lay) + 256;
}

int dtb_tiff_encode_chunks(const dtb_tiff_layout *lay, const void *raster, int64_t first_chunk, int64_t n_chunks, uint8_t *enc,
                           long long *sizes, void *ws, size_t ws_bytes, void *stream)
{
    const int v = te_validate(lay);
    if (v != DTB_OK) return v;
    if (n_chunks == 0) return DTB_OK;
    if (!raster || !enc || !sizes || !ws) return DTB_ERR_INVALID;
    const int r = te_validate_range(lay, first_chunk, n_chunks);
    if (r != DTB_OK) return r;
    const size_t per = te_scratch_bytes(*lay);
    if (ws_bytes < per + 256) return DTB_ERR_WORKSPACE;
    int64_t warps = (int64_t)((ws_bytes - 256) / per);
    const bool smem = tc_tables_in_smem(n_chunks);
    const int64_t cap = smem ? (int64_t)kNumSMs * TS_WARPS : td_warp_cap();
    if (warps > cap) warps = cap;
    if (warps > n_chunks) warps = n_chunks;
    uint8_t *base = reinterpret_cast<uint8_t *>(((uintptr_t)ws + 255) & ~(uintptr_t)255);
    cudaStream_t st = as_stream(stream);
    if (smem) {
        static bool allowed = false;
        DTB_CUDA(tc_allow_smem(tiff_encode_kernel<TS_WARPS, true>, allowed));
        const unsigned blocks = (unsigned)((warps + TS_WARPS - 1) / TS_WARPS);
        DTB_KERNEL("tiff_encode_kernel<shared>", st,
                   tiff_encode_kernel<TS_WARPS, true><<<blocks, TS_WARPS * TD_LANES, TS_WARPS * TS_TABLE_BYTES, st>>>(
                       *lay, (const uint8_t *)raster, first_chunk, n_chunks, enc, sizes, base, warps));
    } else {
        const unsigned blocks = (unsigned)((warps + TD_WARPS - 1) / TD_WARPS);
        DTB_KERNEL("tiff_encode_kernel", st,
                   tiff_encode_kernel<TD_WARPS, false><<<blocks, TD_WARPS * TD_LANES, 0, st>>>(
                       *lay, (const uint8_t *)raster, first_chunk, n_chunks, enc, sizes, base, warps));
    }
    return DTB_OK;
}

int dtb_tiff_pack_chunks(const uint8_t *enc, size_t bound, const long long *sizes, const long long *offsets, int64_t n_chunks,
                         uint8_t *blob, void *stream)
{
    if (n_chunks == 0) return DTB_OK;
    if (!enc || !sizes || !offsets || !blob || n_chunks < 0 || bound == 0) return DTB_ERR_INVALID;
    const int64_t cap = (int64_t)kNumSMs * 8;
    const unsigned blocks = (unsigned)(n_chunks < cap ? n_chunks : cap);
    cudaStream_t st = as_stream(stream);
    DTB_KERNEL("tiff_pack_kernel", st, tiff_pack_kernel<<<blocks, TP_THREADS, 0, st>>>(enc, bound, sizes, offsets, n_chunks, blob));
    return DTB_OK;
}

int dtb_selftest_tiff_encode_host(const dtb_tiff_layout *lay, const void *raster_host, int64_t first_chunk, int64_t n_chunks,
                                  uint8_t *enc_host, long long *sizes_host)
{
    const int v = te_validate(lay);
    if (v != DTB_OK) return v;
    if (!raster_host || !enc_host || !sizes_host) return DTB_ERR_INVALID;
    const int r = te_validate_range(lay, first_chunk, n_chunks);
    if (r != DTB_OK) return r;
    const dtb_tiff_layout &L = *lay;
    const size_t per = te_scratch_bytes(L), bound = te_bound(L);
    std::vector<uint8_t> scratch(per, 0);
    uint8_t *buf = scratch.data();
    uint64_t *tab = reinterpret_cast<uint64_t *>(buf + (per - sizeof(uint32_t) * kLzwHashSlots));
    for (int64_t c = 0; c < n_chunks; ++c) {
        const ChunkGeom g = td_geom(L, first_chunk + c);
        for (int lane = 0; lane < TD_LANES; ++lane) te_gather(L, g, (const uint8_t *)raster_host, buf, lane);
        for (int lane = 0; lane < TD_LANES; ++lane) te_predict(L, g, buf, lane);
        sizes_host[c] = te_encode(L, g, buf, enc_host + (size_t)c * bound, bound, tab, 0, TD_LANES);
    }
    return DTB_OK;
}

}  // extern "C"
