// synth.cu -- benchmark support: synthetic DEM "dtb-synth-v1" and depression filling.
//
// No reference counterpart: the reference's fixtures were hydrologically conditioned by an
// external GIS (Example/example.py:33-39).  BASELINE.json asks for synthetic conditioned DEMs
// up to 40k x 40k (1.6e9 cells); a host priority-flood over that many cells takes minutes, so
// the benchmark generates and conditions its DEM on the device.  Both kernels are
// bit-identical to their host statements in oracle/dt_condition.cpp (tests compare them).
//
//  * dtb_synth_dem_f32: per-cell counter-based value noise (10 octaves) on a tilted plane
//    with carved channels; every f32 operation is individually rounded (__f*_rn, no FMA) so
//    host and device agree bit for bit.
//  * dtb_fill_depressions_f32: the priority-flood+epsilon result is the unique fixed point of
//        W(c) = max(z(c), min over the 8 neighbours n of succ(W(n)))      (succ = next float up)
//    with W = z on seed cells (raster edge / next to nodata).  Start from an upper bound
//    (column and row scans U(c) = max(z(c), succ(U(prev)))), then relax tiles in shared memory
//    (TILE_ITERS sweeps per pass) until a pass changes nothing.
#include "common.cuh"

namespace dtb {
namespace {

struct SynthParams {
    float amp[10];
    float z0, sr, sc, depth;
    uint32_t seed;
};

__device__ __forceinline__ uint32_t lattice_hash(uint32_t ix, uint32_t iy, uint32_t oct, uint32_t seed)
{
    uint32_t h = seed ^ (ix * 0x9E3779B1u) ^ (iy * 0x85EBCA77u) ^ (oct * 0xC2B2AE3Du);
    h ^= h >> 16; h *= 0x7FEB352Du;
    h ^= h >> 15; h *= 0x846CA68Bu;
    h ^= h >> 16;
    return h;
}
__device__ __forceinline__ float lattice_val(uint32_t ix, uint32_t iy, uint32_t oct, uint32_t seed)
{
    return __fsub_rn(__fmul_rn((float)(lattice_hash(ix, iy, oct, seed) >> 8), 1.0f / 8388608.0f), 1.0f);
}
__device__ __forceinline__ float smooth(float t)
{
    const float t2 = __fmul_rn(t, t);
    const float b = __fsub_rn(3.0f, __fmul_rn(2.0f, t));
    return __fmul_rn(t2, b);
}
__device__ __forceinline__ float vnoise(int64_t r, int64_t c, int L, uint32_t oct, uint32_t seed)
{
    const uint32_t ix = (uint32_t)(c / L), iy = (uint32_t)(r / L);
    const float fx = __fdiv_rn((float)(c % L), (float)L), fy = __fdiv_rn((float)(r % L), (float)L);
    const float sx = smooth(fx), sy = smooth(fy);
    const float v00 = lattice_val(ix, iy, oct, seed), v10 = lattice_val(ix + 1, iy, oct, seed);
    const float v01 = lattice_val(ix, iy + 1, oct, seed), v11 = lattice_val(ix + 1, iy + 1, oct, seed);
    const float d0 = __fsub_rn(v10, v00), d1 = __fsub_rn(v11, v01);
    const float a = __fadd_rn(v00, __fmul_rn(sx, d0));
    const float b = __fadd_rn(v01, __fmul_rn(sx, d1));
    const float d = __fsub_rn(b, a);
    return __fadd_rn(a, __fmul_rn(sy, d));
}

__global__ void __launch_bounds__(256)
synth_kernel(int64_t rows, int64_t cols, int64_t row0, SynthParams p, float *__restrict__ out)
{
    const int64_t n = rows * cols;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
        const int64_t rl = i / cols, c = i - rl * cols, r = row0 + rl;
        float z = __fadd_rn(p.z0, __fmul_rn(p.sr, (float)r));
        z = __fadd_rn(z, __fmul_rn(p.sc, (float)c));
#pragma unroll
        for (int k = 0; k < 10; ++k) z = __fadd_rn(z, __fmul_rn(p.amp[k], vnoise(r, c, 2048 >> k, (uint32_t)k, p.seed)));
        const float n2 = vnoise(r, c, 1024, 31u, p.seed);
        float ridge = __fsub_rn(1.0f, __fmul_rn(8.0f, fabsf(n2)));
        if (ridge < 0.0f) ridge = 0.0f;
        z = __fsub_rn(z, __fmul_rn(p.depth, __fmul_rn(ridge, ridge)));
        out[i] = z;
    }
}

// ---- depression filling ---------------------------------------------------------------
__device__ __forceinline__ float succ(float x)
{
    uint32_t u = __float_as_uint(x);
    if (x > 0.0f) u += 1;
    else if (x < 0.0f) u -= 1;
    else u = 1u;
    return __uint_as_float(u);
}
__device__ __forceinline__ bool is_nd(float z) { return z == ND_F || z != z; }

// fixed[p] = 1 for nodata cells and seeds (raster edge or touching nodata); z copied to zsrc
__global__ void __launch_bounds__(256)
fill_mask_kernel(const float *__restrict__ dem, int64_t rows, int64_t cols, float *__restrict__ zsrc,
                 uint8_t *__restrict__ fixed)
{
    const int64_t n = rows * cols;
    const int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (p >= n) return;
    const int64_t r = p / cols, c = p - r * cols;
    const float z = dem[p];
    zsrc[p] = z;
    bool fx = is_nd(z) || r == 0 || c == 0 || r == rows - 1 || c == cols - 1;
    if (!fx) {
#pragma unroll
        for (int dr = -1; dr <= 1; ++dr)
#pragma unroll
            for (int dc = -1; dc <= 1; ++dc) fx |= is_nd(dem[p + dr * cols + dc]);
    }
    fixed[p] = fx ? 1 : 0;
}

// upper bound, one thread per column walking down the rows: W = max(z, succ(W_above))
__global__ void __launch_bounds__(128)
fill_colscan_kernel(const float *__restrict__ zsrc, const uint8_t *__restrict__ fixed, int64_t rows, int64_t cols,
                    float *__restrict__ w)
{
    const int64_t c = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (c >= cols) return;
    float prev = 0.0f;
    for (int64_t r = 0; r < rows; ++r) {
        const int64_t p = r * cols + c;
        const float z = zsrc[p];
        float v = z;
        if (!fixed[p]) v = fmaxf(z, succ(prev));
        w[p] = v;
        prev = v;
    }
}

// tighten with a west-to-east scan, one thread per row
__global__ void __launch_bounds__(128)
fill_rowscan_kernel(const float *__restrict__ zsrc, const uint8_t *__restrict__ fixed, int64_t rows, int64_t cols,
                    float *__restrict__ w)
{
    const int64_t r = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (r >= rows) return;
    float prev = 0.0f;
    for (int64_t c = 0; c < cols; ++c) {
        const int64_t p = r * cols + c;
        float v = w[p];
        if (!fixed[p]) {
            v = fminf(v, fmaxf(zsrc[p], succ(prev)));
            w[p] = v;
        }
        prev = v;
    }
}

constexpr int FT = 32;          // tile edge
constexpr int TILE_ITERS = 24;  // in-tile sweeps per pass

// One pass over one tile.  BAND: w points at row 0 of a band whose halo rows -1 / rows (the neighbours' current
// seam rows) are read where the band has a neighbour -- as constants, never stored -- and *seam is set when a cell
// of the band's first or last row is lowered.  The single-raster instantiation is the original kernel body.
template <bool BAND>
__device__ __forceinline__ void fill_relax_tile(const float *__restrict__ zsrc, const uint8_t *__restrict__ fixed, int64_t rows,
                                                int64_t cols, float *w, int tiles_x, unsigned *__restrict__ changed,
                                                int64_t row_lo, int64_t row_hi, unsigned *__restrict__ seam)
{
    __shared__ float sw[FT + 2][FT + 3];
    const int ty = blockIdx.x / tiles_x, tx = blockIdx.x - ty * tiles_x;
    const int64_t r0 = (int64_t)ty * FT, c0 = (int64_t)tx * FT;
    const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;  // 32 x 8 threads, 4 rows each
    for (int idx = threadIdx.x; idx < (FT + 2) * (FT + 2); idx += 256) {
        const int j = idx / (FT + 2), k = idx - j * (FT + 2);
        const int64_t r = r0 - 1 + j, c = c0 - 1 + k;
        float v = __int_as_float(0x7f800000);  // +inf outside: never the minimum
        bool rin;
        if constexpr (BAND) rin = r >= row_lo && r < row_hi;
        else rin = r >= 0 && r < rows;
        if (rin && c >= 0 && c < cols) v = __ldcg(&w[r * cols + c]);
        sw[j][k] = v;
    }
    float z[4];
    bool fx[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t r = r0 + ly + 8 * i, c = c0 + lx;
        const bool in = r < rows && c < cols;
        fx[i] = !in || fixed[r * cols + c];
        z[i] = in ? zsrc[r * cols + c] : 0.0f;
    }
    __syncthreads();
    bool any = false, edge = false;
    for (int it = 0; it < TILE_ITERS; ++it) {
        bool ch = false;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (fx[i]) continue;
            const int j = ly + 8 * i + 1, k = lx + 1;
            float m = fminf(fminf(sw[j - 1][k - 1], sw[j - 1][k]), fminf(sw[j - 1][k + 1], sw[j][k - 1]));
            m = fminf(m, fminf(fminf(sw[j][k + 1], sw[j + 1][k - 1]), fminf(sw[j + 1][k], sw[j + 1][k + 1])));
            const float v = fmaxf(z[i], succ(m));
            if (v < sw[j][k]) {
                sw[j][k] = v;
                ch = true;
                if constexpr (BAND) {
                    const int64_t r = r0 + ly + 8 * i;
                    edge |= r == 0 || r == rows - 1;
                }
            }
        }
        any |= ch;
        if (!__syncthreads_or(ch)) break;
    }
    if (any) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (!fx[i]) __stcg(&w[(r0 + ly + 8 * i) * cols + c0 + lx], sw[ly + 8 * i + 1][lx + 1]);
    }
    if (__syncthreads_or(any) && threadIdx.x == 0) atomicAdd(changed, 1u);
    if constexpr (BAND) {
        if (__syncthreads_or(edge) && threadIdx.x == 0) atomicOr(seam, 1u);
    }
}

__global__ void __launch_bounds__(256)
fill_relax_kernel(const float *__restrict__ zsrc, const uint8_t *__restrict__ fixed, int64_t rows, int64_t cols,
                  float *w, int tiles_x, unsigned *__restrict__ changed)
{
    fill_relax_tile<false>(zsrc, fixed, rows, cols, w, tiles_x, changed, 0, 0, nullptr);
}

// ---- depression filling over row bands ----------------------------------------------------------
// A band's buffer is (rows + 2) x cols: rows 0 and rows + 1 are halo rows (the neighbours' rows next to the seams),
// the kernels get w = row 1.  Block-Jacobi over bands: every band relaxes to its own fixed point with the halo rows
// held constant; the driver exchanges the seam rows and repeats until no seam row changes (descriptools_b200/bands.py).

// as fill_mask_kernel, but the top / bottom row is a seed only where the band has no neighbour; elsewhere the halo
// row decides whether a cell touches nodata across the seam
__global__ void __launch_bounds__(256)
fill_band_mask_kernel(const float *__restrict__ w, int64_t rows, int64_t cols, int has_above, int has_below,
                      float *__restrict__ zsrc, uint8_t *__restrict__ fixed)
{
    const int64_t n = rows * cols;
    const int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (p >= n) return;
    const int64_t r = p / cols, c = p - r * cols;
    const float z = w[p];
    zsrc[p] = z;
    bool fx = is_nd(z) || c == 0 || c == cols - 1 || (r == 0 && !has_above) || (r == rows - 1 && !has_below);
    if (!fx) {  // rows -1 and `rows` are read only where the band has that neighbour
#pragma unroll
        for (int dr = -1; dr <= 1; ++dr)
#pragma unroll
            for (int dc = -1; dc <= 1; ++dc) fx |= is_nd(w[p + dr * cols + dc]);
    }
    fixed[p] = fx ? 1 : 0;
}

// a band below another one has no column of seeds above it: its non-seed cells start at +inf, and the row scan (every
// row starts at the seed in column 0) brings them down to an upper bound
__global__ void __launch_bounds__(256)
fill_band_inf_kernel(const uint8_t *__restrict__ fixed, int64_t n, float *__restrict__ w)
{
    const int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (p < n && !fixed[p]) w[p] = __int_as_float(0x7f800000);
}

__global__ void __launch_bounds__(256)
fill_relax_band_kernel(const float *__restrict__ zsrc, const uint8_t *__restrict__ fixed, int64_t rows, int64_t cols,
                       float *w, int tiles_x, unsigned *__restrict__ changed, int64_t row_lo, int64_t row_hi,
                       unsigned *__restrict__ seam)
{
    fill_relax_tile<true>(zsrc, fixed, rows, cols, w, tiles_x, changed, row_lo, row_hi, seam);
}

}  // namespace
}  // namespace dtb

using namespace dtb;

extern "C" int dtb_synth_dem_f32(int64_t rows, int64_t cols, int64_t row0, uint32_t seed, const float *amp10_host, float z0,
                                 float sr, float sc, float depth, float *out, void *stream)
{
    if (!out || !amp10_host || rows <= 0 || cols <= 0) return DTB_ERR_INVALID;
    SynthParams p;
    for (int k = 0; k < 10; ++k) p.amp[k] = amp10_host[k];
    p.z0 = z0; p.sr = sr; p.sc = sc; p.depth = depth; p.seed = seed;
    synth_kernel<<<kNumSMs * 8, 256, 0, as_stream(stream)>>>(rows, cols, row0, p, out);
    DTB_LAUNCH_CHECK("synth_kernel");
    return DTB_OK;
}

extern "C" size_t dtb_fill_workspace_bytes(int64_t rows, int64_t cols)
{
    if (rows <= 0 || cols <= 0) return 0;
    const size_t n = (size_t)rows * (size_t)cols;
    return n * 4 + ((n + 255) / 256) * 256 + 256;
}

extern "C" int dtb_fill_depressions_f32(float *dem, int64_t rows, int64_t cols, void *ws, size_t ws_bytes,
                                        int *iterations_host, void *stream)
{
    if (!dem || !ws || rows <= 0 || cols <= 0) return DTB_ERR_INVALID;
    if (ws_bytes < dtb_fill_workspace_bytes(rows, cols)) return DTB_ERR_WORKSPACE;
    cudaStream_t st = as_stream(stream);
    const int64_t n = rows * cols;
    unsigned *changed = reinterpret_cast<unsigned *>(ws);
    float *zsrc = reinterpret_cast<float *>((char *)ws + 256);
    uint8_t *fixed = reinterpret_cast<uint8_t *>((char *)ws + 256 + (size_t)n * 4);
    const unsigned blocks = (unsigned)((n + 255) / 256);
    fill_mask_kernel<<<blocks, 256, 0, st>>>(dem, rows, cols, zsrc, fixed);
    DTB_LAUNCH_CHECK("fill_mask_kernel");
    fill_colscan_kernel<<<(unsigned)((cols + 127) / 128), 128, 0, st>>>(zsrc, fixed, rows, cols, dem);
    DTB_LAUNCH_CHECK("fill_colscan_kernel");
    fill_rowscan_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, st>>>(zsrc, fixed, rows, cols, dem);
    DTB_LAUNCH_CHECK("fill_rowscan_kernel");
    const int tiles_x = (int)((cols + FT - 1) / FT);
    const int64_t ntiles = (int64_t)tiles_x * ((rows + FT - 1) / FT);
    if (ntiles > 0x7fffffff) return DTB_ERR_UNSUPPORTED;
    int passes = 0;
    const int kMaxPasses = 200000;
    for (;;) {
        DTB_CUDA(cudaMemsetAsync(changed, 0, 4, st));
        const int burst = passes < 64 ? 4 : 16;  // check the flag every `burst` passes
        for (int b = 0; b < burst; ++b) {
            fill_relax_kernel<<<(unsigned)ntiles, 256, 0, st>>>(zsrc, fixed, rows, cols, dem, tiles_x, changed);
            DTB_LAUNCH_CHECK("fill_relax_kernel");
        }
        passes += burst;
        unsigned h = 0;
        DTB_CUDA(cudaMemcpyAsync(&h, changed, 4, cudaMemcpyDeviceToHost, st));
        DTB_CUDA(cudaStreamSynchronize(st));
        if (h == 0) break;
        if (passes > kMaxPasses) return DTB_ERR_UNSUPPORTED;
    }
    if (iterations_host) *iterations_host = passes;
    return DTB_OK;
}

// workspace layout as dtb_fill_workspace_bytes: flags (changed at byte 0, seam at byte 4), zsrc, fixed
extern "C" size_t dtb_fill_band_workspace_bytes(int64_t rows, int64_t cols) { return dtb_fill_workspace_bytes(rows, cols); }

extern "C" int dtb_fill_band_f32(float *dem_halo, int64_t rows, int64_t cols, int has_above, int has_below, int mode, void *ws,
                                 size_t ws_bytes, int *passes_host, int *seam_changed_host, void *stream)
{
    if (!dem_halo || !ws || rows <= 0 || cols <= 0) return DTB_ERR_INVALID;
    if ((has_above != 0 && has_above != 1) || (has_below != 0 && has_below != 1)) return DTB_ERR_INVALID;
    if (mode != DTB_FILL_INIT && mode != DTB_FILL_SOLVE) return DTB_ERR_INVALID;
    if (ws_bytes < dtb_fill_band_workspace_bytes(rows, cols)) return DTB_ERR_WORKSPACE;
    const int tiles_x = (int)((cols + FT - 1) / FT);
    const int64_t ntiles = (int64_t)tiles_x * ((rows + FT - 1) / FT);
    if (ntiles > 0x7fffffff) return DTB_ERR_UNSUPPORTED;
    cudaStream_t st = as_stream(stream);
    const int64_t n = rows * cols;
    unsigned *flags = reinterpret_cast<unsigned *>(ws);  // [0] a tile changed, [1] a seam row changed
    float *zsrc = reinterpret_cast<float *>((char *)ws + 256);
    uint8_t *fixed = reinterpret_cast<uint8_t *>((char *)ws + 256 + (size_t)n * 4);
    float *w = dem_halo + cols;
    int passes = 0;
    unsigned seam = 0;
    if (mode == DTB_FILL_INIT) {
        const unsigned blocks = (unsigned)((n + 255) / 256);
        fill_band_mask_kernel<<<blocks, 256, 0, st>>>(w, rows, cols, has_above, has_below, zsrc, fixed);
        DTB_LAUNCH_CHECK("fill_band_mask_kernel");
        if (!has_above) {  // the band holds the raster's top row: the column scan starts at its seeds
            fill_colscan_kernel<<<(unsigned)((cols + 127) / 128), 128, 0, st>>>(zsrc, fixed, rows, cols, w);
            DTB_LAUNCH_CHECK("fill_colscan_kernel");
        } else {
            fill_band_inf_kernel<<<blocks, 256, 0, st>>>(fixed, n, w);
            DTB_LAUNCH_CHECK("fill_band_inf_kernel");
        }
        fill_rowscan_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, st>>>(zsrc, fixed, rows, cols, w);
        DTB_LAUNCH_CHECK("fill_rowscan_kernel");
        DTB_CUDA(cudaStreamSynchronize(st));
    } else {
        const int64_t row_lo = has_above ? -1 : 0, row_hi = has_below ? rows + 1 : rows;
        DTB_CUDA(cudaMemsetAsync(flags, 0, 8, st));
        const int kMaxPasses = 200000;
        for (;;) {
            DTB_CUDA(cudaMemsetAsync(flags, 0, 4, st));
            const int burst = passes < 64 ? 4 : 16;  // check the flag every `burst` passes
            for (int b = 0; b < burst; ++b) {
                fill_relax_band_kernel<<<(unsigned)ntiles, 256, 0, st>>>(zsrc, fixed, rows, cols, w, tiles_x, flags, row_lo, row_hi,
                                                                         flags + 1);
                DTB_LAUNCH_CHECK("fill_relax_band_kernel");
            }
            passes += burst;
            unsigned h[2] = {0, 0};
            DTB_CUDA(cudaMemcpyAsync(h, flags, 8, cudaMemcpyDeviceToHost, st));
            DTB_CUDA(cudaStreamSynchronize(st));
            seam = h[1];
            if (h[0] == 0) break;
            if (passes > kMaxPasses) return DTB_ERR_UNSUPPORTED;
        }
    }
    if (passes_host) *passes_host = passes;
    if (seam_changed_host) *seam_changed_host = seam ? 1 : 0;
    return DTB_OK;
}
