// flats.cu -- flat resolution: D8 codes for the cells a fill without epsilon left exactly flat, the DEM untouched.
//
// Semantics (the host statement the tests compare against is tests/flats_ref.cpp; SURVEY App. A2 for codes and scan
// order).  A flat cell is a valid cell (z > -100, not NaN) whose D8 code is 0.  With the stencil's codes for this DEM it
// has no strictly lower and no undefined neighbour, so 8-adjacent flat cells have equal z and none lies on the raster's
// edge; any other D8 raster is taken as well (off-raster neighbours are skipped, as in the reference).  A flat F is an
// 8-connected component of flat cells; an outlet of a cell of F is a valid neighbour with a code at that cell's
// elevation; a high edge is a cell of F with a strictly higher neighbour.  towards(p) = steps through F to the nearest outlet (1 next to one), away(p) = steps through F to the
// nearest high edge (0 on one), A(F) = max away over F (0 without a high edge).  Each cell of a flat with an outlet
// points at the neighbour of least mask = 2 towards + (A(F) - away) (the second term 0 without a high edge; -1 for an
// outlet), the first in scan order on ties (Garbrecht & Martz 1997, Barnes, Lehman & Mulla 2014: towards the outlets
// and away from the higher ground).  That neighbour's mask is strictly below the cell's own, so every path ends at an
// outlet.  Flats without an outlet keep code 0 and are counted as unresolved.
//
// Device plan (int32 labels and distances, so rows * cols < 2^31):
//   1. count the flat cells (reads the codes; z only where the code is 0) -- nothing else runs when there are none;
//   2. per 32 x 32 tile, seed the three fields (label = own linear index, towards = 1 next to an outlet, away = 0 on a
//      high edge, everything else INF; -1 off the flats) and list the tiles that hold a flat cell;
//   3. relax each field to its fixed point v(p) = min(v(p), min over flat neighbours of v(q) + INC) -- INC 0 gives the
//      least linear index of the flat, INC 1 the breadth-first distance -- with one shared-memory tile kernel in the
//      style of the depression fill (csrc/synth.cu): listed tiles only, passes until one changes nothing;
//   4. A(F) by atomicMax into a label-indexed array;
//   5. write the codes of flat cells only.
#include <climits>

#include "common.cuh"

namespace dtb {
namespace {

constexpr int FT = 32;             // tile edge
constexpr int FLAT_ITERS = 64;     // in-tile sweeps per pass
constexpr int32_t OFF = -1;        // not a flat cell: as unsigned, above every value of a flat cell
constexpr int32_t INF = INT_MAX;   // not reached (yet)
constexpr int kMaxPasses = 200000; // per field, as the depression fill

struct FlatHeader {
    unsigned changed;
    unsigned tiles;                // tiles holding a flat cell
    unsigned long long flat_cells;
    unsigned long long unresolved;
};

__device__ __constant__ int kDR[8] = {-1, -1, -1, 0, 0, 1, 1, 1};
__device__ __constant__ int kDC[8] = {-1, 0, 1, -1, 1, -1, 0, 1};
__device__ __constant__ uint8_t kCode[8] = {32, 64, 128, 16, 1, 8, 4, 2};

template <typename T> __device__ __forceinline__ bool valid(T z) { return z > (T)-100; }  // false for NaN

__device__ __forceinline__ void add_u64(unsigned long long *dst, unsigned long long v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(dst, v);
}

// 1. flat cells: code 0 and a valid elevation.  Sixteen codes per load when the codes are 16-byte aligned.
template <typename T>
__global__ void __launch_bounds__(256)
flats_count_kernel(const T *__restrict__ dem, const uint8_t *__restrict__ d8, int64_t n, FlatHeader *hdr)
{
    const int64_t stride = (int64_t)gridDim.x * 256, t = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int64_t nv = ((uintptr_t)d8 & 15) == 0 ? n / 16 : 0;
    unsigned long long cnt = 0;
    for (int64_t v = t; v < nv; v += stride) {
        const uint4 w = __ldg(reinterpret_cast<const uint4 *>(d8) + v);
        const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (!((ws[k] - 0x01010101u) & ~ws[k] & 0x80808080u)) continue;  // no zero byte
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int64_t p = v * 16 + 4 * k + b;
                cnt += ((ws[k] >> (8 * b)) & 0xFFu) == 0 && valid(dem[p]);
            }
        }
    }
    for (int64_t p = nv * 16 + t; p < n; p += stride) cnt += d8[p] == 0 && valid(dem[p]);
    add_u64(&hdr->flat_cells, cnt);
}

// 2. seed the fields of one tile; list it when it holds a flat cell
template <typename T>
__global__ void __launch_bounds__(256)
flats_init_kernel(const T *__restrict__ dem, const uint8_t *__restrict__ d8, int64_t rows, int64_t cols, int tiles_x,
                  int32_t *__restrict__ lab, int32_t *__restrict__ tow, int32_t *__restrict__ away, int32_t *__restrict__ amax,
                  int *__restrict__ tile_list, FlatHeader *hdr)
{
    const int ty = blockIdx.x / tiles_x, tx = blockIdx.x - ty * tiles_x;
    const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;  // 32 x 8 threads, 4 rows each
    bool any = false;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t r = (int64_t)ty * FT + ly + 8 * i, c = (int64_t)tx * FT + lx;
        if (r >= rows || c >= cols) continue;
        const int64_t p = r * cols + c;
        const T z = dem[p];
        int32_t l = OFF, t = OFF, a = OFF;
        if (d8[p] == 0 && valid(z)) {
            bool outlet = false, high = false;
            for (int k = 0; k < 8; ++k) {
                const int64_t rr = r + kDR[k], cc = c + kDC[k];
                if (rr < 0 || rr >= rows || cc < 0 || cc >= cols) continue;  // d8 need not be the stencil's: edge cells may be flat
                const int64_t q = rr * cols + cc;
                const T zq = dem[q];
                high |= zq > z;
                outlet |= zq == z && d8[q] != 0;  // zq == z: valid
            }
            l = (int32_t)p;
            t = outlet ? 1 : INF;
            a = high ? 0 : INF;
            amax[p] = 0;
            any = true;
        }
        lab[p] = l;
        tow[p] = t;
        away[p] = a;
    }
    if (__syncthreads_or(any) && threadIdx.x == 0) tile_list[atomicAdd(&hdr->tiles, 1u)] = blockIdx.x;
}

// 3. one pass over one listed tile: v(p) = min(v(p), min over flat neighbours of v(q) + INC).  As unsigned, OFF (-1) is
// above every value of a flat cell, so the minimum over all eight neighbours is the minimum over the flat ones.
template <int INC>
__global__ void __launch_bounds__(256)
flats_relax_kernel(int32_t *v, int64_t rows, int64_t cols, int tiles_x, const int *__restrict__ tile_list, unsigned *__restrict__ changed)
{
    __shared__ uint32_t sv[FT + 2][FT + 2];
    const int tile = tile_list[blockIdx.x];
    const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
    const int64_t r0 = (int64_t)ty * FT, c0 = (int64_t)tx * FT;
    const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;
    for (int idx = threadIdx.x; idx < (FT + 2) * (FT + 2); idx += 256) {
        const int j = idx / (FT + 2), k = idx - j * (FT + 2);
        const int64_t r = r0 - 1 + j, c = c0 - 1 + k;
        uint32_t x = (uint32_t)OFF;
        if (r >= 0 && r < rows && c >= 0 && c < cols) x = (uint32_t)__ldcg(&v[r * cols + c]);
        sv[j][k] = x;
    }
    __syncthreads();
    bool mine[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) mine[i] = sv[ly + 8 * i + 1][lx + 1] != (uint32_t)OFF;
    bool any = false;
    for (int it = 0; it < FLAT_ITERS; ++it) {
        bool ch = false;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (!mine[i]) continue;
            const int j = ly + 8 * i + 1, k = lx + 1;
            uint32_t m = min(min(sv[j - 1][k - 1], sv[j - 1][k]), min(sv[j - 1][k + 1], sv[j][k - 1]));
            m = min(m, min(min(sv[j][k + 1], sv[j + 1][k - 1]), min(sv[j + 1][k], sv[j + 1][k + 1])));
            if (m < (uint32_t)INF && m + INC < sv[j][k]) {
                sv[j][k] = m + INC;
                ch = true;
            }
        }
        any |= ch;
        if (!__syncthreads_or(ch)) break;
    }
    if (any) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (mine[i]) __stcg(&v[(r0 + ly + 8 * i) * cols + c0 + lx], (int32_t)sv[ly + 8 * i + 1][lx + 1]);
    }
    if (__syncthreads_or(any) && threadIdx.x == 0) atomicAdd(changed, 1u);
}

// 4. A(F) = max away over F, into amax[label]; a warp whose cells share one label reduces first
__global__ void __launch_bounds__(256)
flats_amax_kernel(const int32_t *__restrict__ lab, const int32_t *__restrict__ away, int64_t rows, int64_t cols, int tiles_x,
                  const int *__restrict__ tile_list, int32_t *amax)
{
    const int tile = tile_list[blockIdx.x];
    const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
    const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t r = (int64_t)ty * FT + ly + 8 * i, c = (int64_t)tx * FT + lx;
        int32_t l = OFF, a = INF;
        if (r < rows && c < cols) {
            l = lab[r * cols + c];
            if (l != OFF) a = away[r * cols + c];
        }
        const bool on = l != OFF && a != INF;
        const unsigned act = __ballot_sync(0xffffffffu, on);
        if (!on) continue;
        if (__match_any_sync(act, l) == act) {
            const unsigned m = __reduce_max_sync(act, (unsigned)a);
            if (lx == __ffs(act) - 1) atomicMax(&amax[l], (int32_t)m);
        } else {
            atomicMax(&amax[l], a);
        }
    }
}

// 5. the codes of flat cells; the neighbours' classes come from the fields, not from d8, which this pass rewrites
template <typename T>
__global__ void __launch_bounds__(256)
flats_code_kernel(const T *__restrict__ dem, uint8_t *d8, int64_t rows, int64_t cols, int tiles_x, const int *__restrict__ tile_list,
                  const int32_t *__restrict__ lab, const int32_t *__restrict__ tow, const int32_t *__restrict__ away,
                  const int32_t *__restrict__ amax, FlatHeader *hdr)
{
    const int tile = tile_list[blockIdx.x];
    const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
    const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;
    unsigned long long left = 0;
#pragma unroll 1
    for (int i = 0; i < 4; ++i) {
        const int64_t r = (int64_t)ty * FT + ly + 8 * i, c = (int64_t)tx * FT + lx;
        if (r >= rows || c >= cols) continue;
        const int64_t p = r * cols + c;
        const int32_t l = lab[p];
        if (l == OFF) continue;
        if (tow[p] == INF) {
            ++left;
            continue;
        }
        const int64_t A = amax[l];
        const T z = dem[p];
        int64_t best = LLONG_MAX;
        uint8_t code = 0;
#pragma unroll 1
        for (int k = 0; k < 8; ++k) {
            const int64_t rr = r + kDR[k], cc = c + kDC[k];
            if (rr < 0 || rr >= rows || cc < 0 || cc >= cols) continue;
            const int64_t q = rr * cols + cc;
            int64_t m;
            if (lab[q] != OFF) {
                const int32_t aq = away[q];
                m = 2 * (int64_t)tow[q] + (aq == INF ? 0 : A - aq);
            } else {
                m = dem[q] == z && d8[q] != 0 ? -1 : LLONG_MAX;  // an outlet (d8 of a cell off the flats is not rewritten)
            }
            if (m < best) {
                best = m;
                code = kCode[k];
            }
        }
        d8[p] = code;
    }
    add_u64(&hdr->unresolved, left);
}

template <typename T>
int resolve_flats(const T *dem, uint8_t *d8, int64_t rows, int64_t cols, void *ws, size_t ws_bytes, int64_t *unresolved_host,
                  cudaStream_t st)
{
    const int64_t n = rows * cols;
    const int tiles_x = (int)((cols + FT - 1) / FT);
    const int64_t ntiles = (int64_t)tiles_x * ((rows + FT - 1) / FT);
    FlatHeader *hdr = reinterpret_cast<FlatHeader *>(ws);
    int32_t *lab = reinterpret_cast<int32_t *>((char *)ws + 256);
    int32_t *tow = lab + n, *away = tow + n, *amax = away + n;
    int *tile_list = reinterpret_cast<int *>(amax + n);
    DTB_CUDA(cudaMemsetAsync(hdr, 0, sizeof(FlatHeader), st));
    const int64_t want = (n + 16 * 256 - 1) / (16 * 256);
    DTB_KERNEL("flats_count_kernel", st,
               flats_count_kernel<T><<<(unsigned)(want < kNumSMs * 16 ? want : kNumSMs * 16), 256, 0, st>>>(dem, d8, n, hdr));
    FlatHeader h;
    DTB_CUDA(cudaMemcpyAsync(&h, hdr, sizeof(h), cudaMemcpyDeviceToHost, st));
    DTB_CUDA(cudaStreamSynchronize(st));
    if (h.flat_cells != 0) {
        DTB_KERNEL("flats_init_kernel", st,
                   flats_init_kernel<T><<<(unsigned)ntiles, 256, 0, st>>>(dem, d8, rows, cols, tiles_x, lab, tow, away, amax, tile_list, hdr));
        DTB_CUDA(cudaMemcpyAsync(&h, hdr, sizeof(h), cudaMemcpyDeviceToHost, st));
        DTB_CUDA(cudaStreamSynchronize(st));
        const unsigned active = h.tiles;
        int32_t *fields[3] = {lab, tow, away};
        for (int f = 0; f < 3; ++f) {
            int passes = 0;
            for (;;) {
                DTB_CUDA(cudaMemsetAsync(&hdr->changed, 0, 4, st));
                const int burst = passes < 64 ? 4 : 16;  // check the flag every `burst` passes
                for (int b = 0; b < burst; ++b) {
                    if (f == 0)
                        DTB_KERNEL("flats_relax_kernel<0>", st,
                                   flats_relax_kernel<0><<<active, 256, 0, st>>>(fields[f], rows, cols, tiles_x, tile_list, &hdr->changed));
                    else
                        DTB_KERNEL("flats_relax_kernel<1>", st,
                                   flats_relax_kernel<1><<<active, 256, 0, st>>>(fields[f], rows, cols, tiles_x, tile_list, &hdr->changed));
                }
                passes += burst;
                unsigned ch = 0;
                DTB_CUDA(cudaMemcpyAsync(&ch, &hdr->changed, 4, cudaMemcpyDeviceToHost, st));
                DTB_CUDA(cudaStreamSynchronize(st));
                if (ch == 0) break;
                if (passes > kMaxPasses) return DTB_ERR_UNSUPPORTED;
            }
        }
        DTB_KERNEL("flats_amax_kernel", st,
                   flats_amax_kernel<<<active, 256, 0, st>>>(lab, away, rows, cols, tiles_x, tile_list, amax));
        DTB_KERNEL("flats_code_kernel", st,
                   flats_code_kernel<T><<<active, 256, 0, st>>>(dem, d8, rows, cols, tiles_x, tile_list, lab, tow, away, amax, hdr));
        DTB_CUDA(cudaMemcpyAsync(&h, hdr, sizeof(h), cudaMemcpyDeviceToHost, st));
        DTB_CUDA(cudaStreamSynchronize(st));
    }
    if (unresolved_host) *unresolved_host = (int64_t)h.unresolved;
    return DTB_OK;
}

}  // namespace
}  // namespace dtb

using namespace dtb;

extern "C" size_t dtb_resolve_flats_workspace_bytes(int64_t rows, int64_t cols)
{
    if (rows <= 0 || cols <= 0) return 0;
    const size_t n = (size_t)rows * (size_t)cols;
    const size_t ntiles = (size_t)((rows + FT - 1) / FT) * (size_t)((cols + FT - 1) / FT);
    return 256 + n * 16 + ntiles * 4;
}

extern "C" int dtb_resolve_flats(const void *dem, int dem_dtype, uint8_t *d8, int64_t rows, int64_t cols, void *ws, size_t ws_bytes,
                                 int64_t *unresolved_host, void *stream)
{
    if (!dem || !d8 || !ws || rows <= 0 || cols <= 0) return DTB_ERR_INVALID;
    if (dem_dtype != DTB_F32 && dem_dtype != DTB_I16) return DTB_ERR_INVALID;
    if (rows > INT_MAX || cols > INT_MAX || rows * cols >= ((int64_t)1 << 31)) return DTB_ERR_UNSUPPORTED;
    if (ws_bytes < dtb_resolve_flats_workspace_bytes(rows, cols)) return DTB_ERR_WORKSPACE;
    cudaStream_t st = as_stream(stream);
    if (dem_dtype == DTB_F32)
        return resolve_flats(static_cast<const float *>(dem), d8, rows, cols, ws, ws_bytes, unresolved_host, st);
    return resolve_flats(static_cast<const int16_t *>(dem), d8, rows, cols, ws, ws_bytes, unresolved_host, st);
}
