// evaluation.cu -- threshold calibration of a descriptor against a benchmark flood map
// (SURVEY.md 8 f1: evaluation.py:5-9 minMaxScale, :12-87 calibration, :90-123 binary_map, :126-171 avaliacao).
//
// The reference evaluates one threshold per full-raster NumPy pass (np.where + np.unique, 61 passes per
// calibration).  Here one pass serves a whole stage of the search: every cell finds the first threshold of the
// ascending stage list that classifies it as flooded, a per-benchmark-class histogram over that position is
// accumulated in shared memory, and prefix sums on the host give the confusion counts of every threshold.
//
// The device / row-band calibration (dtb_eval_extrema, dtb_eval_hist, dtb_eval_class_scaled) never materialises the
// float64 raster of minMaxScale: the two ends of np.unique come from one reduction pass, and the histogram and class-map
// kernels read the raw descriptor and scale every cell on load with the very expression minmax_scale_kernel uses.
#include "common.cuh"

namespace dtb {
namespace {

constexpr int EV_MAXK = 32;
constexpr int EV_THREADS = 256;
constexpr int EV_BLOCKS = kNumSMs * 8;

struct Thresholds {
    double th[EV_MAXK];
    int k;
};

// minMaxScale of one cell (evaluation.py:6-7): nodata -> NaN; NaN stays NaN; everything else (v - mn) / (mx - mn) in f64.
// The one definition the materialising kernel and the fused loads share: a true division, as NumPy does it.
struct EvScale {
    double mn, mx, nodata;
};
__device__ __forceinline__ double minmax_scaled(double v, const EvScale &s)
{
    return (v == s.nodata || v != v) ? __longlong_as_double(0x7ff8000000000000LL) : (v - s.mn) / (s.mx - s.mn);
}

// Source type of the fused kernels: a raw descriptor cell (float or int16) that is min-max scaled when it is loaded.
template <typename S> struct MinMaxScaled {
    S raw;
};
template <typename T> struct EvIsScaled { static constexpr bool value = false; };
template <typename S> struct EvIsScaled<MinMaxScaled<S>> { static constexpr bool value = true; };

// the compared value of a loaded cell
template <typename CT, typename T> __device__ __forceinline__ CT ev_load(T d, const EvScale &) { return (CT)d; }
template <typename CT, typename S> __device__ __forceinline__ CT ev_load(MinMaxScaled<S> d, const EvScale &s)
{
    return minmax_scaled((double)d.raw, s);
}
// binary_map's nodata value (descriptor_matrix[0,0]): a scaled source receives the RAW corner cell and scales it here,
// with the same function as every other cell, so the comparison matches the materialised raster's bit for bit
template <typename T> __device__ __forceinline__ double ev_nodata(double nodata, const EvScale &s)
{
    if constexpr (EvIsScaled<T>::value) return minmax_scaled(nodata, s);
    else return nodata;
}

// binary_map (evaluation.py:90-123): cells equal to `nodata` (= descriptor_matrix[0,0]) and NaNs are never flooded
template <typename T>
__device__ __forceinline__ bool usable(T d, double nodata) { return !((double)d != (double)d) && !((double)d == nodata); }

// avaliacao's remapping of the benchmark (evaluation.py:149-150): 1 -> 2, -100 -> 0
__device__ __forceinline__ int remap(int f) { return f == 1 ? 2 : (f == ND_I ? 0 : f); }

// hist[c][j], c = remapped benchmark value 0..3, j = 0..k: number of thresholds of the list that do NOT flag the cell
// before the first one that does (under: first i with d <= th[i], i.e. j = #{th < d}; over: thresholds th[0..j-1] satisfy
// d >= th, i.e. j = #{th <= d}).
// Four cells per thread and pass (one 16 / 32-byte load of the descriptor, one 4-byte load of the benchmark); j by a
// branch-free binary search over the threshold list in shared memory (padded to 32 entries with +inf); the lanes of a warp
// that hit the same bin as the first of them are summed and added by it (eval_count).  CT = float when the descriptor is f32 and every threshold (and the nodata value)
// is a float exactly: the comparison is the same, without a conversion to f64 per cell.
template <typename T> struct alignas(sizeof(T) * 4) EvPack4 { T v[4]; };

// bin of one cell, or -1 for a benchmark value outside {0, 1, 2, 3, -100}.  Branch-free: the class slot is the low three
// bits of the benchmark byte (-100 = 0x9c -> 4; slots become avaliacao's classes when the block adds its counts to the global histogram);
// a search step is one shared load at [offset + constant], one compare and one predicated add of the byte offset.
// `nodata` arrives as NaN when it cannot equal a CT descriptor.
template <typename CT, bool UNDER>
__device__ __forceinline__ int eval_bin(CT d, int f, CT nodata, const CT *__restrict__ th, int k)
{
    unsigned off = 0;
    const char *base = reinterpret_cast<const char *>(th);
#pragma unroll
    for (int step = EV_MAXK / 2; step >= 1; step >>= 1) {
        const CT t = *reinterpret_cast<const CT *>(base + off + (step - 1) * sizeof(CT));
        if (UNDER ? t < d : t <= d) off += step * (unsigned)sizeof(CT);
    }
    const CT t = *reinterpret_cast<const CT *>(base + off);
    if (UNDER ? t < d : t <= d) off += (unsigned)sizeof(CT);
    int j = min((int)(off / sizeof(CT)), k);  // (d = +inf counts the +inf padding as well)
    if (d != d || d == nodata) j = UNDER ? k : 0;  // never flagged
    const bool valid = (unsigned)f <= 3u || f == ND_I;
    return valid ? (f & 7) * (EV_MAXK + 1) + j : -1;
}

// One histogram update for the four cells of every lane: the cells that fall into the bin of the first lane's first valid
// cell -- in a raster nearly all of them -- are counted with one redux and added by one lane; the others add on their own
// (same-address shared atomics serialise, so per-cell atomics cost 32 passes per warp and cell).
__device__ __forceinline__ void eval_count4(unsigned *sh, const int (&key)[4])
{
    const unsigned act = __activemask();
    int first = key[0];
#pragma unroll
    for (int i = 1; i < 4; ++i) first = first >= 0 ? first : key[i];
    const unsigned want = __ballot_sync(act, first >= 0);
    if (!want) return;
    const int lead = __ffs((int)want) - 1;
    const int cand = __shfl_sync(act, first, lead);
    unsigned hits = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) hits += key[i] == cand ? 1u : 0u;
    const unsigned sum = __reduce_add_sync(act, hits);
    if ((int)(threadIdx.x & 31) == lead) atomicAdd(&sh[cand], sum);
    if (hits != 4u) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (key[i] >= 0 && key[i] != cand) atomicAdd(&sh[key[i]], 1u);
    }
}

constexpr int EV_SLOTS = 5;  // benchmark bytes 0, 1, 2, 3 and -100 (& 7 = 4)

template <typename T, typename CT, bool VEC, bool UNDER>
__global__ void __launch_bounds__(EV_THREADS)
eval_hist_kernel(const T *__restrict__ desc, const int8_t *__restrict__ flood, int64_t n, double nodata, Thresholds t,
                 EvScale sc, unsigned long long *__restrict__ hist)
{
    __shared__ unsigned sh[EV_SLOTS * (EV_MAXK + 1)];
    __shared__ CT th[EV_MAXK + 1];
    for (int i = threadIdx.x; i < EV_SLOTS * (EV_MAXK + 1); i += EV_THREADS) sh[i] = 0;
    if (threadIdx.x <= EV_MAXK) {
        const int i = threadIdx.x;
        th[i] = i < t.k ? (CT)t.th[i] : (CT)__longlong_as_double(0x7ff0000000000000LL);  // +inf: never below a value
    }
    __syncthreads();
    // (a nodata value that is not a CT never equals a CT descriptor: compare with NaN then)
    const double ndv = ev_nodata<T>(nodata, sc);
    const CT nd = (double)(CT)ndv == ndv ? (CT)ndv : (CT)__longlong_as_double(0x7ff8000000000000LL);
    const int64_t t0 = (int64_t)blockIdx.x * EV_THREADS + threadIdx.x, nt = (int64_t)gridDim.x * EV_THREADS;
    const int64_t nv = VEC ? n / 4 : 0;
    for (int64_t q = t0; q < nv; q += nt) {
        const EvPack4<T> d = *reinterpret_cast<const EvPack4<T> *>(desc + 4 * q);
        const char4 f = *reinterpret_cast<const char4 *>(flood + 4 * q);
        const int fv[4] = {f.x, f.y, f.z, f.w};
        int key[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) key[i] = eval_bin<CT, UNDER>(ev_load<CT>(d.v[i], sc), fv[i], nd, th, t.k);
        eval_count4(sh, key);
    }
    for (int64_t p = 4 * nv + t0; p < n; p += nt) {
        const int key = eval_bin<CT, UNDER>(ev_load<CT>(desc[p], sc), (int)flood[p], nd, th, t.k);
        if (key >= 0) atomicAdd(&sh[key], 1u);
    }
    __syncthreads();
    // slots -> avaliacao's classes (evaluation.py:149-150): 1 -> 2, -100 -> 0
    for (int i = threadIdx.x; i < EV_SLOTS * (EV_MAXK + 1); i += EV_THREADS) {
        if (!sh[i]) continue;
        const int slot = i / (EV_MAXK + 1), j = i - slot * (EV_MAXK + 1);
        const int c = slot == 1 ? 2 : (slot == 4 ? 0 : slot);
        atomicAdd(&hist[c * (EV_MAXK + 1) + j], (unsigned long long)sh[i]);
    }
}

template <typename T>
__global__ void __launch_bounds__(EV_THREADS)
eval_class_kernel(const T *__restrict__ desc, const int8_t *__restrict__ flood, int64_t n, double nodata, double th, int under,
                  EvScale sc, int8_t *__restrict__ binary, int8_t *__restrict__ cls)
{
    const double nd = ev_nodata<T>(nodata, sc);
    for (int64_t p = (int64_t)blockIdx.x * EV_THREADS + threadIdx.x; p < n; p += (int64_t)gridDim.x * EV_THREADS) {
        const double d = ev_load<double>(desc[p], sc);
        const int b = usable(d, nd) && (under ? d <= th : d >= th);
        if (binary) binary[p] = (int8_t)b;
        if (cls) cls[p] = (int8_t)(b + remap((int)flood[p]));
    }
}

template <typename T>
__global__ void __launch_bounds__(EV_THREADS)
minmax_scale_kernel(const T *__restrict__ mat, int64_t n, EvScale sc, double *__restrict__ out)
{
    for (int64_t p = (int64_t)blockIdx.x * EV_THREADS + threadIdx.x; p < n; p += (int64_t)gridDim.x * EV_THREADS)
        out[p] = minmax_scaled((double)mat[p], sc);
}

// ---- the two ends of np.unique (evaluation.py's caller, example.py:113-115) in one pass --------------------------------
// Per thread, then per warp, block and grid: the two smallest DISTINCT non-NaN values (a < b; `cnt` of them are set, so
// +-inf stay ordinary values), the largest non-NaN value (valid when cnt > 0) and whether a NaN occurs.  The values are
// compared as float: float32 and int16 cells are floats exactly.  -0 is stored as +0 (np.unique keeps one of them; the
// scaled rasters and counts are the same for either).
struct EvExt {
    float a, b, hi;
    int cnt, nan;
};

__device__ __forceinline__ void ext_insert(EvExt &e, float v)  // v not NaN
{
    v = v + 0.0f;  // -0 -> +0
    if (e.cnt == 0) { e.a = v; e.hi = v; e.cnt = 1; return; }
    e.hi = fmaxf(e.hi, v);
    if (v == e.a) return;
    if (v < e.a) { e.b = e.a; e.a = v; e.cnt = 2; }
    else if (e.cnt == 1 || v < e.b) { e.b = v; e.cnt = 2; }
}

__device__ __forceinline__ void ext_merge(EvExt &e, const EvExt &o)
{
    // the two smallest distinct values of a union are among the two smallest of each part
    if (o.cnt >= 1) ext_insert(e, o.a);
    if (o.cnt >= 2) ext_insert(e, o.b);
    if (o.cnt >= 1) e.hi = fmaxf(e.hi, o.hi);
    e.nan |= o.nan;
}

__device__ __forceinline__ void ext_cell(EvExt &e, float v)
{
    if (v != v) e.nan = 1;
    else ext_insert(e, v);
}

// the block's merged state in thread 0
__device__ __forceinline__ EvExt ext_block(EvExt e)
{
    __shared__ EvExt sh[EV_THREADS / 32];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        EvExt o;
        o.a = __shfl_down_sync(0xffffffffu, e.a, off);
        o.b = __shfl_down_sync(0xffffffffu, e.b, off);
        o.hi = __shfl_down_sync(0xffffffffu, e.hi, off);
        o.cnt = __shfl_down_sync(0xffffffffu, e.cnt, off);
        o.nan = __shfl_down_sync(0xffffffffu, e.nan, off);
        ext_merge(e, o);
    }
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = e;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int w = 1; w < EV_THREADS / 32; ++w) ext_merge(e, sh[w]);
    return e;
}

template <typename T> struct alignas(sizeof(T) * 4) ExtPack4 { T v[4]; };

template <typename T, bool VEC>
__global__ void __launch_bounds__(EV_THREADS) eval_extrema_kernel(const T *__restrict__ desc, int64_t n, EvExt *__restrict__ part)
{
    EvExt e{0.f, 0.f, 0.f, 0, 0};
    const int64_t t0 = (int64_t)blockIdx.x * EV_THREADS + threadIdx.x, nt = (int64_t)gridDim.x * EV_THREADS;
    const int64_t nv = VEC ? n / 4 : 0;
    for (int64_t q = t0; q < nv; q += nt) {
        const ExtPack4<T> d = *reinterpret_cast<const ExtPack4<T> *>(desc + 4 * q);
#pragma unroll
        for (int i = 0; i < 4; ++i) ext_cell(e, (float)d.v[i]);
    }
    for (int64_t p = 4 * nv + t0; p < n; p += nt) ext_cell(e, (float)desc[p]);
    e = ext_block(e);
    if (threadIdx.x == 0) part[blockIdx.x] = e;
}

// one block over the per-block partials -> out[5] = lo, second lo, hi, distinct values (0..2), NaN seen (0 / 1)
__global__ void __launch_bounds__(EV_THREADS) eval_extrema_finish_kernel(const EvExt *__restrict__ part, int nparts, double *__restrict__ out)
{
    EvExt e{0.f, 0.f, 0.f, 0, 0};
    for (int i = threadIdx.x; i < nparts; i += EV_THREADS) ext_merge(e, part[i]);
    e = ext_block(e);
    if (threadIdx.x == 0) {
        out[0] = e.cnt >= 1 ? (double)e.a : 0.0;
        out[1] = e.cnt >= 2 ? (double)e.b : 0.0;
        out[2] = e.cnt >= 1 ? (double)e.hi : 0.0;
        out[3] = (double)e.cnt;
        out[4] = (double)e.nan;
    }
}

// launch the histogram kernel of source type T, compared as CT, on the aligned / scalar and under / over variant
template <typename T, typename CT>
int launch_hist(const char *name, const void *desc, const int8_t *flood, int64_t n, double nodata, const Thresholds &t, const EvScale &sc,
                unsigned long long *hist, bool vec, bool under, cudaStream_t st)
{
#define DTB_EVH(VEC, UNDER) \
    DTB_KERNEL(name, st, (eval_hist_kernel<T, CT, VEC, UNDER><<<EV_BLOCKS, EV_THREADS, 0, st>>>((const T *)desc, flood, n, nodata, t, sc, hist)))
    if (vec && under) DTB_EVH(true, true);
    else if (vec) DTB_EVH(true, false);
    else if (under) DTB_EVH(false, true);
    else DTB_EVH(false, false);
#undef DTB_EVH
    return DTB_OK;
}

int thresholds_of(const double *thresholds_host, int k, Thresholds &t)
{
    if (!thresholds_host || k <= 0 || k > EV_MAXK) return DTB_ERR_INVALID;
    for (int i = 1; i < k; ++i)
        if (!(thresholds_host[i - 1] < thresholds_host[i])) return DTB_ERR_INVALID;  // strictly ascending
    t.k = k;
    for (int i = 0; i < EV_MAXK; ++i) t.th[i] = i < k ? thresholds_host[i] : 0.0;
    return DTB_OK;
}

}  // namespace
}  // namespace dtb

extern "C" int dtb_eval_counts_from_hist(const unsigned long long *hist_host, int k, int under, int64_t *counts_host)
{
    using namespace dtb;
    if (!hist_host || !counts_host || k <= 0 || k > EV_MAXK) return DTB_ERR_INVALID;
    const unsigned long long *h = hist_host;
    for (int i = 0; i < k; ++i) {
        int64_t cnt[5] = {0, 0, 0, 0, 0};  // classes 0..4 (binary + remapped benchmark)
        for (int c = 0; c < 4; ++c) {
            int64_t flagged = 0, total = 0;
            for (int j = 0; j <= k; ++j) {
                total += (int64_t)h[c * (EV_MAXK + 1) + j];
                if (under ? j <= i : j > i) flagged += (int64_t)h[c * (EV_MAXK + 1) + j];
            }
            cnt[c] += total - flagged;
            cnt[c + 1] += flagged;
        }
        for (int c = 0; c < 4; ++c) counts_host[4 * i + c] = cnt[c];  // tn, fp, fn, tp (evaluation.py:152-166)
    }
    return DTB_OK;
}

extern "C" int dtb_eval_counts(const void *desc, int desc_is_f64, const int8_t *flood, int64_t n, double nodata,
                               const double *thresholds_host, int k, int under, int64_t *counts_host, void *ws, size_t ws_bytes,
                               void *stream)
{
    using namespace dtb;
    Thresholds t;
    if (!desc || !flood || !counts_host || !ws || n <= 0 || thresholds_of(thresholds_host, k, t) != DTB_OK) return DTB_ERR_INVALID;
    if (ws_bytes < 4 * (EV_MAXK + 1) * sizeof(unsigned long long)) return DTB_ERR_WORKSPACE;
    cudaStream_t st = as_stream(stream);
    unsigned long long *hist = reinterpret_cast<unsigned long long *>(ws);
    DTB_CUDA(cudaMemsetAsync(hist, 0, 4 * (EV_MAXK + 1) * sizeof(unsigned long long), st));
    const bool vec = (reinterpret_cast<uintptr_t>(desc) % (desc_is_f64 ? 32 : 16)) == 0 && (reinterpret_cast<uintptr_t>(flood) % 4) == 0;
    bool as_float = !desc_is_f64 && (double)(float)nodata == nodata;
    for (int i = 0; i < k && as_float; ++i) as_float = (double)(float)thresholds_host[i] == thresholds_host[i];
    const EvScale none{0.0, 0.0, 0.0};  // unused: these sources are compared as they are
    int rc;
    if (desc_is_f64) rc = launch_hist<double, double>("eval_hist_kernel<f64>", desc, flood, n, nodata, t, none, hist, vec, under, st);
    else if (as_float) rc = launch_hist<float, float>("eval_hist_kernel<f32>", desc, flood, n, nodata, t, none, hist, vec, under, st);
    else rc = launch_hist<float, double>("eval_hist_kernel<f32,f64>", desc, flood, n, nodata, t, none, hist, vec, under, st);
    if (rc != DTB_OK) return rc;
    unsigned long long h[4 * (EV_MAXK + 1)];
    DTB_CUDA(cudaMemcpyAsync(h, hist, sizeof(h), cudaMemcpyDeviceToHost, st));
    DTB_CUDA(cudaStreamSynchronize(st));
    return dtb_eval_counts_from_hist(h, k, under, counts_host);
}

extern "C" int dtb_eval_hist(const void *desc, int desc_dtype, const int8_t *flood, int64_t n, double mn, double mx, double nodata,
                             double corner, const double *thresholds_host, int k, int under, unsigned long long *hist, void *stream)
{
    using namespace dtb;
    Thresholds t;
    if (!desc || !flood || !hist || n <= 0 || thresholds_of(thresholds_host, k, t) != DTB_OK) return DTB_ERR_INVALID;
    if (desc_dtype != DTB_EV_F32 && desc_dtype != DTB_EV_I16) return DTB_ERR_INVALID;
    cudaStream_t st = as_stream(stream);
    const EvScale sc{mn, mx, nodata};
    const size_t pack = desc_dtype == DTB_EV_F32 ? 16 : 8;
    const bool vec = (reinterpret_cast<uintptr_t>(desc) % pack) == 0 && (reinterpret_cast<uintptr_t>(flood) % 4) == 0;
    if (desc_dtype == DTB_EV_F32)
        return launch_hist<MinMaxScaled<float>, double>("eval_hist_kernel<scaled f32>", desc, flood, n, corner, t, sc, hist, vec, under, st);
    return launch_hist<MinMaxScaled<int16_t>, double>("eval_hist_kernel<scaled i16>", desc, flood, n, corner, t, sc, hist, vec, under, st);
}

extern "C" size_t dtb_eval_extrema_workspace_bytes(void) { return (size_t)dtb::EV_BLOCKS * sizeof(dtb::EvExt); }

extern "C" int dtb_eval_extrema(const void *desc, int desc_dtype, int64_t n, double *out, void *ws, size_t ws_bytes, void *stream)
{
    using namespace dtb;
    if (!desc || !out || !ws || n <= 0) return DTB_ERR_INVALID;
    if (desc_dtype != DTB_EV_F32 && desc_dtype != DTB_EV_I16) return DTB_ERR_INVALID;
    if (ws_bytes < dtb_eval_extrema_workspace_bytes()) return DTB_ERR_WORKSPACE;
    cudaStream_t st = as_stream(stream);
    EvExt *part = reinterpret_cast<EvExt *>(ws);
    const bool vec = reinterpret_cast<uintptr_t>(desc) % (desc_dtype == DTB_EV_F32 ? 16 : 8) == 0;
#define DTB_EXT(NAME, T)                                                                                                            \
    do {                                                                                                                            \
        if (vec) DTB_KERNEL(NAME, st, (eval_extrema_kernel<T, true><<<EV_BLOCKS, EV_THREADS, 0, st>>>((const T *)desc, n, part)));  \
        else DTB_KERNEL(NAME, st, (eval_extrema_kernel<T, false><<<EV_BLOCKS, EV_THREADS, 0, st>>>((const T *)desc, n, part)));    \
    } while (0)
    if (desc_dtype == DTB_EV_F32) DTB_EXT("eval_extrema_kernel<f32>", float);
    else DTB_EXT("eval_extrema_kernel<i16>", int16_t);
#undef DTB_EXT
    DTB_KERNEL("eval_extrema_finish_kernel", st, eval_extrema_finish_kernel<<<1, EV_THREADS, 0, st>>>(part, EV_BLOCKS, out));
    return DTB_OK;
}

extern "C" int dtb_eval_class_map(const void *desc, int desc_is_f64, const int8_t *flood, int64_t n, double nodata, double threshold,
                                  int under, int8_t *binary, int8_t *cls, void *stream)
{
    using namespace dtb;
    if (!desc || n <= 0 || (!binary && !cls) || (cls && !flood)) return DTB_ERR_INVALID;
    cudaStream_t st = as_stream(stream);
    const EvScale none{0.0, 0.0, 0.0};
    if (desc_is_f64) DTB_KERNEL("eval_class_kernel<f64>", st, eval_class_kernel<double><<<EV_BLOCKS, EV_THREADS, 0, st>>>((const double *)desc, flood, n, nodata, threshold, under, none, binary, cls));
    else DTB_KERNEL("eval_class_kernel<f32>", st, eval_class_kernel<float><<<EV_BLOCKS, EV_THREADS, 0, st>>>((const float *)desc, flood, n, nodata, threshold, under, none, binary, cls));
    return DTB_OK;
}

extern "C" int dtb_eval_class_scaled(const void *desc, int desc_dtype, const int8_t *flood, int64_t n, double mn, double mx, double nodata,
                                     double corner, double threshold, int under, int8_t *cls, void *stream)
{
    using namespace dtb;
    if (!desc || !flood || !cls || n <= 0) return DTB_ERR_INVALID;
    cudaStream_t st = as_stream(stream);
    const EvScale sc{mn, mx, nodata};
    if (desc_dtype == DTB_EV_F32)
        DTB_KERNEL("eval_class_kernel<scaled f32>", st, eval_class_kernel<MinMaxScaled<float>><<<EV_BLOCKS, EV_THREADS, 0, st>>>(
            (const MinMaxScaled<float> *)desc, flood, n, corner, threshold, under, sc, nullptr, cls));
    else if (desc_dtype == DTB_EV_I16)
        DTB_KERNEL("eval_class_kernel<scaled i16>", st, eval_class_kernel<MinMaxScaled<int16_t>><<<EV_BLOCKS, EV_THREADS, 0, st>>>(
            (const MinMaxScaled<int16_t> *)desc, flood, n, corner, threshold, under, sc, nullptr, cls));
    else return DTB_ERR_INVALID;
    return DTB_OK;
}

extern "C" int dtb_minmax_scale(const void *mat, int mat_dtype, int64_t n, double mn, double mx, double nodata, double *out, void *stream)
{
    using namespace dtb;
    if (!mat || !out || n <= 0) return DTB_ERR_INVALID;
    cudaStream_t st = as_stream(stream);
    const EvScale sc{mn, mx, nodata};
    if (mat_dtype == DTB_EV_F64) DTB_KERNEL("minmax_scale_kernel<f64>", st, minmax_scale_kernel<double><<<EV_BLOCKS, EV_THREADS, 0, st>>>((const double *)mat, n, sc, out));
    else if (mat_dtype == DTB_EV_F32) DTB_KERNEL("minmax_scale_kernel<f32>", st, minmax_scale_kernel<float><<<EV_BLOCKS, EV_THREADS, 0, st>>>((const float *)mat, n, sc, out));
    else if (mat_dtype == DTB_EV_I16) DTB_KERNEL("minmax_scale_kernel<i16>", st, minmax_scale_kernel<int16_t><<<EV_BLOCKS, EV_THREADS, 0, st>>>((const int16_t *)mat, n, sc, out));
    else return DTB_ERR_INVALID;
    return DTB_OK;
}
