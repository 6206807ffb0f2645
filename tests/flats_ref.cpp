// flats_ref.cpp -- host reference for exact depression filling (F1) and flat resolution (F2).
//
// The statement the device kernels (descriptools_b200/csrc/synth.cu fill_relax_flat_kernel, csrc/flats.cu) are tested
// against, written the plain way: a heap-based priority flood and breadth-first searches with queues.
//
// F1: priority flood without epsilon.  Seeds = valid cells on the raster edge or next to a nodata cell (== -100 or NaN)
//     keep z; every other cell reachable from a seed is raised to the lowest level from which it drains.  Nodata cells
//     are untouched.
// F2: on a DEM z and its D8 codes c (SURVEY App. A2), a flat cell is a valid cell (z > -100, not NaN) with c == 0.
//     Flats are 8-connected components of flat cells; an outlet of a flat is a valid cell with c != 0 at the flat's
//     elevation next to one of its cells; a high edge is a flat cell with a strictly higher neighbour.
//     towards = steps to the nearest outlet through the flat (1 next to an outlet), away = steps to the nearest high
//     edge (0 on one), A = max away over the flat (0 without a high edge).  mask = 2 towards + (A - away) (second term
//     0 without a high edge), -1 for an outlet; each cell of a drained flat points at the neighbour of least mask among
//     its flat and its outlets, first in scan order NW N NE W E SW S SE on ties.  Flats without an outlet keep code 0.
#include <cmath>
#include <cstdint>
#include <functional>
#include <queue>
#include <vector>

namespace {

const int DR[8] = {-1, -1, -1, 0, 0, 1, 1, 1}, DC[8] = {-1, 0, 1, -1, 1, -1, 0, 1};
const uint8_t CODE[8] = {32, 64, 128, 16, 1, 8, 4, 2};

template <class T> bool valid(T z) { return z > (T)-100; }  // false for NaN

template <class T>
int64_t resolve(const T *z, uint8_t *d8, int64_t rows, int64_t cols, int64_t *n_flat, int64_t *mask_out)
{
    const int64_t n = rows * cols;
    const int64_t INF = INT64_MAX;
    std::vector<uint8_t> flat((size_t)n);
    for (int64_t p = 0; p < n; ++p) flat[p] = valid(z[p]) && d8[p] == 0;
    auto for_nb = [&](int64_t p, const std::function<void(int, int64_t)> &f) {
        const int64_t r = p / cols, c = p % cols;
        for (int k = 0; k < 8; ++k) {
            const int64_t rr = r + DR[k], cc = c + DC[k];
            if (rr < 0 || rr >= rows || cc < 0 || cc >= cols) continue;
            f(k, rr * cols + cc);
        }
    };
    auto outlet_of = [&](int64_t p, int64_t q) { return !flat[q] && valid(z[q]) && d8[q] != 0 && z[q] == z[p]; };

    // flats: breadth-first labelling
    std::vector<int64_t> label((size_t)n, -1);
    std::vector<int64_t> queue;
    int64_t nf = 0;
    for (int64_t s = 0; s < n; ++s) {
        if (!flat[s] || label[s] >= 0) continue;
        label[s] = s;
        queue.assign(1, s);
        for (size_t i = 0; i < queue.size(); ++i)
            for_nb(queue[i], [&](int, int64_t q) {
                if (flat[q] && label[q] < 0) { label[q] = s; queue.push_back(q); }
            });
        nf += (int64_t)queue.size();
    }
    if (n_flat) *n_flat = nf;

    // multi-source breadth-first distances through flat cells
    auto bfs = [&](std::vector<int64_t> &dist, const std::function<bool(int64_t)> &source, int64_t d0) {
        dist.assign((size_t)n, INF);
        queue.clear();
        for (int64_t p = 0; p < n; ++p)
            if (flat[p] && source(p)) { dist[p] = d0; queue.push_back(p); }
        for (size_t i = 0; i < queue.size(); ++i) {
            const int64_t p = queue[i];
            for_nb(p, [&](int, int64_t q) {
                if (flat[q] && dist[q] == INF) { dist[q] = dist[p] + 1; queue.push_back(q); }
            });
        }
    };
    std::vector<int64_t> towards, away;
    bfs(towards, [&](int64_t p) { bool o = false; for_nb(p, [&](int, int64_t q) { o |= outlet_of(p, q); }); return o; }, 1);
    bfs(away, [&](int64_t p) { bool h = false; for_nb(p, [&](int, int64_t q) { h |= z[q] > z[p]; }); return h; }, 0);
    std::vector<int64_t> amax((size_t)n, 0);
    for (int64_t p = 0; p < n; ++p)
        if (flat[p] && away[p] != INF && away[p] > amax[label[p]]) amax[label[p]] = away[p];
    auto mask = [&](int64_t p) { return 2 * towards[p] + (away[p] == INF ? 0 : amax[label[p]] - away[p]); };

    if (mask_out)
        for (int64_t p = 0; p < n; ++p) mask_out[p] = !flat[p] ? -1 : (towards[p] == INF ? INF : mask(p));

    int64_t unresolved = 0;
    std::vector<uint8_t> code((size_t)n, 0);
    for (int64_t p = 0; p < n; ++p) {
        if (!flat[p]) continue;
        if (towards[p] == INF) { ++unresolved; continue; }
        int64_t best = INF;
        for_nb(p, [&](int k, int64_t q) {
            const int64_t m = flat[q] ? mask(q) : (outlet_of(p, q) ? -1 : INF);
            if (m < best) { best = m; code[p] = CODE[k]; }
        });
    }
    for (int64_t p = 0; p < n; ++p)
        if (flat[p]) d8[p] = code[p];
    return unresolved;
}

}  // namespace

extern "C" {

// priority flood without epsilon, in place
void ref_priority_flood_f32(float *dem, int64_t rows, int64_t cols)
{
    const int64_t n = rows * cols;
    std::vector<uint8_t> closed((size_t)n, 0);
    typedef std::pair<float, int64_t> item;
    std::priority_queue<item, std::vector<item>, std::greater<item>> pq;
    auto is_nd = [&](int64_t p) { return dem[p] == -100.0f || dem[p] != dem[p]; };
    for (int64_t r = 0; r < rows; ++r)
        for (int64_t c = 0; c < cols; ++c) {
            const int64_t p = r * cols + c;
            if (is_nd(p)) { closed[p] = 1; continue; }
            bool seed = (r == 0 || c == 0 || r == rows - 1 || c == cols - 1);
            for (int k = 0; k < 8 && !seed; ++k) {
                const int64_t rr = r + DR[k], cc = c + DC[k];
                seed = is_nd(rr * cols + cc);
            }
            if (seed) { closed[p] = 1; pq.push(item(dem[p], p)); }
        }
    while (!pq.empty()) {
        const item it = pq.top();
        pq.pop();
        const int64_t p = it.second, r = p / cols, c = p % cols;
        for (int k = 0; k < 8; ++k) {
            const int64_t rr = r + DR[k], cc = c + DC[k];
            if (rr < 0 || rr >= rows || cc < 0 || cc >= cols) continue;
            const int64_t q = rr * cols + cc;
            if (closed[q]) continue;
            closed[q] = 1;
            if (dem[q] < it.first) dem[q] = it.first;
            pq.push(item(dem[q], q));
        }
    }
}

// flat resolution of d8 in place; returns the number of unresolved flat cells, *n_flat the number of flat cells.
// mask_out (may be NULL): mask of every flat cell (INT64_MAX in a flat without outlet), -1 on every other cell
int64_t ref_resolve_flats_f32(const float *dem, uint8_t *d8, int64_t rows, int64_t cols, int64_t *n_flat, int64_t *mask_out)
{
    return resolve(dem, d8, rows, cols, n_flat, mask_out);
}
int64_t ref_resolve_flats_i16(const int16_t *dem, uint8_t *d8, int64_t rows, int64_t cols, int64_t *n_flat, int64_t *mask_out)
{
    return resolve(dem, d8, rows, cols, n_flat, mask_out);
}

}  // extern "C"
