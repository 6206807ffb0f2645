// hand.cu -- flow distance to the nearest drainage, river-cell index, HAND (+ fused GFI).
//
// Semantics: flow_distance_index_gpu (flowhand.py:599-846, unpartitioned: out[*] = 0) and
// hand_calculator (flowhand.py:431-442); optional fused river_accumulation + GFI
// (gfi.py:136-147, 287-294).  Restated in oracle/dt_oracle.c.
//
// The reference walks every cell down the D8 pointers (O(path length) dependent loads per
// cell, mean 214 on its example).  Here the D8 forest is resolved by pointer jumping over a
// packed 64-bit state per cell
//     [63..62 kind | 61..47 diagonal moves | 46..32 cardinal moves | 31..0 target]
// in two levels that share the 64x64 tiling of flowacc.cu (tiles.cuh):
//   H1  hand_entry_kernel: per tile, only the perimeter cells that receive flow from outside
//       (entry nodes) walk their in-tile path: it ends on a river cell, fails, or leaves the tile
//       into another entry node.  One 64-bit state per node.
//   H2  hand_node_jump_kernel: pointer jumping over the entry nodes in global memory.  In-place and
//       asynchronous: any state read is a valid description of that node's path, every launch of
//       2 compositions per node covers at least 3x the hops, so ceil(log3(max_moves+1)) launches
//       (10 for the reference's 20 000 moves) decide every node;
//       what is still ACTIVE then needs more than max_moves moves or sits on / drains into a
//       cycle -> FAIL, the reference's outcomes (flowhand.py:826 code-0 landing, :830 cycle
//       detector, :835 move cap, border exits :623-764).  A launch whose predecessor left
//       nothing ACTIVE returns at once.
//   H3  hand_tile_kernel: per tile, pointer jumping over all 4096 cells in shared memory (targets:
//       river cell, failure, or the tile's exit cell), composition with the resolved state of the
//       entry node behind each exit, then the epilogue: idx, flow distance, HAND = z - z[idx]
//       and GFI from the gathered accumulation of the river cell, written once.
// Distance = n_card*px + n_diag*(px*sqrt(2)) in f64 (the reference adds the same terms one
// move at a time, flowhand.py:803-824; the two agree far below f32 resolution).
// GFI = ln(b) + n*ln(A_r*size^2) - ln(H + 0.01) in f64 with the short logarithms of common.cuh: the
// reference's log(b*pow(A_r*size^2, n)/(H+0.01)) (gfi.py:292-294) rearranged to drop the pow.  The two
// agree to (|n| + 2) * 3e-9 plus the f32 rounding of the stored result where |n| <= 8 and 1e-30 < b < 1e30
// (the domain pointwise.cu's log form serves), including n = 0 with A_r = 0 and NaN / infinite HAND values.
// Outside that domain the rearranged form stays finite where the reference's pow overflows.
#include <math.h>
#include <stdlib.h>

#include "tiles.cuh"

namespace dtb {
namespace {

constexpr int H_THREADS = 256;
struct RiverSrc {
    const int8_t *river;  // 0/1 mask (flowhand.py:609) or NULL
    const void *acc;      // river = acc > thr (example.py:52)
    int64_t thr;
};

// 16-bit river mask of the 16 cells (row lr, columns lcb..lcb+15) of the tile at (r0, c0)
template <typename ACC>
__device__ __forceinline__ unsigned river_bits(const RiverSrc &rs, const TileView &v, int64_t r0, int64_t c0, int lr, int lcb,
                                               bool fast)
{
    const int64_t gr = r0 + lr;
    unsigned m = 0;
    if (gr >= v.rows) return 0;
    const int64_t o = gr * v.cols + c0 + lcb;
    if (rs.river) {
        if (fast && ((reinterpret_cast<uintptr_t>(rs.river) & 15u) == 0)) {
            const uint4 w = __ldg(reinterpret_cast<const uint4 *>(rs.river + o));
            const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int i = 0; i < 16; ++i) m |= (((ww[i >> 2] >> (8 * (i & 3))) & 0xFFu) == 1u) << i;
        } else {
            for (int i = 0; i < 16; ++i)
                if (c0 + lcb + i < v.cols) m |= (unsigned)(rs.river[o + i] == 1) << i;
        }
    } else {
        const ACC *a = reinterpret_cast<const ACC *>(rs.acc);
        if (fast && ((reinterpret_cast<uintptr_t>(a) & 15u) == 0)) {
            constexpr int V = 16 / sizeof(ACC);
#pragma unroll
            for (int i = 0; i < 16; i += V) {
                const uint4 w = __ldg(reinterpret_cast<const uint4 *>(a + o + i));
                const ACC *e = reinterpret_cast<const ACC *>(&w);
#pragma unroll
                for (int j = 0; j < V; ++j) m |= (unsigned)((int64_t)e[j] > rs.thr) << (i + j);
            }
        } else {
            for (int i = 0; i < 16; ++i)
                if (c0 + lcb + i < v.cols) m |= (unsigned)((int64_t)a[o + i] > rs.thr) << i;
        }
    }
    return m;
}

// ---- H1: entry nodes walk their in-tile path -------------------------------------------------------
template <typename ACC>
__global__ void __launch_bounds__(H_THREADS)
hand_entry_kernel(TileView v, RiverSrc rs, unsigned long long *__restrict__ nstate, unsigned *__restrict__ active)
{
    __shared__ __align__(16) uint8_t codes[(T + 2) * CP + 16];
    __shared__ uint16_t rivm[H_THREADS];
    const int tid = threadIdx.x;
    const int tile = blockIdx.x;
    const int ty = tile / v.tiles_x, tx = tile - ty * v.tiles_x;
    const int64_t r0 = (int64_t)ty * T, c0 = (int64_t)tx * T;
    const bool fast = stage_codes(v, r0, c0, codes, tid, H_THREADS);
    rivm[tid] = (uint16_t)river_bits<ACC>(rs, v, r0, c0, tid >> 2, (tid & 3) * CPT, fast);
    __syncthreads();
    auto C = [&](int lr, int lc) -> unsigned { return codes[(lr + 1) * CP + 16 + lc]; };

    uint64_t s = 0ull;  // inactive slot (never referenced)
    int is_active = 0;
    if (tid < USED_SLOTS) {
        int lr, lc;
        slot_cell(tid, lr, lc);
        if (C(lr, lc) != 0 && (in_mask(codes, lr, lc) & out_mask(lr, lc))) {
            uint32_t nc = 0, nd = 0;
            s = pack(KIND_FAIL, 0, 0, 0);  // in-tile cycle if the loop runs out
            for (int steps = 0; steps <= TCELLS; ++steps) {
                const int p = lr * T + lc;
                if ((rivm[p >> 4] >> (p & 15)) & 1u) {  // flowhand.py:622
                    s = pack(KIND_RIVER, nd, nc, (uint32_t)((r0 + lr) * v.cols + c0 + lc));
                    break;
                }
                const unsigned code = C(lr, lc);
                int dr, dc;
                if (!d8_offset(code, dr, dc)) break;             // unknown code: "did not move", flowhand.py:830
                const int tr = lr + dr, tc = lc + dc;
                if (C(tr, tc) == 0) break;                        // off-raster or code 0, flowhand.py:623-764, 826
                if (d8_is_diag(code)) ++nd; else ++nc;
                if ((unsigned)tr >= (unsigned)T || (unsigned)tc >= (unsigned)T) {
                    const int64_t gr = r0 + tr, gc = c0 + tc;
                    if (gr < 0) s = pack(KIND_EXIT, nd, nc, LINK_OUT | (uint32_t)gc);
                    else if (gr >= v.rows) s = pack(KIND_EXIT, nd, nc, LINK_OUT | LINK_BELOW | (uint32_t)gc);
                    else { s = pack(KIND_ACTIVE, nd, nc, (uint32_t)node_of_cell(gr, gc, v.tiles_x)); is_active = 1; }
                    break;
                }
                lr = tr;
                lc = tc;
            }
        }
    }
    nstate[(size_t)tile * SLOTS + tid] = s;
    const unsigned ballot = __ballot_sync(0xffffffffu, is_active);
    if ((tid & 31) == 0 && ballot) atomicAdd(&active[0], (unsigned)__popc(ballot));
}

// ---- H2: pointer jumping over the entry nodes ------------------------------------------------------
// round `rnd` (1-based): reads active[rnd-1], adds the number of nodes still ACTIVE to active[rnd]
__global__ void __launch_bounds__(H_THREADS)
hand_node_jump_kernel(int64_t nnodes, unsigned long long *nstate, unsigned *__restrict__ active, int rnd, int jumps)
{
    if (active[rnd - 1] == 0) return;
    unsigned still = 0;
    // two states per thread and pass (16-byte loads): most of a launch is the scan over all slots (nnodes is a multiple of 256)
    for (int64_t q = ((int64_t)blockIdx.x * H_THREADS + threadIdx.x) * 2; q < nnodes; q += (int64_t)gridDim.x * H_THREADS * 2) {
        const ulonglong2 two = __ldcg(reinterpret_cast<const ulonglong2 *>(&nstate[q]));
        const uint64_t in[2] = {two.x, two.y};
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            uint64_t s = in[k];
            if (kind_of(s) != KIND_ACTIVE || s == 0ull) continue;  // 0 = inactive slot
            for (int j = 0; j < jumps; ++j) {
                s = compose(s, __ldcg(&nstate[ptr_of(s)]));
                if (kind_of(s) != KIND_ACTIVE) break;
            }
            __stcg(&nstate[q + k], s);
            still += kind_of(s) == KIND_ACTIVE;
        }
    }
    still = __reduce_add_sync(0xffffffffu, still);
    if ((threadIdx.x & 31) == 0 && still) atomicAdd(&active[rnd], still);
}

template <typename T> struct HandOps;
template <> struct HandOps<float> {
    static __device__ __forceinline__ bool is_nd(float z) { return z == ND_F; }
    static __device__ __forceinline__ float sub(float a, float b) { return a - b; }
    static __device__ __forceinline__ float nd() { return ND_F; }
    // fast_log_pos needs a finite argument (it reads +inf as 1024 ln 2): for a NaN / +inf HAND (a non-finite DEM cell)
    // subtracting H gives the reference's NaN / -inf (NaN where ln b + n ln(A_r size^2) is +inf too).  Two f32
    // instructions per cell; correcting the f64 log instead cost the issue-bound tile pass ~3 % (B200, 40k x 40k).
    static __device__ __forceinline__ void fix_nonfinite(float &g, float h) { if (!(fabsf(h) < INFINITY)) g -= h; }
};
template <> struct HandOps<int16_t> {
    static __device__ __forceinline__ bool is_nd(int16_t z) { return z == ND_I; }
    static __device__ __forceinline__ int16_t sub(int16_t a, int16_t b) { return (int16_t)(a - b); }  // numpy i16 wrap
    static __device__ __forceinline__ int16_t nd() { return (int16_t)ND_I; }
    static __device__ __forceinline__ void fix_nonfinite(float &, int16_t) {}
};

// flowhand.py:436-438
template <typename T>
__device__ __forceinline__ T hand_value(T z, bool resolved, const T *__restrict__ dem, int64_t idx)
{
    T h = HandOps<T>::nd();
    if (!HandOps<T>::is_nd(z) && resolved) h = HandOps<T>::sub(z, dem[idx]);
    if (h < (T)0 && h != HandOps<T>::nd()) h = (T)0;
    return h;
}



// ---- H3: per-tile resolution + epilogue ---------------------------------------------------------
struct HandOut {
    float *fdist;
    void *idx;
    void *hand;
    float *gfi;
    double px, pd;
    uint32_t max_moves;
    double gfi_logb, gfi_n, gfi_s2;
    // row bands: global index offset and the resolved paths behind the halo rows (side 0 above, 1 below)
    int64_t idx_offset;
    const unsigned long long *res_state[2];
    const int64_t *res_idx[2];
    const double *res_z[2];
    const int64_t *res_acc[2];
};

// four consecutive cells of one row, as one vector store when the row is 16-byte tileable
template <typename V>
__device__ __forceinline__ void store4(V *dst, const V (&val)[4], bool vec, int64_t c_first, int64_t cols)
{
    if (vec) {
        if (sizeof(V) == 2) *reinterpret_cast<uint2 *>(dst) = *reinterpret_cast<const uint2 *>(&val[0]);
        else if (sizeof(V) == 4) *reinterpret_cast<uint4 *>(dst) = *reinterpret_cast<const uint4 *>(&val[0]);
        else {
            *reinterpret_cast<uint4 *>(dst) = *reinterpret_cast<const uint4 *>(&val[0]);
            *reinterpret_cast<uint4 *>(dst + 2) = *reinterpret_cast<const uint4 *>(&val[2]);
        }
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (c_first + i < cols) dst[i] = val[i];
    }
}
template <typename V>
__device__ __forceinline__ void load4(const V *src, V (&val)[4], bool vec, int64_t c_first, int64_t cols, V fill)
{
    if (vec) {
        if (sizeof(V) == 2) *reinterpret_cast<uint2 *>(&val[0]) = __ldg(reinterpret_cast<const uint2 *>(src));
        else *reinterpret_cast<uint4 *>(&val[0]) = __ldg(reinterpret_cast<const uint4 *>(src));
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) val[i] = (c_first + i < cols) ? src[i] : fill;
    }
}

// What lies behind exit cell (plr, plc) of the tile at (r0, c0), leaving with direction (dr, dc) / code `code`:
// the state of the entry node it lands on (or of the halo cell, for a band), composed with the exit move.
template <typename TD, typename IDX, typename ACC>
__device__ __forceinline__ void resolve_exit(const TileView &v, int64_t r0, int64_t c0, int slot, int plr, int plc, bool is_exit,
                                             unsigned code, int dr, int dc, const TD *__restrict__ dem,
                                             const ACC *__restrict__ acc, const unsigned long long *__restrict__ nstate,
                                             const HandOut &o, uint32_t *exit_hi, IDX *exit_idx, TD *exit_z, double *exit_l1)
{
    uint64_t e = pack(KIND_FAIL, 0, 0, 0);
    unsigned remote = 0;
    if (is_exit) {
        const int64_t gr = r0 + plr + dr, gc = c0 + plc + dc;
        const bool diag = d8_is_diag(code);
        const uint64_t mv = pack(KIND_ACTIVE, diag ? 1u : 0u, diag ? 0u : 1u, 0);
        uint64_t ns = pack(KIND_FAIL, 0, 0, 0);
        if (gr >= 0 && gr < v.rows) ns = nstate[node_of_cell(gr, gc, v.tiles_x)];
        if (kind_of(ns) == KIND_EXIT || gr < 0 || gr >= v.rows) {
            // the path leaves the band (now, or further down inside the band): continue with the
            // resolved path of the halo cell it lands on
            int side;
            int64_t col;
            uint64_t pre = mv;
            if (gr < 0 || gr >= v.rows) { side = gr < 0 ? 0 : 1; col = gc; }
            else { side = (ptr_of(ns) & LINK_BELOW) ? 1 : 0; col = ptr_of(ns) & 0x3FFFFFFFu; pre = compose(mv, ns); }
            ns = o.res_state[side] ? o.res_state[side][col] : pack(KIND_FAIL, 0, 0, 0);
            ns = (ns & ~0xFFFFFFFFull) | (uint64_t)(uint32_t)col;
            e = compose(pack(KIND_ACTIVE, nd_of(pre), nc_of(pre), 0), ns);
            remote = 1u + (unsigned)side;
        } else {
            e = compose(mv, ns);
        }
        if (kind_of(e) != KIND_RIVER) { e = pack(KIND_FAIL, 0, 0, 0); remote = 0; }  // ACTIVE left over: cycle or > cap
    }
    exit_hi[slot] = ((uint32_t)kind_of(e) << 30) | (nd_of(e) << 15) | nc_of(e);
    if (kind_of(e) == KIND_RIVER) {
        const int64_t loc = (int64_t)ptr_of(e);  // local index of the river cell, or (remote) a column of the halo tables
        double racc = 1.0;
        if (remote) {
            exit_idx[slot] = (IDX)o.res_idx[remote - 1][loc];
            exit_z[slot] = (TD)o.res_z[remote - 1][loc];
            if (o.gfi) racc = (double)o.res_acc[remote - 1][loc];
        } else {
            exit_idx[slot] = (IDX)(loc + o.idx_offset);
            exit_z[slot] = (o.hand || o.gfi) ? dem[loc] : (TD)0;
            if (o.gfi) racc = (double)acc[loc];  // river_accumulation, gfi.py:141-143
        }
        // n = 0: ln b for every A_r, as pow(A_r size^2, 0) = 1 is in the reference (n * ln 0 would be NaN); same at the two sites below
        exit_l1[slot] = o.gfi ? (o.gfi_n == 0.0 ? o.gfi_logb : o.gfi_logb + o.gfi_n * fast_log(racc * o.gfi_s2)) : 0.0;
    }
}

template <typename TD, typename IDX> struct alignas(8) ExitRec {
    uint32_t hi;  // [31..30 kind | 29..15 diagonal moves | 14..0 cardinal moves] from the exit cell on
    TD z;         // elevation of the river cell
    IDX idx;      // its global index
    double l1;    // ln b + n ln(A_r size^2)
};
template <typename TD, typename IDX, typename ACC>
__device__ __forceinline__ void resolve_exit(const TileView &v, int64_t r0, int64_t c0, int slot, int plr, int plc, bool is_exit,
                                             unsigned code, int dr, int dc, const TD *__restrict__ dem,
                                             const ACC *__restrict__ acc, const unsigned long long *__restrict__ nstate,
                                             const HandOut &o, ExitRec<TD, IDX> *exits)
{
    uint32_t hi;
    IDX idx = (IDX)ND_I;
    TD z = (TD)0;
    double l1 = 0.0;
    resolve_exit<TD, IDX, ACC>(v, r0, c0, 0, plr, plc, is_exit, code, dr, dc, dem, acc, nstate, o, &hi, &idx, &z, &l1);
    ExitRec<TD, IDX> x;
    x.hi = hi;
    x.z = z;
    x.idx = idx;
    x.l1 = l1;
    exits[slot] = x;
}

// outputs of one cell from its resolved path
template <typename TD, typename IDX>
__device__ __forceinline__ void finish_cell(const HandOut &o, const bool want_h, const bool want_g, uint32_t kind, uint32_t nd,
                                            uint32_t nc, int64_t idx, TD zr, double l1, TD z, float &fd, IDX &ix, TD &hd, float &gf)
{
    const bool ok = kind == KIND_RIVER && nc + nd <= o.max_moves;  // flowhand.py:835
    fd = ok ? (float)((double)nc * o.px + (double)nd * o.pd) : ND_F;  // flowhand.py:840-843
    ix = ok ? (IDX)idx : (IDX)ND_I;
    TD h = HandOps<TD>::nd();
    float g = ND_F;
    if (want_h && ok && !HandOps<TD>::is_nd(z)) {  // flowhand.py:436-438
        h = HandOps<TD>::sub(z, zr);
        if (h < (TD)0 && h != HandOps<TD>::nd()) h = (TD)0;
        if (want_g && !(h <= HandOps<TD>::nd())) {  // gfi.py:289-294
            g = (float)(l1 - fast_log_pos((double)h + 0.01));
            HandOps<TD>::fix_nonfinite(g, h);
        }
    }
    hd = h;
    gf = g;
}

template <typename TD, typename IDX, typename ACC, bool TABLE>
__device__ __forceinline__ void hand_tile_body(const int tile, const TileView &v, const RiverSrc &rs, const TD *__restrict__ dem,
                                               const ACC *__restrict__ acc, const unsigned long long *__restrict__ nstate,
                                               const uint16_t *__restrict__ table, const HandOut &o)
{
    // TABLE: the successor table the fused finish pass of flowacc.cu left behind (one 16-bit entry per cell in
    // cell order: [15 river | 14 diagonal move | 13..0 successor slot / W_EXIT / W_TERM]) replaces staging the
    // codes, reading the river source and decoding the moves again.
    __shared__ __align__(16) uint8_t codes[TABLE ? 16 : (T + 2) * CP + 16];
    // in-tile state, slot layout of tiles.cuh: x = target (slot of the next cell while ACTIVE, global index of the
    // river cell, perimeter slot of the exit cell), y = [31..30 kind | 29..15 n_diag | 14..0 n_card]
    __shared__ uint2 st[TCELLS];
    // what lies behind each exit cell of the perimeter: resolved once per slot, shared by every cell that
    // leaves the tile through it (kind/moves, global river index, river elevation, ln b + n ln(A_r s^2))
    __shared__ uint32_t exit_hi[SLOTS];
    __shared__ IDX exit_idx[SLOTS];
    __shared__ TD exit_z[SLOTS];
    __shared__ double exit_l1[SLOTS];
    const int tid = threadIdx.x;
    const int ty = tile / v.tiles_x, tx = tile - ty * v.tiles_x;
    const int64_t r0 = (int64_t)ty * T, c0 = (int64_t)tx * T;
    const int lr = tid >> 2, lcb = (tid & 3) * CPT;
    bool fast;
    unsigned myriv = 0;
    if (TABLE) {
        fast = (v.cols % 16 == 0) && (c0 + T <= v.cols);
    } else {
        fast = stage_codes(v, r0, c0, codes, tid, H_THREADS);
        myriv = river_bits<ACC>(rs, v, r0, c0, lr, lcb, fast);
        __syncthreads();
    }
    auto C = [&](int r, int c) -> unsigned {
        if (TABLE) return fetch_code(v, r0 + r, c0 + c);
        return codes[(r + 1) * CP + 16 + c];
    };

    // ---- initial state of my 16 cells ----
    // Inside the tile a path is at most 4095 moves, so the two 15-bit counters never carry and composing
    // "s then t" is one 32-bit add (s is ACTIVE = kind 0) plus taking t's target.
    unsigned activemask = 0;
    if (TABLE) {
        const uint4 *tp = reinterpret_cast<const uint4 *>(table + (size_t)tile * TCELLS + tid * CPT);
        const uint4 ta = __ldg(tp), tb = __ldg(tp + 1);
        const uint32_t tw[8] = {ta.x, ta.y, ta.z, ta.w, tb.x, tb.y, tb.z, tb.w};
#pragma unroll
        for (int i = 0; i < CPT; ++i) {
            const uint32_t e = (tw[i >> 1] >> (16 * (i & 1))) & 0xFFFFu, n = e & 0x3FFFu;
            uint2 s = make_uint2(0u, (uint32_t)KIND_FAIL << 30);  // W_TERM: code 0, unknown code, bad landing
            if (e & 0x8000u) s = make_uint2((uint32_t)((r0 + lr) * v.cols + c0 + lcb + i), (uint32_t)KIND_RIVER << 30);
            else if (n == 0x3FFEu) s = make_uint2((uint32_t)slot_of(lr, lcb + i), (uint32_t)KIND_EXIT << 30);
            else if (n != 0x3FFFu) {  // 0x3FFF: terminal (valid outlet, or nodata when bit 14 is set)
                s = make_uint2(n, (e & 0x4000u) ? (1u << 15) : 1u);
                activemask |= 1u << i;
            }
            st[i * H_THREADS + tid] = s;
        }
    } else {
        const uint8_t *crow = codes + (lr + 1) * CP + 16 + lcb;
        const uint4 cw = *reinterpret_cast<const uint4 *>(crow);
        const uint32_t cws[4] = {cw.x, cw.y, cw.z, cw.w};
#pragma unroll
        for (int i = 0; i < CPT; ++i) {
            const int lc = lcb + i, p = lr * T + lc;
            const unsigned code = (cws[i >> 2] >> (8 * (i & 3))) & 0xFFu;
            uint2 s = make_uint2(0u, (uint32_t)KIND_FAIL << 30);  // code 0 (flowhand.py:601), unknown code, bad landing
            int dloc, dcode;
            if ((myriv >> i) & 1u) {
                if (code != 0) s = make_uint2((uint32_t)((r0 + lr) * v.cols + c0 + lc), (uint32_t)KIND_RIVER << 30);  // flowhand.py:609-612
            } else if (d8_delta(code, dloc, dcode)) {
                if (crow[i + dcode] != 0) {  // landing cell valid (flowhand.py:623-764, 826)
                    if (code & exit_codes(lr, lc)) {
                        s = make_uint2((uint32_t)slot_of(lr, lc), (uint32_t)KIND_EXIT << 30);  // x = perimeter slot; the exit move is added with the node state
                    } else {
                        s = make_uint2(phys_of((uint32_t)(p + dloc)), (code & 0xAAu) ? (1u << 15) : 1u);
                        activemask |= 1u << i;
                    }
                }
            }
            st[i * H_THREADS + tid] = s;
        }
    }
    __syncthreads();

    // ---- in-tile pointer jumping (in place, asynchronous) ----
    // A field reaching 2^14 means the cell sits on / drains into an in-tile cycle (a simple path has < 4096
    // moves): FAIL (flowhand.py:830/835).  Checking before every add keeps the 15-bit fields from carrying.
    constexpr uint32_t CYC = 0x20004000u;
    for (int round = 0; round < 16; ++round) {
#pragma unroll
        for (int i = 0; i < CPT; ++i) {
            if (!((activemask >> i) & 1u)) continue;
            uint2 s = st[i * H_THREADS + tid];
            uint2 t = st[s.x];
            s.x = t.x;
            s.y += t.y;
            if ((s.y >> 30) == 0u && !(s.y & CYC)) {
                t = st[s.x];
                s.x = t.x;
                s.y += t.y;
            }
            if ((s.y >> 30) == 0u && (s.y & CYC)) s.y = (uint32_t)KIND_FAIL << 30;
            st[i * H_THREADS + tid] = s;
            if (s.y >> 30) activemask &= ~(1u << i);
        }
        if (!__syncthreads_or(activemask != 0)) break;
    }

    // ---- resolved state behind every exit cell of the perimeter ----
    if (tid < USED_SLOTS) {
        int plr, plc;
        slot_cell(tid, plr, plc);
        int dr = 0, dc = 0;
        bool is_exit;
        if (TABLE) {
            is_exit = (__ldg(table + (size_t)tile * TCELLS + plr * T + plc) & 0xBFFFu) == 0x3FFEu;  // W_EXIT, not a river cell
            if (is_exit) d8_offset(C(plr, plc), dr, dc);
        } else {
            is_exit = d8_offset(C(plr, plc), dr, dc) &&
                      ((unsigned)(plr + dr) >= (unsigned)T || (unsigned)(plc + dc) >= (unsigned)T) && C(plr + dr, plc + dc) != 0;
        }
        const unsigned code = is_exit ? C(plr, plc) : 0u;
        resolve_exit<TD, IDX, ACC>(v, r0, c0, tid, plr, plc, is_exit, code, dr, dc, dem, acc, nstate, o, exit_hi, exit_idx, exit_z, exit_l1);
    }
    __syncthreads();

    // ---- epilogue: idx, flow distance, HAND, GFI for my 16 cells ----
    const int64_t gr = r0 + lr;
    if (gr >= v.rows) return;
    const bool vec = fast && (((reinterpret_cast<uintptr_t>(dem) | reinterpret_cast<uintptr_t>(o.fdist) |
                                reinterpret_cast<uintptr_t>(o.idx) | reinterpret_cast<uintptr_t>(o.hand) |
                                reinterpret_cast<uintptr_t>(o.gfi)) & 15u) == 0);
#pragma unroll 1
    for (int g4 = 0; g4 < CPT; g4 += 4) {
        const int64_t c_first = c0 + lcb + g4, obase = gr * v.cols + c_first;
        alignas(16) TD z[4];
        alignas(16) float fd[4], gf[4];
        alignas(16) IDX ix[4];
        alignas(16) TD hd[4];
        if (o.hand || o.gfi) load4<TD>(dem + obase, z, vec, c_first, v.cols, HandOps<TD>::nd());
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint2 s2 = st[(g4 + i) * H_THREADS + tid];
            uint32_t kind = s2.y >> 30, nd = (s2.y >> 15) & 0x7FFFu, nc = s2.y & 0x7FFFu;
            int64_t idx = (int64_t)ND_I;
            TD zr = (TD)0;
            double l1 = 0.0;
            if (kind == KIND_EXIT) {  // continue with the resolved path behind the tile's exit cell
                const uint32_t eh = exit_hi[s2.x];
                kind = eh >> 30;
                nd += (eh >> 15) & 0x7FFFu;
                nc += eh & 0x7FFFu;
                if (kind == KIND_RIVER) { idx = exit_idx[s2.x]; zr = exit_z[s2.x]; l1 = exit_l1[s2.x]; }
            } else if (kind == KIND_RIVER) {  // river cell inside this tile: s2.x = its local index in the band
                idx = (int64_t)s2.x + o.idx_offset;
                if (o.hand || o.gfi) zr = dem[s2.x];
                if (o.gfi) l1 = (o.gfi_n == 0.0 ? o.gfi_logb : o.gfi_logb + o.gfi_n * fast_log((double)acc[s2.x] * o.gfi_s2));  // gfi.py:141-143
            }
            finish_cell<TD, IDX>(o, o.hand || o.gfi, o.gfi != nullptr, kind, nd, nc, idx, zr, l1, z[i], fd[i], ix[i], hd[i], gf[i]);
        }
        if (o.fdist) store4<float>(o.fdist + obase, fd, vec, c_first, v.cols);
        if (o.idx) store4<IDX>(reinterpret_cast<IDX *>(o.idx) + obase, ix, vec, c_first, v.cols);
        if (o.hand) store4<TD>(reinterpret_cast<TD *>(o.hand) + obase, hd, vec, c_first, v.cols);
        if (o.gfi) store4<float>(o.gfi + obase, gf, vec, c_first, v.cols);
    }
}

// tiles == nullptr: one CTA per tile of the grid; otherwise the CTAs share the *ntiles tiles listed (the tiles the
// compact pass below had to give up on)
template <typename TD, typename IDX, typename ACC, bool TABLE>
__global__ void __launch_bounds__(H_THREADS)
hand_tile_kernel(TileView v, RiverSrc rs, const TD *__restrict__ dem, const ACC *__restrict__ acc,
                 const unsigned long long *__restrict__ nstate, const uint16_t *__restrict__ table, HandOut o,
                 const unsigned *__restrict__ tiles, const unsigned *__restrict__ ntiles)
{
    if (!tiles) {
        hand_tile_body<TD, IDX, ACC, TABLE>((int)blockIdx.x, v, rs, dem, acc, nstate, table, o);
        return;
    }
    const unsigned n = *ntiles;
    for (unsigned k = blockIdx.x; k < n; k += gridDim.x) {
        hand_tile_body<TD, IDX, ACC, TABLE>((int)tiles[k], v, rs, dem, acc, nstate, table, o);
        __syncthreads();
    }
}

// ---- H3, compact form (over the successor table): one 32-bit word per cell -----------------------------------
//     [31 root | 30 target is a root | 29 guard | 28..21 diagonal moves | 20 guard | 19..12 cardinal moves | 11..0 target]
// (target = a cell of the tile, slot layout).  A root (river cell, exit cell, dead end) points at itself and keeps
// its kind in bits 30..29 (KIND_*) and, for an exit cell, its perimeter slot in bits 19..12.  Composing "s then t"
// is s = (s & ~0xFFF) + t, which also hands t's "target is a root" flag to s: a cell is done when that flag is set.
// Half the shared-memory traffic of the 64-bit form above -- this stage is bound by shared-memory wavefronts -- at
// the price of 8-bit counters: a tile with an in-tile path of 256 or more moves of one kind (or an in-tile cycle)
// is handed to the 64-bit kernel through a list.
constexpr uint32_t C_ROOT = 0x80000000u, C_FLAG = 0x40000000u, C_GUARDS = (1u << 29) | (1u << 20), C_CARD = 1u << 12, C_DIAG = 1u << 21;
constexpr int OVF_SLOT = 32;  // word of the workspace header that counts the listed tiles

// Shared-memory position of a state word.  On top of the slot layout of tiles.cuh (cell p at (p % 16) * 256 + p / 16:
// conflict-free when thread t works on cell 16 t + i) bits 4..3 are XORed with bits 3..2 of the cell number, which
// keeps that property and also makes "lane l works on cell 4 l + k of a 128-cell span" conflict-free -- the
// epilogue's mapping, where a warp reads and writes whole 256-byte raster rows.  An involution.
__device__ __forceinline__ uint32_t swz(uint32_t q) { return q ^ (((q >> 10) & 3u) << 3); }

#ifndef H3C_MINB
#define H3C_MINB 6
#endif
// ALL: every output raster is wanted (the chain) -- spares the per-cell tests of the output pointers
template <typename TD, typename IDX, typename ACC, bool ALL>
__global__ void __launch_bounds__(H_THREADS, H3C_MINB)
hand_tile_compact_kernel(TileView v, const TD *__restrict__ dem, const ACC *__restrict__ acc,
                         const unsigned long long *__restrict__ nstate, const uint16_t *__restrict__ table, HandOut o,
                         unsigned *__restrict__ ovf_tiles, unsigned *__restrict__ ovf_count)
{
    __shared__ uint32_t st[TCELLS];
    __shared__ ExitRec<TD, IDX> exits[SLOTS];
    const int tid = threadIdx.x;
    const int tile = blockIdx.x;
    const int ty = tile / v.tiles_x, tx = tile - ty * v.tiles_x;
    const int64_t r0 = (int64_t)ty * T, c0 = (int64_t)tx * T;
    const int lr = tid >> 2, lcb = (tid & 3) * CPT;
    const bool fast = (v.cols % 16 == 0) && (c0 + T <= v.cols);
    const bool w_fd = ALL || o.fdist, w_ix = ALL || o.idx, w_hd = ALL || o.hand, w_gf = ALL || o.gfi;

    {
        const uint4 *tp = reinterpret_cast<const uint4 *>(table + (size_t)tile * TCELLS + tid * CPT);
        const uint4 ta = __ldg(tp), tb = __ldg(tp + 1);
        const uint32_t tw[8] = {ta.x, ta.y, ta.z, ta.w, tb.x, tb.y, tb.z, tb.w};
        // perimeter slot of my cells (tiles.cuh slot_of, with the per-thread part hoisted): on the first / last row of
        // the tile every cell has one, elsewhere only column 0 (my cell 0) and column T-1 (my cell 15) do
        const bool rowedge = lr == 0 || lr == T - 1;
        const uint32_t slot_row = (uint32_t)(lr == T - 1 ? T + lcb : lcb);
        const uint32_t slot_first = rowedge ? slot_row : (uint32_t)(2 * T + lr - 1);
        const uint32_t slot_last = rowedge ? slot_row + 15u : (uint32_t)(2 * T + (T - 2) + lr - 1);
#pragma unroll
        for (int i = 0; i < CPT; ++i) {
            const uint32_t e = (tw[i >> 1] >> (16 * (i & 1))) & 0xFFFFu, n = e & 0x3FFFu;
            const uint32_t self = swz((uint32_t)(i * H_THREADS + tid));
            const uint32_t slot = i == 0 ? slot_first : (i == CPT - 1 ? slot_last : slot_row + (uint32_t)i);
            // W_TERM: dead end (code 0, unknown code, bad landing); W_EXIT: leaves the tile; bit 15: river cell
            uint32_t s = C_ROOT | self | (n == 0x3FFEu ? ((uint32_t)KIND_EXIT << 29) | (slot << 12) : (uint32_t)KIND_FAIL << 29);
            if (e & 0x8000u) s = C_ROOT | ((uint32_t)KIND_RIVER << 29) | self;
            else if (n < 0x3FFEu) s = ((e & 0x4000u) ? C_DIAG : C_CARD) | swz(n);
            st[self] = s;
        }
    }
    __syncthreads();

    // ---- in-tile pointer jumping (in place, asynchronous) ----
    // Two hops per visit.  A cell is done when its word says "root" or "target is a root"; a guard bit means 256
    // moves of one kind or more: not representable here, the tile is listed (whatever its cells hold by then).
    uint32_t over = 0;
    for (int round = 0; round < 16; ++round) {
        uint32_t all = ~0u;  // AND of the words seen this round: bit 30 / 31 survive iff every cell is done
#pragma unroll
        for (int i = 0; i < CPT; ++i) {
            const uint32_t me = swz((uint32_t)(i * H_THREADS + tid));
            uint32_t s = st[me];
            if (s & (C_ROOT | C_FLAG)) continue;
            const uint32_t t1 = st[s & 0xFFFu];
            s = (t1 & C_ROOT) ? (s | C_FLAG) : ((s & ~0xFFFu) + t1);
            const uint32_t t2 = st[s & 0xFFFu];
            if (!(s & (C_FLAG | C_GUARDS))) s = (t2 & C_ROOT) ? (s | C_FLAG) : ((s & ~0xFFFu) + t2);
            st[me] = s;
            over |= s;
            all &= s;
        }
        if (!__syncthreads_or(!(all & C_FLAG) && !(over & C_GUARDS))) break;
    }
    if (__syncthreads_or((over & C_GUARDS) != 0u)) {
        if (tid == 0) ovf_tiles[atomicAdd(ovf_count, 1u)] = (unsigned)tile;
        return;
    }

    // ---- resolved state behind every exit cell of the perimeter ----
    if (tid < USED_SLOTS) {
        int plr, plc;
        slot_cell(tid, plr, plc);
        const uint32_t w = st[swz(phys_of((uint32_t)(plr * T + plc)))];
        const bool is_exit = (w >> 29) == (4u | (uint32_t)KIND_EXIT);
        int dr = 0, dc = 0;
        unsigned code = 0;
        if (is_exit) {
            code = fetch_code(v, r0 + plr, c0 + plc);
            d8_offset(code, dr, dc);
        }
        resolve_exit<TD, IDX, ACC>(v, r0, c0, tid, plr, plc, is_exit, code, dr, dc, dem, acc, nstate, o, exits);
    }
    __syncthreads();

    // ---- epilogue: idx, flow distance, HAND, GFI ----
    // A warp takes two 64-cell rows per pass (lane l: 4 cells at column 4 (l % 16)), so every load / store
    // instruction covers whole 128-byte lines.
    const bool vec = fast && (((reinterpret_cast<uintptr_t>(dem) | reinterpret_cast<uintptr_t>(o.fdist) |
                                reinterpret_cast<uintptr_t>(o.idx) | reinterpret_cast<uintptr_t>(o.hand) |
                                reinterpret_cast<uintptr_t>(o.gfi)) & 15u) == 0);
    const int ecol = 4 * (tid & 15);
#pragma unroll 1
    for (int pass = 0; pass < 4; ++pass) {
        const int erow = 8 * (tid >> 5) + 2 * pass + ((tid >> 4) & 1);
        const int64_t gr = r0 + erow;
        if (gr >= v.rows) continue;
        const int64_t c_first = c0 + ecol, obase = gr * v.cols + c_first;
        const uint32_t p = (uint32_t)(erow * T + ecol);
        alignas(16) TD z[4];
        alignas(16) float fd[4], gf[4];
        alignas(16) IDX ix[4];
        alignas(16) TD hd[4];
        if (w_hd || w_gf) load4<TD>(dem + obase, z, vec, c_first, v.cols, HandOps<TD>::nd());
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t s = st[swz((((p & 15u) + i) << 8) | (p >> 4))];
            uint32_t r = s, nd = 0, nc = 0;
            if (!(s & C_ROOT)) {
                r = st[s & 0xFFFu];
                nd = (s >> 21) & 0xFFu;
                nc = (s >> 12) & 0xFFu;
            }
            uint32_t kind = (r >> 29) & 3u;
            int64_t idx = (int64_t)ND_I;
            TD zr = (TD)0;
            double l1 = 0.0;
            if (kind == KIND_EXIT) {  // continue with the resolved path behind the tile's exit cell
                const ExitRec<TD, IDX> x = exits[(r >> 12) & 0xFFu];  // (idx, z, l1 only meaningful for a river)
                kind = x.hi >> 30;
                nd += (x.hi >> 15) & 0x7FFFu;
                nc += x.hi & 0x7FFFu;
                idx = x.idx;
                zr = x.z;
                l1 = x.l1;
            } else if (kind == KIND_RIVER) {  // river cell inside this tile
                const uint32_t rp = logical_of(swz(r & 0xFFFu));
                const int64_t loc = (r0 + (int64_t)(rp >> 6)) * v.cols + c0 + (int64_t)(rp & 63u);
                idx = loc + o.idx_offset;
                if (w_hd || w_gf) zr = dem[loc];
                if (w_gf) l1 = (o.gfi_n == 0.0 ? o.gfi_logb : o.gfi_logb + o.gfi_n * fast_log((double)acc[loc] * o.gfi_s2));  // gfi.py:141-143
            }
            finish_cell<TD, IDX>(o, w_hd || w_gf, w_gf, kind, nd, nc, idx, zr, l1, z[i], fd[i], ix[i], hd[i], gf[i]);
        }
        if (w_fd) store4<float>(o.fdist + obase, fd, vec, c_first, v.cols);
        if (w_ix) store4<IDX>(reinterpret_cast<IDX *>(o.idx) + obase, ix, vec, c_first, v.cols);
        if (w_hd) store4<TD>(reinterpret_cast<TD *>(o.hand) + obase, hd, vec, c_first, v.cols);
        if (w_gf) store4<float>(o.gfi + obase, gf, vec, c_first, v.cols);
    }
}

// ---- band summary: the path that starts at each boundary-row cell fed by the halo row ----
template <typename TD, typename ACC>
__global__ void __launch_bounds__(H_THREADS)
hand_band_summary_kernel(TileView v, int side, const unsigned long long *__restrict__ nstate, const TD *__restrict__ dem,
                         const ACC *__restrict__ acc, int64_t idx_offset, unsigned long long *__restrict__ sum_state,
                         int64_t *__restrict__ sum_idx, double *__restrict__ sum_z, int64_t *__restrict__ sum_acc)
{
    const int64_t c = (int64_t)blockIdx.x * H_THREADS + threadIdx.x;
    if (c >= v.cols) return;
    const int64_t r = side ? v.rows - 1 : 0, hr = side ? v.rows : -1;
    uint64_t s = 0ull;
    int64_t gi = ND_I, ga = 0;
    double gz = 0.0;
    if (v.d8[r * v.cols + c] != 0) {
        const bool fed = side ? (fetch_code(v, hr, c - 1) == 128u || fetch_code(v, hr, c) == 64u || fetch_code(v, hr, c + 1) == 32u)
                              : (fetch_code(v, hr, c - 1) == 2u || fetch_code(v, hr, c) == 4u || fetch_code(v, hr, c + 1) == 8u);
        if (fed) {
            s = nstate[node_of_cell(r, c, v.tiles_x)];
            if (kind_of(s) == KIND_ACTIVE) s = pack(KIND_FAIL, 0, 0, 0);  // unresolved inside the band: cycle / cap
            if (kind_of(s) == KIND_RIVER) {
                const int64_t p = (int64_t)ptr_of(s);
                gi = p + idx_offset;
                if (dem) gz = (double)dem[p];
                if (acc) ga = (int64_t)acc[p];
            }
        }
    }
    sum_state[c] = s;
    sum_idx[c] = gi;
    sum_z[c] = gz;
    sum_acc[c] = ga;
}

template <typename T, typename IDX>
__global__ void __launch_bounds__(H_THREADS)
hand_from_index_kernel(const T *__restrict__ dem, const IDX *__restrict__ idx, int64_t n, T *__restrict__ hand, int32_t *__restrict__ oob)
{
    const int64_t p = (int64_t)blockIdx.x * H_THREADS + threadIdx.x;
    if (p >= n) return;
    int64_t i = (int64_t)idx[p];
    bool ok = i != ND_I;      // -100 is masked out (flowhand.py:436)
    if (ok && i < 0) i += n;  // numpy fancy indexing wraps negative indices
    if (ok && (i < 0 || i >= n)) {  // an IndexError in the reference: never dereferenced here
        if (oob) *oob = 1;
        ok = false;
    }
    hand[p] = hand_value<T>(dem[p], ok, dem, ok ? i : 0);
}

// ---- band boundary graph (multi-GPU): what lies behind the halo rows of every band -------------------
// Node (b, side, c) = cell c of the first (side 0) / last (side 1) row of band b, with the summary state
// hand_band_summary_kernel left for it: RIVER / FAIL, or EXIT = "leaves band b towards side t of column col", i.e.
// continues at node (b -+ 1, other side, col).  Same in-place asynchronous pointer jumping as H2; a resolved node
// carries in its pointer field the node whose payload (river index, elevation, accumulation) it ends on.
__global__ void __launch_bounds__(H_THREADS)
hb_init_kernel(const long long *__restrict__ summ, int64_t n, int64_t cols, unsigned long long *__restrict__ w,
               unsigned *__restrict__ active)
{
    const int64_t node = (int64_t)blockIdx.x * H_THREADS + threadIdx.x;
    int live = 0;
    if (node < 2 * n * cols) {
        const int64_t b = node / (2 * cols), rem = node - b * 2 * cols, side = rem / cols, c = rem - side * cols;
        const uint64_t st = (uint64_t)summ[(b * 8 + side * 4) * cols + c];
        uint64_t s = pack(KIND_FAIL, nd_of(st), nc_of(st), (uint32_t)node);  // 0 = not an entry (never referenced)
        if (st != 0ull && kind_of(st) == KIND_RIVER) s = pack(KIND_RIVER, nd_of(st), nc_of(st), (uint32_t)node);
        else if (st != 0ull && kind_of(st) == KIND_EXIT) {
            const int64_t t_side = (ptr_of(st) >> 30) & 1u, t_col = ptr_of(st) & 0x3FFFFFFFu;
            const int64_t b2 = t_side ? b + 1 : b - 1;
            if (b2 >= 0 && b2 < n && t_col < cols) {
                s = pack(KIND_EXIT, nd_of(st), nc_of(st), (uint32_t)((b2 * 2 + (1 - t_side)) * cols + t_col));
                live = 1;
            }
        }
        w[node] = s;
    }
    const unsigned ballot = __ballot_sync(0xffffffffu, live);
    if ((threadIdx.x & 31) == 0 && ballot) atomicAdd(&active[0], (unsigned)__popc(ballot));
}

__global__ void __launch_bounds__(H_THREADS)
hb_jump_kernel(int64_t nnodes, unsigned long long *w, unsigned *__restrict__ active, int rnd)
{
    if (active[rnd - 1] == 0) return;
    unsigned still = 0;
    for (int64_t q = (int64_t)blockIdx.x * H_THREADS + threadIdx.x; q < nnodes; q += (int64_t)gridDim.x * H_THREADS) {
        uint64_t s = __ldcg(&w[q]);
        if (kind_of(s) != KIND_EXIT) continue;
        for (int j = 0; j < 2 && kind_of(s) == KIND_EXIT; ++j) {
            const uint64_t t = __ldcg(&w[ptr_of(s)]);
            s = pack(kind_of(t), sat_add(nd_of(s), nd_of(t)), sat_add(nc_of(s), nc_of(t)), ptr_of(t));
        }
        __stcg(&w[q], s);
        still += kind_of(s) == KIND_EXIT;
    }
    still = __reduce_add_sync(0xffffffffu, still);
    if ((threadIdx.x & 31) == 0 && still) atomicAdd(&active[rnd], still);
}

__global__ void __launch_bounds__(H_THREADS)
hb_out_kernel(const long long *__restrict__ summ, int64_t n, int64_t cols, const unsigned long long *__restrict__ w,
              long long *__restrict__ res, int *__restrict__ flag)
{
    const int64_t i = (int64_t)blockIdx.x * H_THREADS + threadIdx.x;
    if (i >= 2 * n * cols) return;
    const int64_t b = i / (2 * cols), rem = i - b * 2 * cols, out = rem / cols, c = rem - out * cols;  // out 0: above, 1: below
    const int64_t nb = out ? b + 1 : b - 1;
    long long v[4] = {(long long)pack(KIND_FAIL, 0, 0, 0), 0, 0, 0};
    if (nb >= 0 && nb < n) {
        uint64_t s = w[(nb * 2 + (1 - out)) * cols + c];  // above band b = last row of band b-1; below = first row of band b+1
        if (kind_of(s) == KIND_EXIT) {  // still travelling: a cycle across seams, or more seam crossings than the rounds cover
            s = pack(KIND_FAIL, nd_of(s), nc_of(s), ptr_of(s));
            *flag = 1;
        }
        const int64_t src = (int64_t)ptr_of(s), sb = src / (2 * cols), srem = src - sb * 2 * cols, ss = srem / cols, sc = srem - ss * cols;
        v[0] = (long long)(s & ~0xFFFFFFFFull);
#pragma unroll
        for (int k = 1; k < 4; ++k) v[k] = summ[(sb * 8 + ss * 4 + k) * cols + sc];
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) res[(b * 8 + out * 4 + k) * cols + c] = v[k];
}

// A launch in which every thread composes `jumps` times multiplies the hops every ACTIVE state covers by at least
// jumps + 1 (each composed state covers at least what the shortest state covered when the launch began), so
// ceil(log_{jumps+1}(max_moves + 1)) launches decide every node that max_moves moves can decide.
inline int node_jumps()
{
    static const int j = [] {
        const char *e = getenv("DTB_NODE_JUMPS");  // measurement aid
        const int v = e ? atoi(e) : 0;
        return v >= 1 && v <= 16 ? v : 2;  // measured at 40k x 40k (profiles/r2z_node_jumps.txt): 2 is the fastest
    }();
    return j;
}
inline int rounds_for(int64_t max_moves, int jumps)
{
    int r = 0;
    for (double cover = 1.0; cover < (double)max_moves + 1.0; cover *= jumps + 1) ++r;
    return r;
}

template <typename TD, typename IDX, typename ACC>
int run_tiles(const dtb_hand_args *a, const TileView &v, const RiverSrc &rs, const unsigned long long *nstate, int64_t tiles,
              uint32_t max_moves, cudaStream_t st)
{
    HandOut o;
    o.fdist = a->fdist;
    o.idx = a->idx;
    o.hand = a->hand;
    o.gfi = a->gfi;
    o.px = a->px;
    o.pd = a->px * sqrt(2.0);
    o.max_moves = max_moves;
    o.gfi_logb = log(a->gfi_b);
    o.gfi_n = a->gfi_n;
    o.gfi_s2 = a->gfi_size * a->gfi_size;
    o.idx_offset = 0;
    for (int k = 0; k < 2; ++k) { o.res_state[k] = nullptr; o.res_idx[k] = nullptr; o.res_z[k] = nullptr; o.res_acc[k] = nullptr; }
    if (a->band) {
        o.idx_offset = a->band->row_offset * a->cols;
        const dtb_hand_seam *sm[2] = {&a->band->above, &a->band->below};
        for (int k = 0; k < 2; ++k) {
            o.res_state[k] = reinterpret_cast<const unsigned long long *>(sm[k]->res_state);
            o.res_idx[k] = sm[k]->res_idx;
            o.res_z[k] = sm[k]->res_z;
            o.res_acc[k] = sm[k]->res_acc;
        }
    }
    // the successor table of the fused finish pass sits behind the node states in the workspace
    const uint16_t *table = reinterpret_cast<const uint16_t *>(nstate + tiles * SLOTS);
    if (a->entry_done) {
        // compact pass over every tile, then the 64-bit pass over the few tiles it could not represent
        unsigned *ovf_count = reinterpret_cast<unsigned *>(const_cast<unsigned long long *>(nstate)) - 64 + OVF_SLOT;
        unsigned *ovf_tiles = reinterpret_cast<unsigned *>(const_cast<uint16_t *>(table) + tiles * TCELLS);
        DTB_CUDA(cudaMemsetAsync(ovf_count, 0, sizeof(unsigned), st));
        if (a->fdist && a->idx && a->hand && a->gfi)
            DTB_KERNEL("hand_tile_kernel<table>", st, hand_tile_compact_kernel<TD, IDX, ACC, true><<<(unsigned)tiles, H_THREADS, 0, st>>>(
                           v, (const TD *)a->dem, (const ACC *)a->acc, nstate, table, o, ovf_tiles, ovf_count));
        else
            DTB_KERNEL("hand_tile_kernel<table>", st, hand_tile_compact_kernel<TD, IDX, ACC, false><<<(unsigned)tiles, H_THREADS, 0, st>>>(
                           v, (const TD *)a->dem, (const ACC *)a->acc, nstate, table, o, ovf_tiles, ovf_count));
        const unsigned grid = (unsigned)(tiles < kNumSMs * 4 ? tiles : kNumSMs * 4);
        DTB_KERNEL("hand_tile_kernel<listed>", st, hand_tile_kernel<TD, IDX, ACC, true><<<grid, H_THREADS, 0, st>>>(
                       v, rs, (const TD *)a->dem, (const ACC *)a->acc, nstate, table, o, ovf_tiles, ovf_count));
    } else
        DTB_KERNEL("hand_tile_kernel", st, hand_tile_kernel<TD, IDX, ACC, false><<<(unsigned)tiles, H_THREADS, 0, st>>>(
                       v, rs, (const TD *)a->dem, (const ACC *)a->acc, nstate, nullptr, o, nullptr, nullptr));
    return DTB_OK;
}

template <typename TD, typename IDX>
int run_tiles_acc(const dtb_hand_args *a, const TileView &v, const RiverSrc &rs, const unsigned long long *ns, int64_t tiles,
                  uint32_t mm, cudaStream_t st)
{
    return a->acc_dtype == DTB_I64 ? run_tiles<TD, IDX, int64_t>(a, v, rs, ns, tiles, mm, st)
                                   : run_tiles<TD, IDX, int32_t>(a, v, rs, ns, tiles, mm, st);
}

template <typename TD>
int run_tiles_idx(const dtb_hand_args *a, const TileView &v, const RiverSrc &rs, const unsigned long long *ns, int64_t tiles,
                  uint32_t mm, cudaStream_t st)
{
    return a->idx_dtype == DTB_I64 ? run_tiles_acc<TD, int64_t>(a, v, rs, ns, tiles, mm, st)
                                   : run_tiles_acc<TD, int32_t>(a, v, rs, ns, tiles, mm, st);
}

}  // namespace
}  // namespace dtb

extern "C" size_t dtb_hand_workspace_bytes(int64_t rows, int64_t cols)
{
    if (rows <= 0 || cols <= 0) return 0;
    const int64_t tiles = ((rows + dtb::T - 1) / dtb::T) * ((cols + dtb::T - 1) / dtb::T);
    // node states + the per-cell successor table of the fused flow-accumulation finish pass (flowacc.cu)
    // + the list of tiles the compact tile pass hands to the 64-bit one
    return 256 + (size_t)tiles * dtb::SLOTS * 8 + (size_t)tiles * dtb::TCELLS * 2 + (size_t)tiles * 4;
}

extern "C" int dtb_hand(const dtb_hand_args *a, void *ws, size_t ws_bytes, void *stream)
{
    using namespace dtb;
    if (!a || !a->fdr || !ws || a->rows <= 0 || a->cols <= 0 || !(a->px > 0.0)) return DTB_ERR_INVALID;
    if (!a->river && !a->acc) return DTB_ERR_INVALID;
    if ((a->hand || a->gfi) && !a->dem) return DTB_ERR_INVALID;
    if (a->gfi && !a->acc) return DTB_ERR_INVALID;
    if (a->dem_dtype != DTB_F32 && a->dem_dtype != DTB_I16) return DTB_ERR_INVALID;
    if (ws_bytes < dtb_hand_workspace_bytes(a->rows, a->cols)) return DTB_ERR_WORKSPACE;
    const int64_t n = a->rows * a->cols;
    if (n > 0xffffffffLL) return DTB_ERR_UNSUPPORTED;  // 32-bit targets: shard larger rasters into bands
    if (a->idx && a->idx_dtype == DTB_I32 && n > 0x7fffffffLL) return DTB_ERR_UNSUPPORTED;
    const int64_t max_moves = a->max_moves > 0 ? a->max_moves : 20000;  // flowhand.py:835
    if (max_moves > 32000) return DTB_ERR_UNSUPPORTED;
    cudaStream_t st = as_stream(stream);
    unsigned *active = reinterpret_cast<unsigned *>(ws);
    unsigned long long *nstate = reinterpret_cast<unsigned long long *>((char *)ws + 256);
    const dtb_hand_band *band = a->band;
    const int mode = band ? band->mode : DTB_HAND_FULL;
    if (mode < DTB_HAND_FULL || mode > DTB_HAND_FINISH) return DTB_ERR_INVALID;
    if (band && band->below.halo && a->rows % T != 0) return DTB_ERR_INVALID;  // band seams sit on tile seams
    TileView v{a->fdr, band ? band->above.halo : nullptr, band ? band->below.halo : nullptr, a->rows, a->cols,
               (int)((a->cols + T - 1) / T)};
    const int64_t tiles = (int64_t)v.tiles_x * ((a->rows + T - 1) / T);
    const int64_t nnodes = tiles * SLOTS;
    if (nnodes >= (int64_t)1 << 30) return DTB_ERR_UNSUPPORTED;
    RiverSrc rs{a->river, a->acc, a->river_threshold};

    if (a->entry_done && a->river) return DTB_ERR_INVALID;  // the fused entry pass knows only acc > threshold
    if (mode != DTB_HAND_FINISH) {
        if (!a->entry_done) {
            DTB_CUDA(cudaMemsetAsync(active, 0, 256, st));
            DTB_KERNEL("hand_entry_kernel", st, {
                if (a->acc_dtype == DTB_I64) hand_entry_kernel<int64_t><<<(unsigned)tiles, H_THREADS, 0, st>>>(v, rs, nstate, active);
                else hand_entry_kernel<int32_t><<<(unsigned)tiles, H_THREADS, 0, st>>>(v, rs, nstate, active);
            });
        }
        const int jumps = node_jumps(), rounds = rounds_for(max_moves, jumps);
        for (int r = 1; r <= rounds; ++r) {
            DTB_KERNEL("hand_node_jump_kernel", st, hand_node_jump_kernel<<<JUMP_BLOCKS, H_THREADS, 0, st>>>(nnodes, nstate, active, r, jumps));
        }
    }
    if (mode == DTB_HAND_SUMMARY) {
        const unsigned nbc = (unsigned)((a->cols + H_THREADS - 1) / H_THREADS);
        const int64_t off = band->row_offset * a->cols;
        const dtb_hand_seam *sm[2] = {&band->above, &band->below};
        for (int side = 0; side < 2; ++side) {
            const dtb_hand_seam *q = sm[side];
            if (!q->sum_state) continue;
            if (!q->sum_idx || !q->sum_z || !q->sum_acc) return DTB_ERR_INVALID;
            unsigned long long *ss = reinterpret_cast<unsigned long long *>(q->sum_state);
#define DTB_SUMMARY(TD, ACC)                                                                                            \
    hand_band_summary_kernel<TD, ACC><<<nbc, H_THREADS, 0, st>>>(v, side, nstate, (const TD *)a->dem, (const ACC *)a->acc, off, \
                                                                 ss, q->sum_idx, q->sum_z, q->sum_acc)
            if (a->dem_dtype == DTB_I16) { if (a->acc_dtype == DTB_I64) DTB_SUMMARY(int16_t, int64_t); else DTB_SUMMARY(int16_t, int32_t); }
            else { if (a->acc_dtype == DTB_I64) DTB_SUMMARY(float, int64_t); else DTB_SUMMARY(float, int32_t); }
#undef DTB_SUMMARY
            DTB_LAUNCH_CHECK("hand_band_summary_kernel");
        }
        return DTB_OK;
    }
    if (!a->fdist && !a->idx && !a->hand && !a->gfi) return DTB_OK;
    return a->dem_dtype == DTB_I16 ? run_tiles_idx<int16_t>(a, v, rs, nstate, tiles, (uint32_t)max_moves, st)
                                   : run_tiles_idx<float>(a, v, rs, nstate, tiles, (uint32_t)max_moves, st);
}

extern "C" int dtb_hand_from_index(const void *dem, int dem_dtype, const void *idx, int idx_dtype, int64_t n, void *hand,
                                   int32_t *oob, void *stream)
{
    using namespace dtb;
    if (!dem || !idx || !hand || n < 0) return DTB_ERR_INVALID;
    if (n == 0) return DTB_OK;
    cudaStream_t st = as_stream(stream);
    const unsigned blocks = (unsigned)((n + H_THREADS - 1) / H_THREADS);
    if (dem_dtype == DTB_F32 && idx_dtype == DTB_I64)
        hand_from_index_kernel<float, int64_t><<<blocks, H_THREADS, 0, st>>>((const float *)dem, (const int64_t *)idx, n, (float *)hand, oob);
    else if (dem_dtype == DTB_F32 && idx_dtype == DTB_I32)
        hand_from_index_kernel<float, int32_t><<<blocks, H_THREADS, 0, st>>>((const float *)dem, (const int32_t *)idx, n, (float *)hand, oob);
    else if (dem_dtype == DTB_I16 && idx_dtype == DTB_I64)
        hand_from_index_kernel<int16_t, int64_t><<<blocks, H_THREADS, 0, st>>>((const int16_t *)dem, (const int64_t *)idx, n, (int16_t *)hand, oob);
    else if (dem_dtype == DTB_I16 && idx_dtype == DTB_I32)
        hand_from_index_kernel<int16_t, int32_t><<<blocks, H_THREADS, 0, st>>>((const int16_t *)dem, (const int32_t *)idx, n, (int16_t *)hand, oob);
    else
        return DTB_ERR_INVALID;
    DTB_LAUNCH_CHECK("hand_from_index_kernel");
    return DTB_OK;
}

extern "C" size_t dtb_hand_boundary_workspace_bytes(int64_t nbands, int64_t cols)
{
    if (nbands <= 0 || cols <= 0) return 0;
    return 256 + (size_t)(2 * nbands * cols) * 8;
}

extern "C" int dtb_hand_boundary_solve(const int64_t *summ, int64_t nbands, int64_t cols, int rounds, int64_t *res,
                                       int *unresolved, void *ws, size_t ws_bytes, void *stream)
{
    using namespace dtb;
    if (!summ || !res || !unresolved || !ws || nbands <= 0 || cols <= 0 || rounds < 1 || rounds > 32) return DTB_ERR_INVALID;
    if (cols >= (int64_t)1 << 30 || 2 * nbands * cols > 0xffffffffLL) return DTB_ERR_UNSUPPORTED;
    if (ws_bytes < dtb_hand_boundary_workspace_bytes(nbands, cols)) return DTB_ERR_WORKSPACE;
    cudaStream_t st = as_stream(stream);
    unsigned *active = reinterpret_cast<unsigned *>(ws);
    unsigned long long *w = reinterpret_cast<unsigned long long *>((char *)ws + 256);
    const int64_t nn = 2 * nbands * cols;
    const unsigned blocks = (unsigned)((nn + H_THREADS - 1) / H_THREADS);
    DTB_CUDA(cudaMemsetAsync(active, 0, 256, st));
    DTB_CUDA(cudaMemsetAsync(unresolved, 0, sizeof(int), st));
    DTB_KERNEL("hb_init_kernel", st, hb_init_kernel<<<blocks, H_THREADS, 0, st>>>(reinterpret_cast<const long long *>(summ), nbands, cols, w, active));
    const unsigned jb = blocks < (unsigned)JUMP_BLOCKS ? blocks : (unsigned)JUMP_BLOCKS;
    for (int r = 1; r <= rounds; ++r)
        DTB_KERNEL("hb_jump_kernel", st, hb_jump_kernel<<<jb, H_THREADS, 0, st>>>(nn, w, active, r));
    DTB_KERNEL("hb_out_kernel", st, hb_out_kernel<<<blocks, H_THREADS, 0, st>>>(reinterpret_cast<const long long *>(summ), nbands, cols, w,
                                                                             reinterpret_cast<long long *>(res), unresolved));
    return DTB_OK;
}
