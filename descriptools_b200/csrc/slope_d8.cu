// slope_d8.cu -- fused slope (%) + D8 flow direction, one 3x3 stencil pass.
//
// Semantics: slope.py:228-259 (slope_gpu) with the -100 padding ring of slope.py:175-182
// replaced by "off-raster neighbours are skipped"; D8 per SURVEY.md App. A2 (direction of
// the neighbour that last raised the running maximum in scan order NW,N,NE,W,E,SW,S,SE;
// outlets point at their first undefined neighbour).  Bit-exact against oracle/dt_oracle.c.
//
// B200 design: persistent CTAs (3 per SM) draw 128x32-cell tiles from an atomic counter in
// row-major order; each tile plus its halo (a 136x34 f32 box starting 4 columns left of the
// tile: the TMA unit faults unless the box's innermost start coordinate is 16-byte aligned --
// measured on B200, scripts/tma_probe.cu) is staged in shared memory by TMA
// (cp.async.bulk.tensor.2d, out-of-bounds elements filled with NaN, which stands in for the
// reference's -100 padding ring) through a 3-stage ring of full / empty mbarriers: the eight
// warps of a CTA consume a tile independently, only the producer lane waits for "all warps
// are done with this stage" before it refills it, two tiles ahead.  With the arithmetic
// stubbed out this skeleton moves 9 B/cell at the measured HBM copy peak (0.137 ms for
// 10 000 x 10 000); the kernel is bound by instruction issue, so the strip below is written
// for instruction count and pipe balance (see "lean strip").  A thread owns 4 columns x 4
// rows and slides a 3-row register window down its strip: LDS.128 + 2 LDS.32 per row, results
// leave as one STG.128 (slope) and one STG.32 (four D8 codes) per row.
//
// Exactness without f64 in the hot loop (the reference divides in f64 inside the 8-neighbour
// loop, slope.py:249-257):
//   * within a class (cardinal / diagonal) the divisor is a common positive constant, so
//     comparing the f32 differences is equivalent to comparing the f64 gradients;
//   * slope = f32(f64(diff)/d*100) is bracketed by two fused multiply-adds with a two-term
//     f32 constant for 100/d; when both ends round to the same f32 that is the answer, else
//     the row goes to the literal f64 loop (slow_row);
//   * cardinal-vs-diagonal is decided on those exact f32 slopes (all roundings are monotone);
//     equal non-zero slopes go to slow_row.
#include <math.h>

#include <atomic>

#include "common.cuh"

namespace dtb {
namespace {

constexpr int TW = 128;           // tile width  (cells)
constexpr int TH = 32;            // tile height (cells)
constexpr int HALO_L = 4;         // staged columns start at c0-4 (TMA: 16-byte aligned box start)
constexpr int BOXW = TW + 8;      // staged columns c0-4 .. c0+TW+3
constexpr int BOXH = TH + 2;      // staged rows    r0-1 .. r0+TH
constexpr int NTHREADS = 256;     // 32 column groups x 8 row groups
constexpr int RPT = TH / 8;       // rows per thread
constexpr int STAGES = 3;
constexpr int STAGE_BYTES = ((BOXW * BOXH * 4 + 127) / 128) * 128;
constexpr int TMA_BYTES = BOXW * BOXH * 4;
constexpr size_t SMEM_TMA = (size_t)STAGES * STAGE_BYTES + 256;  // + full / empty barriers + tile ids

struct SlopeConsts {
    double px;   // cardinal step            (slope.py:250)
    double pd;   // px * sqrt(2.0)           (slope.py:255)
    float spacer;  // unused: keeps the floats below 4 bytes off 8-byte alignment; moved, they change the TMA kernel's register allocation
    float kc_hi, kc_lop, kc_lom, kd_hi, kd_lop, kd_lom;  // k = 100/px, 100/pd: k = k_hi + k_lo to 2^-48; k_lo+- = k_lo +- 2^-44 k
};

// ---- PTX wrappers ------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, int x, int y, uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(dst)),
        "l"(map), "r"(x), "r"(y), "r"(smem_u32(bar))
        : "memory");
}

// ---- output ------------------------------------------------------------------------------------
// One row of four cells: slopes s4 and D8 codes (one per byte) to the row pointers slope / d8 (nullptr: not wanted).
// VEC: one 16-byte and one 4-byte store (the TMA kernel: cols % 4 == 0, aligned outputs).  Otherwise cell by cell, and
// only the cells col .. cols-1 (col: raster column of the first cell; the ragged last group of a row has fewer than four).
// s4 and codes by reference: slow_row_store's copy then reads them from its stack only after the null tests.
template <bool VEC>
__device__ __forceinline__ void store_row4(float *slope, uint8_t *d8, const float4 &s4, const uint32_t &codes, int64_t col, int64_t cols)
{
    if (VEC) {
        if (slope) *reinterpret_cast<float4 *>(slope) = s4;
        if (d8) *reinterpret_cast<uint32_t *>(d8) = codes;
    } else {
        const float s[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
        for (int c = 0; c < 4; ++c)
            if (col + c < cols) {
                if (slope) slope[c] = s[c];
                if (d8) d8[c] = (uint8_t)(codes >> (8 * c));
            }
    }
}

// ---- the exact path ----------------------------------------------------------------------------
// Everything that is rare in the lean strip below -- a cell with no positive gradient next to an undefined value
// (outlet rule), a slope product within 2^-44 of an f32 rounding boundary, equal cardinal and diagonal slopes,
// sub-range values -- is delegated, one row of four cells at a time, to slow_row(): the literal per-neighbour
// loop of slope.py:244-258 over the staged raw values.
__device__ __noinline__ void slow_row(const float *tile, int trow, int tcol0, double px, double pd, float4 &slope4, uint32_t &codes)
{
    // trow/tcol0: position of the first of the four cells inside the staged box
    const int DR[8] = {-1, -1, -1, 0, 0, 1, 1, 1}, DC[8] = {-1, 0, 1, -1, 1, -1, 0, 1};
    const int CODE[8] = {32, 64, 128, 16, 1, 8, 4, 2};
    float out[4];
    codes = 0;
    for (int c = 0; c < 4; ++c) {
        const int tcol = tcol0 + c;
        const float zc = tile[trow * BOXW + tcol];
        if (zc <= ND_F) { out[c] = ND_F; continue; }  // slope.py:231 (a NaN centre is off-raster: never stored)
        double m = 0.0;
        int code = 0, first_undef = 0;
        for (int k = 0; k < 8; ++k) {
            const float zq = tile[(trow + DR[k]) * BOXW + tcol + DC[k]];
            const float diff = zc - zq;
            if (zq == ND_F || diff != diff) {  // skipped neighbour (slope.py:247) / off-raster
                if (!first_undef) first_undef = CODE[k];
                continue;
            }
            const double g = (double)diff / ((DR[k] == 0 || DC[k] == 0) ? px : pd);
            if (m < g) { m = g; code = CODE[k]; }  // slope.py:250,255
        }
        out[c] = (float)(m * 100.0);  // slope.py:259
        if (code == 0) code = first_undef;  // outlet rule, SURVEY.md App. A2
        codes |= (uint32_t)code << (8 * c);
    }
    slope4 = make_float4(out[0], out[1], out[2], out[3]);
}

// ---- lean strip (v2): packed f32x2 arithmetic, no f64, no conversions --------------------------------
// Issue-rate facts measured on B200 (scripts/pipe_probe.cu, profiles/r2b_pipe_probe.txt; clocks per warp
// instruction per SM sub-partition): FADD/FFMA 1, FADD2/FFMA2 2 (two results per issue slot), FMNMX3 / FSET /
// FSETP / FSEL / LOP3 / SHF / PRMT / IMAD 2, FLO 8, F2F (f32<->f64) 8.5.  The v1 strip spent 2 F2F + 1 FLO (25
// clocks of the XU pipe) and ~34 half-rate ALU instructions per cell.  v2, per PAIR of horizontally adjacent cells:
//   * the 8 elevation differences of both cells by 8 FADD2 (operands are register pairs: a row is held both as
//     cell-aligned pairs P and as the pairs M shifted by one column);
//   * class maxima by FMNMX3 (never NaN: an undefined neighbour -- off-raster NaN, NaN in the data -- is
//     skipped exactly like slope.py:247 skips -100);
//   * first maximum in scan order (strict '<', slope.py:250,255): l_k = [d_k != max] by FSET, then the index
//     of the first winner j = l0 (1 + l1 (1 + l2)) by two FFMA2 per class;
//   * slope of BOTH classes without f64: s+- = RN(a k_hi + RN(a k_lo+-)) (one FMUL2 + one FFMA2 each), where
//     k_hi + k_lo = 100/d to 2^-48 and k_lo+- = k_lo +- 2^-44 (100/d).  The fused multiply-add rounds the exact
//     sum once, so s- <= f32(f64(a)/d*100) <= s+ (the reference's three roundings move the real value by < 2^-50
//     relative, the bracket is 2^-44 wide); s+ == s- pins the result, otherwise the row takes the exact path
//     (about one cell in 10^6).  S = max(S_card, S_diag) (all roundings are monotone); cardinal wins iff
//     S_card > S_diag; S_card == S_diag > 0 cannot be decided in f32 and takes the exact path;
//   * no positive gradient (S == 0): q = 1 adds 8 to the cell's nibble, the byte permute below then yields code
//     0 (selector nibbles 8..15 replicate the sign bit of a table byte; the cardinal bytes have none), the
//     slope is +0; the outlet rule (first undefined neighbour) needs the exact path only if the window holds a
//     NaN, which is tested only for rows that have a pit;
//   * 0 < S < 2^-30 (where the products above could lose bits to underflow) makes q fractional; q (q - 1) != 0
//     is accumulated on the FMA pipe and tested once per row of four cells.
typedef unsigned long long p2;  // two packed f32 (an aligned register pair)
__device__ __forceinline__ p2 pk(float lo, float hi) { p2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void upk(p2 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ p2 add2(p2 a, p2 b) { p2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ p2 sub2(p2 a, p2 b) { p2 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ p2 mul2(p2 a, p2 b) { p2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ p2 fma2(p2 a, p2 b, p2 c) { p2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ float max3(float a, float b, float c) { float r; asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c)); return r; }
__device__ __forceinline__ float min3(float a, float b, float c) { float r; asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c)); return r; }
__device__ __forceinline__ float set_neu(float a, float b) { float r; asm("set.neu.f32.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float fma_sat(float a, float b, float c) { float r; asm("fma.rn.sat.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c)); return r; }
__device__ __forceinline__ float mul_sat(float a, float b) { float r; asm("mul.sat.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ bool equ(float a, float b) { return !(a < b || a > b); }  // equal or unordered
__device__ __forceinline__ float lds_f32(uint32_t addr)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}

struct Row2 {
    float w[6];  // w[1..4]: the thread's four cells (one LDS.128: aligned register pairs), w[0], w[5]: the halo columns
};

// lo: running minimum of everything the strip has loaded (NaN ignored): <= -100 means nodata somewhere in it
__device__ __forceinline__ void load_row2(uint32_t a /* shared address of the thread's first cell */, Row2 &r, float &lo)
{
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.w[1]), "=f"(r.w[2]), "=f"(r.w[3]), "=f"(r.w[4]) : "r"(a));
    r.w[0] = lds_f32(a - 4);
    r.w[5] = lds_f32(a + 16);
    lo = min3(min3(min3(lo, r.w[0], r.w[1]), r.w[2], r.w[3]), r.w[4], r.w[5]);
}

struct FastK {
    p2 kc_hi, kc_lop, kc_lom, kd_hi, kd_lop, kd_lom;  // 100/px and 100/(px sqrt2): f32 hi, and lo +- 2^-44 k
    p2 one, four, neg8, w256;
};

__device__ __forceinline__ FastK fast_k(const SlopeConsts &c)
{
    FastK k;
    k.kc_hi = pk(c.kc_hi, c.kc_hi); k.kc_lop = pk(c.kc_lop, c.kc_lop); k.kc_lom = pk(c.kc_lom, c.kc_lom);
    k.kd_hi = pk(c.kd_hi, c.kd_hi); k.kd_lop = pk(c.kd_lop, c.kd_lop); k.kd_lom = pk(c.kd_lom, c.kd_lom);
    k.one = pk(1.0f, 1.0f); k.four = pk(4.0f, 4.0f); k.neg8 = pk(-8.0f, -8.0f); k.w256 = pk(256.0f, 256.0f);
    return k;
}

// one pair of horizontally adjacent cells: columns j, j+1 (1 or 3) of the window rows U (above), M, D (below);
// H[t] = M.w[t] - M.w[t+1]: the horizontal differences of the centre row, each used by both of its cells.
// Only the vertical differences are packed (their operands are the aligned pairs of the LDS.128 results); the
// shifted directions would need copies into new register pairs, which cost more issue slots than scalar FADDs.
// (Sharing the vertical / diagonal differences between consecutive rows as well was measured: the 12 carried
// registers spill at 80 registers per thread and cost more than the 11 FADDs per row they save.)
// N accumulates the two cells' selector nibbles (lane 0: even cell, lane 1: odd cell), scaled by W (1 or 256).
template <int W, bool CX>
__device__ __forceinline__ void cell_pair2(const Row2 &U, const Row2 &M, const Row2 &D, const float (&H)[5], const int j, const FastK &k,
                                           float &Sa, float &Sb, p2 &N, p2 &acc, bool &redo)
{
    float nA, nB, sA, sB;
    const p2 C = pk(M.w[j], M.w[j + 1]);
    upk(sub2(C, pk(U.w[j], U.w[j + 1])), nA, nB);
    upk(sub2(C, pk(D.w[j], D.w[j + 1])), sA, sB);
    const float cA = M.w[j], cB = M.w[j + 1];
    const float wA = -H[j - 1], wB = -H[j], eA = H[j], eB = H[j + 1];
    const float nwA = cA - U.w[j - 1], nwB = cB - U.w[j], neA = cA - U.w[j + 1], neB = cB - U.w[j + 2];
    const float swA = cA - D.w[j - 1], swB = cB - D.w[j], seA = cA - D.w[j + 1], seB = cB - D.w[j + 2];
    // class maxima, floor 0 (slope.py:244: m starts at 0); NaN differences are ignored by FMNMX
    const float acA = max3(max3(nA, wA, eA), sA, 0.0f), acB = max3(max3(nB, wB, eB), sB, 0.0f);
    const float adA = max3(max3(nwA, neA, swA), seA, 0.0f), adB = max3(max3(nwB, neB, swB), seB, 0.0f);
    // losers among the first three of each class in scan order (N,W,E,[S]) / (NW,NE,SW,[SE]); NaN loses
    const p2 lN = pk(set_neu(nA, acA), set_neu(nB, acB)), lW = pk(set_neu(wA, acA), set_neu(wB, acB)),
             lE = pk(set_neu(eA, acA), set_neu(eB, acB));
    const p2 lNW = pk(set_neu(nwA, adA), set_neu(nwB, adB)), lNE = pk(set_neu(neA, adA), set_neu(neB, adB)),
             lSW = pk(set_neu(swA, adA), set_neu(swB, adB));
    const p2 jc = fma2(lN, fma2(lW, lE, lW), lN);                      // 0..3 = N W E S
    const p2 jd4 = add2(fma2(lNW, fma2(lNE, lSW, lNE), lNW), k.four);  // 4..7 = NW NE SW SE
    // slope bracket of both classes
    const p2 ac = pk(acA, acB), ad = pk(adA, adB);
    float cpA, cpB, cmA, cmB, dpA, dpB, dmA, dmB;
    if (CX) {
        // 100/px is a power of two (px = 12.5, 25, 50, ...): a * (100/px) is exact in f32, and f32(f64(a)/px*100) is that
        // number (the reference's two f64 roundings move it by < 2^-51 relative, far inside half an f32 ulp)
        upk(mul2(ac, k.kc_hi), cpA, cpB);
        cmA = cpA;
        cmB = cpB;
    } else {
        upk(fma2(ac, k.kc_hi, mul2(ac, k.kc_lop)), cpA, cpB);
        upk(fma2(ac, k.kc_hi, mul2(ac, k.kc_lom)), cmA, cmB);
    }
    upk(fma2(ad, k.kd_hi, mul2(ad, k.kd_lop)), dpA, dpB);
    upk(fma2(ad, k.kd_hi, mul2(ad, k.kd_lom)), dmA, dmB);
    if (CX) redo |= (dpA != dmA) | (dpB != dmB);  // the cardinal product is one correctly rounded multiplication, like the reference's
    else redo |= (cpA != cmA) | (cpB != cmB) | (dpA != dmA) | (dpB != dmB);               // rounding in doubt (or NaN / inf)
    Sa = fmaxf(cpA, dpA);
    Sb = fmaxf(cpB, dpB);
    // p = [positive gradient] = sat(S 2^100): exactly 0 iff S == 0, exactly 1 iff S >= 2^-100, fractional in between (the
    // sub-range where the products above lose bits to underflow: exact path) -- accumulate p (p - 1) <= 0, exactly 0 for
    // p in {0, 1} (nothing is absorbed, unlike (acc + p^2) - p)
    const p2 pp = pk(mul_sat(Sa, 1.2676506e30f), mul_sat(Sb, 1.2676506e30f));
    const p2 pm1 = sub2(pp, k.one);
    acc = fma2(pp, pm1, acc);
    // class: u = [S_card >= S_diag]; undecidable here: S_card == S_diag > 0 (z == 0 and p == 1), and both infinite (z NaN)
    float zA, zB, mA, mB;
    upk(sub2(pk(cpA, cpB), pk(dpA, dpB)), zA, zB);
    upk(pm1, mA, mB);
    redo |= equ(zA, mA) | equ(zB, mB);
    const p2 u = pk(fma_sat(zA, 8.507059e37f, 1.0f), fma_sat(zB, 8.507059e37f, 1.0f));
    // selector nibble - 8: -8..-1 for a direction, 0..3 for a pit (the strip adds the 8 back: 8..11 select "code 0")
    const p2 m = fma2(pp, k.neg8, fma2(u, sub2(jc, jd4), jd4));
    if (W == 1) N = add2(N, m);
    else N = fma2(m, k.w256, N);
}

// the exact path for one row of four cells, stored straight to the outputs
template <bool VEC>
__device__ __noinline__ void slow_row_store(const float *tile, int trow, int tcol0, double px, double pd, float *slope, uint8_t *d8,
                                            int64_t col, int64_t cols)
{
    float4 s4;
    uint32_t codes;
    slow_row(tile, trow, tcol0, px, pd, s4, codes);
    store_row4<VEC>(slope, d8, s4, codes, col, cols);
}

// One row of four cells, given the three window rows.  Returns true when the exact path has to redo the row.
template <bool CX>
__device__ __forceinline__ bool fast_row2(const Row2 &U, const Row2 &M, const Row2 &D, const FastK &k, float4 &s4, uint32_t &codes,
                                          uint32_t &sel)
{
    float H[5];
#pragma unroll
    for (int t = 0; t <= 4; ++t) H[t] = M.w[t] - M.w[t + 1];
    p2 N = pk(0.0f, 0.0f), acc = pk(0.0f, 0.0f);
    bool redo = false;
    cell_pair2<1, CX>(U, M, D, H, 1, k, s4.x, s4.y, N, acc, redo);
    cell_pair2<256, CX>(U, M, D, H, 3, k, s4.z, s4.w, N, acc, redo);
    float n0, n1, a0, a1;
    upk(N, n0, n1);
    upk(acc, a0, a1);
    // 2^23 + sum of nibble_c 16^c (the 8 every cell_pair2 left out: 0x8888): the low mantissa bits are the byte-permute selector
    sel = __float_as_uint(fmaf(n1, 16.0f, n0 + (8388608.0f + 34952.0f)));
    // selector nibble 0..7 picks a table byte; 8..11 (a pit) replicates the sign bit of a cardinal byte = 0.
    // (PTX prmt; CUDA's __byte_perm masks the nibbles to three bits.)
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(codes) : "r"(0x04011040u), "r"(0x02088020u), "r"(sel));  // S E W N | SE SW NE NW
    return redo | !(a0 + a1 == 0.0f);
}

// a pit's code is its first undefined neighbour (SURVEY.md App. A2): does the window hold a NaN (off-raster, NaN in
// the data, nodata rewritten by robust_row_store)?
__device__ __forceinline__ bool window_has_nan(const Row2 &U, const Row2 &M, const Row2 &D)
{
    float x = 0.0f;
#pragma unroll
    for (int t = 0; t < 6; ++t) x += (U.w[t] + M.w[t]) + D.w[t];
    return !(x == x);
}

// A row whose window holds nodata (<= -100).  Values equal to -100 are rewritten as NaN, which the fast arithmetic
// skips exactly like the reference skips a -100 neighbour (slope.py:247: FMNMX ignores NaN, FSET.NEU makes it a
// loser); values below -100 stay what they are for their neighbours (the reference does not skip them either);
// nodata centres (<= -100, slope.py:231) get slope -100, code 0.  Only what is still undecided (a pit next to an
// undefined neighbour, a rounding in doubt) goes on to the exact path.
template <bool VEC>
__device__ __noinline__ void robust_row_store(const float *tile, int trow, int tcol0, SlopeConsts kk, float *slope, uint8_t *d8,
                                              int64_t col, int64_t cols)
{
    const FastK k = fast_k(kk);
    const float qnan = __int_as_float(0x7fc00000);
    Row2 R[3];
    unsigned nd = 0;
#pragma unroll
    for (int j = 0; j < 3; ++j)
#pragma unroll
        for (int t = 0; t < 6; ++t) {
            const float v = tile[(trow - 1 + j) * BOXW + tcol0 - 1 + t];
            if (j == 1 && t >= 1 && t <= 4 && v <= ND_F) nd |= 1u << (t - 1);
            R[j].w[t] = v == ND_F ? qnan : v;
        }
    float4 s4 = make_float4(ND_F, ND_F, ND_F, ND_F);
    uint32_t codes = 0, sel = 0;
    bool redo = false;
    if (nd != 15u) {
        redo = fast_row2<false>(R[0], R[1], R[2], k, s4, codes, sel);
        if (nd & 1u) { s4.x = ND_F; codes &= 0xFFFFFF00u; sel &= ~0x000Fu; }
        if (nd & 2u) { s4.y = ND_F; codes &= 0xFFFF00FFu; sel &= ~0x00F0u; }
        if (nd & 4u) { s4.z = ND_F; codes &= 0xFF00FFFFu; sel &= ~0x0F00u; }
        if (nd & 8u) { s4.w = ND_F; codes &= 0x00FFFFFFu; sel &= ~0xF000u; }
        if (!redo && (sel & 0x8888u)) redo = window_has_nan(R[0], R[1], R[2]);
    }
    if (redo) slow_row_store<VEC>(tile, trow, tcol0, kk.px, kk.pd, slope, d8, col, cols);
    else store_row4<VEC>(slope, d8, s4, codes, col, cols);
}

// 4 columns x RPT rows of one staged tile.  sbase / dbase: the outputs; off: element offset of the strip's first
// cell; col: its raster column; nrows: how many of the strip's rows are inside the output (0..RPT).
// WS / WD: the output is wanted.  VEC: the stores of store_row4; with VEC = false a null output base is also skipped.
template <bool WS, bool WD, bool CX, bool VEC>
__device__ __forceinline__ void stencil_strip_v2(const float *tile, int gx, int ry0, const SlopeConsts &kk, const FastK &k,
                                                 float *__restrict__ sbase, uint8_t *__restrict__ dbase, int64_t off, int64_t col,
                                                 int64_t cols, int nrows)
{
    const bool ws = WS && (VEC || sbase), wd = WD && (VEC || dbase);
    const int tcol0 = 4 * gx + HALO_L;
    const uint32_t a = smem_u32(tile + ry0 * BOXW + tcol0);
    Row2 U, M, D;
    float lo = 3.0e38f;
    load_row2(a, U, lo);
    load_row2(a + BOXW * 4, M, lo);
    const int64_t off0 = off;
    unsigned later = 0;  // bit i: row i of the strip goes to the exact path (after the loop: keeps the calls out of it)
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
        load_row2(a + (2 + i) * BOXW * 4, D, lo);
        float4 s4;
        uint32_t codes, sel;
        bool redo = fast_row2<CX>(U, M, D, k, s4, codes, sel);
        if (i < nrows) store_row4<VEC>(ws ? sbase + off : nullptr, wd ? dbase + off : nullptr, s4, codes, col, cols);
#ifdef DTB_DEBUG_FORCE_REDO
        redo = true;
#endif
        if (!redo && (sel & 0x8888u)) redo = window_has_nan(U, M, D);
        if (redo) later |= 1u << i;
        off += cols;
        U = M;
        M = D;
    }
    // Nodata (<= -100, slope.py:231,247) anywhere in the 6 x 6 values this strip has seen: what the loop stored for it is
    // discarded and every row is redone by the nodata path (one test per strip instead of one per row; nodata comes in
    // blobs, and the lean arithmetic cannot fault on it).
    const bool nodata = lo <= ND_F;
    if (nodata) later = 0xFu;
    later &= (1u << nrows) - 1u;
    if (later) {
#pragma unroll 1
        for (int i = 0; i < RPT; ++i) {
            if (!(later >> i & 1u)) continue;
            float *sp = ws ? sbase + off0 + i * cols : nullptr;
            uint8_t *dp = wd ? dbase + off0 + i * cols : nullptr;
            if (nodata) robust_row_store<VEC>(tile, ry0 + 1 + i, tcol0, kk, sp, dp, col, cols);
            else slow_row_store<VEC>(tile, ry0 + 1 + i, tcol0, kk.px, kk.pd, sp, dp, col, cols);
        }
    }
}

// ---- TMA persistent kernels (f32, cols % 4 == 0, 16-byte aligned bases) -----------------------------
// Tile scheduler state: one (next tile, CTAs done) pair per launch slot; the last CTA to run dry resets its slot.
__device__ unsigned int g_tile_sched[64][2];

// v2: warps consume tiles independently.  full[s]: the TMA load of stage s has landed (and tile_xy[s] is valid);
// empty[s]: all eight warps are done reading stage s.  Lane 0 of warp 0 is the producer: before its own strip of
// tile number `it` it refills the stage of tile it-1 (two tiles of look-ahead), so only that one warp ever waits
// for the others, and nobody at a CTA-wide barrier.  Tiles are handed out by an atomic counter (row-major order:
// the CTAs of the grid sweep the raster together, which keeps the DRAM pages and the L2 halo reuse local).
template <bool WS, bool WD, bool CX, int MINB>
__global__ void __launch_bounds__(NTHREADS, MINB)
slope_d8_tma2_kernel(const __grid_constant__ CUtensorMap dem_map, int64_t row_begin, int64_t row_end, int64_t cols, int tiles_x,
                     int ntiles, SlopeConsts k, float *__restrict__ slope, uint8_t *__restrict__ d8, int sched_slot)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    if ((smem_u32(smem) & 127u) != 0u) __trap();  // TMA destination alignment
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + (size_t)STAGES * STAGE_BYTES);
    uint64_t *empty = full + STAGES;
    int *tile_xy = reinterpret_cast<int *>(empty + STAGES);  // (tx, ty) per stage; tx < 0: no more tiles
    const int tid = threadIdx.x;
    unsigned int *sched = g_tile_sched[sched_slot];

    // producer only (tid 0): fetch the next tile, publish it in `stage`, start its load
    auto produce = [&](int stage) -> bool {
        const int tile = (int)atomicAdd(&sched[0], 1u);
        if (tile >= ntiles) {
            tile_xy[2 * stage] = -1;
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&full[stage])) : "memory");
            if (atomicAdd(&sched[1], 1u) == gridDim.x - 1) {  // every CTA has drawn its last ticket
                sched[0] = 0;
                sched[1] = 0;
            }
            return false;
        }
        const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
        tile_xy[2 * stage] = tx;
        tile_xy[2 * stage + 1] = ty;
        mbar_expect_tx(&full[stage], TMA_BYTES);
        tma_load_2d(smem + (size_t)stage * STAGE_BYTES, &dem_map, tx * TW - HALO_L, (int)(row_begin + (int64_t)ty * TH - 1), &full[stage]);
        return true;
    };

    bool more = true;
    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], NTHREADS / 32);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        for (int s = 0; s < STAGES && more; ++s) more = produce(s);
    }
    __syncthreads();

    const int gx = tid & 31, gy = tid >> 5;
    // the host launches each form with the outputs it writes: store_row4's null tests fold away
    if (WS) __builtin_assume(slope != nullptr);
    if (WD) __builtin_assume(d8 != nullptr);
    const FastK fk = fast_k(k);
    const int64_t out_rows = row_end - row_begin;

    for (int it = 0;; ++it) {
        const int stage = it % STAGES;
        mbar_wait(&full[stage], (uint32_t)(it / STAGES) & 1u);
        const int tx = tile_xy[2 * stage], ty = tile_xy[2 * stage + 1];
        if (tx < 0) break;
        if (tid == 0 && more && it >= 1) {  // refill the stage of the previous tile before computing this one: two tiles ahead
            const int ps = (it - 1) % STAGES;
            mbar_wait(&empty[ps], (uint32_t)((it - 1) / STAGES) & 1u);
            more = produce(ps);  // tile number it-1+STAGES
        }
        const float *tbuf = reinterpret_cast<const float *>(smem + (size_t)stage * STAGE_BYTES);
        const int64_t orow = (int64_t)ty * TH + gy * RPT, ocol = (int64_t)tx * TW + 4 * gx;
        const int64_t left = out_rows - orow;
        const int nrows = ocol < cols ? (left < RPT ? (left < 0 ? 0 : (int)left) : RPT) : 0;
        stencil_strip_v2<WS, WD, CX, true>(tbuf, gx, gy * RPT, k, fk, slope, d8, orow * cols + ocol, ocol, cols, nrows);
        __syncwarp();
        if (gx == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&empty[stage])) : "memory");
    }
}

// ---- generic kernel (any width / alignment, f32 or i16 DEM) --------------------------------
// One CTA per tile, staged by plain loads into the same box the TMA kernel stages (NaN off the raster), then the same
// strip with per-cell stores.  Either output may be null.
template <typename T, bool CX>
__global__ void __launch_bounds__(NTHREADS)
slope_d8_generic_kernel(const T *__restrict__ dem, int64_t buf_rows, int64_t row_begin, int64_t row_end, int64_t cols,
                        int tiles_x, SlopeConsts k, float *__restrict__ slope, uint8_t *__restrict__ d8)
{
    __shared__ __align__(16) float tile[BOXH * BOXW];
    const int tid = threadIdx.x;
    const int ty = blockIdx.x / tiles_x, tx = blockIdx.x - ty * tiles_x;
    const int64_t r0 = row_begin + (int64_t)ty * TH - 1, c0 = (int64_t)tx * TW - HALO_L;
    const float qnan = __int_as_float(0x7fc00000);
    for (int idx = tid; idx < BOXH * BOXW; idx += NTHREADS) {
        const int j = idx / BOXW, kk = idx - j * BOXW;
        const int64_t r = r0 + j, c = c0 + kk;
        float v = qnan;
        if (r >= 0 && r < buf_rows && c >= 0 && c < cols) v = (float)dem[r * cols + c];
        tile[idx] = v;
    }
    __syncthreads();
    const int gx = tid & 31, gy = tid >> 5;
    const int64_t orow = (int64_t)ty * TH + gy * RPT, ocol = (int64_t)tx * TW + 4 * gx;
    const int64_t left = (row_end - row_begin) - orow;
    const int nrows = ocol < cols ? (left < RPT ? (left < 0 ? 0 : (int)left) : RPT) : 0;
    stencil_strip_v2<true, true, CX, false>(tile, gx, gy * RPT, k, fast_k(k), slope, d8, orow * cols + ocol, ocol, cols, nrows);
}

// ---- tensor map (driver entry point fetched at run time: libdtb200 does not link libcuda) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn()
{
    static EncodeTiledFn fn = nullptr;
    if (fn) return fn;
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
        return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(p);
    return fn;
}

}  // namespace
}  // namespace dtb

extern "C" int dtb_slope_d8(const void *dem, int dem_dtype, int64_t buf_rows, int64_t cols, int64_t row_begin,
                            int64_t row_end, double px, float *slope, uint8_t *d8, void *stream)
{
    using namespace dtb;
    if (!dem || buf_rows <= 0 || cols <= 0 || row_begin < 0 || row_end > buf_rows || row_begin > row_end || !(px > 0.0))
        return DTB_ERR_INVALID;
    if (dem_dtype != DTB_F32 && dem_dtype != DTB_I16) return DTB_ERR_INVALID;
    if (row_begin == row_end || (!slope && !d8)) return DTB_OK;
    if (cols > (int64_t)1 << 30 || buf_rows > (int64_t)1 << 30) return DTB_ERR_UNSUPPORTED;
    cudaStream_t st = as_stream(stream);

    SlopeConsts k;
    k.px = px;
    k.pd = px * sqrt(2.0);
    const double kc = 100.0 / k.px, kd = 100.0 / k.pd;
    k.kc_hi = (float)kc;
    k.kc_lop = (float)(kc - (double)k.kc_hi + ldexp(kc, -44));
    k.kc_lom = (float)(kc - (double)k.kc_hi - ldexp(kc, -44));
    k.kd_hi = (float)kd;
    k.kd_lop = (float)(kd - (double)k.kd_hi + ldexp(kd, -44));
    k.kd_lom = (float)(kd - (double)k.kd_hi - ldexp(kd, -44));
    // 100/px a power of two: the cardinal slope product is exact (see cell_pair2)
    int e2 = 0;
    const bool cx = frexp(kc, &e2) == 0.5 && kc >= 1.0 / 1048576.0 && kc <= 1048576.0;

    const int64_t nrows = row_end - row_begin;
    const int tiles_x = (int)((cols + TW - 1) / TW);
    const int64_t tiles_y = (nrows + TH - 1) / TH;
    const int64_t ntiles64 = tiles_y * tiles_x;
    if (ntiles64 > 0x7fffffff) return DTB_ERR_UNSUPPORTED;
    const int ntiles = (int)ntiles64;

    const bool aligned = dem_dtype == DTB_F32 && (cols % 4 == 0) && (((uintptr_t)dem) % 16 == 0) &&
                         (!slope || ((uintptr_t)slope) % 16 == 0) && (!d8 || ((uintptr_t)d8) % 4 == 0);
    if (aligned) {
        EncodeTiledFn enc = get_encode_fn();
        if (!enc) return cuda_fail_msg("cuTensorMapEncodeTiled entry point not available");
        CUtensorMap map;
        const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)buf_rows};
        const cuuint64_t gstride[1] = {(cuuint64_t)cols * 4};
        const cuuint32_t box[2] = {BOXW, BOXH};
        const cuuint32_t estr[2] = {1, 1};
        const CUresult r = enc(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void *>(dem), gdim, gstride, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NAN_REQUEST_ZERO_FMA);
        if (r != CUDA_SUCCESS) return cuda_fail_msg("cuTensorMapEncodeTiled failed");
        static std::atomic<unsigned> slot_ctr{0};
        const int slot = (int)(slot_ctr.fetch_add(1) % 64u);
        const int per_sm = 3;  // 79 registers; 4 CTAs at 64 registers measured the same (profiles/r2p_stencil.txt)
        const int grid = ntiles < per_sm * kNumSMs ? ntiles : per_sm * kNumSMs;
#define DTB_LAUNCH_TMA2(WS, WD, CX, MINB)                                                                                              \
    do {                                                                                                                               \
        static bool attr = false;                                                                                                      \
        if (!attr) {                                                                                                                   \
            DTB_CUDA(cudaFuncSetAttribute(slope_d8_tma2_kernel<WS, WD, CX, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize,        \
                                          (int)SMEM_TMA));                                                                            \
            attr = true;                                                                                                               \
        }                                                                                                                              \
        DTB_KERNEL("slope_d8_tma_kernel", st, (slope_d8_tma2_kernel<WS, WD, CX, MINB><<<grid, NTHREADS, SMEM_TMA, st>>>(              \
                                                  map, row_begin, row_end, cols, tiles_x, ntiles, k, slope, d8, slot)));              \
    } while (0)
        if (slope && d8) {
            if (cx) DTB_LAUNCH_TMA2(true, true, true, 3);
            else DTB_LAUNCH_TMA2(true, true, false, 3);
        } else if (slope) {
            DTB_LAUNCH_TMA2(true, false, false, 3);
        } else {
            DTB_LAUNCH_TMA2(false, true, false, 3);
        }
#undef DTB_LAUNCH_TMA2
    } else {
#define DTB_LAUNCH_GENERIC(T, NAME)                                                                                                    \
    DTB_KERNEL(NAME, st, ((cx ? slope_d8_generic_kernel<T, true> : slope_d8_generic_kernel<T, false>)<<<ntiles, NTHREADS, 0, st>>>( \
                             (const T *)dem, buf_rows, row_begin, row_end, cols, tiles_x, k, slope, d8)))
        if (dem_dtype == DTB_F32) DTB_LAUNCH_GENERIC(float, "slope_d8_generic_kernel<f32>");
        else DTB_LAUNCH_GENERIC(int16_t, "slope_d8_generic_kernel<i16>");
#undef DTB_LAUNCH_GENERIC
    }
    return DTB_OK;
}
