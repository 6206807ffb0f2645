"""GFI, ln(hl/H), TI and MTI against the f64 oracle on every kernel instantiation and at the edges of the log form.

pointwise.cu evaluates log(b * pow(x, n) / y) as ln b + n ln x - ln y with short logarithms (common.cuh fast_log_pos,
|error| < 3e-9) where 1e-30 < b < 1e30, |n| <= 8 and both x and y lie in (1e-30, 1e30), and the reference's expression
elsewhere; the fused HAND tile pass (hand.cu) uses the same form.  Every finite result must be within the suite's
RTOL / ATOL and, tighter, within spacing(f32) + (|n| + 2) * 3e-9 of the oracle's; NaN and +-inf must sit where the
oracle has them.

Which kernel an input reaches follows from the launchers in pointwise.cu: the vector kernel (4 cells per thread and
pass) when every pointer is 16-byte aligned, the scalar kernel otherwise.  The vector kernel's grid is at most
148 * 16 CTAs of 256 threads, so it covers 4 * 606 208 = 2 424 832 cells per pass; a raster above that takes a second
grid-stride pass.  Its last n % 4 cells go through the scalar tail loop.
"""
import math
import zlib

import numpy as np
import pytest
import torch

import oracle
from helpers import ATOL, PX, RTOL, hand_fused_vs_oracle, misaligned, synth

pytestmark = pytest.mark.gpu

VEC_CELLS_PER_PASS = 4 * 148 * 16 * 256

# (name, shape): big is 16-byte aligned and needs two grid-stride passes of the vector kernel; tail is aligned with
# n % 4 == 3, so the vector kernel's scalar tail loop runs; misaligned is the tail shape in views that start one element
# into their buffers, which only the scalar kernel takes
LAYOUTS = {"big": (2000, 1500), "tail": (61, 67), "misaligned": (61, 67)}
assert 2000 * 1500 > VEC_CELLS_PER_PASS and (61 * 67) % 4 == 3

HAND_EDGES_F32 = [-100, -100.5, -250, 0, -0.005, -0.5, 1e29, 1e31, np.nan, np.inf, -np.inf, 0.3, 7.25, 120.0, -99.9]
HAND_EDGES_I16 = [-32768, -101, -100, -99, 32767, 0, 1, 3, 250, -1]
ACC_EDGES_I32 = [0, -100, -101, 1, 2**31 - 1, 7, 130000, 5]
ACC_EDGES_I64 = ACC_EDGES_I32 + [10**10, 4 * 10**18]
HALF_PI = np.float32(math.pi / 2)


def _seed(*key):
    return zlib.crc32(repr(key).encode())


def _acc_edges(dtype):
    return ACC_EDGES_I64 if dtype == np.int64 else ACC_EDGES_I32


def _slope_edges():
    """radians: -100 (nodata), 0, beta with beta + 0.01 just below / just above pi/2 (tan flips sign), NaN, ordinary"""
    below, above = np.float32(math.pi / 2 - 0.01 - 1e-6), np.float32(math.pi / 2 - 0.01 + 1e-6)
    assert float(below) + 0.01 < math.pi / 2 < float(above) + 0.01
    return np.array([-100, 0, below, above, np.nan, 0.05, 0.4, 1.2, HALF_PI], np.float32)


def _fill(n, edges, typical, rng):
    """n values: the edge values every 3rd cell (so they land in both grid-stride passes, the tail and every lane of a
    4-cell pack), random typical values between"""
    out = typical(n)
    e = np.asarray(edges, dtype=out.dtype)
    k = np.arange(0, n, 3)
    out[k] = e[(k // 3 + rng.integers(0, len(e))) % len(e)]
    out[-len(e):] = e  # the tail holds every edge as well
    return out


def _hand(n, dtype, rng):
    if dtype == np.int16:
        return _fill(n, HAND_EDGES_I16, lambda m: rng.integers(0, 400, m).astype(np.int16), rng)
    return _fill(n, HAND_EDGES_F32, lambda m: (rng.random(m) * 60).astype(np.float32), rng)


def _acc(n, dtype, rng):
    return _fill(n, _acc_edges(dtype), lambda m: rng.integers(0, 50000, m).astype(dtype), rng)


def _slope(n, rng):
    return _fill(n, _slope_edges(), lambda m: (rng.random(m) * 1.4).astype(np.float32), rng)


def _dev(a, layout):
    """device copy of a host array in the given layout, and the kernel form it reaches"""
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    if layout == "misaligned":
        t = misaligned(t)
    return t


def _kernel_form(*ts):
    """what the launcher picks: 'vector' if every pointer is 16-byte aligned, else 'scalar' (pointwise.cu aligned4)"""
    return "vector" if all(t.data_ptr() % 16 == 0 for t in ts) else "scalar"


def _expect_form(layout, ts):
    form = _kernel_form(*ts)
    assert form == ("scalar" if layout == "misaligned" else "vector"), (layout, form)
    n = ts[0].numel()
    if layout == "big":
        assert n > VEC_CELLS_PER_PASS  # a second grid-stride pass of the vector kernel
    if layout == "tail":
        assert n % 4 != 0  # the vector kernel's scalar tail loop


def _poison_like(n):
    """leave a freed block of n float32 cells filled with a value no index produces, so a cell a kernel fails to write
    cannot read as right by reusing an earlier correct output"""
    p = torch.full((n,), -12345.678, dtype=torch.float32, device="cuda")
    del p


def assert_log_close(got, want, n, what=""):
    """NaN / +-inf positions equal, finite values within RTOL / ATOL, and within the short logs' error bound"""
    got = np.asarray(got)
    want = np.asarray(want)
    assert got.dtype == np.float32 and want.dtype == np.float32
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=ATOL, err_msg=what)
    # past |log| = 708 the reference's quotient is subnormal (only the reference's expression gets there: the log form's
    # terms keep it above 1e-300), and two libms' pow may round it one subnormal step apart
    fin = np.isfinite(got) & np.isfinite(want) & (np.abs(want) < 708)
    g, w = got[fin].astype(np.float64), want[fin].astype(np.float64)
    bound = np.spacing(np.maximum(np.abs(got[fin]), np.abs(want[fin]))).astype(np.float64) + (abs(n) + 2) * 3e-9
    err = np.abs(g - w)
    bad = err > bound
    if bad.any():
        i = int(np.argmax(err - bound))
        raise AssertionError(f"{what}: {int(bad.sum())} cells beyond spacing + (|n|+2)*3e-9, worst got {g[i]!r} want {w[i]!r} "
                             f"|diff| {err[i]:.3e} bound {bound[i]:.3e}")


def _gfi_ref(kind, hand, acc, n, b, size):
    with np.errstate(all="ignore"):
        if kind == "gfi":
            return oracle.gfi(hand, acc.astype(np.int64), np.arange(hand.size).reshape(hand.shape), n, b, size)
        return oracle.ln_hl_H(hand, acc.astype(np.int64), n, b, size)


def _gfi_dev(kind, h, a, n, b, size):
    from descriptools_b200 import device

    _poison_like(h.numel())
    f = device.gfi if kind == "gfi" else device.ln_hl_H
    return f(h, a, n, b, size).cpu().numpy()


# ---- GFI / ln(hl/H): every instantiation x layout --------------------------------------------------------------------
@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("acc_dtype", [np.int32, np.int64], ids=["acc32", "acc64"])
@pytest.mark.parametrize("hand_dtype", [np.float32, np.int16], ids=["f32", "i16"])
@pytest.mark.parametrize("kind", ["gfi", "lnhlh"])
def test_gfi_lnhlh_instantiations(kind, hand_dtype, acc_dtype, layout):
    """dtb_gfi (river accumulation given) and dtb_lnhlh (own accumulation, A == 0 -> 1) for hand f32 / int16 x acc
    int32 / int64 on the vector kernel (two passes, tail) and the scalar kernel"""
    rng = np.random.default_rng(_seed(kind, layout, hand_dtype, acc_dtype))
    shape = LAYOUTS[layout]
    hand = _hand(shape[0] * shape[1], hand_dtype, rng).reshape(shape)
    acc = _acc(hand.size, acc_dtype, rng).reshape(shape)
    h, a = _dev(hand, layout), _dev(acc, layout)
    _expect_form(layout, [h, a])
    params = [(0.4, 0.1, PX), (-8.0, 1e-29, 0.5)] if layout == "big" else [(0.4, 0.1, PX), (0.0, 0.1, PX), (-0.4, 3.0, PX),
                                                                           (8.0, 1e-29, 0.5), (-8.0, 1e29, 2.0)]
    for n, b, size in params:
        want = _gfi_ref(kind, hand, acc, n, b, size)
        assert_log_close(_gfi_dev(kind, h, a, n, b, size), want, n, f"{kind} n={n} b={b} size={size}")


N_EDGES = [0.4, 0.0, -0.4, 8.0, -8.0, float(np.nextafter(8.0, 9.0)), float(np.nextafter(-8.0, -9.0))]
B_EDGES = [0.1, 1e-30, 1e30, float(np.nextafter(1e-30, 1)), float(np.nextafter(1e30, 0)), float(np.nextafter(1e-30, 0)),
           float(np.nextafter(1e30, 2e30)), 0.0]
SIZE_EDGES = [PX, 1e-20, 1e16]


@pytest.mark.parametrize("kind", ["gfi", "lnhlh"])
@pytest.mark.parametrize("n", N_EDGES)
def test_gfi_lnhlh_parameter_edges(kind, n):
    """both sides of the fast / reference boundary in every parameter: |n| = 8 and the next double, b at 1e-30 / 1e30
    and their neighbours, b = 0, size giving A size^2 below 1e-30 (1e-20) and above 1e30 (1e16)"""
    rng = np.random.default_rng(int(abs(n) * 1000) + (kind == "gfi"))
    shape = LAYOUTS["tail"]
    hand = _hand(shape[0] * shape[1], np.float32, rng).reshape(shape)
    acc = _acc(hand.size, np.int64, rng).reshape(shape)
    h, a = _dev(hand, "tail"), _dev(acc, "tail")
    for b in B_EDGES:
        for size in SIZE_EDGES:
            want = _gfi_ref(kind, hand, acc, n, b, size)
            assert_log_close(_gfi_dev(kind, h, a, n, b, size), want, n, f"{kind} n={n!r} b={b!r} size={size!r}")


@pytest.mark.parametrize("kind", ["gfi", "lnhlh"])
def test_gfi_pow_overflow_stays_infinite(kind):
    """n = 30 with accumulation 1e9: (A size^2)^n overflows in the reference's pow, so the result is +inf -- a log form
    that took |n| = 30 would return a finite ~776 instead"""
    shape = LAYOUTS["tail"]
    hand = np.full(shape, 5.0, np.float32)
    acc = np.full(shape, 10**9, np.int64)
    want = _gfi_ref(kind, hand, acc, 30.0, 0.1, PX)
    assert np.isposinf(want).all()
    for layout in ("tail", "misaligned"):
        h, a = _dev(hand, layout), _dev(acc, layout)
        assert_log_close(_gfi_dev(kind, h, a, 30.0, 0.1, PX), want, 30.0, f"{kind} {layout}")


@pytest.mark.parametrize("layout", ["tail", "misaligned"])
@pytest.mark.parametrize("kind", ["gfi", "lnhlh"])
def test_gfi_near_zero_tight_bound(kind, layout):
    """H = f32(b x^n - 0.01) per cell with n = 8: results lie within about +-1e-6 of zero, where the suite's ATOL is
    loose and spacing + (|n| + 2) * 3e-9 is what holds the short logarithms to their stated error"""
    rng = np.random.default_rng(8)
    n, b, size = 8.0, 0.1, 0.1
    shape = LAYOUTS[layout]
    acc = rng.integers(100, 1500, shape).astype(np.int64)  # x = A size^2 in [1, 15]: b x^8 in [0.1, 2.6e8]
    x = acc.astype(np.float64) * size * size
    hand = (b * x ** n - 0.01).astype(np.float32)
    want = _gfi_ref(kind, hand, acc, n, b, size)
    assert np.abs(want).max() < 0.25
    h, a = _dev(hand, layout), _dev(acc, layout)
    assert_log_close(_gfi_dev(kind, h, a, n, b, size), want, n, f"{kind} near zero")


# ---- TI / MTI ---------------------------------------------------------------------------------------------------------
def _ti_ref(acc, slope, px, n):
    with np.errstate(all="ignore"):
        return oracle.ti_mti(acc.astype(np.int64), slope, px, n)


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("outputs", ["both", "ti", "mti"])
@pytest.mark.parametrize("acc_dtype", [np.int32, np.int64], ids=["acc32", "acc64"])
def test_ti_mti_instantiations(acc_dtype, outputs, layout):
    """dtb_ti_mti for acc int32 / int64, asked for both outputs, TI only and MTI only, on every layout; the parameter
    sets include the reference's expression (px = 1e16 puts A px^2 above 1e30)"""
    from descriptools_b200 import device

    rng = np.random.default_rng(_seed(outputs, layout, acc_dtype))
    shape = LAYOUTS[layout]
    acc = _acc(shape[0] * shape[1], acc_dtype, rng).reshape(shape)
    slope = _slope(acc.size, rng).reshape(shape)
    a, s = _dev(acc, layout), _dev(slope, layout)
    _expect_form(layout, [a, s])
    want_ti, want_mti = outputs in ("both", "ti"), outputs in ("both", "mti")
    params = [(PX, 0.1), (1e16, 0.4)] if layout == "big" else [(PX, 0.1), (PX, 0.0), (PX, -8.0), (1e-20, 8.0), (1e16, 0.4),
                                                                  (PX, float(np.nextafter(8.0, 9.0))), (3.0, 30.0)]
    for px, n in params:
        ti_ref, mti_ref = _ti_ref(acc, slope, px, n)
        _poison_like(acc.size)
        ti, mti = device.ti_mti(a, s, px, n, want_ti=want_ti, want_mti=want_mti)
        assert (ti is None) != want_ti and (mti is None) != want_mti
        if want_ti:
            assert_log_close(ti.cpu().numpy(), ti_ref, 1.0, f"TI px={px} n={n}")
        if want_mti:
            assert_log_close(mti.cpu().numpy(), mti_ref, n, f"MTI px={px} n={n}")


# ---- river accumulation gather, slope to radians ----------------------------------------------------------------------
@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("idx_dtype", [np.int32, np.int64], ids=["idx32", "idx64"])
@pytest.mark.parametrize("acc_dtype", [np.int32, np.int64], ids=["acc32", "acc64"])
def test_river_accumulation_instantiations(acc_dtype, idx_dtype, layout):
    """dtb_river_accumulation, all four integer widths: -100 reads cell 0 (gfi.py:141-143), -1 and -n wrap like NumPy's
    flat indexing (last and first cell)"""
    from descriptools_b200 import device

    rng = np.random.default_rng(_seed(layout, acc_dtype, idx_dtype))
    shape = LAYOUTS[layout]
    n = shape[0] * shape[1]
    acc = _acc(n, acc_dtype, rng).reshape(shape)
    idx = rng.integers(0, n, n).astype(idx_dtype)
    k = np.arange(0, n, 5)
    idx[k] = np.array([-100, -1, -n], idx_dtype)[k % 3]
    idx[-3:] = [-100, -1, -n]
    idx = idx.reshape(shape)
    wrapped = np.where((idx < 0) & (idx != -100), idx.astype(np.int64) + n, idx)  # NumPy's rule, then the oracle's gather
    want = oracle.river_accumulation(acc.astype(np.int64), wrapped).astype(acc_dtype)
    a, i = _dev(acc, layout), _dev(idx, layout)
    got = device.river_accumulation(a, i).cpu().numpy()
    assert got.dtype == acc_dtype
    np.testing.assert_array_equal(got, want)


@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_slope_to_radians_layouts(layout):
    """dtb_slope_to_radians on the vector kernel (two passes, tail) and the scalar kernel: arctan(S / 100) in f32,
    nodata kept at -100 (example.py:63-64), within the tolerance of test_slope_to_radians_matches_example_glue"""
    from descriptools_b200 import device

    rng = np.random.default_rng(3)
    shape = LAYOUTS[layout]
    slope = (rng.random(shape) * 300).astype(np.float32)
    slope.reshape(-1)[::7] = -100
    s = _dev(slope, layout)
    _expect_form(layout, [s])
    want = np.where(slope == -100, np.float32(-100), np.arctan(slope / np.float32(100))).astype(np.float32)
    _poison_like(slope.size)
    got = device.slope_to_radians(s).cpu().numpy()
    np.testing.assert_array_equal(got == -100, want == -100)
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-7)


def test_numpy_modules_follow_the_oracle():
    """one pass through the drop-in NumPy modules with the same edge inputs"""
    import descriptools_b200.gfi as gfi
    import descriptools_b200.topoindexes as topoindexes

    rng = np.random.default_rng(21)
    shape = LAYOUTS["tail"]
    hand = _hand(shape[0] * shape[1], np.float32, rng).reshape(shape)
    acc = _acc(hand.size, np.int64, rng).reshape(shape)
    idx = rng.integers(0, hand.size, shape).astype(np.int64)
    idx.reshape(-1)[::11] = -100
    slope = _slope(hand.size, rng).reshape(shape)
    n, b = 0.4, 0.1
    with np.errstate(all="ignore"):
        g_ref = oracle.gfi(hand, acc, idx, n, b, PX)
        l_ref = oracle.ln_hl_H(hand, acc, n, b, PX)
    g = gfi.gfi_calculator(hand, acc, idx, n, b, PX)
    l = gfi.ln_hl_H_calculator(hand, acc, n, b, PX)
    assert g.dtype == np.float64 and l.dtype == np.float64
    assert_log_close(g.astype(np.float32), g_ref, n, "gfi_calculator")
    assert_log_close(l.astype(np.float32), l_ref, n, "ln_hl_H_calculator")
    ti_ref, mti_ref = _ti_ref(acc, slope, PX, n)
    ti, mti = topoindexes.topographic_index(acc, slope, PX, n)
    assert_log_close(ti.astype(np.float32), ti_ref, 1.0, "TI")
    assert_log_close(mti.astype(np.float32), mti_ref, n, "MTI")


# ---- the fused epilogue of the HAND tile pass -------------------------------------------------------------------------
FUSED_PARAMS = [(0.4, 0.1, PX), (0.0, 0.1, PX), (-0.4, 0.1, PX), (8.0, 1e-29, 0.5), (-8.0, 1e29, 2.0), (0.0, 7.0, 3.0)]


def _nonfinite_dem(rows, cols, seed):
    """a conditioned DEM, its D8 codes and accumulation (from the clean DEM), and the DEM HAND reads: NaN, +inf and -inf
    cells on river cells and on the paths that drain to them"""
    dem = synth(rows, cols, seed)
    _, d8 = oracle.slope_d8(dem, PX)
    acc, left = oracle.flow_accumulation(d8)
    assert left == 0
    rng = np.random.default_rng(seed)
    bad = dem.copy()
    for thr_mask in (acc > 300, (acc >= 0) & (acc <= 300)):
        cells = np.flatnonzero(thr_mask)
        pick = rng.choice(cells, size=min(60, cells.size), replace=False)
        bad.reshape(-1)[pick] = np.array([np.nan, np.inf, -np.inf], np.float32)[np.arange(pick.size) % 3]
    return bad, d8, acc


@pytest.mark.parametrize("n,b,size", FUSED_PARAMS)
def test_fused_gfi_nonfinite_hand_and_zero_accumulation(n, b, size):
    """the fused GFI of the HAND tile pass (fused with flow accumulation, the stand-alone HAND kernels, and a river mask
    holding cells of accumulation 0) against the oracle, on a DEM with NaN / +-inf cells on and off the river: NaN HAND
    gives NaN, +inf HAND gives -inf (NaN where ln b + n ln(A size^2) is +inf too), and n = 0 gives ln(b / (H + 0.01))
    for A_r = 0 as the reference's pow(0, 0) = 1 does"""
    from descriptools_b200 import device

    thr = 300
    dem, d8, acc_ref = _nonfinite_dem(300, 420, 41)
    hand_fused_vs_oracle(d8, dem, thr, n=n, b=b, size=size)

    t8, td = torch.from_numpy(d8).cuda(), torch.from_numpy(dem).cuda()
    acc = device.flow_accumulation(t8)
    np.testing.assert_array_equal(acc.cpu().numpy(), acc_ref)
    rng = np.random.default_rng(5)
    river = (acc_ref > thr).astype(np.int8)
    zero = np.flatnonzero(acc_ref == 0)
    river.reshape(-1)[rng.choice(zero, size=400, replace=False)] = 1  # river cells with accumulation 0
    for name, mask in (("threshold", (acc_ref > thr).astype(np.int8)), ("mask with A = 0", river)):
        _, i_ref, h_ref = oracle.flow_hand_index(dem, d8, mask, PX)
        with np.errstate(all="ignore"):
            g_ref = oracle.gfi(h_ref, acc_ref, i_ref, n, b, size)
        if name == "threshold":
            out = device.hand(t8, td, PX, acc=acc, river_threshold=thr, gfi_params=(n, b, size))
        else:
            out = device.hand(t8, td, PX, river=torch.from_numpy(mask).cuda(), acc=acc, gfi_params=(n, b, size))
            assert (np.isnan(g_ref) | np.isinf(g_ref)).any()
        np.testing.assert_array_equal(out["idx"].cpu().numpy(), i_ref, err_msg=name)
        np.testing.assert_array_equal(out["hand"].cpu().numpy(), h_ref, err_msg=name)
        assert_log_close(out["gfi"].cpu().numpy(), g_ref, n, f"{name} n={n} b={b} size={size}")


@pytest.mark.parametrize("n", [0.0, 0.4])
def test_run_device_every_cell_a_river(n):
    """pipeline.run_device with river_threshold = -1: every valid cell is a river cell, including those of accumulation
    0, so GFI is log(b (A size^2)^n / 0.01) there -- ln(b / 0.01) for n = 0, -inf for A = 0 and n > 0"""
    from descriptools_b200 import pipeline

    dem = synth(260, 330, 17)
    got = pipeline.run_device(torch.from_numpy(dem).cuda(), PX, -1, n_gfi=n, scale_factor=0.1)
    _, d8 = oracle.slope_d8(dem, PX)
    acc, _ = oracle.flow_accumulation(d8)
    river = (acc > -1).astype(np.int8)
    assert (acc == 0).sum() > 1000
    fdist, idx, hand = oracle.flow_hand_index(dem, d8, river, PX)
    with np.errstate(all="ignore"):
        gfi = oracle.gfi(hand, acc, idx, n, 0.1, PX)
    np.testing.assert_array_equal(got["acc"].cpu().numpy(), acc)
    np.testing.assert_array_equal(got["idx"].cpu().numpy(), idx)
    np.testing.assert_array_equal(got["hand"].cpu().numpy(), hand)
    assert_log_close(got["gfi"].cpu().numpy(), gfi, n, f"run_device n={n}")


@pytest.mark.parametrize("n", [0.0, 0.4])
def test_bands_equal_single_gpu_nonfinite_dem(n):
    """3 row bands == the single-raster run bit for bit (NaN where it has NaN) on a DEM with NaN / +inf cells, whose
    paths reach river cells of other bands (hand.cu: the remote river's accumulation from the halo tables)"""
    from descriptools_b200 import bands, pipeline

    rows, cols, thr = 384, 300, 150
    dem = synth(rows, cols, 29)
    rng = np.random.default_rng(29)
    pick = rng.choice(dem.size, size=90, replace=False)
    dem.reshape(-1)[pick] = np.array([np.nan, np.inf], np.float32)[np.arange(pick.size) % 2]
    ref = pipeline.run_device(torch.from_numpy(dem).cuda(), PX, thr, n_gfi=n, scale_factor=0.1)
    runner = bands.BandRunner(rows, cols, PX, thr, n, 0.1, nbands=3)
    runner.load([torch.from_numpy(dem[a:b]) for a, b in zip(runner.edges, runner.edges[1:])])
    runner.step()
    torch.cuda.synchronize()
    outs = runner.outputs()
    got = {name: torch.cat([o[name] for o in outs], 0).cpu().numpy() for name in outs[0]}
    for name in ("d8", "acc", "idx", "fdist", "hand", "gfi"):
        np.testing.assert_array_equal(got[name], ref[name].cpu().numpy(), err_msg=name)
    g = got["gfi"]
    assert np.isnan(g).any() or np.isneginf(g).any()
