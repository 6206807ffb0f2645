"""GPU parity tests: the CUDA path (through libdtb200's C ABI) against the CPU oracle on the same
inputs, against the committed golden fixtures, and -- at larger sizes -- through size-independent
properties.  Integer / index / D8 outputs must be bit-exact; floats are within the north-star
tolerance (1e-5 relative; atol 1e-6 for indices that cross zero), and bit-exact where stated.
"""
import numpy as np
import pytest
import torch

import oracle
from helpers import example_inputs, hand_fused_vs_oracle, listed_tiles, load, serpentine_d8, sha, synth

pytestmark = pytest.mark.gpu

PX = 12.5
RTOL, ATOL = 1e-5, 1e-6


@pytest.fixture(scope="module")
def mods():
    import descriptools_b200.downslope as downslope
    import descriptools_b200.flowhand as flowhand
    import descriptools_b200.gfi as gfi
    import descriptools_b200.slope as slope
    import descriptools_b200.topoindexes as topoindexes

    return dict(slope=slope, flowhand=flowhand, downslope=downslope, gfi=gfi, topoindexes=topoindexes)


@pytest.fixture(scope="module")
def ex():
    return example_inputs()


# ---- slope + D8 -------------------------------------------------------------------------------
def misaligned(t):
    """the same values in a contiguous view that starts 4 bytes into its buffer: not 16-byte aligned"""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 != 0
    return v


def check_slope_d8(mods, dem, px):
    """all three launch forms (slope only, D8 only, both outputs -- the fused kernel of the chain) against the oracle;
    then all three again on a DEM that is not 16-byte aligned, which only the generic kernel takes"""
    from descriptools_b200 import device

    with np.errstate(all="ignore"):
        s_ref, d_ref = oracle.slope_d8(dem, px)
    np.testing.assert_array_equal(mods["slope"].sloper(dem, px).astype(np.float32), s_ref)
    np.testing.assert_array_equal(mods["flowhand"].flow_direction_d8(dem, px), d_ref)
    t = torch.from_numpy(np.ascontiguousarray(dem)).cuda()
    s, d = device.slope_d8(t, px)
    np.testing.assert_array_equal(s.cpu().numpy(), s_ref)
    np.testing.assert_array_equal(d.cpu().numpy(), d_ref)
    g = misaligned(t)
    s, d = device.slope_d8(g, px)
    np.testing.assert_array_equal(s.cpu().numpy(), s_ref, err_msg="generic kernel, both outputs")
    np.testing.assert_array_equal(d.cpu().numpy(), d_ref, err_msg="generic kernel, both outputs")
    s, _ = device.slope_d8(g, px, want_d8=False)
    np.testing.assert_array_equal(s.cpu().numpy(), s_ref, err_msg="generic kernel, slope only")
    _, d = device.slope_d8(g, px, want_slope=False)
    np.testing.assert_array_equal(d.cpu().numpy(), d_ref, err_msg="generic kernel, D8 only")


@pytest.mark.parametrize("shape", [(1, 1), (1, 7), (5, 1), (3, 3), (64, 128), (65, 129), (130, 260), (257, 516), (100, 1534 // 2)])
def test_slope_d8_f32_bit_exact(mods, shape):
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    dem = (rng.standard_normal(shape) * 20 + 300).astype(np.float32)
    if dem.size > 20:
        dem.reshape(-1)[rng.integers(0, dem.size, dem.size // 15)] = -100
        dem.reshape(-1)[rng.integers(0, dem.size, 3)] = -250.0
        dem.reshape(-1)[rng.integers(0, dem.size, 3)] = np.nan
    s_ref, d_ref = oracle.slope_d8(dem, PX)
    np.testing.assert_array_equal(mods["slope"].sloper(dem, PX), s_ref.astype(np.float64))
    np.testing.assert_array_equal(mods["flowhand"].flow_direction_d8(dem, PX), d_ref)


def test_slope_d8_ties_and_flats(mods):
    """integer-valued and plateau DEMs: many exact ties inside a class and flats (m == 0)."""
    rng = np.random.default_rng(9)
    dem = rng.integers(0, 4, (200, 260)).astype(np.float32)
    dem[50:90, 60:120] = 2.0
    s_ref, d_ref = oracle.slope_d8(dem, 10.0)
    np.testing.assert_array_equal(mods["slope"].sloper(dem, 10.0), s_ref.astype(np.float64))
    np.testing.assert_array_equal(mods["flowhand"].flow_direction_d8(dem, 10.0), d_ref)


@pytest.mark.parametrize("px", [12.5, 30.0, 1.0, 0.3, 7.77])
def test_slope_d8_near_tie_card_vs_diag(mods, px):
    """cardinal-vs-diagonal gradients engineered to be within/around the f32 guard band."""
    rng = np.random.default_rng(3)
    rows, cols = 96, 128
    dem = np.full((rows, cols), 500.0, np.float32)
    s2 = np.sqrt(2.0)
    for r in range(1, rows - 1, 3):
        for c in range(1, cols - 1, 3):
            a = np.float32(rng.uniform(0.5, 30))
            eps = np.float32(rng.choice([0, 1, -1, 2, -2, 50, -50])) * np.spacing(a)
            dem[r, c + 1] = np.float32(500.0) - a            # cardinal drop a
            dem[r + 1, c + 1] = np.float32(500.0) - np.float32(np.float32(a * s2) + eps)  # diagonal drop ~ a*sqrt2
    s_ref, d_ref = oracle.slope_d8(dem, px)
    np.testing.assert_array_equal(mods["slope"].sloper(dem, px), s_ref.astype(np.float64))
    np.testing.assert_array_equal(mods["flowhand"].flow_direction_d8(dem, px), d_ref)


@pytest.mark.parametrize("px", [12.5, 25.0, 0.5, 30.0, 1.0, 7.77])
def test_slope_d8_tma_path_exact(mods, px):
    """the lean strip on both kernels: power-of-two and general 100/px, several tiles, pits everywhere; crops to widths
    4k + 1, 4k + 2 and 4k + 3 (generic kernel only) end every row in a ragged group of fewer than four cells."""
    rng = np.random.default_rng(int(px * 100))
    dem = (np.cumsum(rng.standard_normal((300, 512)), axis=1) * 3 + rng.standard_normal((300, 512)) + 400).astype(np.float32)
    for cols in (512, 509, 510, 511):
        check_slope_d8(mods, np.ascontiguousarray(dem[:, :cols]), px)


@pytest.mark.parametrize("scale", [1e-30, 1e-38, 1e-42, 1e25, 1e36])
def test_slope_d8_extreme_ranges(mods, scale):
    """sub-range and huge elevations (products that underflow / overflow in f32): the lean strip must hand them to the
    exact path, results stay bit-exact (incl. inf slopes where the reference overflows f32)."""
    rng = np.random.default_rng(11)
    with np.errstate(over="ignore", under="ignore"):
        dem = (rng.standard_normal((96, 256)) * scale).astype(np.float32)
    dem[10:14, 20:28] = 0.0
    dem[40, 100] = np.inf
    dem[60, 30] = -np.inf
    check_slope_d8(mods, dem, 12.5)
    check_slope_d8(mods, dem, 30.0)


def test_slope_d8_rounding_ties(mods):
    """differences whose slope product is exactly half-way between two f32 (px = 1: a * 100 with a on a coarse grid) --
    the bracket of the lean strip straddles the boundary and the exact path must decide (round-half-even)."""
    rng = np.random.default_rng(5)
    dem = np.full((128, 256), 500.0, np.float32)
    dem[1::2, 1::2] = np.float32(500.0) - (rng.integers(1, 1 << 20, (64, 128)) * np.float32(2.0 ** -15)).astype(np.float32)
    for px in (1.0, 2.0, 12.5, 0.25):
        check_slope_d8(mods, dem, px)


def test_slope_d8_nodata_holes_and_outlets(mods):
    """nodata blobs (-100 and values below -100), NaNs and pits next to them: the nodata row path and the outlet rule."""
    rng = np.random.default_rng(21)
    dem = (np.cumsum(rng.standard_normal((260, 384)), axis=0) * 2 + 300).astype(np.float32)
    yy, xx = np.mgrid[0:260, 0:384]
    for (cy, cx, r) in [(60, 70, 30), (150, 200, 55), (200, 350, 40), (10, 380, 15)]:
        dem[(yy - cy) ** 2 + (xx - cx) ** 2 <= r * r] = -100
    dem[100:104, 10:30] = -250.0
    dem[rng.integers(0, 260, 40), rng.integers(0, 384, 40)] = np.nan
    dem[120:140, 300:320] = 123.0  # a flat: pits with defined neighbours only
    check_slope_d8(mods, dem, 12.5)
    check_slope_d8(mods, dem, 10.0)


def test_slope_example_int16_golden(mods, ex):
    """int16 example DEM (generic, non-TMA kernel: 1534 columns) against the reference's own output."""
    gold = load("example_cpujit.npz")
    s = mods["slope"].sloper(ex["dem"], PX)
    assert s.dtype == np.float64
    assert sha(s.astype(np.float32)) == str(gold["slope_sha256"])


def test_slope_cpu_wrapper(mods):
    dem = synth(40, 52, 5)
    full = mods["slope"].sloper(dem, PX).astype(np.float32)
    # tile = rows 10..30 with real halo above/below, raster edge left/right
    tile = mods["slope"].slope_cpu(dem[9:31, :], PX, np.array([0, 1, 1, 0]))
    np.testing.assert_array_equal(tile, full[10:30, :])


def test_slope_d8_band_rows(mods):
    """rows [row_begin,row_end) of a buffer with halo rows == the same rows of the full raster."""
    from descriptools_b200 import device

    dem = synth(300, 256, 8)
    s_ref, d_ref = oracle.slope_d8(dem, PX)
    t = torch.from_numpy(dem).cuda()
    for (a, b) in [(0, 100), (100, 217), (217, 300)]:
        lo, hi = max(a - 1, 0), min(b + 1, 300)
        buf = t[lo:hi].contiguous()
        s, d = device.slope_d8(buf, PX, row_begin=a - lo, row_end=(a - lo) + (b - a))
        # interior band edges see real halo rows; raster edges are off-raster in both
        np.testing.assert_array_equal(s.cpu().numpy(), s_ref[a:b])
        np.testing.assert_array_equal(d.cpu().numpy(), d_ref[a:b])


# ---- flow accumulation ------------------------------------------------------------------------
@pytest.mark.parametrize("shape,seed", [((1, 1), 1), ((7, 5), 2), ((128, 200), 3), ((300, 411), 4)])
def test_flowacc_bit_exact(mods, shape, seed):
    dem = synth(*shape, seed, holes=shape[0] > 20)
    _, d8 = oracle.slope_d8(dem, PX)
    acc_ref, left = oracle.flow_accumulation(d8)
    assert left == 0
    acc = mods["flowhand"].flow_accumulation(d8)
    assert acc.dtype == np.int64
    np.testing.assert_array_equal(acc, acc_ref)


def test_flowacc_random_codes_with_cycles(mods):
    """arbitrary D8 grids (cycles, unknown codes, exits): partial counts on cycles match the oracle."""
    from descriptools_b200 import device

    rng = np.random.default_rng(11)
    d8 = rng.choice(np.array([0, 1, 2, 4, 8, 16, 32, 64, 128, 3, 255], np.uint8), (90, 130))
    acc_ref, left_ref = oracle.flow_accumulation(d8)
    acc, left = device.flow_accumulation(torch.from_numpy(d8).cuda(), dtype=torch.int64, check_cycles=True)
    assert left == left_ref and left_ref > 0
    np.testing.assert_array_equal(acc.cpu().numpy(), acc_ref)


def test_flowacc_kat2_example(mods, ex):
    acc = mods["flowhand"].flow_accumulation(ex["fdr"])
    acc_ref, _ = oracle.flow_accumulation(ex["fdr"])
    np.testing.assert_array_equal(acc, acc_ref)
    valid = ex["fdr"] != 0
    assert (acc[valid] == ex["fac"][valid]).mean() > 0.98 and (acc[valid] <= ex["fac"][valid]).all()


# ---- flow distance / index / HAND ---------------------------------------------------------------
def test_hand_example_golden(mods, ex):
    """full bundled example (int16 DEM): idx and hand bit-exact against the reference's output."""
    gold = load("example_cpujit.npz")
    fdist, idx, hand = mods["flowhand"].flow_hand_index(ex["dem"], ex["fdr"], ex["river"], PX)
    assert fdist.dtype == np.float32 and idx.dtype == np.int64 and hand.dtype == np.int16
    assert sha(idx) == str(gold["idx_sha256"])
    assert sha(hand) == str(gold["hand_sha256"])
    np.testing.assert_allclose(fdist.reshape(-1)[::37], gold["fdist_sample"], rtol=RTOL, atol=0)
    f_ref, _ = oracle.flow_distance_index(ex["fdr"], ex["river"], PX)
    np.testing.assert_allclose(fdist, f_ref, rtol=RTOL, atol=0)
    np.testing.assert_array_equal(mods["flowhand"].hand_calculator(ex["dem"], idx), hand)


@pytest.mark.parametrize("name", ["cudasim_example_crop.npz", "cudasim_synth_f32.npz"])
def test_all_descriptors_vs_reference_kernels(mods, name):
    """every public entry point against the reference's own GPU kernels (CUDASIM goldens)."""
    g = load(name)
    dem, fdr, fac, river = g["dem"], g["fdr"], g["fac"], g["river"]
    delta = 5 if dem.dtype == np.int16 else 0.5
    np.testing.assert_array_equal(mods["slope"].sloper(dem, PX).astype(np.float32), g["slope"])
    fdist, idx, hand = mods["flowhand"].flow_hand_index(dem, fdr, river, PX)
    np.testing.assert_array_equal(idx, g["idx"])
    np.testing.assert_array_equal(hand, g["hand"])
    assert hand.dtype == g["hand"].dtype
    np.testing.assert_allclose(fdist, g["fdist"], rtol=RTOL, atol=0)
    np.testing.assert_array_equal(mods["downslope"].downsloper(dem, fdr, PX, delta), g["downslope"])
    ti, mti = mods["topoindexes"].topographic_index(fac, g["slope_rad"], PX, 0.1)
    assert ti.dtype == np.float64
    np.testing.assert_allclose(ti, g["ti"], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(mti, g["mti"], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(mods["gfi"].gfi_calculator(hand, fac, idx, 0.4, 0.1, PX), g["gfi"], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(mods["gfi"].ln_hl_H_calculator(hand, fac, 0.4, 0.1, PX), g["lnhlh"], rtol=RTOL, atol=ATOL)
    np.testing.assert_array_equal(mods["gfi"].river_accumulation(fac, idx), oracle.river_accumulation(fac, idx))


def test_hand_special_cases(mods):
    g = load("cudasim_special.npz")
    fdist, idx, hand = mods["flowhand"].flow_hand_index(g["dem"], g["fdr"], g["river"], PX)
    np.testing.assert_array_equal(idx, g["idx"])
    np.testing.assert_array_equal(hand, g["hand"])
    np.testing.assert_allclose(fdist, g["fdist"], rtol=RTOL, atol=0)
    np.testing.assert_array_equal(mods["downslope"].downsloper(g["dem_ds"], g["fdr"], PX, 4), g["downslope"])


def test_hand_move_cap(mods):
    """flowhand.py:835: 20001 moves fail, 20000 succeed (serpentine fixture from the reference kernel)."""
    g = load("cudasim_cap.npz")
    n = int(g["n_cells"])
    fdr, river = g["fdr"], g["river"]
    dem = np.full(fdr.shape, 50, np.float32)
    fdist, idx, _ = mods["flowhand"].flow_hand_index(dem, fdr, river, PX)
    np.testing.assert_array_equal(idx.reshape(-1)[:n], g["idx"])
    np.testing.assert_allclose(fdist.reshape(-1)[:n], g["fdist"], rtol=RTOL)
    f_ref, i_ref = oracle.flow_distance_index(fdr, river, PX)
    np.testing.assert_array_equal(idx, i_ref)
    np.testing.assert_allclose(fdist, f_ref, rtol=RTOL)


def test_hand_random_codes(mods):
    """arbitrary D8 grids: cycles of every length, unknown codes, rivers with code 0."""
    rng = np.random.default_rng(21)
    fdr = rng.choice(np.array([0, 1, 2, 4, 8, 16, 32, 64, 128, 3, 255], np.uint8), (120, 150),
                     p=[.03, .2, .1, .2, .1, .1, .08, .08, .08, .015, .015])
    river = (rng.random(fdr.shape) < 0.02).astype(np.int8)
    dem = (rng.standard_normal(fdr.shape) * 10 + 100).astype(np.float32)
    dem[rng.random(fdr.shape) < 0.02] = -100
    f_ref, i_ref, h_ref = oracle.flow_hand_index(dem, fdr, river, PX)
    fdist, idx, hand = mods["flowhand"].flow_hand_index(dem, fdr, river, PX)
    np.testing.assert_array_equal(idx, i_ref)
    np.testing.assert_array_equal(hand, h_ref)
    np.testing.assert_allclose(fdist, f_ref, rtol=RTOL, atol=0)


def test_hand_small_cap_parameter():
    from descriptools_b200 import device

    dem = synth(150, 190, 31)
    _, d8 = oracle.slope_d8(dem, PX)
    acc, _ = oracle.flow_accumulation(d8)
    river = (acc > 2000).astype(np.int8)
    for cap in (5, 37, 64):
        f_ref, i_ref = oracle.flow_distance_index(d8, river, PX, max_moves=cap)
        out = device.hand(torch.from_numpy(d8).cuda(), None, PX, river=torch.from_numpy(river).cuda(), max_moves=cap,
                          want_hand=False)
        np.testing.assert_array_equal(out["idx"].cpu().numpy(), i_ref)
        np.testing.assert_allclose(out["fdist"].cpu().numpy(), f_ref, rtol=RTOL, atol=0)
        assert (i_ref == -100).sum() > (river == 0).sum() * 0.05  # the cap really bites


# ---- downslope, pointwise ----------------------------------------------------------------------
def test_downslope_example_golden(mods, ex):
    gold = load("example_cpujit.npz")
    d = mods["downslope"].downsloper(ex["dem"], ex["fdr"], PX, 5)
    assert d.dtype == np.float32
    assert sha(d) == str(gold["downslope_sha256"])


def test_downslope_synth_bit_exact(mods):
    dem = synth(200, 333, 17)
    _, d8 = oracle.slope_d8(dem, PX)
    for delta in (0.5, 5):
        np.testing.assert_array_equal(mods["downslope"].downsloper(dem, d8, PX, delta), oracle.downslope(dem, d8, PX, delta))


def test_downslope_drop_limits_and_odd_codes(mods):
    """the kernel tests "drop < delta" in the DEM's own type against a limit derived from delta on the host: deltas that
    are not float32 values, tiny, zero, negative and NaN; int16 elevations with fractional deltas; grids with cells that
    carry no or several direction bits (the walk stops there) -- all bit-exact against the oracle's f64 comparison"""
    dem = synth(160, 211, 29)
    _, d8 = oracle.slope_d8(dem, PX)
    rng = np.random.default_rng(5)
    odd = d8.copy()
    hit = rng.random(odd.shape) < 0.02
    odd[hit] = rng.choice(np.array([0, 3, 129, 255, 96], np.uint8), size=int(hit.sum()))
    for delta in (5.1, 0.1 + 1e-9, 1e-50, 0.0, -3.0, float("nan"), 1e30):
        for codes in (d8, odd):
            np.testing.assert_array_equal(mods["downslope"].downsloper(dem, codes, PX, delta), oracle.downslope(dem, codes, PX, delta),
                                          err_msg=f"delta={delta}")
    # elevation differences that land exactly on float32 neighbours of delta
    step = np.float32(5.1)
    ramp = (np.float32(1000.0) - np.arange(64, dtype=np.float32)[None, :] * step) + np.zeros((8, 1), np.float32)
    east = np.full(ramp.shape, 1, np.uint8)
    for delta in (float(step), float(np.nextafter(step, np.float32(0))), float(np.nextafter(step, np.float32(10))), 5.1):
        np.testing.assert_array_equal(mods["downslope"].downsloper(ramp, east, PX, delta), oracle.downslope(ramp, east, PX, delta),
                                      err_msg=f"ramp delta={delta}")
    dem16 = np.round(dem).astype(np.int16)
    _, d16 = oracle.slope_d8(dem16, PX)
    for delta in (4.5, 5, 5.0000001, -1.5, 1e9):
        np.testing.assert_array_equal(mods["downslope"].downsloper(dem16, d16, PX, delta), oracle.downslope(dem16, d16, PX, delta),
                                      err_msg=f"int16 delta={delta}")


def test_gfi_lnhlh_example_golden(mods, ex):
    gold = load("example_cpujit.npz")
    _, idx, hand = oracle.flow_hand_index(ex["dem"], ex["fdr"], ex["river"], PX)
    g = mods["gfi"].gfi_calculator(hand, ex["fac"], idx, 0.4, 0.1, PX)
    l = mods["gfi"].ln_hl_H_calculator(hand, ex["fac"], 0.4, 0.1, PX)
    assert g.dtype == np.float64 and l.dtype == np.float64
    np.testing.assert_allclose(g.reshape(-1)[::37], gold["gfi_sample"], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(l.reshape(-1)[::37], gold["lnhlh_sample"], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(g, oracle.gfi(hand, ex["fac"], idx, 0.4, 0.1, PX), rtol=RTOL, atol=ATOL)


def test_ti_mti_example(mods, ex):
    s, _ = oracle.slope_d8(ex["dem"], PX)
    rad = np.arctan(s / 100).astype(np.float32)
    rad = np.where(ex["dem"] == -100, -100, rad).astype(np.float32)  # example.py:63-64
    ti_ref, mti_ref = oracle.ti_mti(ex["fac"], rad, PX, 0.1)
    ti, mti = mods["topoindexes"].topographic_index(ex["fac"], rad, PX, 0.1)
    np.testing.assert_allclose(ti, ti_ref, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(mti, mti_ref, rtol=RTOL, atol=ATOL)


# ---- the fused chain ----------------------------------------------------------------------------
def test_slope_to_radians_matches_example_glue():
    """dtb_slope_to_radians == the host glue of example.py:63-64: arctan(S / 100) in f32, nodata patched back to -100."""
    from descriptools_b200 import device

    rng = np.random.default_rng(4)
    dem = (rng.standard_normal((96, 160)) * 30 + 200).astype(np.float32)
    dem[rng.random(dem.shape) < 0.1] = -100
    slope = oracle.slope_d8(dem, PX)[0]
    want = np.arctan(slope / np.float32(100)).astype(np.float32)  # example.py:63
    want = np.where(dem == -100, np.float32(-100), want).astype(np.float32)  # example.py:64
    got = device.slope_to_radians(torch.from_numpy(slope).cuda()).cpu().numpy()
    assert got.dtype == np.float32
    np.testing.assert_array_equal(got == -100, want == -100)
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-7)  # CUDA atanf vs NumPy arctan: 1-2 ulp


def test_gathers_follow_numpy_index_rules(mods):
    """hand_calculator / river_accumulation on caller-supplied indices: -100 is the mask, other negative indices wrap like
    NumPy's, an index outside the raster raises IndexError (as the reference's fancy indexing does), and rasters of
    different shapes are refused before anything is launched."""
    rng = np.random.default_rng(12)
    rows, cols = 40, 56
    n = rows * cols
    dem = (rng.standard_normal((rows, cols)) * 10 + 100).astype(np.float32)
    fac = rng.integers(0, 5000, (rows, cols)).astype(np.int64)
    idx = rng.integers(0, n, (rows, cols)).astype(np.int64)
    idx[rng.random(idx.shape) < 0.2] = -100
    idx[3, 4], idx[7, 9] = -1, -n  # NumPy: last element, first element
    ref_hand = np.where((dem != -100) & (idx != -100), dem - dem.reshape(-1)[idx], -100).astype(np.float32)  # flowhand.py:436
    ref_hand = np.where((ref_hand < 0) & (ref_hand != -100), 0, ref_hand).astype(np.float32)               # flowhand.py:438
    np.testing.assert_array_equal(mods["flowhand"].hand_calculator(dem, idx), ref_hand)
    ref_racc = np.where(idx != -100, fac.reshape(-1)[idx], fac.reshape(-1)[0])  # gfi.py:141-143
    np.testing.assert_array_equal(mods["gfi"].river_accumulation(fac, idx), ref_racc)
    for bad in (n, n + 12345, -n - 1):
        idx2 = idx.copy()
        idx2[5, 5] = bad
        with pytest.raises(IndexError):
            mods["flowhand"].hand_calculator(dem, idx2)
        with pytest.raises(IndexError):
            mods["gfi"].river_accumulation(fac, idx2)
    with pytest.raises(ValueError):
        mods["gfi"].river_accumulation(fac, idx[:-1])
    with pytest.raises(ValueError):
        mods["flowhand"].hand_calculator(dem[:, :-1], idx)


@pytest.mark.parametrize("shape,thr", [((512, 640), 300), ((1000, 1200), 2000)])
def test_pipeline_vs_oracle(shape, thr):
    from descriptools_b200 import pipeline

    dem = synth(*shape, seed=shape[0])
    got = pipeline.pipeline(dem, PX, thr, 0.4, 0.1)
    slope, d8 = oracle.slope_d8(dem, PX)
    acc, left = oracle.flow_accumulation(d8)
    assert left == 0
    river = (acc > thr).astype(np.int8)
    fdist, idx, hand = oracle.flow_hand_index(dem, d8, river, PX)
    gfi = oracle.gfi(hand, acc, idx, 0.4, 0.1, PX)
    np.testing.assert_array_equal(got["slope"], slope)
    np.testing.assert_array_equal(got["d8"], d8)
    np.testing.assert_array_equal(got["acc"], acc)
    np.testing.assert_array_equal(got["idx"], idx)
    np.testing.assert_array_equal(got["hand"], hand)
    np.testing.assert_allclose(got["fdist"], fdist, rtol=RTOL, atol=0)
    np.testing.assert_allclose(got["gfi"], gfi, rtol=RTOL, atol=ATOL)


def test_synth_and_fill_match_host():
    """device DEM generator and depression filling are bit-identical to oracle/dt_condition.cpp."""
    from descriptools_b200 import device

    rows, cols = 700, 900
    d = device.synth_dem(rows, cols, 0, 123)
    h = oracle.synth_dem(rows, cols, 0, 123)
    np.testing.assert_array_equal(d.cpu().numpy(), h)
    band = device.synth_dem(100, cols, 250, 123)
    np.testing.assert_array_equal(band.cpu().numpy(), h[250:350])
    passes = device.fill_depressions(d)
    np.testing.assert_array_equal(d.cpu().numpy(), oracle.priority_flood_eps(h))
    assert passes > 0
    # with nodata holes
    h2 = h.copy()
    h2[300:340, 400:470] = -100
    d2 = torch.from_numpy(h2).cuda()
    device.fill_depressions(d2)
    np.testing.assert_array_equal(d2.cpu().numpy(), oracle.priority_flood_eps(h2))


def test_pipeline_properties_large():
    """size-independent properties on a DEM too large for the CPU oracle to be the only check:
    sum of source-free accumulation identities, idempotence of HAND from idx, idx points at rivers."""
    from descriptools_b200 import device, pipeline

    rows, cols = 4096, 4096
    dem = device.conditioned_dem(rows, cols, seed=77)
    thr = 2000
    res = pipeline.run_device(dem, PX, thr)
    d8, acc, idx, hand = res["d8"], res["acc"], res["idx"], res["hand"]
    assert int((d8 == 0).sum()) == 0  # conditioned DEM: every cell drains
    # every cell is counted once by each of its downstream cells: sum(acc) == sum over cells of path length to outlet
    # cheaper identity: cells draining off-raster are the roots; sum over roots of (acc+1) == number of cells
    r = torch.arange(rows, device="cuda").view(-1, 1).expand(rows, cols)
    c = torch.arange(cols, device="cuda").view(1, -1).expand(rows, cols)
    dr = torch.zeros_like(r)
    dc = torch.zeros_like(c)
    for code, (a, b) in {1: (0, 1), 2: (1, 1), 4: (1, 0), 8: (1, -1), 16: (0, -1), 32: (-1, -1), 64: (-1, 0), 128: (-1, 1)}.items():
        m = d8 == code
        dr[m], dc[m] = a, b
    rr, cc = r + dr, c + dc
    root = (rr < 0) | (rr >= rows) | (cc < 0) | (cc >= cols)
    assert int((acc[root].long() + 1).sum()) == rows * cols
    # acc of a non-root cell's downstream neighbour is strictly larger
    nxt = (rr.clamp(0, rows - 1) * cols + cc.clamp(0, cols - 1)).view(-1)
    assert bool((acc.view(-1)[nxt][~root.view(-1)] > acc.view(-1)[~root.view(-1)]).all())
    # idx points at river cells; hand recomputed from idx is identical; river cells have hand 0, idx = self
    ok = idx >= 0
    river = acc > thr
    assert bool(river.view(-1)[idx[ok].long()].all())
    lin = torch.arange(rows * cols, device="cuda", dtype=idx.dtype).view(rows, cols)
    assert bool((idx[river] == lin[river]).all()) and bool((hand[river] == 0).all())
    np.testing.assert_array_equal(device.hand_from_index(dem, idx).cpu().numpy(), hand.cpu().numpy())
    assert bool((hand[ok] >= 0).all())
    # against the oracle on a corner crop is not possible (paths leave the crop); check slope/D8 rows instead
    s_ref, d_ref = oracle.slope_d8(dem[:300].cpu().numpy(), PX, 0, 299)
    np.testing.assert_array_equal(res["slope"][:299].cpu().numpy(), s_ref)
    np.testing.assert_array_equal(d8[:299].cpu().numpy(), d_ref)


def test_chain_check_identities_and_detection():
    """dtb_chain_check (what bench.py prints as "verified"): green on a correct chain -- whole raster and summed over
    row bands -- and red when one accumulation count, one river index or one HAND value is off."""
    from descriptools_b200 import device, pipeline

    rows, cols, thr = 1024, 768, 500
    dem = device.conditioned_dem(rows, cols, seed=5)
    res = pipeline.run_device(dem, PX, thr)
    full = device.chain_check(res["d8"], res["acc"], thr, idx=res["idx"], dem=dem, hand=res["hand"]).tolist()
    v = device.chain_verdict(full)
    assert v["verified"] and v["valid_cells"] == rows * cols and v["idx_in_other_band"] == 0
    # the same rasters cut into three bands: the counters add up to the whole-raster ones (except the cross-band ones)
    tot = torch.zeros(8, dtype=torch.int64, device="cuda")
    for a, b in [(0, 320), (320, 704), (704, rows)]:
        tot += device.chain_check(res["d8"][a:b].contiguous(), res["acc"][a:b].contiguous(), thr, idx=res["idx"][a:b].contiguous(),
                                  dem=dem[a:b].contiguous(), hand=res["hand"][a:b].contiguous(), row0=a, total_rows=rows)
    vb = device.chain_verdict(tot.tolist())
    assert vb["verified"] and vb["valid_cells"] == rows * cols and vb["root_mass"] == rows * cols
    # against the oracle's own accumulation: the identity really is "every cell counted once at its root"
    acc_ref, left = oracle.flow_accumulation(res["d8"].cpu().numpy())
    assert left == 0
    np.testing.assert_array_equal(res["acc"].cpu().numpy(), acc_ref)
    # detection
    bad = res["acc"].clone()
    bad[rows // 2, cols // 2] += 1
    assert not device.chain_verdict(device.chain_check(res["d8"], bad, thr, idx=res["idx"], dem=dem, hand=res["hand"]).tolist())["verified"]
    ok = torch.nonzero((res["idx"] >= 0) & (res["acc"] <= thr))
    r, c = int(ok[len(ok) // 2][0]), int(ok[len(ok) // 2][1])
    bad_idx = res["idx"].clone()
    bad_idx[r, c] = r * cols + c  # itself: not a river cell
    assert device.chain_verdict(device.chain_check(res["d8"], res["acc"], thr, idx=bad_idx, dem=dem, hand=res["hand"]).tolist())["idx_not_river"] == 1
    bad_hand = res["hand"].clone()
    bad_hand[r, c] += 1.0
    assert device.chain_verdict(device.chain_check(res["d8"], res["acc"], thr, idx=res["idx"], dem=dem, hand=bad_hand).tolist())["hand_mismatch"] == 1


def test_chain_above_2_31_cells_int64_verified():
    """46 400 x 46 400 = 2.15e9 cells (> 2**31): counts and river indices are int64; the device-side identities of
    dtb_chain_check stand in for the oracle at this size (they pin every accumulation count, the river index targets and
    HAND).  Needs ~110 GB of device memory: skipped on smaller GPUs."""
    from descriptools_b200 import device, pipeline

    if torch.cuda.get_device_properties(0).total_memory < 150e9:
        pytest.skip("needs a 180 GB GPU")
    n = 46400
    assert n * n > 2**31
    dem = device.conditioned_dem(n, n, seed=3)
    device.workspace.release()
    torch.cuda.empty_cache()
    res = pipeline.run_device(dem, PX, 128000)
    assert res["acc"].dtype == torch.int64 and res["idx"].dtype == torch.int64
    v = device.chain_verdict(device.chain_check(res["d8"], res["acc"], 128000, idx=res["idx"], dem=dem, hand=res["hand"]).tolist())
    assert v["verified"], v
    assert v["valid_cells"] == n * n and v["root_mass"] == n * n
    assert int(res["idx"].max()) >= 2**31  # indices beyond int32 really occur
    del res, dem
    device.workspace.release()
    pipeline.release_buffers()
    torch.cuda.empty_cache()


# ---- row bands (multi-GPU decomposition, k logical bands on one GPU) ------------------------------
def weaving_dem(rows, cols, seam, amp=20.0, period=90.0):
    """a valley that weaves across row `seam` many times: every HAND / accumulation path re-enters bands"""
    r = np.arange(rows, dtype=np.float64)[:, None]
    c = np.arange(cols, dtype=np.float64)[None, :]
    centre = seam + amp * np.sin(2 * np.pi * c / period)
    z = 50.0 + 0.35 * np.abs(r - centre) + 0.05 * (cols - c) + 0.001 * ((r * 7 + c * 13) % 11)
    return oracle.priority_flood_eps(z.astype(np.float32))


def _run_bands(dem, k, thr, force_int64=False):
    from descriptools_b200 import bands

    rows, cols = dem.shape
    runner = bands.BandRunner(rows, cols, PX, thr, 0.4, 0.1, nbands=k, force_int64=force_int64)
    runner.load([torch.from_numpy(dem[a:b]) for a, b in zip(runner.edges, runner.edges[1:])])
    runner.step()
    torch.cuda.synchronize()
    outs = runner.outputs()
    return {name: torch.cat([o[name] for o in outs], 0).cpu().numpy() for name in outs[0]}


@pytest.mark.parametrize("shape,k,thr", [((512, 320), 2, 200), ((768, 400), 3, 300), ((1024, 272), 4, 150), ((200, 130), 1, 50),
                                         ((256, 200), 4, 150)])
def test_bands_equal_single_gpu(shape, k, thr):
    """k row bands + boundary-graph solve == the single-raster run, bit for bit (all seven rasters).  Bands of more than
    4 rows take the overlapped stencil (halo on its own stream, interior rows, then edges); 64-row bands are its tightest
    split."""
    from descriptools_b200 import pipeline

    dem = synth(*shape, seed=shape[1])
    ref = pipeline.run_device(torch.from_numpy(dem).cuda(), PX, thr)
    got = _run_bands(dem, k, thr)
    for name in ("slope", "d8", "acc", "idx", "fdist", "hand", "gfi"):
        np.testing.assert_array_equal(got[name], ref[name].cpu().numpy(), err_msg=name)


def test_bands_weaving_valley_vs_oracle():
    """paths that cross the seam many times (river running along a band edge): bands == oracle."""
    rows, cols, thr = 256, 720, 400
    dem = weaving_dem(rows, cols, seam=128)
    got = _run_bands(dem, 2, thr)
    slope, d8 = oracle.slope_d8(dem, PX)
    acc, left = oracle.flow_accumulation(d8)
    assert left == 0
    river = (acc > thr).astype(np.int8)
    assert river.sum() > 100
    fdist, idx, hand = oracle.flow_hand_index(dem, d8, river, PX)
    # the valley (and with it many paths) really crosses the seam repeatedly
    on_seam = river[127:129].sum(axis=0)
    assert (np.diff((river[:128].sum(axis=0) > 0).astype(int)) != 0).sum() >= 6 and on_seam.sum() > 0
    np.testing.assert_array_equal(got["d8"], d8)
    np.testing.assert_array_equal(got["acc"], acc)
    np.testing.assert_array_equal(got["idx"], idx)
    np.testing.assert_array_equal(got["hand"], hand)
    np.testing.assert_allclose(got["fdist"], fdist, rtol=RTOL, atol=0)
    np.testing.assert_allclose(got["gfi"], oracle.gfi(hand, acc, idx, 0.4, 0.1, PX), rtol=RTOL, atol=ATOL)


# ---- tiled kernels: paths the small cases above do not reach ----------------------------------------
def test_chain_int64_counts_and_indices():
    """the int64 instantiations (acc, idx; 64-bit inflow pushes in shared memory) against the oracle"""
    from descriptools_b200 import device

    dem = synth(330, 470, 5)
    thr = 700
    t = torch.from_numpy(dem).cuda()
    slope, d8 = device.slope_d8(t, PX)
    acc = device.flow_accumulation(d8, dtype=torch.int64, fuse_hand_threshold=thr)
    out = device.hand(d8, t, PX, acc=acc, river_threshold=thr, gfi_params=(0.4, 0.1, PX), idx_dtype=torch.int64, entry_done=True)
    _, d8_ref = oracle.slope_d8(dem, PX)
    acc_ref, _ = oracle.flow_accumulation(d8_ref)
    river = (acc_ref > thr).astype(np.int8)
    fdist, idx, hand = oracle.flow_hand_index(dem, d8_ref, river, PX)
    assert acc.dtype == torch.int64 and out["idx"].dtype == torch.int64
    np.testing.assert_array_equal(acc.cpu().numpy(), acc_ref)
    np.testing.assert_array_equal(out["idx"].cpu().numpy(), idx)
    np.testing.assert_array_equal(out["hand"].cpu().numpy(), hand)
    np.testing.assert_allclose(out["fdist"].cpu().numpy(), fdist, rtol=RTOL, atol=0)
    np.testing.assert_allclose(out["gfi"].cpu().numpy(), oracle.gfi(hand, acc_ref, idx, 0.4, 0.1, PX), rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("thr", [10, 4095, 4096, 30000])
def test_fused_and_unfused_hand_agree(thr):
    """river threshold below / at / above the tile size (4096 cells): the fused entry pass + successor table
    must give exactly what the stand-alone HAND kernels give from the same accumulation"""
    from descriptools_b200 import device

    dem = synth(900, 1024, 77)
    t = torch.from_numpy(dem).cuda()
    _, d8 = device.slope_d8(t, PX)
    acc_plain = device.flow_accumulation(d8)
    plain = device.hand(d8, t, PX, acc=acc_plain, river_threshold=thr, gfi_params=(0.4, 0.1, PX))
    acc_fused = device.flow_accumulation(d8, fuse_hand_threshold=thr)
    fused = device.hand(d8, t, PX, acc=acc_fused, river_threshold=thr, gfi_params=(0.4, 0.1, PX), entry_done=True)
    river = (acc_plain > thr).to(torch.int8)
    masked = device.hand(d8, t, PX, river=river, acc=acc_plain, gfi_params=(0.4, 0.1, PX))
    assert torch.equal(acc_plain, acc_fused)
    for name in ("idx", "fdist", "hand", "gfi"):
        assert torch.equal(plain[name], fused[name]), name
        assert torch.equal(plain[name], masked[name]), name
    acc_ref, _ = oracle.flow_accumulation(d8.cpu().numpy())
    np.testing.assert_array_equal(acc_plain.cpu().numpy(), acc_ref)
    _, idx_ref = oracle.flow_distance_index(d8.cpu().numpy(), (acc_ref > thr).astype(np.int8), PX)
    np.testing.assert_array_equal(fused["idx"].cpu().numpy(), idx_ref)


def test_serpentine_across_tiles():
    """one channel snaking through every row of a 200 x 300 raster (19 000+ moves, hundreds of tile crossings):
    accumulation along the stem, HAND to a single outlet river cell, and the 20 000-move cap with a shorter one"""
    from descriptools_b200 import device

    rows, cols = 200, 300
    d8 = np.zeros((rows, cols), np.uint8)
    for r in range(rows):
        east = r % 2 == 0
        d8[r, :] = 1 if east else 16
        d8[r, cols - 1 if east else 0] = 4  # turn down at the end of the row
    d8[rows - 1, cols - 1 if (rows - 1) % 2 == 0 else 0] = 4  # last cell drains off the raster
    acc_ref, left = oracle.flow_accumulation(d8)
    assert left == 0 and acc_ref.max() == rows * cols - 1
    acc = device.flow_accumulation(torch.from_numpy(d8).cuda(), dtype=torch.int32)
    np.testing.assert_array_equal(acc.cpu().numpy(), acc_ref)
    river = np.zeros((rows, cols), np.int8)
    river[rows - 1, 0 if (rows - 1) % 2 else cols - 1] = 1
    for cap in (0, 12345):  # 0 = the reference's 20000
        f_ref, i_ref = oracle.flow_distance_index(d8, river, PX, max_moves=cap or 20000)
        out = device.hand(torch.from_numpy(d8).cuda(), None, PX, river=torch.from_numpy(river).cuda(), max_moves=cap, want_hand=False)
        np.testing.assert_array_equal(out["idx"].cpu().numpy(), i_ref)
        np.testing.assert_allclose(out["fdist"].cpu().numpy(), f_ref, rtol=RTOL, atol=0)
        assert 0 < (i_ref >= 0).sum() < rows * cols  # the cap cuts the upstream part of the channel


def test_flowacc_large_acyclic_partial_tiles():
    from descriptools_b200 import device

    dem = synth(1111, 777, 9)  # neither dimension a multiple of 64 or 16: generic staging path, clipped tiles
    _, d8 = oracle.slope_d8(dem, PX)
    acc_ref, left = oracle.flow_accumulation(d8)
    acc, bad = device.flow_accumulation(torch.from_numpy(d8).cuda(), check_cycles=True)
    assert left == 0 and bad == 0
    np.testing.assert_array_equal(acc.cpu().numpy(), acc_ref)


def test_forest_accumulate_cuda_matches_torch():
    """band boundary solver: the library's sweep == pointer doubling in torch, on a random forest"""
    from descriptools_b200 import bands

    rng = np.random.default_rng(3)
    n = 50000
    nxt = np.full(n, -1, np.int64)
    for i in range(1, n):  # a random forest: every node points at a lower-numbered node or nowhere
        if rng.random() < 0.9:
            nxt[i] = rng.integers(max(0, i - 50), i)
    base = rng.integers(0, 1 << 33, n).astype(np.int64)
    ref, flag_ref = bands.forest_accumulate(torch.from_numpy(nxt), torch.from_numpy(base), rounds=20)
    got, flag = bands.forest_accumulate(torch.from_numpy(nxt).cuda(), torch.from_numpy(base).cuda())
    assert not bool(flag_ref) and not bool(flag)
    assert torch.equal(got.cpu(), ref)
    nxt[0] = 5  # 0 -> 5 -> ... -> 0: a cycle
    _, flag = bands.forest_accumulate(torch.from_numpy(nxt).cuda(), torch.from_numpy(base).cuda())
    assert bool(flag)


def test_band_inflow_beyond_2_32_carries():
    """int64 counts: inflow carried by the halo rows may exceed 2**32 (100 000 x 100 000).  The finish pass adds it in two
    32-bit halves with a carry; acc must be linear in the inflow: acc(k) = acc(0) + k * (number of halo paths through the
    cell), exactly, for k on both sides of 2**32 and for sums that wrap the low word."""
    import ctypes

    from descriptools_b200._lib import DTB_I64, FlowaccArgs, check, lib

    dem = synth(192, 256, 14, holes=False)
    t = torch.from_numpy(dem).cuda()
    _, d8 = __import__("descriptools_b200").device.slope_d8(t, PX)
    rows, cols = d8.shape
    halo = torch.full((cols,), 4, dtype=torch.uint8, device="cuda")  # every halo cell above flows south into row 0
    ws = torch.empty(lib.dtb_flowacc_workspace_bytes(rows, cols), dtype=torch.uint8, device="cuda")

    def run(k):
        acc = torch.empty((rows, cols), dtype=torch.int64, device="cuda")
        inflow = torch.full((cols,), k, dtype=torch.int64, device="cuda")
        a = FlowaccArgs()
        a.d8, a.rows, a.cols, a.halo_above = d8.data_ptr(), rows, cols, halo.data_ptr()
        a.inflow_above, a.acc, a.acc_dtype, a.nodata_fill, a.mode = inflow.data_ptr(), acc.data_ptr(), DTB_I64, -100, 0
        check(lib.dtb_flowacc_band(ctypes.byref(a), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream), "flowacc")
        torch.cuda.synchronize()
        return acc

    a0, a3 = run(0), run(3)
    m = (a3 - a0) // 3
    assert bool(((a3 - a0) % 3 == 0).all()) and int(m.max()) > 1  # several halo paths merge somewhere
    for k in (2**32 - 1, 2**32 + 11, 2**31 + 5, 3 * 2**32 + 7):
        np.testing.assert_array_equal(run(k).cpu().numpy(), (a0 + k * m).cpu().numpy())


def test_bands_int64_equal_single_gpu():
    """the continental configuration's dtypes (int64 accumulation and indices) through the band path"""
    from descriptools_b200 import pipeline

    dem = synth(640, 336, 12)
    thr = 250
    ref = pipeline.run_device(torch.from_numpy(dem).cuda(), PX, thr)
    got = _run_bands(dem, 3, thr, force_int64=True)
    assert got["acc"].dtype == np.int64 and got["idx"].dtype == np.int64
    for name in ("slope", "d8", "acc", "idx", "fdist", "hand", "gfi"):
        np.testing.assert_array_equal(got[name], ref[name].cpu().numpy().astype(got[name].dtype), err_msg=name)


def test_bands_step_host_matches_device_step():
    from descriptools_b200 import bands

    dem = synth(384, 272, 4)
    thr = 150
    rows, cols = dem.shape
    runner = bands.BandRunner(rows, cols, PX, thr, 0.4, 0.1, nbands=2)
    parts = [torch.from_numpy(dem[a:b].copy()).pin_memory() for a, b in zip(runner.edges, runner.edges[1:])]
    pinned = [{k: torch.empty(tuple(t.shape), dtype=t.dtype).pin_memory() for k, t in b.outputs().items()} for b in runner.bands]
    runner.step_host(parts, pinned)
    host = {k: np.concatenate([p[k].numpy() for p in pinned], 0) for k in pinned[0]}
    ref = _run_bands(dem, 2, thr)
    for k in ref:
        np.testing.assert_array_equal(host[k], ref[k], err_msg=k)


# ---- evaluation.py (SURVEY 8 f1): calibration against the benchmark flood map ---------------------
def test_evaluation_kat1_hand_class(mods, ex):
    """example.py:106-147 end to end on the device: flow_hand_index -> minMaxScale -> calibration -> binary_map ->
    avaliacao reproduces Example/output/hand_class.tif (the reference's only golden output) and its indexes."""
    import descriptools_b200.evaluation as evaluation
    from helpers import avaliacao as avaliacao_ref, binary_map as binary_map_ref, calibration as calibration_ref, min_max_scale

    _, _, hand = mods["flowhand"].flow_hand_index(ex["dem"], ex["fdr"], ex["river"], PX)
    elements = np.unique(hand)
    mn, mx = elements[1], elements[-1]
    desc = evaluation.minMaxScale(hand, mn, mx, -100)
    np.testing.assert_array_equal(desc, min_max_scale(hand, mn, mx, -100))
    flood = ex["flood"].copy()
    th = evaluation.calibration(desc, flood, "under")
    assert th == calibration_ref(desc, ex["flood"].copy()) == pytest.approx(0.012)
    assert set(np.unique(flood)) <= {0, 2}  # remapped in place like the reference
    binary = evaluation.binary_map(desc, th, "under")
    np.testing.assert_array_equal(binary, binary_map_ref(desc, th))
    c, f, cls = evaluation.avaliacao(binary, flood)
    c_ref, f_ref, cls_ref = avaliacao_ref(binary_map_ref(desc, th), ex["flood"].copy())
    assert c == c_ref == pytest.approx(0.8581615676712259, abs=1e-12)
    assert f == f_ref == pytest.approx(0.7240945135019289, abs=1e-12)
    np.testing.assert_array_equal(cls, cls_ref)
    np.testing.assert_array_equal(cls.astype(np.uint8), ex["hand_class"])


def test_evaluation_counts_random_over_and_under():
    import descriptools_b200.evaluation as evaluation
    from helpers import binary_map as binary_map_ref

    rng = np.random.default_rng(8)
    desc = rng.random((300, 257))
    desc[rng.random(desc.shape) < 0.1] = np.nan
    desc[0, 0] = np.nan
    flood = (rng.random(desc.shape) < 0.3).astype(np.int8)
    flood[rng.random(desc.shape) < 0.05] = -100
    for under in ("under", "over"):
        th = 0.37
        b = evaluation.binary_map(desc, th, under)
        ref = binary_map_ref(desc, th, under == "under")
        np.testing.assert_array_equal(b, ref)
        c, f, cls = evaluation.avaliacao(b, flood.copy())
        cmp_ = np.where(flood == 1, 2, np.where(flood == -100, 0, flood))
        ref_cls = ref + cmp_
        tn, fp, fn, tp = [(ref_cls == k).sum() for k in range(4)]
        assert c == tp / (tp + fn) and f == tp / (tp + fn + fp)
        np.testing.assert_array_equal(cls, ref_cls)


def test_evaluation_counts_kernel_against_brute_force():
    """dtb_eval_counts (one pass, up to 32 thresholds): float32 / float64 descriptors, under / over, NaN, +-inf, nodata,
    benchmark values outside 0..3, a length that is not a multiple of 4, an unaligned view, thresholds that are floats
    exactly (f32 comparison in the kernel) and thresholds that are not (f64 comparison)"""
    import descriptools_b200.evaluation as ev

    rng = np.random.default_rng(31)
    n = 257 * 301 + 3
    base = rng.random(n + 5) * 2.0 - 0.5
    base[rng.random(n + 5) < 0.05] = np.nan
    base[rng.random(n + 5) < 0.02] = np.inf
    base[rng.random(n + 5) < 0.02] = -np.inf
    base[rng.random(n + 5) < 0.1] = -100.0  # nodata
    flood_all = rng.choice(np.array([0, 1, -100, 3, 7], np.int8), size=n + 5, p=[0.5, 0.3, 0.1, 0.05, 0.05])
    grids = {"exact": np.linspace(-0.5, 1.5, 17), "inexact": np.linspace(-0.45, 1.45, 32) + 1e-9, "one": np.array([0.3])}
    for dt in (np.float32, np.float64):
        for off in (0, 1):  # off = 1: the device pointers are not 16-byte aligned
            desc_t = torch.from_numpy(base.astype(dt)).cuda()[off:off + n]
            flood_t = torch.from_numpy(flood_all).cuda()[off:off + n]
            d = desc_t.cpu().numpy()
            f = flood_t.cpu().numpy()
            cmp_ = np.where(f == 1, 2, np.where(f == -100, 0, f)).astype(np.int64)
            usable = ~np.isnan(d) & (d != dt(-100.0))
            for under in ("under", "over"):
                ctr = ev._Counter(desc_t, dt is np.float64, -100.0, flood_t, under)
                for name, th in grids.items():
                    got = ctr.counts(th.tolist())
                    for i, t in enumerate(th):
                        tt = dt(t)  # NumPy compares a float32 array with a Python float in float32
                        with np.errstate(invalid="ignore"):
                            hit = usable & ((d <= tt) if under == "under" else (d >= tt))
                        cls = hit.astype(np.int64) + cmp_
                        # classes above 3 (benchmark 3 + flagged) are not counted; benchmark values outside 0..3 are skipped
                        ok = (cmp_ >= 0) & (cmp_ <= 3)
                        want = [int(((cls == c) & ok).sum()) for c in range(4)]
                        assert got[i].tolist() == want, (dt.__name__, off, under, name, i)
    # the C ABI itself takes any f64 thresholds: a float32 descriptor is then compared in f64, (double)d <= th
    import ctypes

    from descriptools_b200._lib import check, lib

    desc_t = torch.from_numpy(base[:n].astype(np.float32)).cuda()
    flood_t = torch.from_numpy(flood_all[:n]).cuda()
    d = desc_t.cpu().numpy().astype(np.float64)
    cmp_ = np.where(flood_all[:n] == 1, 2, np.where(flood_all[:n] == -100, 0, flood_all[:n])).astype(np.int64)
    ok = (cmp_ >= 0) & (cmp_ <= 3)
    th = np.ascontiguousarray(grids["inexact"])
    ws = torch.empty(4 * 33 * 8, dtype=torch.uint8, device="cuda")
    for under in (1, 0):
        res = np.zeros((len(th), 4), np.int64)
        check(lib.dtb_eval_counts(desc_t.data_ptr(), 0, flood_t.data_ptr(), n, -100.0, th.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                  len(th), under, res.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), ws.data_ptr(), ws.numel(),
                                  torch.cuda.current_stream().cuda_stream), "dtb_eval_counts")
        for i, t in enumerate(th):
            with np.errstate(invalid="ignore"):
                hit = ~np.isnan(d) & (d != -100.0) & ((d <= t) if under else (d >= t))
            cls = hit.astype(np.int64) + cmp_
            assert res[i].tolist() == [int(((cls == c) & ok).sum()) for c in range(4)], (under, i)


def test_evaluation_float32_thresholds_compare_like_numpy():
    """cells exactly at float32(threshold): NumPy compares a float32 descriptor with a Python float in float32"""
    import descriptools_b200.evaluation as ev

    th = 0.1  # not representable: float32(0.1) > 0.1
    desc = np.full((8, 16), np.float32(th), np.float32)
    desc[0, 0] = -100.0  # the reference takes the value at [0, 0] for nodata (evaluation.py:110)
    desc[1, :4] = np.float32(0.5)

    def reference(d, under):  # evaluation.py:110-121, verbatim semantics
        d = np.where(d == d[0, 0], np.nan, d)
        hit = d <= th if under == "under" else d >= th
        return np.where(np.isnan(d), 0, np.where(hit, 1, 0))

    want = reference(desc, "under")  # float32 comparison: the cells at float32(0.1) > 0.1 still count as <= 0.1
    assert want.sum() == desc.size - 5
    np.testing.assert_array_equal(ev.binary_map(desc, th, "under"), want)
    np.testing.assert_array_equal(ev.binary_map(desc, th, "over"), reference(desc, "over"))
    d64 = desc.astype(np.float64)
    np.testing.assert_array_equal(ev.binary_map(d64, th, "under"), reference(d64, "under"))  # float64: 0.1000000015 > 0.1


def test_bands_downslope_equals_single_gpu():
    from descriptools_b200 import bands, device

    dem = synth(384, 300, 21)
    rows, cols = dem.shape
    t = torch.from_numpy(dem).cuda()
    _, d8 = device.slope_d8(t, PX)
    ref = device.downslope(t, d8, PX, 5.0).cpu().numpy()
    np.testing.assert_array_equal(ref, oracle.downslope(dem, d8.cpu().numpy(), PX, 5.0))
    runner = bands.BandRunner(rows, cols, PX, 200, nbands=3)
    runner.load([torch.from_numpy(dem[a:b]) for a, b in zip(runner.edges, runner.edges[1:])])
    runner.step()
    got = torch.cat(runner.downslope(5.0), 0).cpu().numpy()
    np.testing.assert_array_equal(got, ref)
    # a tiny halo: walks escape the window, the driver widens it (x4) until none does, then has to fall back to the
    # replicated form when the windows already hold their whole neighbours -- same result every way
    for h in (1, 7, 64):
        np.testing.assert_array_equal(torch.cat(runner.downslope(5.0, halo_rows=h), 0).cpu().numpy(), ref)
    np.testing.assert_array_equal(torch.cat(runner._downslope_replicated(5.0), 0).cpu().numpy(), ref)
    assert not (got == -50).any()


def test_downslope_window_marks_escaping_walks():
    """dtb_downslope_window: cells whose walk leaves through an open side get the reference's -50 marker and are counted;
    everything else equals the whole-raster result."""
    from descriptools_b200 import device
    from descriptools_b200._lib import check, lib

    dem = synth(256, 200, 8, holes=False)
    t = torch.from_numpy(dem).cuda()
    _, d8 = device.slope_d8(t, PX)
    ref = device.downslope(t, d8, PX, 5.0)
    a, b = 96, 160  # window = rows [a-16, b+16), band = [a, b)
    wd, w8 = t[a - 16:b + 16].contiguous(), d8[a - 16:b + 16].contiguous()
    out = torch.empty((b - a, 200), dtype=torch.float32, device="cuda")
    esc = torch.zeros(1, dtype=torch.int64, device="cuda")
    check(lib.dtb_downslope_window(wd.data_ptr(), 0, w8.data_ptr(), b - a + 32, 200, 16, 16 + b - a, PX, 5.0, 0, out.data_ptr(), 1, 1,
                                   esc.data_ptr(), torch.cuda.current_stream().cuda_stream), "dtb_downslope_window")
    flagged = out == -50
    assert int(esc.item()) == int(flagged.sum()) > 0
    np.testing.assert_array_equal(out[~flagged].cpu().numpy(), ref[a:b][~flagged].cpu().numpy())


def test_fused_hand_tiles_beyond_the_compact_counters():
    """in-tile paths of 256+ moves of one kind do not fit the 8-bit counters of the compact tile pass: a serpentine
    narrower than a tile (3 800+ cardinal moves inside one tile) must go through the list to the 64-bit pass and
    still match the oracle.  Serpentines and rows wider than a tile leave every tile within 64 + 64 moves: the
    compact pass keeps them."""
    for rows, cols, listed in ((200, 300, False), (200, 60, True)):
        d8 = serpentine_d8(rows, cols)
        dem = (np.arange(rows * cols, dtype=np.float32)[::-1].reshape(rows, cols) * 0.01 + 5).copy()
        prof = hand_fused_vs_oracle(d8, dem, rows * cols - 500)
        assert prof["hand_tile_kernel<listed>"][0] > 0.0
        assert (listed_tiles(rows, cols) > 0) == listed, (rows, cols)
    # every row flows east across ten tiles
    d8 = np.full((128, 640), 1, np.uint8)
    d8[:, -1] = 4
    d8[-1, -1] = 4
    dem = np.linspace(900, 1, 128 * 640, dtype=np.float32).reshape(128, 640).copy()
    hand_fused_vs_oracle(d8, dem, 128 * 640 - 700)


def test_fused_hand_random_codes_with_cycles():
    """arbitrary D8 grids on the fused path: the flat sweep handles flow accumulation, the compact tile pass must
    hand every tile with an in-tile cycle to the 64-bit pass"""
    rng = np.random.default_rng(5)
    d8 = rng.choice(np.array([0, 1, 2, 4, 8, 16, 32, 64, 128, 3, 255], np.uint8), (150, 200),
                    p=[.03, .2, .1, .2, .1, .1, .08, .08, .08, .015, .015])
    dem = (rng.standard_normal(d8.shape) * 10 + 100).astype(np.float32)
    dem[rng.random(d8.shape) < 0.02] = -100
    hand_fused_vs_oracle(d8, dem, 3)
    assert listed_tiles(150, 200) > 0


def test_hand_boundary_solver_cuda_equals_torch():
    """dtb_hand_boundary_solve (rank 0 of the band driver) against the torch pointer doubling the CPU / gloo tests
    use: random boundary graphs with chains over several seams, dead ends and cycles across seams"""
    from descriptools_b200 import bands

    rng = np.random.default_rng(11)
    for n, cols, p_exit in ((2, 257, 0.5), (5, 1000, 0.7), (8, 640, 0.3)):
        kind = rng.choice([0, 1, 2, 3], size=(n, 2, cols), p=[0.1, 0.72 * (1 - p_exit), 0.18 * (1 - p_exit), 0.9 * p_exit])
        nd = rng.integers(0, 300, (n, 2, cols))
        nc = rng.integers(0, 300, (n, 2, cols))
        t_side = rng.integers(0, 2, (n, 2, cols))
        t_col = rng.integers(0, cols, (n, 2, cols))
        state = (kind.astype(np.int64) << 62) | (nd.astype(np.int64) << 47) | (nc.astype(np.int64) << 32)
        state = np.where(kind == 3, state | (1 << 31) | (t_side.astype(np.int64) << 30) | t_col, state)
        state = np.where(kind == 0, 0, state)  # not an entry
        summ = np.zeros((n, 8, cols), np.int64)
        summ[:, 0], summ[:, 4] = state[:, 0], state[:, 1]
        summ[:, 1:4] = rng.integers(1, 1 << 40, (n, 3, cols))
        summ[:, 5:8] = rng.integers(1, 1 << 40, (n, 3, cols))
        t = torch.from_numpy(summ)
        ref, flag_ref = bands.solve_hand_boundary(t)
        got, flag = bands.solve_hand_boundary(t.cuda())
        ref, got = ref.numpy(), got.cpu().numpy()
        assert bool(flag) == bool(flag_ref)
        for row in (0, 4):
            k_ref, k_got = (ref[:, row] >> 62) & 3, (got[:, row] >> 62) & 3
            np.testing.assert_array_equal(k_got, k_ref)
            river = k_ref == 1
            assert river.any()
            np.testing.assert_array_equal(got[:, row][river], ref[:, row][river])
            for k in (1, 2, 3):
                np.testing.assert_array_equal(got[:, row + k][river], ref[:, row + k][river])
