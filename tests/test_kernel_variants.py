"""Kernel instantiations the public API reaches that the float32 parity tests do not: int16 DEMs through the slope / D8
stencil (both kinds of 100/px, band rows) and through the fused chain (the compact and the listed 64-bit HAND tile
passes, int16 HAND that wraps like NumPy), every output subset of the fused and unfused HAND paths, the accumulation /
index widths, the move cap on the fused path, caller outputs that are not 16-byte aligned, and int16 GeoTIFFs through
pipeline_files.  Every result is compared with the CPU oracle, or bit for bit with a path that is itself compared with
it.  Integer rasters, slope, D8 and HAND are bit-exact; fdist and GFI keep the suite's RTOL / ATOL.
"""
import functools
import itertools
import math

import numpy as np
import pytest
import torch

import oracle
from helpers import ATOL, PX, RTOL, hand_fused_vs_oracle, listed_tiles, serpentine_d8, synth

gpu = pytest.mark.gpu
ND = -100
N_GFI, B_GFI = 0.4, 0.1
HAND_OUTS = ("fdist", "idx", "hand", "gfi")
CHAIN = ("slope", "d8", "acc", "fdist", "idx", "hand", "gfi")
# 100/px is a power of two for 12.5 and 25 (the stencil's exact cardinal product, CX = true), not for the others
STENCIL_PX = (12.5, 25.0, 30.0, 90.0, 1.0, 7.77)


def pow2_cardinal(px):
    """the host's choice of the stencil's exact-cardinal-product form (csrc/slope_d8.cu, dtb_slope_d8)"""
    kc = 100.0 / px
    return math.frexp(kc)[0] == 0.5 and 2.0 ** -20 <= kc <= 2.0 ** 20


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a).copy()).cuda()


def profiled(fn):
    """(fn(), {kernel name: (ms, launches)} of what fn launched)"""
    from descriptools_b200 import _lib

    _lib.profile_enable(True)
    try:
        res = fn()
        torch.cuda.synchronize()
        prof = _lib.profile_collect()
    finally:
        _lib.profile_enable(False)
    return res, prof


# ---- inputs ------------------------------------------------------------------------------------------
def stencil_dem16(rows, cols, seed):
    """int16 stencil input: rough terrain, full-range noise (-32768 next to 32767 included), integer plateaus and a
    patch of values 0..3 (heavy ties inside each class), -100 blobs, and -101 / -9999 / -32768 cells (nodata centres,
    ordinary neighbours)"""
    rng = np.random.default_rng(seed)
    z = np.cumsum(rng.integers(-40, 41, (rows, cols)), axis=1) + np.cumsum(rng.integers(-40, 41, (rows, 1)), axis=0) + 2000
    z = np.clip(z, -32768, 32767)
    noisy = rng.random((rows, cols)) < 0.15
    z[noisy] = rng.integers(-32768, 32768, int(noisy.sum()))
    for _ in range(max(2, rows * cols // 3000)):
        r, c = int(rng.integers(0, rows)), int(rng.integers(0, cols))
        h, w = (int(v) for v in rng.integers(1, 30, 2))
        kind = rng.integers(0, 3)
        if kind == 0:
            z[r:r + h, c:c + w] = ND
        elif kind == 1:
            z[r:r + h, c:c + w] = int(rng.integers(-3000, 3000))
        else:
            z[r:r + h, c:c + w] = rng.integers(0, 4, z[r:r + h, c:c + w].shape)
    special = rng.random((rows, cols)) < 0.03
    z[special] = rng.choice(np.array([-32768, 32767, -101, -9999, ND, 0]), int(special.sum()))
    flat = z.reshape(-1)
    flat[0], flat[-1] = 32767, -32768
    flat[flat.size // 2] = -32768
    if flat.size > 2:
        flat[flat.size // 2 + 1] = 32767
    return z.astype(np.int16)


@functools.lru_cache(maxsize=None)
def valley16(rows, cols, seed=1):
    """int16 valley that drains everything: z = lateral(|c - centre(r)|) + (rows-1-r) * 2 + noise{0,1} - 99, centre(r) =
    cols/2 + round(20 sin(r/25)).  The lateral rise of each row tops out at the int16 maximum, so in the lowest ~50 rows
    (valley floor below 0) the farthest cells drop more than 32767 to the floor: their int16 HAND wraps."""
    rng = np.random.default_rng(seed)
    r = np.arange(rows)[:, None]
    c = np.arange(cols)[None, :]
    centre = cols // 2 + np.round(20 * np.sin(r / 25)).astype(np.int64)
    dist = np.abs(c - centre)
    down = (rows - 1 - r) * 2
    wall = (32767 - 1 - (down - 99)) / np.maximum(dist.max(axis=1, keepdims=True), 1)
    z = np.floor(dist * wall).astype(np.int64) + down + rng.integers(0, 2, (rows, cols)) - 99
    assert z.max() <= 32767 and z.min() >= -99
    return z.astype(np.int16)


@functools.lru_cache(maxsize=None)
def rough16(rows, cols, seed=7):
    """int16 DEM that no GIS has conditioned: the synthetic terrain in decimetres (flats, pits) with -100 blobs"""
    z = np.round(oracle.synth_dem(rows, cols, 0, seed) * 10).astype(np.int16)
    rng = np.random.default_rng(seed)
    for _ in range(5):
        r, c = int(rng.integers(0, rows)), int(rng.integers(0, cols))
        z[r:r + int(rng.integers(1, 12)), c:c + int(rng.integers(1, 12))] = ND
    return z


@functools.lru_cache(maxsize=None)
def synth_f32(rows, cols, seed=3):
    return synth(rows, cols, seed)


@functools.lru_cache(maxsize=None)
def snake16(rows=251, cols=256):
    """one channel through every second row (walls of 32767 between), joined at alternate ends: a path of
    (rows+1)/2 * cols + (rows-1)/2 cells, longer than the largest move cap (32000), crossing a 64-cell tile seam
    every 64 moves"""
    z = np.full((rows, cols), 32767, np.int64)
    order = []
    for r in range(0, rows, 2):
        east = (r // 2) % 2 == 0
        order += [(r, c) for c in (range(cols) if east else range(cols - 1, -1, -1))]
        if r + 1 < rows:
            order.append((r + 1, cols - 1 if east else 0))
    for p, (r, c) in enumerate(order):
        z[r, c] = -99 + (len(order) - 1 - p)
    assert z.max() <= 32767 and len(order) - 1 > 32000
    return z.astype(np.int16)


DEMS = {"valley": valley16, "rough": rough16, "synth_f32": synth_f32, "snake": snake16}


def chain_oracle(dem, px, thr, max_moves=oracle.MAX_MOVES_HAND):
    slope, d8 = oracle.slope_d8(dem, px)
    acc, _ = oracle.flow_accumulation(d8)
    fdist, idx = oracle.flow_distance_index(d8, (acc > thr).astype(np.int8), px, max_moves)
    hand = oracle.hand(dem, idx)
    gfi = oracle.gfi(hand, acc, idx, N_GFI, B_GFI, px)
    return dict(slope=slope, d8=d8, acc=acc, fdist=fdist, idx=idx, hand=hand, gfi=gfi)


@pytest.fixture(scope="module")
def ref():
    """ref(kind, shape, thr, max_moves) -> (dem, oracle chain), each computed once per module: the oracle's HAND walk
    is O(cells x path length)"""
    cache = {}

    def get(kind, shape, thr, max_moves=oracle.MAX_MOVES_HAND):
        dem = DEMS[kind](*shape)
        key = (kind, shape, thr, max_moves)
        if key not in cache:
            cache[key] = chain_oracle(dem, PX, thr, max_moves)
        return dem, cache[key]

    return get


def host(t):
    return t.cpu().numpy() if isinstance(t, torch.Tensor) else t


def assert_outputs(got, want, names, msg=""):
    for name in names:
        g = host(got[name])
        if name == "fdist":
            np.testing.assert_allclose(g, want[name], rtol=RTOL, atol=0, err_msg=f"{name} {msg}")
        elif name == "gfi":
            np.testing.assert_allclose(g, want[name], rtol=RTOL, atol=ATOL, err_msg=f"{name} {msg}")
        else:
            np.testing.assert_array_equal(g, want[name], err_msg=f"{name} {msg}")


# ---- 1. int16 stencil ----------------------------------------------------------------------------------
STENCIL_SHAPES = [(260, 516), (260, 517), (260, 518), (260, 519), (1, 300), (1, 7), (300, 1), (5, 1), (3, 3)]


@pytest.mark.parametrize("px", STENCIL_PX + (0.25,))
def test_oracle_int16_stencil_equals_float32(px):
    """the oracle's int16 stencil is its float32 stencil on the same values: what lets the TMA kernel (float32 only)
    stand in for the oracle on int16 inputs below"""
    for k, shape in enumerate(STENCIL_SHAPES):
        z = stencil_dem16(*shape, seed=100 + k)
        s16, d16 = oracle.slope_d8(z, px)
        s32, d32 = oracle.slope_d8(z.astype(np.float32), px)
        np.testing.assert_array_equal(s16, s32, err_msg=str(shape))
        np.testing.assert_array_equal(d16, d32, err_msg=str(shape))
    # the stencil tests below reach both forms of the cardinal product
    assert {pow2_cardinal(p) for p in STENCIL_PX} == {True, False}


@gpu
@pytest.mark.parametrize("px", STENCIL_PX)
def test_int16_stencil_vs_oracle(px):
    """slope_d8_generic_kernel<int16_t, CX> (CX = 100/px is a power of two) on widths 4k .. 4k+3, 1 x N and N x 1, in
    all three launch forms"""
    from descriptools_b200 import device

    for k, shape in enumerate(STENCIL_SHAPES):
        z = stencil_dem16(*shape, seed=100 + k)
        s_ref, d_ref = oracle.slope_d8(z, px)
        t = cuda(z)
        (s, d), prof = profiled(lambda: device.slope_d8(t, px))
        assert "slope_d8_generic_kernel<i16>" in prof and "slope_d8_tma_kernel" not in prof
        np.testing.assert_array_equal(host(s), s_ref, err_msg=f"slope {shape}")
        np.testing.assert_array_equal(host(d), d_ref, err_msg=f"d8 {shape}")
        s, _ = device.slope_d8(t, px, want_d8=False)
        np.testing.assert_array_equal(host(s), s_ref, err_msg=f"slope only {shape}")
        _, d = device.slope_d8(t, px, want_slope=False)
        np.testing.assert_array_equal(host(d), d_ref, err_msg=f"d8 only {shape}")


@gpu
@pytest.mark.parametrize("px", [12.5, 30.0])
def test_int16_stencil_band_rows(px):
    """int16 rows [row_begin, row_end) of a buffer with halo rows == the same rows of the whole raster (the form
    pipeline.pipeline launches on each row block of the DEM)"""
    from descriptools_b200 import device

    rows, cols = 300, 259
    z = stencil_dem16(rows, cols, seed=5)
    s_ref, d_ref = oracle.slope_d8(z, px)
    t = cuda(z)
    for a, b in [(0, 100), (100, 217), (217, 300), (150, 151)]:
        lo, hi = max(a - 1, 0), min(b + 1, rows)
        s, d = device.slope_d8(t[lo:hi].contiguous(), px, row_begin=a - lo, row_end=b - lo)
        np.testing.assert_array_equal(host(s), s_ref[a:b], err_msg=f"rows {a}:{b}")
        np.testing.assert_array_equal(host(d), d_ref[a:b], err_msg=f"rows {a}:{b}")
        # and over the whole buffer
        s, d = device.slope_d8(t, px, row_begin=a, row_end=b)
        np.testing.assert_array_equal(host(s), s_ref[a:b])
        np.testing.assert_array_equal(host(d), d_ref[a:b])


@gpu
@pytest.mark.parametrize("px", STENCIL_PX)
def test_int16_generic_equals_float32_tma(px):
    """no oracle involved: the int16 values as float32 in an aligned buffer with cols % 4 == 0 go through the TMA
    kernel, and must give exactly what the int16 generic kernel gives (all three launch forms)"""
    from descriptools_b200 import device

    z = stencil_dem16(300, 512, seed=9)
    t16, t32 = cuda(z), cuda(z.astype(np.float32))
    assert t32.data_ptr() % 16 == 0 and z.shape[1] % 4 == 0
    for ws, wd in [(True, True), (True, False), (False, True)]:
        (s16, d16), p16 = profiled(lambda: device.slope_d8(t16, px, want_slope=ws, want_d8=wd))
        (s32, d32), p32 = profiled(lambda: device.slope_d8(t32, px, want_slope=ws, want_d8=wd))
        assert "slope_d8_generic_kernel<i16>" in p16 and "slope_d8_tma_kernel" in p32 and "slope_d8_generic_kernel<f32>" not in p32
        if ws:
            assert torch.equal(s16, s32), (ws, wd)
        if wd:
            assert torch.equal(d16, d32), (ws, wd)


# ---- 2. int16 through the fused chain ------------------------------------------------------------------
# 640 x 1024: every tile full and 16-byte tileable; 577 x 976: last tile column 16- but not 64-aligned, partial last
# tile row; 300 x 411: width not a multiple of 16; 40 x 50: less than one tile
CHAIN_SHAPES = [(640, 1024), (577, 976), (300, 411), (40, 50)]


def _above_max(kind, shape):
    _, d8 = oracle.slope_d8(DEMS[kind](*shape), PX)
    return int(oracle.flow_accumulation(d8)[0].max()) + 1


@gpu
@pytest.mark.parametrize("kind", ["valley", "rough"])
@pytest.mark.parametrize("shape", CHAIN_SHAPES)
@pytest.mark.parametrize("thr", [10, 4095, 4096, "above_max"])
def test_int16_run_device_vs_oracle(ref, kind, shape, thr):
    """pipeline.run_device on an int16 DEM: all seven rasters against the oracle chain, HAND stays int16; the host
    row-block path (pipeline.pipeline) on the same NumPy DEM gives the same rasters"""
    from descriptools_b200 import pipeline

    if thr == "above_max":
        thr = _above_max(kind, shape)
    dem, want = ref(kind, shape, thr)
    assert dem.dtype == np.int16
    res, prof = profiled(lambda: pipeline.run_device(cuda(dem), PX, thr))
    assert res["hand"].dtype == torch.int16
    assert "slope_d8_generic_kernel<i16>" in prof and "hand_tile_kernel<table>" in prof
    assert_outputs(res, want, CHAIN, f"{kind} {shape} thr={thr}")
    got = pipeline.pipeline(dem, PX, thr, N_GFI, B_GFI)
    assert got["hand"].dtype == np.int16
    for name in CHAIN:
        np.testing.assert_array_equal(got[name], host(res[name]), err_msg=f"pipeline.pipeline {name}")


@gpu
def test_int16_hand_wraps_like_numpy(ref):
    """HAND = z - z[idx] in int16 wraps as NumPy's does (then negative -> 0): cells whose true drop exceeds 32767 exist
    and come out as NumPy computes them on the fused path"""
    from descriptools_b200 import pipeline

    shape, thr = (577, 976), 4096
    dem, want = ref("valley", shape, thr)
    idx = want["idx"]
    ok = idx >= 0
    drop = np.zeros(shape, np.int64)
    drop[ok] = dem[ok].astype(np.int64) - dem.reshape(-1)[idx[ok]].astype(np.int64)
    wrapped = drop > 32767
    assert wrapped.sum() >= 20
    with np.errstate(over="ignore"):
        h = np.where(ok, dem - dem.reshape(-1)[np.where(ok, idx, 0)], np.int16(ND)).astype(np.int16)  # flowhand.py:436
    h = np.where((h < 0) & (h != ND), np.int16(0), h)  # flowhand.py:438
    np.testing.assert_array_equal(want["hand"], h)  # the oracle wraps too
    res = pipeline.run_device(cuda(dem), PX, thr)
    np.testing.assert_array_equal(host(res["hand"]), h)
    np.testing.assert_array_equal(host(res["hand"])[wrapped], h[wrapped])
    assert (h[wrapped] != np.minimum(drop[wrapped], 32767)).all()  # a saturating subtraction would differ on every one


@gpu
def test_int16_fused_listed_64bit_pass():
    """int16 DEM on tiles the compact pass cannot represent (in-tile paths of 256+ cardinal moves, and in-tile cycles
    of random codes): hand_tile_kernel<int16_t, ..., TABLE=true> over the listed tiles, against the oracle"""
    rows, cols = 200, 60  # narrower than a tile: up to 64 x 60 cardinal moves inside one tile
    d8 = serpentine_d8(rows, cols)
    dem = (np.arange(rows * cols)[::-1].reshape(rows, cols) * 2 - 99).astype(np.int16)
    prof = hand_fused_vs_oracle(d8, dem, rows * cols - 500)
    assert "hand_tile_kernel<listed>" in prof and listed_tiles(rows, cols) > 0
    rng = np.random.default_rng(5)
    d8 = rng.choice(np.array([0, 1, 2, 4, 8, 16, 32, 64, 128, 3, 255], np.uint8), (150, 200),
                    p=[.03, .2, .1, .2, .1, .1, .08, .08, .08, .015, .015])
    dem = rng.integers(-2000, 30000, d8.shape).astype(np.int16)
    dem[rng.random(d8.shape) < 0.02] = ND
    hand_fused_vs_oracle(d8, dem, 3)
    assert listed_tiles(150, 200) > 0


# ---- 3. output subsets -----------------------------------------------------------------------------------
SUBSET_SHAPE = (257, 336)  # partial tiles; 336 = 21 x 16: the epilogue's vector form on full tiles


def _poisoned(shape, dtype):
    t = torch.empty(shape, dtype=dtype, device="cuda")
    t.view(torch.uint8).fill_(0x5A)
    return t


def _hand_outputs(d8, dem, acc, thr, fused, **kw):
    from descriptools_b200 import device

    if fused:
        acc = device.flow_accumulation(d8, dtype=acc.dtype, fuse_hand_threshold=thr)
        return device.hand(d8, dem, PX, acc=acc, river_threshold=thr, entry_done=True, **kw)
    return device.hand(d8, dem, PX, acc=acc, river_threshold=thr, **kw)


@gpu
@pytest.mark.parametrize("kind,thr", [("synth_f32", 300), ("valley", 4096)])
@pytest.mark.parametrize("fused", [True, False], ids=["fused", "unfused"])
def test_hand_output_subsets(ref, kind, thr, fused):
    """every request of fdist / idx / hand / gfi (gfi without hand included; the compact tile pass takes its ALL=false
    form for all but the full one): each wanted raster equals what the all-outputs call writes, bit for bit, the others
    come back absent and their caller buffers untouched"""
    from descriptools_b200 import device

    dem, want = ref(kind, SUBSET_SHAPE, thr)
    t = cuda(dem)
    _, d8 = device.slope_d8(t, PX)
    acc = device.flow_accumulation(d8)
    (full, prof) = profiled(lambda: _hand_outputs(d8, t, acc, thr, fused, gfi_params=(N_GFI, B_GFI, PX)))
    assert ("hand_tile_kernel<table>" in prof) == fused and full["hand"].dtype == t.dtype
    assert_outputs(full, want, HAND_OUTS, f"{kind} all outputs")
    dts = dict(fdist=torch.float32, idx=full["idx"].dtype, hand=t.dtype, gfi=torch.float32)
    for wanted in itertools.product([False, True], repeat=4):
        names = [n for n, w in zip(HAND_OUTS, wanted) if w]
        given = {n: _poisoned(SUBSET_SHAPE, dts[n]) for n in HAND_OUTS}
        poison = {n: given[n].clone() for n in HAND_OUTS}
        got = _hand_outputs(d8, t, acc, thr, fused, want_fdist=wanted[0], want_idx=wanted[1], want_hand=wanted[2],
                            gfi_params=(N_GFI, B_GFI, PX) if wanted[3] else None, out=given)
        assert sorted(got) == sorted(names), names
        for n in HAND_OUTS:
            if n in names:
                assert got[n] is given[n] and torch.equal(got[n], full[n]), (n, names)
            else:
                assert torch.equal(given[n], poison[n]), (n, names)


# ---- 4. accumulation x index x DEM widths ---------------------------------------------------------------------
WIDTH_SHAPE = (333, 976)


@gpu
@pytest.mark.parametrize("kind,thr", [("synth_f32", 300), ("valley", 4096)])
@pytest.mark.parametrize("acc_dt", [torch.int32, torch.int64], ids=["acc32", "acc64"])
@pytest.mark.parametrize("idx_dt", [torch.int32, torch.int64], ids=["idx32", "idx64"])
@pytest.mark.parametrize("fused", [True, False], ids=["fused", "unfused"])
def test_hand_acc_idx_widths(ref, kind, thr, acc_dt, idx_dt, fused):
    """fused (flow_accumulation(fuse_hand_threshold) + hand(entry_done)) and unfused (hand_entry_kernel<ACC> on
    river = acc > threshold) HAND for every accumulation / index width against the oracle"""
    from descriptools_b200 import device

    dem, want = ref(kind, WIDTH_SHAPE, thr)
    t = cuda(dem)
    _, d8 = device.slope_d8(t, PX)

    def run():
        if fused:
            acc = device.flow_accumulation(d8, dtype=acc_dt, fuse_hand_threshold=thr)
        else:
            acc = device.flow_accumulation(d8, dtype=acc_dt)
        out = device.hand(d8, t, PX, acc=acc, river_threshold=thr, gfi_params=(N_GFI, B_GFI, PX), idx_dtype=idx_dt,
                          entry_done=fused)
        out["acc"] = acc
        return out

    out, prof = profiled(run)
    assert ("hand_entry_kernel" in prof) != fused and ("fa_tile_finish_kernel<hand>" in prof) == fused
    assert out["acc"].dtype == acc_dt and out["idx"].dtype == idx_dt and out["hand"].dtype == t.dtype
    assert_outputs(out, want, ("acc",) + HAND_OUTS, f"{kind} {acc_dt} {idx_dt}")


# ---- 5. move cap on the fused path --------------------------------------------------------------------------
CAPS = (1, 5, 63, 64, 65, 255, 256, 4096, 20000, 32000)


@pytest.fixture(scope="module")
def snake_runs():
    """snake DEM: threshold that makes the last cells of the channel the river, and the uncapped run of both DEM types"""
    from descriptools_b200 import pipeline

    dem = snake16()
    _, d8 = oracle.slope_d8(dem, PX)
    thr = int(oracle.flow_accumulation(d8)[0].max()) - 20
    free = {dt: {k: host(v) for k, v in pipeline.run_device(cuda(dem.astype(dt)), PX, thr).items()} for dt in (np.int16, np.float32)}
    return dem, thr, free


@gpu
@pytest.mark.parametrize("cap", CAPS)
def test_fused_move_cap(ref, snake_runs, cap):
    """run_device(max_moves=k) against oracle.flow_distance_index(..., max_moves=k) on a channel of 32 000+ moves that
    crosses a tile seam every 64 moves: every cap cuts paths, and changes nothing but fdist, idx, hand and gfi"""
    from descriptools_b200 import pipeline

    dem, thr, free = snake_runs
    _, want = ref("snake", dem.shape, thr, cap)
    resolved = int((want["idx"] >= 0).sum())
    assert 0 < resolved < dem.size  # the cap cuts the upstream part of the channel
    if cap > 1:
        assert resolved > int((ref("snake", dem.shape, thr, CAPS[CAPS.index(cap) - 1])[1]["idx"] >= 0).sum())
    for dt in (np.int16, np.float32):
        res = {k: host(v) for k, v in pipeline.run_device(cuda(dem.astype(dt)), PX, thr, max_moves=cap).items()}
        assert res["hand"].dtype == dt
        for name in ("slope", "d8", "acc"):
            np.testing.assert_array_equal(res[name], free[dt][name], err_msg=f"{name} changed by the cap ({dt.__name__})")
        w = dict(want, hand=oracle.hand(dem.astype(dt), want["idx"]))
        w["gfi"] = oracle.gfi(w["hand"], want["acc"], want["idx"], N_GFI, B_GFI, PX)
        assert_outputs(res, w, HAND_OUTS, f"cap={cap} {dt.__name__}")


# ---- 6. caller outputs that are not 16-byte aligned ---------------------------------------------------------
def _offset_views(rows, cols, dtypes):
    """contiguous views one element into their buffers (4 bytes for float32 / int32, 2 for int16, ...), poisoned"""
    out = {}
    for name, dt in dtypes.items():
        buf = torch.empty(rows * cols + 1, dtype=dt, device="cuda")
        buf.view(torch.uint8).fill_(0x5A)
        out[name] = buf[1:].view(rows, cols)
        assert out[name].data_ptr() % 16 != 0
    return out


@gpu
@pytest.mark.parametrize("kind,thr", [("synth_f32", 300), ("valley", 4096)])
def test_unaligned_caller_outputs(ref, kind, thr):
    """out= views that start one element into their buffers, on a width that is a multiple of 16 (tiles take the fast
    path, the epilogue its per-cell stores): fused path and run_device equal the aligned call and the oracle"""
    from descriptools_b200 import device, pipeline

    shape = (577, 976)
    assert shape[1] % 16 == 0
    dem, want = ref(kind, shape, thr)
    t = cuda(dem)
    aligned = pipeline.run_device(t, PX, thr)
    assert all(v.data_ptr() % 16 == 0 for v in aligned.values())
    assert_outputs(aligned, want, CHAIN, kind)
    dts = {k: v.dtype for k, v in aligned.items()}
    views = _offset_views(*shape, dts)
    got = pipeline.run_device(t, PX, thr, out=views)
    for name in CHAIN:
        assert got[name] is views[name] and torch.equal(got[name], aligned[name]), name
    views = _offset_views(*shape, {k: dts[k] for k in ("acc",) + HAND_OUTS})
    acc = device.flow_accumulation(aligned["d8"], fuse_hand_threshold=thr, out=views)
    got = device.hand(aligned["d8"], t, PX, acc=acc, river_threshold=thr, gfi_params=(N_GFI, B_GFI, PX), entry_done=True, out=views)
    assert acc is views["acc"] and torch.equal(acc, aligned["acc"])
    for name in HAND_OUTS:
        assert got[name] is views[name] and torch.equal(got[name], aligned[name]), name


# ---- 7. int16 GeoTIFF in, GeoTIFFs out ---------------------------------------------------------------------
@gpu
def test_pipeline_files_int16_geotiff(ref, tmp_path):
    """an LZW-tiled int16 DEM whose nodata is -32768 (the reference example's DEM type): pipeline_files with the host
    and the device codecs keeps it int16 and writes what pipeline.pipeline gives for the array with -32768 -> -100,
    which matches the oracle"""
    import descriptools_b200.raster as rio
    from descriptools_b200 import pipeline

    rows, cols, thr = 300, 420, 2000
    dem = valley16(rows, cols).copy()
    hole = np.zeros(dem.shape, bool)
    hole[40:70, 100:160] = True
    hole[200:205, 300:420] = True
    stored = np.where(hole, np.int16(-32768), dem).astype(np.int16)
    masked = np.where(hole, np.int16(ND), dem).astype(np.int16)
    p = tmp_path / "dem.tif"
    with rio.open(p, "w", width=cols, height=rows, dtype="int16", compress="lzw", predictor=2, tiled=True, blockxsize=128,
                  blockysize=128, nodata=-32768, transform=rio.Affine(PX, 0, 1000.0, 0, -PX, 9000.0)) as dst:
        dst.write(stored)
    with rio.open(p) as src:
        assert src.dtypes[0] == "int16" and src.nodata == -32768 and src.compression == "lzw"
    want = pipeline.pipeline(masked, PX, thr, N_GFI, B_GFI)
    assert want["hand"].dtype == np.int16
    assert_outputs(want, chain_oracle(masked, PX, thr), CHAIN, "pipeline.pipeline")
    for decode, encode in itertools.product(("host", "device"), repeat=2):
        paths = pipeline.pipeline_files(p, tmp_path / f"out_{decode}_{encode}", river_threshold=thr, block_bytes=100_000,
                                        decode=decode, encode=encode)
        assert sorted(paths) == sorted(CHAIN)
        for name, path in paths.items():
            with rio.open(path) as src:
                got = src.read(1)
            assert got.dtype == want[name].dtype, name
            np.testing.assert_array_equal(got, want[name], err_msg=f"{name} ({decode} / {encode})")
