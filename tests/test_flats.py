"""Exact depression filling (fill without epsilon) and flat resolution: the host reference (flats_ref.cpp) against
hand-worked cases and a heapq priority flood, and the device kernels (csrc/synth.cu, csrc/flats.cu) against the
reference bit for bit."""
import heapq
import os
import sys

import numpy as np
import pytest

import oracle

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import flats_ref  # noqa: E402
from helpers import PX, RTOL, ATOL, example_inputs  # noqa: E402

NB = [(-1, -1), (-1, 0), (-1, 1), (0, -1), (0, 1), (1, -1), (1, 0), (1, 1)]
CODE = {32: (-1, -1), 64: (-1, 0), 128: (-1, 1), 16: (0, -1), 1: (0, 1), 8: (1, -1), 4: (1, 0), 2: (1, 1)}


def heap_flood(dem):
    """priority flood without epsilon, in Python"""
    w = dem.astype(np.float32).copy()
    rows, cols = w.shape
    nd = (w == -100) | np.isnan(w)
    done = nd.copy()
    heap = []
    for r in range(rows):
        for c in range(cols):
            if nd[r, c]:
                continue
            seed = r in (0, rows - 1) or c in (0, cols - 1) or any(nd[r + a, c + b] for a, b in NB)
            if seed:
                done[r, c] = True
                heap.append((float(w[r, c]), r, c))
    heapq.heapify(heap)
    while heap:
        z, r, c = heapq.heappop(heap)
        for a, b in NB:
            rr, cc = r + a, c + b
            if 0 <= rr < rows and 0 <= cc < cols and not done[rr, cc]:
                done[rr, cc] = True
                w[rr, cc] = max(w[rr, cc], np.float32(z))
                heapq.heappush(heap, (float(w[rr, cc]), rr, cc))
    return w


def quantised_synth(rows, cols, seed, holes=True, nan=True):
    """the synthetic DEM rounded to 0.1 m, which makes flats; -100 blobs unless holes=False, NaN cells unless nan=False"""
    z = oracle.synth_dem(rows, cols, 0, seed)
    z = (np.round(z.astype(np.float64) * 10) / 10).astype(np.float32)
    if holes:
        rng = np.random.default_rng(seed)
        for _ in range(6):
            r, c = int(rng.integers(2, rows - 12)), int(rng.integers(2, cols - 12))
            z[r:r + int(rng.integers(1, 10)), c:c + int(rng.integers(1, 10))] = -100
        if nan:
            z[rng.integers(0, rows, 20), rng.integers(0, cols, 20)] = np.nan
    return z


def resolved_chain(dem):
    """F1 -> stencil -> F2 with the reference: (filled DEM in the input's dtype, d8 before, d8 after, unresolved, mask)"""
    f = flats_ref.priority_flood(dem)
    if dem.dtype == np.int16:
        f = f.astype(np.int16)
    _, c = oracle.slope_d8(f, PX)
    r, left, _, mask = flats_ref.resolve_flats(f, c, with_mask=True)
    return f, c, r, left, mask


def check_resolution(dem, c, r, mask):
    """no valid cell keeps code 0, non-flat codes stay, every flat cell points at a neighbour of strictly smaller mask
    (another cell of its flat or an outlet: a coded cell at its elevation), and the accumulation finalises every cell"""
    valid = dem > -100
    flat = valid & (c == 0)
    assert not np.any(valid & (r == 0))
    np.testing.assert_array_equal(r[~flat], c[~flat])
    rr, cc = np.nonzero(flat)
    dr = np.array([CODE[int(k)][0] for k in r[flat]])
    dc = np.array([CODE[int(k)][1] for k in r[flat]])
    qr, qc = rr + dr, cc + dc
    assert np.all(mask[qr, qc] < mask[rr, cc])
    off = ~flat[qr, qc]
    assert np.all(dem[qr, qc][off] == dem[rr, cc][off]) and np.all(c[qr, qc][off] != 0)
    _, left = oracle.flow_accumulation(r)
    assert left == 0


# ---- the reference ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_reference_fill_is_the_heap_priority_flood(seed):
    rng = np.random.default_rng(seed)
    dem = (rng.random((37, 53)) * 20).astype(np.float32)
    dem[rng.random(dem.shape) < 0.03] = -100
    dem[rng.random(dem.shape) < 0.01] = np.nan
    dem[10:14, 20:25] = -100
    got = flats_ref.priority_flood(dem)
    np.testing.assert_array_equal(got, heap_flood(dem))
    assert np.all((got >= dem) | np.isnan(dem))


def _resolve(z):
    z = np.asarray(z, np.float32)
    _, c = oracle.slope_d8(z, PX)
    r, left, nflat = flats_ref.resolve_flats(z, c)
    return c, r, left, nflat


ONE_OUTLET = [[9, 9, 9, 9, 9],
              [9, 5, 5, 5, 9],
              [9, 5, 5, 5, 5],
              [9, 5, 5, 5, 9],
              [9, 9, 9, 9, 9]]
# towards 3 2 1 by column, away 0 on the ring and 1 in the centre (A = 1): masks 7 5 3 / 7 4 3 / 7 5 3, the outlet -1
ONE_OUTLET_CODES = [[2, 1, 2],
                    [1, 128, 1],
                    [128, 128, 128]]


def test_reference_flat_with_one_edge_outlet():
    c, r, left, nflat = _resolve(ONE_OUTLET)
    assert left == 0 and nflat == 9
    np.testing.assert_array_equal(r[1:4, 1:4], ONE_OUTLET_CODES)
    r[1:4, 1:4] = 0
    np.testing.assert_array_equal(r, c)


def test_reference_filled_bowl():
    bowl = np.array([[9, 9, 9, 9, 9],
                     [9, 3, 2, 3, 9],
                     [9, 2, 1, 2, 6],
                     [9, 3, 2, 3, 9],
                     [9, 9, 9, 9, 9]], np.float32)
    f = flats_ref.priority_flood(bowl)
    want = bowl.copy()
    want[1:4, 1:4] = 6
    np.testing.assert_array_equal(f, want)
    _, r, left, nflat = _resolve(f)
    assert left == 0 and nflat == 9
    np.testing.assert_array_equal(r[1:4, 1:4], ONE_OUTLET_CODES)


def test_reference_two_flats_at_one_elevation_behind_a_ridge():
    z = [[9, 9, 9, 9, 9, 9, 9, 9],
         [5, 5, 5, 5, 9, 5, 5, 5],
         [9, 9, 9, 9, 9, 9, 9, 9]]
    _, r, left, nflat = _resolve(z)
    assert left == 0 and nflat == 5
    # left flat drains west to (1, 0), right flat east to (1, 7); nothing crosses the ridge
    np.testing.assert_array_equal(r[1, 1:4], [16, 16, 16])
    np.testing.assert_array_equal(r[1, 5:7], [1, 1])


def test_reference_flat_without_high_edge():
    z = np.full((5, 5), 5, np.float32)  # every edge cell is an outlet at the flat's elevation
    _, r, left, nflat = _resolve(z)
    assert left == 0 and nflat == 9
    # ring: towards 1 (mask 2) -> first outlet in scan order; centre: towards 2 -> first ring cell (NW)
    np.testing.assert_array_equal(r[1:4, 1:4], [[32, 32, 32], [32, 32, 128], [32, 8, 128]])


def test_reference_tie_goes_to_the_first_neighbour_in_scan_order():
    z = [[9, 9, 9, 9, 9],
         [5, 5, 5, 5, 5],
         [9, 9, 9, 9, 9]]
    _, r, left, nflat = _resolve(z)
    assert left == 0 and nflat == 3
    # masks 2 4 2: the middle cell has W and E at 2 and takes W
    np.testing.assert_array_equal(r[1, 1:4], [16, 16, 1])


def test_reference_pit_without_outlet_is_unresolved():
    z = np.full((4, 4), 9, np.float32)
    z[1:3, 1:3] = 2   # a pit: no outlet
    c, r, left, nflat = _resolve(z)
    assert left == 4 and nflat == 4
    np.testing.assert_array_equal(r, c)
    assert np.all(r[1:3, 1:3] == 0)


def test_reference_drains_the_example_dem_in_its_own_type():
    ex = example_inputs()
    dem = ex["dem"]
    f, c, r, left, mask = resolved_chain(dem)
    assert f.dtype == np.int16
    np.testing.assert_array_equal(f, dem)  # the example has flats, no depressions
    assert int(((c == 0) & (dem > -100)).sum()) == 221011
    assert left == 0
    check_resolution(f, c, r, mask)
    # reported only: agreement of the codes on the flat cells with the GIS's 12_fdr.tif, next to the epsilon fill's
    flat = (c == 0) & (dem > -100)
    _, ce = oracle.slope_d8(oracle.priority_flood_eps(dem.astype(np.float32)), PX)
    print(f"\nexample flat cells: {int(flat.sum())}; D8 equal to 12_fdr.tif on them: flat resolution "
          f"{(r[flat] == ex['fdr'][flat]).mean():.4f}, epsilon fill {(ce[flat] == ex['fdr'][flat]).mean():.4f}")


def test_reference_drains_a_quantised_synthetic_dem():
    # no NaN cells: the stencil points a NaN cell at a neighbour, which can close a cycle whatever the conditioning
    dem = quantised_synth(600, 700, 5, nan=False)
    f, c, r, left, mask = resolved_chain(dem)
    assert left == 0 and int(((c == 0) & (f > -100)).sum()) > 1000
    check_resolution(f, c, r, mask)


# ---- the device -----------------------------------------------------------------------------------------------
def spiral(n):
    """a corridor of elevation 0 winding inwards through walls of 10, open at (1, 0) on the raster's edge"""
    z = np.full((n, n), 10, np.float32)
    r, c, d = 1, 1, 0
    steps = [(0, 1), (1, 0), (0, -1), (-1, 0)]
    z[r, c] = 0
    turns = 0
    while turns < 2:
        dr, dc = steps[d]
        rr, cc = r + 2 * dr, c + 2 * dc
        if 1 <= rr < n - 1 and 1 <= cc < n - 1 and z[rr, cc] != 0:
            z[r + dr, c + dc] = 0
            z[rr, cc] = 0
            r, c, turns = rr, cc, 0
        else:
            d, turns = (d + 1) % 4, turns + 1
    z[1, 0] = 0
    return z


def edge_nodata_flats():
    """flats next to outlets on the raster's edge, next to -100 and next to NaN cells"""
    z = np.full((70, 90), 20, np.float32)
    z[1:12, 0:30] = 5          # touches the west edge: its edge cells are outlets
    z[30:40, 30:60] = 7
    z[34, 29] = -100           # a nodata cell on its west side
    z[50:62, 60:89] = 3
    z[55, 89] = np.nan         # an outlet next to NaN on the east edge
    z[20:25, 70:80] = 8        # a pit: no outlet
    return z


def _device_resolve(dem):
    import torch

    from descriptools_b200 import device

    t = torch.from_numpy(dem).cuda()
    _, d8 = device.slope_d8(t, PX, want_slope=False)
    left = device.resolve_flats(t, d8)
    return d8.cpu().numpy(), left


def _compare(dem):
    _, c = oracle.slope_d8(dem, PX)
    want, left_ref, nflat = flats_ref.resolve_flats(dem, c)
    got, left = _device_resolve(dem)
    np.testing.assert_array_equal(got, want)
    assert left == left_ref
    return nflat, left


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.int16])
def test_device_fill_without_epsilon_equals_the_reference(dtype):
    import torch

    from descriptools_b200 import device

    if dtype == np.int16:
        dem = example_inputs()["dem"].copy()
        dem[600:640, 700:760] = 40  # a depression the example lacks
    else:
        dem = quantised_synth(1100, 1300, 7)
    t = torch.from_numpy(dem).cuda()
    device.fill_depressions(t, epsilon=False)
    got = t.cpu().numpy()
    assert got.dtype == dtype
    np.testing.assert_array_equal(got.astype(np.float32), flats_ref.priority_flood(dem))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.int16, np.float32])
@pytest.mark.parametrize("filled", [True, False])
def test_device_resolve_flats_on_the_example(dtype, filled):
    dem = example_inputs()["dem"].copy()
    dem[600:640, 700:760] = 40
    if filled:
        dem = flats_ref.priority_flood(dem).astype(np.int16)
    nflat, left = _compare(dem.astype(dtype))
    assert nflat > 221000 and (left == 0) == filled


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1024, 2048), (1537, 2311)])
@pytest.mark.parametrize("filled", [True, False])
def test_device_resolve_flats_on_quantised_synthetic(shape, filled):
    dem = quantised_synth(*shape, 11)
    if filled:
        dem = flats_ref.priority_flood(dem)
    nflat, left = _compare(dem)
    assert nflat > 0 and (left == 0) == filled


@pytest.mark.gpu
def test_device_resolve_one_flat_over_4096_squared_with_one_outlet():
    z = np.zeros((4096, 4096), np.float32)
    z[0, :] = z[-1, :] = z[:, 0] = z[:, -1] = 10
    z[2000, 0] = 0
    nflat, left = _compare(z)
    assert nflat == 4094 * 4094 and left == 0


@pytest.mark.gpu
def test_device_resolve_spiral_corridor():
    z = spiral(513)
    nflat, left = _compare(z)
    assert nflat > 100000 and left == 0


@pytest.mark.gpu
def test_device_resolve_flats_at_edges_nodata_and_nan():
    nflat, left = _compare(edge_nodata_flats())
    assert left == 5 * 10 and nflat > left


def _any_d8_cases():
    """D8 rasters that are not the stencil's output for the DEM: code 0 on the raster's edge, codes of another DEM,
    codes that are no direction at all"""
    z = np.full((4, 4), 5, np.float32)
    d8 = np.zeros((4, 4), np.uint8)
    d8[3, 3] = 2
    yield z, d8
    rng = np.random.default_rng(3)
    for dtype, shape in ((np.float32, (67, 45)), (np.int16, (300, 517)), (np.float32, (1100, 1300))):
        z = rng.integers(0, 4, shape).astype(dtype)  # four levels: many equal neighbours
        z[rng.random(shape) < 0.02] = -100
        if dtype == np.float32:
            z[rng.random(shape) < 0.01] = np.nan
        d8 = rng.choice(np.array([0, 1, 2, 4, 8, 16, 32, 64, 128, 3, 255], np.uint8), shape,
                        p=[0.6] + [0.04] * 8 + [0.04, 0.04])
        d8[0, :] = d8[-1, :] = d8[:, 0] = d8[:, -1] = 0
        d8[0, ::7] = 1
        yield z, d8


@pytest.mark.gpu
def test_device_resolve_flats_takes_any_d8_raster():
    import torch

    from descriptools_b200 import device

    for z, d8 in _any_d8_cases():
        want, left_ref, nflat = flats_ref.resolve_flats(z, d8)
        got = torch.from_numpy(d8).cuda()
        left = device.resolve_flats(torch.from_numpy(z).cuda(), got)
        np.testing.assert_array_equal(got.cpu().numpy(), want)
        assert left == left_ref and nflat > left


@pytest.mark.gpu
def test_device_resolve_leaves_an_epsilon_filled_dem_alone():
    import torch

    from descriptools_b200 import device

    dem = torch.from_numpy(quantised_synth(900, 1000, 13)).cuda()
    device.fill_depressions(dem)
    _, d8 = device.slope_d8(dem, PX, want_slope=False)
    before = d8.clone()
    assert device.resolve_flats(dem, d8) == 0
    assert torch.equal(d8, before)


@pytest.mark.gpu
def test_run_device_with_resolved_flats_equals_the_oracle_chain():
    import torch

    from descriptools_b200 import device, pipeline

    thr = 300
    dem = quantised_synth(1200, 1500, 17, nan=False)
    t = torch.from_numpy(dem).cuda()
    device.fill_depressions(t, epsilon=False)
    f = flats_ref.priority_flood(dem)
    _, c = oracle.slope_d8(f, PX)
    d8, _, _ = flats_ref.resolve_flats(f, c)
    got = pipeline.run_device(t, PX, thr, resolve_flats=True)
    acc, left = oracle.flow_accumulation(d8)
    assert left == 0
    river = (acc > thr).astype(np.int8)
    fdist, idx, hand = oracle.flow_hand_index(f, d8, river, PX)
    with np.errstate(all="ignore"):
        gfi = oracle.gfi(hand, acc, idx, 0.4, 0.1, PX)
    np.testing.assert_array_equal(got["d8"].cpu().numpy(), d8)
    np.testing.assert_array_equal(got["acc"].cpu().numpy(), acc)
    np.testing.assert_array_equal(got["idx"].cpu().numpy(), idx)
    np.testing.assert_array_equal(got["hand"].cpu().numpy(), hand)
    np.testing.assert_allclose(got["fdist"].cpu().numpy(), fdist, rtol=RTOL, atol=0)
    np.testing.assert_allclose(got["gfi"].cpu().numpy(), gfi, rtol=RTOL, atol=ATOL)


@pytest.mark.gpu
def test_run_device_with_resolved_flats_verifies_at_20k():
    import torch

    from descriptools_b200 import device, pipeline

    n, thr = 20000, 1000
    dem = device.synth_dem(n, n)
    dem = torch.round(dem * 10) / 10
    device.fill_depressions(dem, epsilon=False)
    res = pipeline.run_device(dem, PX, thr, resolve_flats=True)
    valid = dem > -100
    assert int(((res["d8"] == 0) & valid).sum()) == 0
    v = device.chain_verdict(device.chain_check(res["d8"], res["acc"], thr, res["idx"], dem, res["hand"]).cpu())
    assert v["verified"], v
    del res, dem
    device.workspace.release()
    torch.cuda.empty_cache()


def _write_tif(path, arr, nodata):
    from descriptools_b200 import raster as rio

    rows, cols = arr.shape
    with rio.open(path, "w", width=cols, height=rows, dtype=arr.dtype.name, compress="lzw", tiled=True, blockxsize=256,
                  blockysize=256, nodata=nodata, transform=rio.Affine(PX, 0, 500000.0, 0, -PX, 7000000.0)) as dst:
        dst.write(arr)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["example_int16", "synth_f32"])
def test_pipeline_files_condition_flats(tmp_path, kind):
    from descriptools_b200 import pipeline
    from descriptools_b200 import raster as rio

    if kind == "example_int16":
        dem = example_inputs()["dem"].copy()
        dem[600:640, 700:760] = 40
        nodata = -100
    else:
        dem = quantised_synth(700, 530, 23, holes=False)
        dem[170:215, 40:120] = -9999.0
        nodata = -9999.0
    src = tmp_path / "dem.tif"
    _write_tif(src, dem, nodata)
    paths = pipeline.pipeline_files(src, tmp_path / "out", river_threshold=300, px=PX, condition="flats")
    z = np.where(dem == nodata, -100, dem).astype(dem.dtype)
    f = flats_ref.priority_flood(z).astype(dem.dtype)
    _, c = oracle.slope_d8(f, PX)
    d8, left, _ = flats_ref.resolve_flats(f, c)
    assert left == 0
    np.testing.assert_array_equal(rio.read_to_device(paths["d8"]).cpu().numpy(), d8)
    # HAND is the oracle's on the resolved codes; -100 is left only where a path leaves the raster or meets nodata
    # before it meets a river, and no longer on every cell of a flat
    hand = rio.read_to_device(paths["hand"]).cpu().numpy()
    valid = f > -100
    hands = []
    for codes in (d8, c):
        acc, _ = oracle.flow_accumulation(codes)
        hands.append(oracle.flow_hand_index(f, codes, (acc > 300).astype(np.int8), PX)[2])
    np.testing.assert_array_equal(hand, hands[0])
    assert np.count_nonzero(hand[valid] == -100) < np.count_nonzero(hands[1][valid] == -100)
    if kind == "synth_f32":  # the epsilon route is unchanged
        eps = pipeline.pipeline_files(src, tmp_path / "eps", river_threshold=300, px=PX, condition=True, outputs=("d8", "hand"))
        fe = oracle.priority_flood_eps(z)
        _, ce = oracle.slope_d8(fe, PX)
        np.testing.assert_array_equal(rio.read_to_device(eps["d8"]).cpu().numpy(), ce)


@pytest.mark.gpu
def test_numpy_drop_ins():
    from descriptools_b200 import flowhand

    dem = example_inputs()["dem"].copy()
    dem[600:640, 700:760] = 40
    f = flowhand.fill_depressions(dem, epsilon=False)
    assert f.dtype == np.int16
    np.testing.assert_array_equal(f, flats_ref.priority_flood(dem).astype(np.int16))
    c = flowhand.flow_direction_d8(f, PX)
    want, _, _ = flats_ref.resolve_flats(f, c)
    np.testing.assert_array_equal(flowhand.resolve_flats(f, c), want)
    np.testing.assert_array_equal(flowhand.fill_depressions(dem.astype(np.float32)),
                                  oracle.priority_flood_eps(dem.astype(np.float32)))


def test_resolve_flats_argument_checks_need_no_device():
    from descriptools_b200 import _lib

    L = _lib.lib
    assert L.dtb_resolve_flats_workspace_bytes(100, 70) == 256 + 100 * 70 * 16 + 4 * 3 * 4
    assert L.dtb_resolve_flats(None, 0, None, 10, 10, None, 0, None, None) == -1
    assert L.dtb_resolve_flats(1, 7, 1, 10, 10, 1, 1 << 20, None, None) == -1              # bad dtype
    assert L.dtb_resolve_flats(1, 0, 1, 1 << 16, 1 << 15, 1, 1 << 62, None, None) == -4   # 2^31 cells
    assert L.dtb_resolve_flats(1, 1, 1, 10, 10, 1, 100, None, None) == -3                  # workspace
    assert L.dtb_fill_flat_f32(None, 10, 10, None, 0, None, None) == -1
