"""flowhand.py -- drop-in for descriptools/flowhand.py (reference: flowhand.py:242-846), plus the
two stages the reference's workflow needs but does not implement: D8 flow direction and D8 flow
accumulation (it loads both from disk, Example/example.py:36,39).
"""
import numpy as np

from . import device
from ._convert import dem_to_native, fdr_to_u8, ints_to_native, river_to_i8, to_dev, to_host


def flow_hand_index(dem_raster, flow_direction_matrix, river_matrix, px, division_column=0, division_row=0):
    """Flow distance, river-cell index and HAND -- flowhand.py:242-411.

    Returns (flow_distance float32, indices int64, hand in the DEM's dtype), flowhand.py:279-280,
    436, 411.  `division_*` are accepted and ignored (result == the unpartitioned reference path;
    the reference's partitioned mode is broken, SURVEY.md 5.7).
    """
    dem_in = np.asarray(dem_raster)
    d = dem_to_native(dem_in)
    out = device.hand(to_dev(fdr_to_u8(flow_direction_matrix)), to_dev(d), px, river=to_dev(river_to_i8(river_matrix)))
    hand = to_host(out["hand"])
    if hand.dtype != dem_in.dtype:
        hand = hand.astype(dem_in.dtype)
    return to_host(out["fdist"]), to_host(out["idx"]).astype(np.int64), hand


def hand_calculator(dem, indices):
    """HAND from a river-cell index raster -- flowhand.py:414-442."""
    dem_in = np.asarray(dem)
    d = dem_to_native(dem_in)
    idx = ints_to_native(np.asarray(indices).reshape(d.shape), "indices")
    hand = to_host(device.hand_from_index(to_dev(d), to_dev(idx)))
    return hand if hand.dtype == dem_in.dtype else hand.astype(dem_in.dtype)


def flow_distance_index_cpu(dem, flow_direction, river_matrix, px, boundary_distance, boundary_index, out,
                            row_start, col_start, matrix_columns, blocks=0, threads=0):
    """Host wrapper of the flow-distance kernel -- flowhand.py:476-562.

    Only the unpartitioned call (all `out` flags 0) is supported; it returns
    (flow_distance float32, indices float64) with the index offset arithmetic of flowhand.py:612,845.
    """
    if np.any(np.asarray(out) != 0):
        raise NotImplementedError("tile-partitioned flow distance is not supported: the reference's partitioned mode "
                                  "is broken (SURVEY.md 5.7); call flow_hand_index on the whole raster")
    fdr = fdr_to_u8(flow_direction)
    res = device.hand(to_dev(fdr), None, px, river=to_dev(river_to_i8(river_matrix)), want_hand=False)
    idx = to_host(res["idx"]).astype(np.int64)
    rows, cols = fdr.shape
    ok = idx != -100
    r, c = np.divmod(np.where(ok, idx, 0), cols)
    idx_g = np.where(ok, (row_start + r) * matrix_columns + col_start + c, -100).astype(np.float64)
    return to_host(res["fdist"]), idx_g


# ---- stages the reference consumes but does not implement ---------------------------------
def flow_direction_d8(dem, px):
    """D8 flow direction (uint8, ESRI codes 1..128, 0 = nodata) -- SURVEY.md App. A2; encoding
    per flowhand.py:801-824."""
    _, d8 = device.slope_d8(to_dev(dem_to_native(dem)), px, want_slope=False, want_d8=True)
    return to_host(d8)


def flow_accumulation(flow_direction, nodata=-100):
    """D8 flow accumulation (int64; number of strictly-upstream cells; `nodata` where the direction
    code is 0) -- SURVEY.md App. A3; convention of Example/input/12_fac.tif."""
    import torch

    fdr = fdr_to_u8(flow_direction)
    dt = torch.int32 if fdr.size < 2**31 else torch.int64
    return to_host(device.flow_accumulation(to_dev(fdr), dtype=dt, nodata_fill=nodata)).astype(np.int64)


def fill_depressions(dem, epsilon=True):
    """Hydrological conditioning (SURVEY.md section 8 f4): every cell is raised to the lowest level from which water can
    leave the raster (or reach a nodata cell).  epsilon=True: priority-flood + epsilon, every filled or flat cell one
    float32 step above the cell it drains to, so D8 drains it.  The reference's fixtures were conditioned by an external
    GIS before example.py:33-39 reads them; an unconditioned DEM leaves interior pits, where D8 has no code and the
    accumulation stops.  float32 in (other dtypes are converted if exact), float32 out.
    epsilon=False: the priority flood alone; filled areas stay exactly flat (give them codes with resolve_flats).  An
    int16 DEM stays int16.  -100 / NaN cells stay as they are."""
    d = dem_to_native(dem)
    if d.dtype != np.float32 and (epsilon or d.dtype != np.int16):
        d = d.astype(np.float32)  # int16 elevations: exact
    t = to_dev(d).clone()
    device.fill_depressions(t, epsilon=epsilon)
    return to_host(t)


def resolve_flats(dem, flow_direction):
    """D8 codes for the flat cells (valid cells with code 0) of `flow_direction`, the D8 raster of `dem`
    (flow_direction_d8): each flat drains towards its outlets and away from the higher ground around it (Garbrecht &
    Martz 1997; Barnes, Lehman & Mulla 2014).  Returns a new uint8 raster; the DEM and every other code are unchanged.
    Flats without an outlet (pits of an unfilled DEM) keep code 0."""
    t = to_dev(fdr_to_u8(flow_direction)).clone()
    device.resolve_flats(to_dev(dem_to_native(dem)), t)
    return to_host(t)
