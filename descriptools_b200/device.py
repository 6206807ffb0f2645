"""Device-resident entry points: torch CUDA tensors in, torch CUDA tensors out.

These are thin argument marshallers around the C ABI (include/dtb200.h); the arithmetic is in
descriptools_b200/csrc/*.cu.  The NumPy drop-in modules (slope.py, flowhand.py, ...) and the
benchmark both go through here.  All calls are enqueued on torch's current CUDA stream.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import DTB_F32, DTB_I16, DTB_I32, DTB_I64, HandArgs, check, lib

_DEM_DT = {torch.float32: DTB_F32, torch.int16: DTB_I16}
_INT_DT = {torch.int32: DTB_I32, torch.int64: DTB_I64}


def require_cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise _lib.DtbError("descriptools_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _stream() -> int:  # the current stream of the current device: compute calls run under torch.cuda.device(tensor.device)
    return torch.cuda.current_stream().cuda_stream


def _ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


def _chk2d(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor")
    if t.dim() != 2:
        raise ValueError(f"{name} must be 2-D")
    return t.contiguous()


def _dem_dtype(t: torch.Tensor) -> int:
    try:
        return _DEM_DT[t.dtype]
    except KeyError:
        raise TypeError(f"DEM/HAND tensors must be float32 or int16, got {t.dtype}") from None


def _int_dtype(t: torch.Tensor) -> int:
    try:
        return _INT_DT[t.dtype]
    except KeyError:
        raise TypeError(f"index/accumulation tensors must be int32 or int64, got {t.dtype}") from None


class _Workspace:
    """Cached scratch buffers per (device, stage, stream), grown on demand (caller-owned from the ABI's view)."""

    def __init__(self):
        self.buf = {}
        self.fused = {}  # device index -> what the fused flow-accumulation call left in the "hand" workspace

    def get(self, nbytes: int, stage: str = "shared", device=None) -> torch.Tensor:
        """scratch on `device` (default: the current one) for the stream the call is enqueued on: calls on one stream are
        ordered, two streams each get a buffer of their own."""
        index = torch.cuda.current_device() if device is None else torch.device(device).index
        key = (index, stage, torch.cuda.current_stream(index).cuda_stream)
        b = self.buf.get(key)
        if b is None or b.numel() < nbytes:
            self.buf[key] = None
            b = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{index}")
            self.buf[key] = b
            if stage == "hand":
                self.fused.pop(index, None)  # a new buffer holds no entry-node states
        return b

    def release(self):
        self.buf.clear()
        self.fused.clear()


workspace = _Workspace()


def _out(out, name, shape, dtype, dev):
    """a caller-supplied output raster (dict `out`, reused across calls: multi-GB allocations per call make the caching
    allocator split and re-malloc blocks, and cudaMalloc / cudaFree synchronise the device) or a fresh one"""
    if out is not None and name in out:
        t = out[name]
        if tuple(t.shape) != tuple(shape) or t.dtype != dtype or not t.is_cuda or not t.is_contiguous():
            raise ValueError(f"out[{name!r}] must be a contiguous CUDA tensor of shape {tuple(shape)} and dtype {dtype}")
        return t
    return torch.empty(shape, dtype=dtype, device=dev)


def slope_d8(dem: torch.Tensor, px: float, want_slope: bool = True, want_d8: bool = True,
             row_begin: int = 0, row_end: int | None = None, out: dict | None = None):
    """Fused slope (%) + D8 over rows [row_begin,row_end) of `dem` (slope.py:152-259 + SURVEY A2)."""
    dem = _chk2d(dem, "dem")
    rows, cols = dem.shape
    row_end = rows if row_end is None else row_end
    nr = row_end - row_begin
    slope = _out(out, "slope", (nr, cols), torch.float32, dem.device) if want_slope else None
    d8 = _out(out, "d8", (nr, cols), torch.uint8, dem.device) if want_d8 else None
    check(lib.dtb_slope_d8(_ptr(dem), _dem_dtype(dem), rows, cols, row_begin, row_end, float(px), _ptr(slope), _ptr(d8),
                           _stream()), "dtb_slope_d8")
    return slope, d8


def flow_accumulation(d8: torch.Tensor, dtype: torch.dtype = torch.int32, nodata_fill: int = -100,
                      check_cycles: bool = False, fuse_hand_threshold: int | None = None, out: dict | None = None):
    """D8 flow accumulation (SURVEY A3).  Returns acc, or (acc, n_cycle_cells) if check_cycles.

    fuse_hand_threshold = t: the final tile pass also runs HAND's entry-node pass for the river mask
    acc > t and leaves the node states in the HAND workspace; follow with hand(..., entry_done=True).
    """
    from ._lib import FlowaccArgs

    d8 = _chk2d(d8, "d8")
    if d8.dtype != torch.uint8:
        raise TypeError("d8 must be uint8")
    rows, cols = d8.shape
    acc = _out(out, "acc", (rows, cols), dtype, d8.device)
    nbytes = lib.dtb_flowacc_workspace_bytes(rows, cols)
    ws = workspace.get(nbytes, "flowacc", d8.device)
    left = ctypes.c_int64(0)
    a = FlowaccArgs()
    a.d8, a.rows, a.cols = _ptr(d8), rows, cols
    a.acc, a.acc_dtype, a.nodata_fill = _ptr(acc), _int_dtype(acc), int(nodata_fill)
    if check_cycles:
        a.unfinalised_host = ctypes.pointer(left)
    if fuse_hand_threshold is not None:
        hb = lib.dtb_hand_workspace_bytes(rows, cols)
        hws = workspace.get(hb, "hand", d8.device)
        a.hand_ws, a.hand_ws_bytes, a.hand_river_threshold = _ptr(hws), hb, int(fuse_hand_threshold)
    with torch.cuda.device(d8.device):
        check(lib.dtb_flowacc_band(ctypes.byref(a), _ptr(ws), nbytes, _stream()), "dtb_flowacc_band")
    if fuse_hand_threshold is not None:  # hand(entry_done=True) honours only exactly this state
        workspace.fused[d8.device.index] = (d8.data_ptr(), acc.data_ptr(), (rows, cols), int(fuse_hand_threshold), _ptr(hws))
    return (acc, int(left.value)) if check_cycles else acc


def hand(fdr: torch.Tensor, dem: torch.Tensor | None, px: float, river: torch.Tensor | None = None,
         acc: torch.Tensor | None = None, river_threshold: int = 0, max_moves: int = 0,
         want_fdist: bool = True, want_idx: bool = True, want_hand: bool = True,
         gfi_params: tuple[float, float, float] | None = None, idx_dtype: torch.dtype | None = None,
         entry_done: bool = False, out: dict | None = None):
    """Flow distance, river index, HAND and (optionally) fused GFI.

    flowhand.py:476-846 + 414-442 (+ gfi.py:118-147, 267-294 when gfi_params=(n, b, size)).
    Returns a dict with the requested tensors: fdist f32, idx int32/int64, hand (DEM dtype), gfi f32.
    """
    fdr = _chk2d(fdr, "fdr")
    if fdr.dtype != torch.uint8:
        raise TypeError("fdr must be uint8")
    rows, cols = fdr.shape
    dev = fdr.device
    a = HandArgs()
    a.fdr = _ptr(fdr)
    if river is not None:
        river = _chk2d(river, "river")
        if river.dtype != torch.int8:
            raise TypeError("river must be int8")
    a.river = _ptr(river)
    if acc is not None:
        acc = _chk2d(acc, "acc")
        a.acc_dtype = _int_dtype(acc)
    a.acc = _ptr(acc)
    a.river_threshold = int(river_threshold)
    if dem is not None:
        dem = _chk2d(dem, "dem")
        a.dem_dtype = _dem_dtype(dem)
    a.dem = _ptr(dem)
    a.rows, a.cols, a.px, a.max_moves = rows, cols, float(px), int(max_moves)
    _same_shape(flow_direction=fdr, river=river, flow_accumulation=acc, dem=dem)
    given, out = out, {}
    if want_fdist:
        out["fdist"] = _out(given, "fdist", (rows, cols), torch.float32, dev)
    if want_idx:
        if idx_dtype is None:
            idx_dtype = torch.int32 if rows * cols < 2**31 else torch.int64
        out["idx"] = _out(given, "idx", (rows, cols), idx_dtype, dev)
        a.idx_dtype = _int_dtype(out["idx"])
    if want_hand:
        if dem is None:
            raise ValueError("hand needs dem")
        out["hand"] = _out(given, "hand", (rows, cols), dem.dtype, dev)
    if gfi_params is not None:
        if dem is None or acc is None:
            raise ValueError("fused gfi needs dem and acc")
        out["gfi"] = _out(given, "gfi", (rows, cols), torch.float32, dev)
        a.gfi_n, a.gfi_b, a.gfi_size = (float(v) for v in gfi_params)
    a.fdist, a.idx, a.hand, a.gfi = _ptr(out.get("fdist")), _ptr(out.get("idx")), _ptr(out.get("hand")), _ptr(out.get("gfi"))
    a.entry_done = 1 if entry_done else 0
    nbytes = lib.dtb_hand_workspace_bytes(rows, cols)
    ws = workspace.get(nbytes, "hand", dev)
    if entry_done:
        # the entry-node states must be the ones the fused flow accumulation of THIS raster and threshold left in THIS buffer
        want = (fdr.data_ptr(), acc.data_ptr() if acc is not None else 0, (rows, cols), int(river_threshold), _ptr(ws))
        if workspace.fused.get(dev.index) != want:
            raise RuntimeError("hand(entry_done=True) must directly follow flow_accumulation(fuse_hand_threshold=...) on the same "
                               "flow-direction raster, accumulation raster and threshold")
    with torch.cuda.device(dev):
        check(lib.dtb_hand(ctypes.byref(a), _ptr(ws), nbytes, _stream()), "dtb_hand")
    if not entry_done:
        workspace.fused.pop(dev.index, None)  # the workspace now holds this call's node states
    return out


def _same_shape(**named):
    """every raster of one call covers the same grid (the kernels index them with one linear index)"""
    it = iter(named.items())
    n0, t0 = next(it)
    for n, t in it:
        if t is not None and (tuple(t.shape) != tuple(t0.shape) or t.device != t0.device):
            raise ValueError(f"{n} {tuple(t.shape)} on {t.device} does not match {n0} {tuple(t0.shape)} on {t0.device}")


def _raise_if_oob(flag: torch.Tensor, what: str):
    if int(flag.item()):  # one 4-byte read back: these two calls return host-visible results anyway
        raise IndexError(f"{what}: index out of bounds for the raster (the reference's NumPy / Numba gather raises here too)")


def hand_from_index(dem: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    dem, idx = _chk2d(dem, "dem"), _chk2d(idx, "idx")
    _same_shape(dem=dem, idx=idx)
    out = torch.empty_like(dem)
    oob = torch.zeros(1, dtype=torch.int32, device=dem.device)
    check(lib.dtb_hand_from_index(_ptr(dem), _dem_dtype(dem), _ptr(idx), _int_dtype(idx), dem.numel(), _ptr(out), _ptr(oob),
                                  _stream()), "dtb_hand_from_index")
    _raise_if_oob(oob, "hand_calculator")
    return out


def downslope(dem: torch.Tensor, fdr: torch.Tensor, px: float, delta: float, max_moves: int = 0) -> torch.Tensor:
    dem, fdr = _chk2d(dem, "dem"), _chk2d(fdr, "fdr")
    _same_shape(dem=dem, fdr=fdr)
    rows, cols = dem.shape
    out = torch.empty((rows, cols), dtype=torch.float32, device=dem.device)
    check(lib.dtb_downslope(_ptr(dem), _dem_dtype(dem), _ptr(fdr), rows, cols, float(px), float(delta), int(max_moves),
                            _ptr(out), _stream()), "dtb_downslope")
    return out


def river_accumulation(acc: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    acc, idx = _chk2d(acc, "acc"), _chk2d(idx, "idx")
    _same_shape(acc=acc, idx=idx)
    out = torch.empty_like(acc)
    oob = torch.zeros(1, dtype=torch.int32, device=acc.device)
    check(lib.dtb_river_accumulation(_ptr(acc), _int_dtype(acc), _ptr(idx), _int_dtype(idx), acc.numel(), _ptr(out), _ptr(oob),
                                     _stream()), "dtb_river_accumulation")
    _raise_if_oob(oob, "river_accumulation")
    return out


def gfi(hand_t: torch.Tensor, racc: torch.Tensor, n: float, b: float, size: float) -> torch.Tensor:
    hand_t, racc = _chk2d(hand_t, "hand"), _chk2d(racc, "racc")
    _same_shape(hand=hand_t, river_accumulation=racc)
    out = torch.empty(hand_t.shape, dtype=torch.float32, device=hand_t.device)
    check(lib.dtb_gfi(_ptr(hand_t), _dem_dtype(hand_t), _ptr(racc), _int_dtype(racc), hand_t.numel(), float(n), float(b),
                      float(size), _ptr(out), _stream()), "dtb_gfi")
    return out


def ln_hl_H(hand_t: torch.Tensor, acc: torch.Tensor, n: float, b: float, size: float) -> torch.Tensor:
    hand_t, acc = _chk2d(hand_t, "hand"), _chk2d(acc, "acc")
    _same_shape(hand=hand_t, flow_accumulation=acc)
    out = torch.empty(hand_t.shape, dtype=torch.float32, device=hand_t.device)
    check(lib.dtb_lnhlh(_ptr(hand_t), _dem_dtype(hand_t), _ptr(acc), _int_dtype(acc), hand_t.numel(), float(n), float(b),
                        float(size), _ptr(out), _stream()), "dtb_lnhlh")
    return out


def ti_mti(acc: torch.Tensor, slope_rad: torch.Tensor, px: float, n: float, want_ti: bool = True, want_mti: bool = True):
    acc, slope_rad = _chk2d(acc, "acc"), _chk2d(slope_rad, "slope")
    if slope_rad.dtype != torch.float32:
        raise TypeError("slope must be float32 (radians)")
    _same_shape(flow_accumulation=acc, slope=slope_rad)
    ti = torch.empty(acc.shape, dtype=torch.float32, device=acc.device) if want_ti else None
    mti = torch.empty(acc.shape, dtype=torch.float32, device=acc.device) if want_mti else None
    check(lib.dtb_ti_mti(_ptr(acc), _int_dtype(acc), _ptr(slope_rad), acc.numel(), float(px), float(n), _ptr(ti), _ptr(mti),
                         _stream()), "dtb_ti_mti")
    return ti, mti


def nodata_to_sentinel(dem: torch.Tensor, nodata: float | None) -> torch.Tensor:
    """in place: cells equal to `nodata` (if given) and NaN cells -> -100 (example.py:42-43); one pass"""
    if dem.dtype != torch.float32 or not dem.is_cuda or not dem.is_contiguous():
        raise ValueError("dem must be a contiguous float32 CUDA tensor")
    check(lib.dtb_nodata_to_sentinel_f32(_ptr(dem), dem.numel(), float(nodata) if nodata is not None else 0.0,
                                         1 if nodata is not None else 0, _stream()), "dtb_nodata_to_sentinel_f32")
    return dem


def slope_to_radians(slope_pct: torch.Tensor) -> torch.Tensor:
    slope_pct = _chk2d(slope_pct, "slope")
    out = torch.empty_like(slope_pct)
    check(lib.dtb_slope_to_radians(_ptr(slope_pct), slope_pct.numel(), _ptr(out), _stream()), "dtb_slope_to_radians")
    return out


# ---- calibration against a benchmark flood map without the float64 raster (csrc/evaluation.cu) ----------------------
_EV_DT = {torch.float32: 0, torch.int16: 2}  # DTB_EV_F32, DTB_EV_I16


def _ev_dtype(t: torch.Tensor) -> int:
    try:
        return _EV_DT[t.dtype]
    except KeyError:
        raise TypeError(f"calibrated descriptors must be float32 or int16, got {t.dtype}") from None


def flood_int8(flood: torch.Tensor, like: torch.Tensor) -> torch.Tensor:
    """a benchmark flood map as the kernels read it: int8, or uint8 viewed as int8 (what .astype("int8") makes of it)"""
    flood = _chk2d(flood, "flood")
    if flood.dtype == torch.uint8:
        flood = flood.view(torch.int8)
    elif flood.dtype != torch.int8:
        raise TypeError(f"the flood map must be int8 or uint8, got {flood.dtype}")
    _same_shape(descriptor=like, flood=flood)
    return flood


def eval_extrema(desc: torch.Tensor) -> torch.Tensor:
    """float64 [5] on the device, no host sync: smallest and second-smallest distinct non-NaN values, largest non-NaN
    value, distinct non-NaN values seen (capped at 2), NaN seen -- the two ends of np.unique(desc) (dtb_eval_extrema)"""
    desc = _chk2d(desc, "descriptor")
    out = torch.empty(5, dtype=torch.float64, device=desc.device)
    nbytes = lib.dtb_eval_extrema_workspace_bytes()
    with torch.cuda.device(desc.device):
        ws = workspace.get(nbytes, "extrema", desc.device)
        check(lib.dtb_eval_extrema(_ptr(desc), _ev_dtype(desc), desc.numel(), _ptr(out), _ptr(ws), nbytes, _stream()), "dtb_eval_extrema")
    return out


def eval_hist(desc: torch.Tensor, flood: torch.Tensor, mn: float, mx: float, corner: float, thresholds, under: str,
              hist: torch.Tensor, nodata: float = -100) -> torch.Tensor:
    """ADD the 4 x 33 confusion histogram of `thresholds` (strictly ascending, at most 32) on minMaxScale(desc, mn, mx,
    nodata) into `hist` (int64 [4 * 33] on desc's device), scaling every cell on load; `corner` is the raw value of the
    raster's cell (0, 0), binary_map's nodata after scaling (dtb_eval_hist).  No host sync."""
    desc = _chk2d(desc, "descriptor")
    flood = flood_int8(flood, desc)
    if hist.dtype != torch.int64 or hist.numel() != 4 * 33 or hist.device != desc.device or not hist.is_contiguous():
        raise ValueError("hist must be a contiguous int64 tensor of 4 x 33 entries on the descriptor's device")
    th = np.ascontiguousarray(thresholds, dtype=np.float64)
    with torch.cuda.device(desc.device):
        check(lib.dtb_eval_hist(_ptr(desc), _ev_dtype(desc), _ptr(flood), desc.numel(), float(mn), float(mx), float(nodata),
                                float(corner), th.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), len(th),
                                1 if under == "under" else 0, _ptr(hist), _stream()), "dtb_eval_hist")
    return hist


def eval_class(desc: torch.Tensor, flood: torch.Tensor, mn: float, mx: float, corner: float, threshold: float, under: str,
               nodata: float = -100, out: torch.Tensor | None = None) -> torch.Tensor:
    """int8 class map (0 tn, 1 fp, 2 fn, 3 tp) = avaliacao(binary_map(minMaxScale(desc, mn, mx, nodata), threshold), flood),
    scaled on load like eval_hist (dtb_eval_class_scaled)"""
    desc = _chk2d(desc, "descriptor")
    flood = flood_int8(flood, desc)
    cls = _out(None if out is None else {"cls": out}, "cls", tuple(desc.shape), torch.int8, desc.device)
    with torch.cuda.device(desc.device):
        check(lib.dtb_eval_class_scaled(_ptr(desc), _ev_dtype(desc), _ptr(flood), desc.numel(), float(mn), float(mx), float(nodata),
                                        float(corner), float(threshold), 1 if under == "under" else 0, _ptr(cls), _stream()),
              "dtb_eval_class_scaled")
    return cls


def calibrate(desc: torch.Tensor, flood: torch.Tensor, under: str = "under", nodata: float = -100) -> dict:
    """Calibrate a descriptor against a benchmark flood map on the device: what example.py:113-147 does with np.unique,
    minMaxScale, calibration, binary_map and avaliacao, without the float64 raster and without modifying `flood`.

    desc: float32 or int16 CUDA tensor; flood: int8 or uint8 of the same shape.  One extrema pass gives
    mn = np.unique(desc)[1] and mx = np.unique(desc)[-1], then one scaled histogram pass per stage of the threshold search
    (evaluation.search_threshold) and one class-map pass.  Returns {"threshold", "correctness", "fit", "mn", "mx",
    "counts": (tn, fp, fn, tp) at the threshold, "class_map": int8 CUDA tensor}.  ValueError if desc has fewer than two
    distinct values."""
    from . import evaluation

    desc = _chk2d(desc, "descriptor")
    _ev_dtype(desc)
    flood = flood_int8(flood, desc)
    if under not in ("under", "over"):
        raise ValueError("under must be 'under' or 'over'")
    with torch.cuda.device(desc.device):
        ext = torch.cat([eval_extrema(desc), desc.reshape(-1)[:1].to(torch.float64)]).cpu().numpy()
        mn, mx = evaluation.unique_ends(ext[:5])
        corner = float(ext[5])
        hist = torch.empty(4 * 33, dtype=torch.int64, device=desc.device)

        def counts(thresholds):
            hist.zero_()
            eval_hist(desc, flood, mn, mx, corner, thresholds, under, hist, nodata)
            return evaluation.counts_from_hist(hist.cpu().numpy(), len(thresholds), under)

        th, c, f, cnt = evaluation.search_threshold(counts)
        cls = eval_class(desc, flood, mn, mx, corner, th, under, nodata)
    return dict(threshold=th, correctness=c, fit=f, mn=mn, mx=mx, counts=cnt, class_map=cls)


def chain_check(d8: torch.Tensor, acc: torch.Tensor, river_threshold: int, idx: torch.Tensor | None = None,
                dem: torch.Tensor | None = None, hand: torch.Tensor | None = None, row0: int = 0,
                total_rows: int | None = None) -> torch.Tensor:
    """Identities of a finished chain over one raster / row band -> 8 uint64 counters on the device (csrc/verify.cu)."""
    d8, acc = _chk2d(d8, "d8"), _chk2d(acc, "acc")
    _same_shape(d8=d8, acc=acc, idx=idx, dem=dem, hand=hand)
    rows, cols = d8.shape
    out = torch.zeros(8, dtype=torch.int64, device=d8.device)
    if (dem is not None and dem.dtype != torch.float32) or (hand is not None and hand.dtype != torch.float32):
        dem = hand = None  # the HAND identity is checked for float32 rasters only
    check(lib.dtb_chain_check(_ptr(d8), _ptr(acc), _int_dtype(acc), _ptr(idx), _int_dtype(idx) if idx is not None else 0, _ptr(dem),
                              _ptr(hand), rows, cols, int(row0), int(rows if total_rows is None else total_rows),
                              int(river_threshold), _ptr(out), _stream()), "dtb_chain_check")
    return out


def chain_verdict(counters) -> dict:
    """counters: the (summed over bands) result of chain_check -> {"verified": bool, ...}"""
    c = [int(v) for v in counters]
    return {"verified": c[0] == c[1] and c[2] == c[3] == c[4] == c[5] == 0, "valid_cells": c[1], "root_mass": c[0],
            "count_not_sum_of_tributaries": c[2], "idx_not_river": c[3], "river_not_self": c[4], "hand_mismatch": c[5], "no_river": c[6],
            "idx_in_other_band": c[7]}


# ---- benchmark support -----------------------------------------------------------------
SYNTH_SEED = 20260101
SYNTH_Z0, SYNTH_SR, SYNTH_SC, SYNTH_DEPTH = 100.0, 0.02, 0.005, 6.0
SYNTH_AMP0, SYNTH_HURST = 15.0, 0.6


def synth_amplitudes() -> np.ndarray:
    k = np.arange(10, dtype=np.float64)
    return (SYNTH_AMP0 * (0.5 ** k) ** SYNTH_HURST).astype(np.float32)


def synth_dem(rows: int, cols: int, row0: int = 0, seed: int = SYNTH_SEED) -> torch.Tensor:
    """Synthetic DEM recipe 'dtb-synth-v1' (SURVEY.md 8d) generated on the device."""
    dev = require_cuda()
    out = torch.empty((rows, cols), dtype=torch.float32, device=dev)
    amp = synth_amplitudes()
    check(lib.dtb_synth_dem_f32(rows, cols, row0, seed, amp.ctypes.data_as(ctypes.POINTER(ctypes.c_float)),
                                SYNTH_Z0, SYNTH_SR, SYNTH_SC, SYNTH_DEPTH, _ptr(out), _stream()), "dtb_synth_dem_f32")
    return out


def fill_depressions(dem: torch.Tensor) -> int:
    """In-place priority-flood+epsilon fixed point; returns the number of relaxation passes."""
    dem_c = _chk2d(dem, "dem")
    if dem_c.data_ptr() != dem.data_ptr() or dem.dtype != torch.float32:
        raise ValueError("dem must be a contiguous float32 CUDA tensor")
    rows, cols = dem.shape
    nbytes = lib.dtb_fill_workspace_bytes(rows, cols)
    ws = workspace.get(nbytes, "fill")
    it = ctypes.c_int(0)
    check(lib.dtb_fill_depressions_f32(_ptr(dem), rows, cols, _ptr(ws), nbytes, ctypes.byref(it), _stream()),
          "dtb_fill_depressions_f32")
    return int(it.value)


def conditioned_dem(rows: int, cols: int, seed: int = SYNTH_SEED) -> torch.Tensor:
    dem = synth_dem(rows, cols, 0, seed)
    fill_depressions(dem)
    return dem
