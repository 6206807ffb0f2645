"""pipeline.py -- the headline chain slope -> D8 -> flow accumulation -> HAND -> GFI.

The reference runs every descriptor as an independent host->device->host round trip
(Example/example.py:59-91) and takes D8 / accumulation rasters from disk (example.py:36,39).
Here the chain stays on the device: three C-ABI calls (dtb_slope_d8, dtb_flowacc, dtb_hand with
the fused HAND/GFI epilogue) over buffers that never leave HBM.

    run_device(dem_cuda_tensor, ...) -> dict of CUDA tensors        (what bench.py times as `value`)
    pipeline(dem_numpy, ...)         -> dict of NumPy arrays        (host in / host out, `e2e`)
    pipeline_files(dem.tif, out_dir) -> GeoTIFF in, GeoTIFFs out            (raster.py codec, section 8 f3)
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import device
from ._convert import dem_to_native

STAGE_OUTPUTS = ("slope", "d8", "acc", "fdist", "idx", "hand", "gfi")
LOG_OUTPUTS = ("ti", "mti", "lnhlh")  # pipeline_files(outputs=...) and BandRunner.log_indices


def alloc_outputs(rows: int, cols: int, dem_dtype: torch.dtype = torch.float32, device=None) -> dict:
    """the seven rasters of the chain, allocated once (pass as `out=` to run_device / pipeline to reuse them)"""
    dev = device if device is not None else torch.device("cuda", torch.cuda.current_device())
    it = torch.int32 if rows * cols < 2**31 else torch.int64
    dts = dict(slope=torch.float32, d8=torch.uint8, acc=it, fdist=torch.float32, idx=it, hand=dem_dtype, gfi=torch.float32)
    return {k: torch.empty((rows, cols), dtype=v, device=dev) for k, v in dts.items()}


def run_device(dem: torch.Tensor, px: float, river_threshold: int, n_gfi: float = 0.4, scale_factor: float = 0.1,
               size: float | None = None, max_moves: int = 0, out: dict | None = None) -> dict:
    """slope(%) f32, d8 u8, acc i32/i64, fdist f32, idx i32/i64, hand (DEM dtype), gfi f32.

    river cells are `acc > river_threshold` (example.py:52); GFI uses `size` = px by default
    (example.py:87).  All tensors stay on the device.
    """
    size = px if size is None else size
    rows, cols = dem.shape
    int_dt = torch.int32 if rows * cols < 2**31 else torch.int64
    slope, d8 = device.slope_d8(dem, px, out=out)
    # the last tile pass of the accumulation also does HAND's entry-node pass (river = acc > threshold)
    acc = device.flow_accumulation(d8, dtype=int_dt, nodata_fill=-100, fuse_hand_threshold=river_threshold, out=out)
    out = device.hand(d8, dem, px, acc=acc, river_threshold=river_threshold, max_moves=max_moves,
                      gfi_params=(n_gfi, scale_factor, size), idx_dtype=int_dt, entry_done=True, out=out)
    out.update(slope=slope, d8=d8, acc=acc)
    return out


_buffers = {}


def _device_buffers(rows, cols, dem_dtype, dev) -> dict:
    """device rasters of the host pipeline, kept between calls (one set per shape; release_buffers() frees them)"""
    key = (rows, cols, dem_dtype, str(dev))
    if key not in _buffers:
        _buffers.clear()
        b = alloc_outputs(rows, cols, dem_dtype, dev)
        b["dem"] = torch.empty((rows, cols), dtype=dem_dtype, device=dev)
        _buffers[key] = b
    return _buffers[key]


def release_buffers() -> None:
    _buffers.clear()


def pipeline(dem, px: float, river_threshold: int, n_gfi: float = 0.4, scale_factor: float = 0.1,
             size: float | None = None, outputs=STAGE_OUTPUTS, pinned_out: dict | None = None, chunks: int = 8) -> dict:
    """Host-side chain: NumPy DEM in, NumPy rasters out (dtypes as the reference returns them on the
    device side: slope/fdist/gfi float32, d8 uint8, acc/idx int32 or int64, hand in the DEM's dtype).

    The reference moves every descriptor host->device->host separately (slope.py:195-200,
    flowhand.py:543-557, gfi.py:252-261).  Here the DEM goes up once, in `chunks` row blocks on a copy
    stream, the slope/D8 stencil starts on a block as soon as the block below it has landed, and every
    finished raster streams back on a second copy stream while the next stage computes.

    `pinned_out` may hold pre-allocated pinned torch CPU tensors keyed by output name (the benchmark
    reuses them across steps); otherwise pageable arrays are returned.
    """
    dev = device.require_cuda()
    size = px if size is None else size
    dem_h = dem if isinstance(dem, torch.Tensor) else torch.from_numpy(dem_to_native(dem))
    if dem_h.is_cuda:
        res = run_device(dem_h, px, river_threshold, n_gfi, scale_factor, size)
        host = {name: res[name].cpu().numpy() for name in outputs}
        return host
    rows, cols = dem_h.shape
    int_dt = torch.int32 if rows * cols < 2**31 else torch.int64
    main = torch.cuda.current_stream()
    up, down = torch.cuda.Stream(), torch.cuda.Stream()
    host, keep = {}, []

    def send_back(name, t, r0=None, r1=None):
        """queue the device->host copy of raster `name` (rows [r0, r1) of it) behind the work recorded so far"""
        if name not in outputs:
            return
        if name not in host:
            if pinned_out is not None and name in pinned_out:
                host[name] = pinned_out[name]
            else:
                host[name] = torch.empty(t.shape, dtype=t.dtype)
        ev = torch.cuda.Event()
        ev.record(main)
        down.wait_event(ev)
        with torch.cuda.stream(down):
            if r0 is None:
                host[name].copy_(t, non_blocking=True)
            else:
                host[name][r0:r1].copy_(t[r0:r1], non_blocking=True)

    # DEM up in row blocks; slope + D8 of a block runs once the block below it (its halo row) is resident
    buf = _device_buffers(rows, cols, dem_h.dtype, dev)
    dem_d, slope, d8 = buf["dem"], buf["slope"], buf["d8"]
    k = max(1, min(chunks, rows // 256 or 1))
    edges = [rows * i // k for i in range(k + 1)]
    arrived = []
    up.wait_stream(main)
    for i in range(k):
        with torch.cuda.stream(up):
            dem_d[edges[i]:edges[i + 1]].copy_(dem_h[edges[i]:edges[i + 1]], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(up)
        arrived.append(ev)
    from ._lib import check, lib

    for i in range(k):
        main.wait_event(arrived[min(i + 1, k - 1)])
        r0, r1 = edges[i], edges[i + 1]
        check(lib.dtb_slope_d8(dem_d.data_ptr(), device._dem_dtype(dem_d), rows, cols, r0, r1, float(px),
                               slope[r0:r1].data_ptr(), d8[r0:r1].data_ptr(), main.cuda_stream), "dtb_slope_d8")
        send_back("slope", slope, r0, r1)
        send_back("d8", d8, r0, r1)
    acc = device.flow_accumulation(d8, dtype=int_dt, nodata_fill=-100, fuse_hand_threshold=river_threshold, out=buf)
    send_back("acc", acc)
    out = device.hand(d8, dem_d, px, acc=acc, river_threshold=river_threshold, gfi_params=(n_gfi, scale_factor, size),
                      idx_dtype=int_dt, entry_done=True, out=buf)
    for name in ("idx", "fdist", "hand", "gfi"):
        keep.append(out[name])
        send_back(name, out[name])
    down.synchronize()
    main.synchronize()
    return {name: host[name].numpy() for name in outputs}


def output_dtypes(dem_dtype: np.dtype, n_cells: int) -> dict:
    it = np.int32 if n_cells < 2**31 else np.int64
    return dict(slope=np.float32, d8=np.uint8, acc=it, fdist=np.float32, idx=it, hand=np.dtype(dem_dtype), gfi=np.float32)


def output_meta(name: str, floating: bool, compress: str = "lzw", blocksize: int = 256) -> dict:
    """file metadata of the chain's raster `name` (pipeline_files, bands.BandRunner.write_files): tiled, the predictor that
    suits the samples (3 floating point, 2 integers), nodata -100 (0 for the D8 codes, like 12_fdr.tif, and for class
    maps, like example.py:206)"""
    return dict(compress=compress, predictor=1 if compress in (None, "none") else (3 if floating else 2), tiled=True, blockxsize=blocksize,
                blockysize=blocksize, nodata=0 if name == "d8" or name.endswith("_class") else -100)


def pipeline_files(dem_path, out_dir, river_threshold: int, px: float | None = None, n_gfi: float = 0.4,
                   scale_factor: float = 0.1, size: float | None = None, outputs=STAGE_OUTPUTS, compress: str = "lzw",
                   blocksize: int = 256, block_bytes: int = 256 << 20, threads: int = 0, decode: str = "auto", encode: str = "auto",
                   condition: bool = False, flood=None, under: str = "under", n_top: float = 0.1) -> dict:
    """The chain from a DEM GeoTIFF to one GeoTIFF per descriptor (`out_dir/<name>.tif`), what a user of the
    reference does around the descriptor calls with rasterio (example.py:33, :42-43, :201-217).

    The DEM is decoded in row blocks into pinned memory and copied to the device as it is decoded
    (raster.read_to_device; `decode="device"` sends the compressed tiles instead and decodes them on the GPU); its nodata value (GDAL_NODATA tag) becomes the path's sentinel -100 on the device
    (example.py:42-43 does that on the host, from the corner cell); `px` defaults to the file's pixel size.
    Results are encoded block by block as they are copied back (raster.write_from_device; `encode="device"` encodes the
    tiles on the GPU and copies only the compressed bytes), tiled and compressed,
    with the DEM's georeferencing; nodata is -100 (0 for the D8 codes, like 12_fdr.tif).
    `condition=True` fills the DEM's depressions on the device first (device.fill_depressions, SURVEY section 8 f4) --
    for DEMs that no GIS has conditioned yet (float32 only).
    `decode` / `encode`: "device", "host", or "auto" (default) = the device codec whenever it can take the file
    (stored or LZW chunks), the host codec for the rest (Deflate, PackBits, chunks over 1 MiB).
    `outputs` may also list "ti", "mti" (example.py:63-69, exponent `n_top`), "lnhlh" (example.py:91) and, with a
    benchmark flood map GeoTIFF `flood` (uint8 / int8, the DEM's shape), "hand_class": HAND calibrated against it
    (device.calibrate, direction `under`; example.py:113-147), written as uint8 with nodata 0 (example.py:201-217).
    Returns {name: path}, plus "calibration": the numbers of device.calibrate when `flood` is given.
    """
    import torch

    from . import raster

    device.require_cuda()
    known = STAGE_OUTPUTS + LOG_OUTPUTS + ("hand_class",)
    for name in outputs:
        if name not in known:
            raise ValueError(f"unknown output {name!r} (one of {', '.join(known)})")
    if "hand_class" in outputs and flood is None:
        raise ValueError("the output 'hand_class' needs a benchmark flood map (flood=...)")
    with raster.open(dem_path) as src:
        geo = dict(crs=src.crs, transform=src.transform)
        if px is None:
            px = src.res[0]
        dem = raster.read_to_device(src, block_bytes=block_bytes, threads=threads, decode=decode)
        nodata = src.nodata
    if dem.dtype not in (torch.float32, torch.int16):
        # the kernels take the two DEM types the reference is used with (f32 rasters, int16 after example.py:33)
        dem = dem.to(torch.float32)
    if dem.dtype == torch.float32:
        device.nodata_to_sentinel(dem, nodata)  # example.py:42-43, one pass (dtb_nodata_to_sentinel_f32)
    elif nodata is not None:
        dem.masked_fill_(dem == nodata, -100)   # int16 DEMs: plumbing only
    if condition:
        if dem.dtype != torch.float32:
            raise TypeError("condition=True needs a float32 DEM (the filling raises cells by single float32 steps)")
        device.fill_depressions(dem)
    res = run_device(dem, float(px), int(river_threshold), n_gfi, scale_factor, size)
    if any(name in outputs for name in ("ti", "mti")):
        res["ti"], res["mti"] = device.ti_mti(res["acc"], device.slope_to_radians(res["slope"]), float(px), n_top)
    if "lnhlh" in outputs:
        res["lnhlh"] = device.ln_hl_H(res["hand"], res["acc"], n_gfi, scale_factor, px if size is None else size)
    calib = None
    if flood is not None:
        fl = raster.read_to_device(flood, block_bytes=block_bytes, threads=threads, decode=decode)
        if tuple(fl.shape) != tuple(dem.shape):
            raise ValueError(f"{flood}: flood map is {tuple(fl.shape)}, the DEM {tuple(dem.shape)}")
        calib = device.calibrate(res["hand"], fl, under)
        res["hand_class"] = calib.pop("class_map").view(torch.uint8)
    os.makedirs(out_dir, exist_ok=True)
    paths = {}
    for name in outputs:
        t = res[name]
        paths[name] = os.path.join(out_dir, name + ".tif")
        raster.write_from_device(paths[name], t, block_bytes=block_bytes, threads=threads, encode=encode,
                                 **output_meta(name, t.dtype.is_floating_point, compress, blocksize), **geo)
    if calib is not None:
        paths["calibration"] = calib
    return paths
