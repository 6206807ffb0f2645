"""GeoTIFF codec (SURVEY.md section 8 f3; include/dtb200_io.h, descriptools_b200/raster.py).

The checker is libtiff as bundled with Pillow: files written by the codec must read back identically through
Pillow, and files written by Pillow (strips, LZW / Deflate / PackBits, with and without the horizontal predictor)
must decode identically through the codec.
"""
import ctypes
import os
import re
import struct

import numpy as np
import pytest

import descriptools_b200.raster as rio

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PIL_MODES = {"uint8": "L", "uint16": "I;16", "int32": "I", "float32": "F"}


def _rand(shape, dtype, seed=0, smooth=True):
    rng = np.random.default_rng(seed)
    dt = np.dtype(dtype)
    if dt.kind == "f":
        a = rng.standard_normal(shape).cumsum(axis=1) if smooth else rng.standard_normal(shape)
        return a.astype(dt)
    info = np.iinfo(dt)
    if smooth:
        a = rng.integers(-3, 4, size=shape).cumsum(axis=1) + (0 if info.min < 0 else 200)
        return np.clip(a, info.min, info.max).astype(dt)
    return rng.integers(info.min, info.max, size=shape, dtype=dt, endpoint=True)


def _pil_read(path):
    from PIL import Image

    Image.MAX_IMAGE_PIXELS = None
    with Image.open(path) as im:
        return np.array(im)


def test_library_exports_every_declared_symbol():
    src = open(os.path.join(REPO, "include", "dtb200_io.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = sorted(set(re.findall(r"\b(dtbio_[a-z0-9_]+)\s*\(", src)))
    assert len(names) >= 14
    raw = ctypes.CDLL(rio.LIB_PATH)
    for n in names:
        assert hasattr(raw, n), f"libdtb200_io.so does not export {n}"
    assert rio.lib.dtbio_abi_version() == 1
    assert [rio.lib.dtbio_dtype_size(i) for i in range(10)] == [1, 1, 2, 2, 4, 4, 8, 8, 4, 8]


@pytest.mark.parametrize("dtype", ["uint8", "int8", "uint16", "int16", "uint32", "int32", "uint64", "int64", "float32", "float64"])
@pytest.mark.parametrize("layout", ["strips", "tiles"])
@pytest.mark.parametrize("compress,predictor", [("none", 1), ("lzw", 1), ("lzw", 2), ("deflate", 1), ("deflate", 2), ("lzw", 3), ("deflate", 3)])
def test_round_trip_every_dtype_layout_and_codec(tmp_path, dtype, layout, compress, predictor):
    if predictor == 3 and np.dtype(dtype).kind != "f":
        pytest.skip("floating-point predictor")
    a = _rand((157, 203), dtype, seed=3)  # ragged against 64 x 48 tiles and 7-row strips
    path = tmp_path / "t.tif"
    kw = dict(tiled=True, blockxsize=48, blockysize=64) if layout == "tiles" else dict(blockysize=7)
    with rio.open(path, "w", driver="GTiff", width=203, height=157, count=1, dtype=dtype, compress=compress, predictor=predictor,
                  nodata=-100 if np.dtype(dtype).kind != "u" else 0, **kw) as dst:
        dst.write(a)
    with rio.open(path) as src:
        assert src.shape == a.shape and src.dtypes == (dtype,) and src.compression == compress
        assert src.nodata == (-100 if np.dtype(dtype).kind != "u" else 0)
        assert src.block_shapes == ([(64, 48)] if layout == "tiles" else [(7, 203)])
        np.testing.assert_array_equal(src.read(1), a)
        np.testing.assert_array_equal(src.read(), a[None])
        # a row block that starts and ends inside chunks, into a wider buffer
        buf = np.full((40, 256), 77, dtype=dtype)
        src.read_rows(59, 40, buf, threads=3)
        np.testing.assert_array_equal(buf[:, :203], a[59:99])
        assert (buf[:, 203:] == 77).all()
    if dtype in PIL_MODES:  # libtiff agrees (it has no mode for the other sample types through Pillow)
        np.testing.assert_array_equal(_pil_read(path), a)


@pytest.mark.parametrize("dtype", ["uint8", "uint16", "int32", "float32"])
@pytest.mark.parametrize("compression,predictor", [("raw", False), ("tiff_lzw", False), ("tiff_lzw", True), ("tiff_adobe_deflate", False),
                                                   ("tiff_adobe_deflate", True), ("packbits", False)])
def test_reads_what_libtiff_writes(tmp_path, dtype, compression, predictor):
    from PIL import Image

    if predictor and dtype == "float32":
        pytest.skip("Pillow cannot ask libtiff for the floating-point predictor")
    a = _rand((301, 333), dtype, seed=5, smooth=(compression != "raw"))
    path = str(tmp_path / "p.tif")
    kw = {} if compression == "raw" else {"compression": compression}
    if predictor:
        kw["tiffinfo"] = {317: 2}
    Image.fromarray(a).save(path, **kw)
    with rio.open(path) as src:
        assert src.dtypes == (dtype,)
        np.testing.assert_array_equal(src.read(1, threads=2), a)
        np.testing.assert_array_equal(src.read_rows(300, 1), a[300:])


def test_lzw_table_resets_and_incompressible_data(tmp_path):
    # 256 KiB of noise per tile: the 12-bit table fills and is cleared dozens of times per chunk
    a = _rand((512, 512), "uint8", seed=9, smooth=False)
    path = tmp_path / "noise.tif"
    with rio.open(path, "w", width=512, height=512, dtype="uint8", compress="lzw", tiled=True, blockxsize=512, blockysize=512) as dst:
        dst.write(a)
    np.testing.assert_array_equal(rio.open(path).read(1), a)
    np.testing.assert_array_equal(_pil_read(path), a)
    # and the other extreme: one value, codes grow to the longest strings
    z = np.zeros((512, 512), np.uint8)
    with rio.open(path, "w", width=512, height=512, dtype="uint8", compress="lzw", blockysize=512) as dst:
        dst.write(z)
    assert os.path.getsize(path) < 2000
    np.testing.assert_array_equal(rio.open(path).read(1), z)
    np.testing.assert_array_equal(_pil_read(path), z)


def test_georeferencing_and_meta_follow_the_example(tmp_path):
    """example.py:201-217: meta of the DEM, dtype / nodata updated, written with the class map"""
    crs = rio.GeoKeys((1, 1, 0, 3, 1024, 0, 1, 1, 1025, 0, 1, 1, 3072, 0, 1, 32722), (), "")
    tr = rio.Affine(12.5, 0.0, 605681.5, 0.0, -12.5, 7010736.25)
    dem = _rand((64, 80), "float32", seed=1)
    p1, p2 = tmp_path / "dem.tif", tmp_path / "class.tif"
    with rio.open(p1, "w", driver="GTiff", width=80, height=64, count=1, dtype=rio.float32, crs=crs, transform=tr,
                  nodata=-3.4028230607370965e38, compress="lzw", tiled=True, blockxsize=32, blockysize=32) as dst:
        dst.write(dem.reshape(1, 64, 80))
    meta = rio.open(p1).meta
    assert meta["dtype"] == "float32" and meta["width"] == 80 and meta["height"] == 64 and meta["count"] == 1
    assert meta["crs"] == crs and meta["crs"].to_epsg() == 32722 and meta["transform"] == tr
    assert meta["nodata"] == pytest.approx(-3.4028230607370965e38)
    meta.update(dtype=rio.uint8)
    meta.update(nodata=0)
    cls = (dem > 0).astype("uint8").reshape(1, 64, 80)
    with rio.open(p2, "w", **meta) as dist:
        dist.write(cls.astype(rio.uint8))
    with rio.open(p2) as src:
        assert src.meta == dict(meta, dtype="uint8", nodata=0.0)
        assert src.transform * (0, 0) == (605681.5, 7010736.25) and src.res == (12.5, 12.5)
        assert not src.is_tiled and src.compression == "none"  # rasterio's default layout for a bare meta
        np.testing.assert_array_equal(src.read(1), cls[0])
    from PIL import Image

    with Image.open(p2) as im:  # a foreign reader sees the same tags
        assert im.tag_v2[33550] == (12.5, 12.5, 0.0) and im.tag_v2[33922] == (0.0, 0.0, 0.0, 605681.5, 7010736.25, 0.0)
        assert im.tag_v2[42113] == "0" and tuple(im.tag_v2[34735]) == crs.directory


def test_predictor_without_a_codec_is_dropped(tmp_path):
    """libtiff and GDAL apply the predictor only inside LZW / Deflate; a stored file never carries one"""
    a = _rand((40, 50), "int16", seed=7)
    p = tmp_path / "s.tif"
    with rio.open(p, "w", width=50, height=40, dtype="int16", compress="none", predictor=2) as dst:
        dst.write(a)
    assert rio.open(p).profile["predictor"] == 1
    np.testing.assert_array_equal(_pil_read(p), a)
    from descriptools_b200 import _lib

    lay = _lib.TiffLayout(rows=40, cols=50, bps=2, predictor=2, compression=1, tiled=0, chunk_rows=8, chunk_cols=50, big_endian=0)
    assert _lib.lib.dtb_tiff_encode_bound(ctypes.byref(lay)) == 0
    assert _lib.lib.dtb_tiff_decode_workspace_bytes(ctypes.byref(lay), 5) == 0


def test_bigtiff_and_big_endian_files(tmp_path):
    a = _rand((90, 70), "int16", seed=2)
    path = tmp_path / "big.tif"
    with rio.open(path, "w", width=70, height=90, dtype="int16", compress="deflate", predictor=2, tiled=True, blockxsize=32, blockysize=32,
                  bigtiff="YES") as dst:
        assert dst.bigtiff
        dst.write(a)
    assert open(path, "rb").read(4) == b"II\x2b\x00"
    with rio.open(path) as src:
        assert src.profile["bigtiff"] and src.profile["predictor"] == 2 and src.profile["blockxsize"] == 32
        np.testing.assert_array_equal(src.read(1), a)
    np.testing.assert_array_equal(_pil_read(path), a)
    # hand-made big-endian classic TIFF: one uncompressed strip of int16
    be = tmp_path / "mm.tif"
    data = a.astype(">i2").tobytes()
    entries = [(256, 3, 1, 70), (257, 3, 1, 90), (258, 3, 1, 16), (259, 3, 1, 1), (262, 3, 1, 1), (273, 4, 1, 8), (277, 3, 1, 1),
               (278, 3, 1, 90), (279, 4, 1, len(data)), (339, 3, 1, 2)]
    ifd = struct.pack(">H", len(entries))
    for tag, typ, cnt, val in entries:
        ifd += struct.pack(">HHI", tag, typ, cnt) + (struct.pack(">HH", val, 0) if typ == 3 else struct.pack(">I", val))
    ifd += struct.pack(">I", 0)
    with open(be, "wb") as f:
        f.write(b"MM" + struct.pack(">HI", 42, 8 + len(data)) + data + ifd)
    with rio.open(be) as src:
        assert src.dtypes == ("int16",)
        np.testing.assert_array_equal(src.read(1), a)
    np.testing.assert_array_equal(_pil_read(be), a)


def test_row_blocks_in_any_order_and_writer_rules(tmp_path):
    a = _rand((200, 96), "float32", seed=4)
    path = tmp_path / "blocks.tif"
    w = rio.open(path, "w", width=96, height=200, dtype="float32", compress="lzw", predictor=3, tiled=True, blockxsize=64, blockysize=64)
    assert w.chunk_rows == 64
    with pytest.raises(rio.RasterError, match="chunk boundary"):
        w.write_rows(10, a[10:74])
    with pytest.raises(rio.RasterError, match="chunk boundary"):
        w.write_rows(0, a[:70])
    w.write_rows(128, a[128:])  # last block first, ragged end
    w.write_rows(0, a[:128])
    with pytest.raises(rio.RasterError, match="twice"):
        w.write_rows(64, a[64:128])
    w.close()
    np.testing.assert_array_equal(rio.open(path).read(1), a)
    np.testing.assert_array_equal(_pil_read(path), a)
    # a writer closed with chunks missing reports it and leaves no file behind
    w = rio.open(path, "w", width=96, height=200, dtype="float32", blockysize=50)
    w.write_rows(0, a[:50])
    with pytest.raises(rio.RasterError, match="never written"):
        w.close()
    assert not os.path.exists(path)


def test_errors_are_reported_not_guessed(tmp_path):
    with pytest.raises(rio.RasterError, match="cannot open"):
        rio.open(tmp_path / "absent.tif")
    junk = tmp_path / "junk.tif"
    junk.write_bytes(b"not a tiff at all")
    with pytest.raises(rio.RasterError, match="not a TIFF"):
        rio.open(junk)
    from PIL import Image

    rgb = tmp_path / "rgb.tif"
    Image.fromarray(np.zeros((8, 8, 3), np.uint8)).save(rgb)
    with pytest.raises(rio.RasterError, match="sample per pixel"):
        rio.open(rgb)
    # a truncated file: the tile data is gone but the IFD survives at the front? (ours sits at the end: cut it)
    good = tmp_path / "good.tif"
    with rio.open(good, "w", width=64, height=64, dtype="uint8", compress="lzw") as dst:
        dst.write(np.zeros((64, 64), np.uint8))
    cut = tmp_path / "cut.tif"
    cut.write_bytes(good.read_bytes()[:40])
    with pytest.raises(rio.RasterError):
        rio.open(cut)
    with pytest.raises(rio.RasterError, match="band 1"):
        rio.open(good).read(2)
    with pytest.raises(rio.RasterError, match="shape"):
        with rio.open(tmp_path / "x.tif", "w", width=4, height=4, dtype="uint8") as dst:
            dst.write(np.zeros((5, 4), np.uint8))
    assert not os.path.exists(tmp_path / "x.tif")
    with pytest.raises(rio.RasterError, match="GeoKeys"):
        rio.open(tmp_path / "y.tif", "w", width=4, height=4, dtype="uint8", crs="EPSG:32722")
    assert not os.path.exists(tmp_path / "y.tif")


def _count_closes(monkeypatch):
    """dtbio_close_writer wrapped: counts the calls per handle and forwards only the first (a second one would free the
    handle twice)"""
    calls, real = {}, rio.lib.dtbio_close_writer

    def close_once(h):
        calls[h.value] = calls.get(h.value, 0) + 1
        return real(h) if calls[h.value] == 1 else 0

    monkeypatch.setattr(rio.lib, "dtbio_close_writer", close_once)
    return calls


def test_writer_closed_inside_its_with_block_is_closed_once(tmp_path, monkeypatch):
    calls = _count_closes(monkeypatch)
    a = _rand((64, 80), "float32", seed=1)
    p = tmp_path / "c.tif"
    with pytest.raises(RuntimeError, match="after close"):
        with rio.open(p, "w", width=80, height=64, dtype="float32", compress="lzw", tiled=True, blockxsize=32, blockysize=32) as w:
            w.write(a)
            w.close()
            raise RuntimeError("after close")
    assert list(calls.values()) == [1]
    np.testing.assert_array_equal(rio.open(p).read(1), a)  # complete, so it stays


def _decode_like_the_device(path, first=0, count=None, rows=None):
    """the tile-decoding kernel's per-lane code (csrc/tiffcodec.cu), run lane by lane on the CPU by the library's self-test
    entry point: same geometry, LZW, byte order, predictor and store code the warps execute"""
    from descriptools_b200 import _lib

    with rio.open(path) as r:
        lay, across, off, cnt = rio.chunk_table(r)
        shape, dtype = r.shape, r.dtypes[0]
    data = np.fromfile(path, dtype=np.uint8)
    if rows is not None:  # a row band: the output holds only those rows
        lay.row_lo, lay.row_hi = rows
        shape = (rows[1] - rows[0], shape[1])
        first, last = rio._band_chunks(rows[0], rows[1], lay.chunk_rows, across)
        count = last - first
    out = np.full(shape, 7, dtype=dtype)
    status = ctypes.c_ulonglong(99)
    n = off.size - first if count is None else count
    rc = _lib.lib.dtb_selftest_tiff_decode_host(ctypes.byref(lay), data.ctypes.data, off[first:].ctypes.data, cnt[first:].ctypes.data,
                                                first, n, out.ctypes.data, ctypes.byref(status))
    assert rc == 0
    return out, status.value, (lay, across)


@pytest.mark.parametrize("dtype", ["uint8", "int16", "uint32", "int64", "float32", "float64"])
@pytest.mark.parametrize("layout", ["strips", "tiles"])
@pytest.mark.parametrize("compress,predictor", [("none", 1), ("lzw", 1), ("lzw", 2), ("lzw", 3)])
def test_device_decoder_lane_code_on_the_cpu(tmp_path, dtype, layout, compress, predictor):
    if predictor == 3 and np.dtype(dtype).kind != "f":
        pytest.skip("floating-point predictor")
    a = _rand((157, 203), dtype, seed=8)
    path = tmp_path / "t.tif"
    kw = dict(tiled=True, blockxsize=48, blockysize=64) if layout == "tiles" else dict(blockysize=7)
    with rio.open(path, "w", width=203, height=157, dtype=dtype, compress=compress, predictor=predictor, **kw) as dst:
        dst.write(a)
    out, status, (lay, across) = _decode_like_the_device(path)
    assert status == 0
    np.testing.assert_array_equal(out, a)
    # a range of chunks in the middle: only their cells are touched
    first = across * 1 if layout == "tiles" else 5
    count = across if layout == "tiles" else 9
    out, status, _ = _decode_like_the_device(path, first, count)
    r0, r1 = (64, 128) if layout == "tiles" else (35, 98)
    assert status == 0
    np.testing.assert_array_equal(out[r0:r1], a[r0:r1])
    assert (out[:r0] == 7).all() and (out[r1:] == 7).all()
    # a row band that starts and ends inside chunks: exactly its rows, nothing written outside the band's buffer
    for band in ((70, 141), (0, 64), (150, 157), (3, 4)):
        out, status, _ = _decode_like_the_device(path, rows=band)
        assert status == 0 and out.shape == (band[1] - band[0], 203)
        np.testing.assert_array_equal(out, a[band[0]:band[1]], err_msg=str(band))


def _encode_like_the_device(path, a, **kw):
    """the tile-encoding kernel's per-lane code (csrc/tiffcodec.cu) on the CPU, then the file is put together the way
    write_from_device(encode="device") does it: one blob of streams, dtbio_write_encoded"""
    from descriptools_b200 import _lib

    w = rio.open(path, "w", width=a.shape[1], height=a.shape[0], dtype=a.dtype.name, **kw)
    lay, across, n = w.chunk_layout()
    bound = _lib.lib.dtb_tiff_encode_bound(ctypes.byref(lay))
    assert bound > 0
    enc = np.zeros(n * bound, np.uint8)
    sizes = np.zeros(n, np.int64)
    a = np.ascontiguousarray(a)
    assert _lib.lib.dtb_selftest_tiff_encode_host(ctypes.byref(lay), a.ctypes.data, 0, n, enc.ctypes.data, sizes.ctypes.data) == 0
    assert (sizes > 0).all() and (sizes <= bound).all()
    half = n // 2  # two groups, the second one first
    for c0, c1 in ((half, n), (0, half)):
        al = (sizes[c0:c1] + 1) & ~1
        offs = np.cumsum(al) - al
        blob = np.zeros(int(al.sum()), np.uint8)
        for i in range(c0, c1):
            blob[offs[i - c0]:offs[i - c0] + sizes[i]] = enc[i * bound:i * bound + sizes[i]]
        w.write_encoded(c0, blob, offs, sizes[c0:c1])
    w.close()
    return sizes


@pytest.mark.parametrize("dtype", ["uint8", "int16", "uint32", "int64", "float32", "float64"])
@pytest.mark.parametrize("layout", ["strips", "tiles"])
@pytest.mark.parametrize("compress,predictor", [("none", 1), ("lzw", 1), ("lzw", 2), ("lzw", 3)])
def test_device_encoder_lane_code_on_the_cpu(tmp_path, dtype, layout, compress, predictor):
    if predictor == 3 and np.dtype(dtype).kind != "f":
        pytest.skip("floating-point predictor")
    a = _rand((157, 203), dtype, seed=21)
    path = tmp_path / "e.tif"
    kw = dict(tiled=True, blockxsize=48, blockysize=64) if layout == "tiles" else dict(blockysize=7)
    _encode_like_the_device(path, a, compress=compress, predictor=predictor, nodata=0, **kw)
    with rio.open(path) as src:
        assert src.compression == compress and src.profile["predictor"] == predictor
        np.testing.assert_array_equal(src.read(1), a)       # the host codec reads it
    if dtype in PIL_MODES:
        np.testing.assert_array_equal(_pil_read(path), a)   # libtiff reads it
    out, status, _ = _decode_like_the_device(path)          # the device decoder's lane code reads it
    assert status == 0
    np.testing.assert_array_equal(out, a)


def test_device_encoder_table_resets_and_compression_ratio(tmp_path):
    noise = _rand((512, 512), "uint8", seed=9, smooth=False)   # the dictionary fills and is cleared ~70 times per tile
    p = tmp_path / "n.tif"
    sizes = _encode_like_the_device(p, noise, compress="lzw", tiled=True, blockxsize=512, blockysize=512)
    assert sizes[0] <= 512 * 512 * 1.5 + 200
    np.testing.assert_array_equal(_pil_read(p), noise)
    np.testing.assert_array_equal(rio.open(p).read(1), noise)
    flat = np.zeros((512, 512), np.uint8)                      # longest strings
    sizes = _encode_like_the_device(p, flat, compress="lzw", blockysize=512)
    assert sizes[0] < 2000
    np.testing.assert_array_equal(_pil_read(p), flat)
    # the forgetful dictionary costs little against the exact one of the host codec
    dem = _rand((512, 512), "float32", seed=4)
    q = tmp_path / "h.tif"
    with rio.open(q, "w", width=512, height=512, dtype="float32", compress="lzw", predictor=3, tiled=True, blockxsize=256, blockysize=256) as d:
        d.write(dem)
    _encode_like_the_device(p, dem, compress="lzw", predictor=3, tiled=True, blockxsize=256, blockysize=256)
    np.testing.assert_array_equal(rio.open(p).read(1), dem)
    assert os.path.getsize(p) < 1.05 * os.path.getsize(q)


@pytest.mark.parametrize("dtype", ["uint8", "int16", "uint32", "float32", "float64"])
@pytest.mark.parametrize("layout", ["strips", "tiles"])
@pytest.mark.parametrize("predictor", [1, 2, 3])
def test_device_inflate_lane_code_on_the_cpu(tmp_path, dtype, layout, predictor):
    """Deflate chunks (zlib streams: dynamic, fixed and stored blocks) through the device decoder's lane code"""
    if predictor == 3 and np.dtype(dtype).kind != "f":
        pytest.skip("floating-point predictor")
    path = tmp_path / "z.tif"
    kw = dict(tiled=True, blockxsize=48, blockysize=64) if layout == "tiles" else dict(blockysize=7)
    for smooth in (True, False):  # compressible (dynamic codes, long matches) and noise (stored / near-stored blocks)
        a = _rand((157, 203), dtype, seed=31, smooth=smooth)
        with rio.open(path, "w", width=203, height=157, dtype=dtype, compress="deflate", predictor=predictor, **kw) as dst:
            dst.write(a)
        out, status, _ = _decode_like_the_device(path)
        assert status == 0
        np.testing.assert_array_equal(out, a)
        out, status, _ = _decode_like_the_device(path, rows=(60, 131))
        assert status == 0
        np.testing.assert_array_equal(out, a[60:131])


@pytest.mark.parametrize("dtype", ["uint8", "uint16", "int32", "float32"])
def test_device_packbits_lane_code_on_the_cpu(tmp_path, dtype):
    """PackBits strips as libtiff writes them, through the device decoder's lane code"""
    from PIL import Image

    p = str(tmp_path / "pb.tif")
    for a in (_rand((301, 333), dtype, seed=5), np.repeat(_rand((301, 9), dtype, seed=6, smooth=False), 37, axis=1)):  # literals; long runs
        Image.fromarray(a).save(p, compression="packbits")
        assert rio.open(p).compression == "packbits"
        out, status, _ = _decode_like_the_device(p)
        assert status == 0
        np.testing.assert_array_equal(out, a)
        out, status, _ = _decode_like_the_device(p, rows=(100, 211))
        assert status == 0
        np.testing.assert_array_equal(out, a[100:211])


def test_device_inflate_block_types_and_damage(tmp_path):
    import zlib

    from descriptools_b200 import _lib

    rng = np.random.default_rng(5)
    raw = {"runs": np.repeat(rng.integers(0, 4, 700, dtype=np.uint8), 27)[:16384],       # overlapping matches, distance 1
           "text": np.frombuffer((b"flow accumulation and HAND " * 700)[:16384], np.uint8),
           "noise": rng.integers(0, 256, 16384, dtype=np.uint8),
           "zeros": np.zeros(16384, np.uint8)}
    lay = _lib.TiffLayout(rows=128, cols=128, bps=1, predictor=1, compression=8, tiled=1, chunk_rows=128, chunk_cols=128, big_endian=0)

    def lane_decode(stream):
        comp = np.frombuffer(stream, np.uint8).copy()
        off, cnt = np.zeros(1, np.uint64), np.array([comp.size], np.uint64)
        out = np.full((128, 128), 7, np.uint8)
        st = ctypes.c_ulonglong(0)
        assert _lib.lib.dtb_selftest_tiff_decode_host(ctypes.byref(lay), comp.ctypes.data, off.ctypes.data, cnt.ctypes.data, 0, 1,
                                                      out.ctypes.data, ctypes.byref(st)) == 0
        return out.ravel(), st.value

    for name, data in raw.items():
        for level, strategy in ((9, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_DEFAULT_STRATEGY), (0, zlib.Z_DEFAULT_STRATEGY),
                                (6, zlib.Z_FIXED), (6, zlib.Z_HUFFMAN_ONLY), (6, zlib.Z_RLE)):
            c = zlib.compressobj(level, zlib.DEFLATED, 15, 9, strategy)
            stream = c.compress(data.tobytes()) + c.flush()
            out, status = lane_decode(stream)
            assert status == 0, (name, level, strategy)
            np.testing.assert_array_equal(out, data, err_msg=f"{name} level {level} strategy {strategy}")
    # several flushed blocks in one stream (stored, fixed and dynamic mixed)
    c = zlib.compressobj(6)
    stream = b"".join(c.compress(raw["text"][i:i + 3000].tobytes()) + c.flush(zlib.Z_FULL_FLUSH) for i in range(0, 16384, 3000)) + c.flush()
    out, status = lane_decode(stream)
    assert status == 0
    np.testing.assert_array_equal(out, raw["text"])
    # damage is reported as a corrupt chunk, never a crash: truncation, flipped bits, a bad header
    good = zlib.compress(raw["text"].tobytes(), 6)
    for bad in (good[:len(good) // 2], good[:2] + bytes([good[2] ^ 0x06]) + good[3:], b"\x78\x9d" + good[2:], b"\x00\x00" + good[2:], good[:1]):
        out, status = lane_decode(bad)
        assert status & 7 in (1, 3) and status >> 3 == 1
    for k in range(40):  # random corruption anywhere in the stream
        b = bytearray(good)
        for _ in range(3):
            b[rng.integers(2, len(b))] ^= 1 << int(rng.integers(0, 8))
        out, status = lane_decode(bytes(b))
        assert status == 0 or (status & 7 in (1, 3))


@pytest.mark.parametrize("name", ["fuzz_lzw", "fuzz_inflate", "fuzz_reader"])
def test_decoders_under_sanitizers(tmp_path, name):
    """the coders shared by host and device (csrc/lzw.cuh, csrc/inflate.cuh), compiled with AddressSanitizer + UBSan and fed
    intact, truncated and bit-flipped streams from exact-size heap blocks: a damaged file may fail to decode, it must never
    read or write outside its buffers (on the device that would be a fault, not an exception).  fuzz_reader does the same
    to the host library as a whole: valid files of every layout with bytes flipped in the header, the IFD and the chunks"""
    import shutil
    import subprocess

    if shutil.which("g++") is None:
        pytest.skip("no g++")
    src = os.path.join(REPO, "tests", "fuzz", name + ".cpp")
    exe = str(tmp_path / name)
    build = subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=all", "-pthread", src, "-o", exe, "-lz"],
                           capture_output=True, text=True, cwd=os.path.dirname(src))
    if build.returncode != 0 and "sanitize" in build.stderr.lower() + build.stdout.lower():
        pytest.skip("sanitizer runtime not installed")
    assert build.returncode == 0, build.stderr
    run = subprocess.run([exe, "500", str(tmp_path)], capture_output=True, text=True, timeout=300)  # fuzz_reader: whole damaged files
    assert run.returncode == 0, run.stdout[-2000:] + run.stderr[-4000:]
    assert "0 problems" in run.stdout


def test_device_decoder_lane_code_big_endian_and_damage(tmp_path):
    from PIL import Image

    a = _rand((90, 70), "uint16", seed=2)
    be = str(tmp_path / "mm.tif")
    data = a.astype(">u2").tobytes()
    entries = [(256, 3, 1, 70), (257, 3, 1, 90), (258, 3, 1, 16), (259, 3, 1, 1), (262, 3, 1, 1), (273, 4, 1, 8), (277, 3, 1, 1),
               (278, 3, 1, 90), (279, 4, 1, len(data)), (339, 3, 1, 1)]
    ifd = struct.pack(">H", len(entries))
    for tag, typ, cnt, val in entries:
        ifd += struct.pack(">HHI", tag, typ, cnt) + (struct.pack(">HH", val, 0) if typ == 3 else struct.pack(">I", val))
    with open(be, "wb") as f:
        f.write(b"MM" + struct.pack(">HI", 42, 8 + len(data)) + data + ifd + struct.pack(">I", 0))
    out, status, _ = _decode_like_the_device(be)
    assert status == 0
    np.testing.assert_array_equal(out, a)
    # libtiff's LZW with the horizontal predictor (strips), decoded by the lane code
    p = str(tmp_path / "p.tif")
    Image.fromarray(a).save(p, compression="tiff_lzw", tiffinfo={317: 2})
    out, status, _ = _decode_like_the_device(p)
    assert status == 0
    np.testing.assert_array_equal(out, a)
    # damage: truncate every chunk's byte count -> the first chunk is reported as short, nothing crashes
    good = tmp_path / "good.tif"
    with rio.open(good, "w", width=70, height=90, dtype="uint16", compress="lzw", tiled=True, blockxsize=32, blockysize=32) as dst:
        dst.write(a)
    from descriptools_b200 import _lib

    with rio.open(good) as r:
        lay, across, off, cnt = rio.chunk_table(r)
    raw = np.fromfile(good, dtype=np.uint8)
    out = np.zeros((90, 70), np.uint16)
    st = ctypes.c_ulonglong(0)
    half = (cnt // 2).astype(np.uint64)
    assert _lib.lib.dtb_selftest_tiff_decode_host(ctypes.byref(lay), raw.ctypes.data, off.ctypes.data, half.ctypes.data, 0, off.size,
                                                  out.ctypes.data, ctypes.byref(st)) == 0
    assert st.value == ((0 + 1) << 3) | 3
    # an absent chunk (byte count 0) reads as zeros, like GDAL's sparse files
    cnt2 = cnt.copy()
    cnt2[4] = 0
    out = np.full((90, 70), 9, np.uint16)
    _lib.lib.dtb_selftest_tiff_decode_host(ctypes.byref(lay), raw.ctypes.data, off.ctypes.data, cnt2.ctypes.data, 0, off.size,
                                           out.ctypes.data, ctypes.byref(st))
    want = a.copy()
    want[32:64, 32:64] = 0
    assert st.value == 0
    np.testing.assert_array_equal(out, want)
    # argument checks need no device
    lay.compression = 8  # Deflate: decoded, never written
    assert _lib.lib.dtb_tiff_decode_workspace_bytes(ctypes.byref(lay), 4) > 0 and _lib.lib.dtb_tiff_encode_bound(ctypes.byref(lay)) == 0
    lay.compression = 32773  # PackBits: decoded, never written
    assert _lib.lib.dtb_tiff_decode_workspace_bytes(ctypes.byref(lay), 4) > 0 and _lib.lib.dtb_tiff_encode_bound(ctypes.byref(lay)) == 0
    lay.compression = 7  # JPEG: neither
    assert _lib.lib.dtb_tiff_decode_workspace_bytes(ctypes.byref(lay), 4) == 0
    assert _lib.lib.dtb_tiff_decode_chunks(ctypes.byref(lay), 1, 1, 1, 0, 1, 1, 1, 1 << 20, 1, None) == -4
    lay.compression = 5
    assert _lib.lib.dtb_tiff_decode_workspace_bytes(ctypes.byref(lay), 4) == 4 * (32 * 32 * 2 + 8 * 4096) + 256
    assert _lib.lib.dtb_tiff_decode_chunks(ctypes.byref(lay), 1, 1, 1, 0, 1, 1, 1, 100, 1, None) == -3
    assert _lib.lib.dtb_tiff_decode_chunks(ctypes.byref(lay), 1, 1, 1, 8, 2, 1, 1, 1 << 20, 1, None) == -1  # 9 chunks only


def test_random_shapes_layouts_and_codecs(tmp_path):
    """seeded sweep over odd shapes (1-pixel rasters, tiles larger than the raster, one-row strips, ...): host codec,
    libtiff, and the device codec's lane code (decode, banded decode, encode) all agree with the array"""
    import random

    rnd = random.Random(20260101)
    dtypes = ["uint8", "int8", "uint16", "int16", "uint32", "int32", "uint64", "int64", "float32", "float64"]
    for it in range(80):
        dt = rnd.choice(dtypes)
        rows, cols = rnd.choice([1, 2, 3, 5, 16, 17, 31, 33, 64, 65, 100, 129]), rnd.choice([1, 2, 3, 7, 16, 17, 33, 64, 65, 100, 200, 257])
        comp = rnd.choice(["none", "lzw", "lzw", "deflate"])
        pred = rnd.choice([1, 2, 3]) if comp != "none" else 1
        if pred == 3 and np.dtype(dt).kind != "f":
            pred = 2
        if rnd.random() < 0.5:
            kw = dict(tiled=True, blockxsize=rnd.choice([16, 32, 64, 128]), blockysize=rnd.choice([16, 32, 64, 128]))
        else:
            kw = dict(blockysize=rnd.choice([0, 1, 3, 8, 64, 1000]))
        a = _rand((rows, cols), dt, seed=it, smooth=rnd.random() < 0.7)
        what = f"case {it}: {dt} {rows}x{cols} {comp} predictor {pred} {kw}"
        p, q = tmp_path / "h.tif", tmp_path / "d.tif"
        with rio.open(p, "w", width=cols, height=rows, dtype=dt, compress=comp, predictor=pred, **kw) as w:
            w.write(a)
        np.testing.assert_array_equal(rio.open(p).read(1, threads=rnd.choice([1, 3])), a, err_msg=what)
        r0 = rnd.randrange(rows)
        r1 = rnd.randrange(r0 + 1, rows + 1)
        np.testing.assert_array_equal(rio.open(p).read_rows(r0, r1 - r0), a[r0:r1], err_msg=what)
        if dt in PIL_MODES:
            np.testing.assert_array_equal(_pil_read(p), a, err_msg=what)
        if comp == "deflate":
            continue
        out, status, _ = _decode_like_the_device(p, rows=(r0, r1))
        assert status == 0, what
        np.testing.assert_array_equal(out, a[r0:r1], err_msg=what)
        _encode_like_the_device(q, a, compress=comp, predictor=pred, **kw)
        np.testing.assert_array_equal(rio.open(q).read(1), a, err_msg=what)
        if dt in PIL_MODES:
            np.testing.assert_array_equal(_pil_read(q), a, err_msg=what)
        out, status, _ = _decode_like_the_device(q)
        assert status == 0, what
        np.testing.assert_array_equal(out, a, err_msg=what)


def test_launch_planning_is_exact():
    """the pure planning helpers behind the device paths: which chunks hold a row band, how many chunks go into a launch"""
    assert rio._band_chunks(0, 640, 128, 3) == (0, 15)
    assert rio._band_chunks(64, 320, 128, 3) == (0, 9)      # seams inside tiles: the tiles on both sides are included
    assert rio._band_chunks(320, 640, 128, 3) == (6, 15)
    assert rio._band_chunks(130, 131, 128, 3) == (3, 6)
    assert rio._band_chunks(5, 6, 7, 1) == (0, 1)
    for n, across, raw, block in [(1024, 32, 262144, 256 << 20), (24649, 157, 262144, 256 << 20), (97969, 313, 65536, 256 << 20),
                                  (4, 2, 262144, 200_000), (63, 1, 99456, 1 << 20), (1, 1, 10, 1), (10**6, 1000, 1 << 20, 1 << 30)]:
        g = rio._chunks_per_group(n, across, raw, block)
        assert 1 <= g <= n and (g % across == 0 or g == n), (n, across, g)
        assert g * raw <= (4 << 30) + across * raw                      # bounded staging
        if n >= 2 * rio._WARPS_IN_FLIGHT:
            assert g >= rio._WARPS_IN_FLIGHT                            # a launch fills the device ...
            assert -(-n // g) >= 2                                      # ... and there are launches to overlap with the copies
    ok_off, ok_cnt = np.array([8, 100, 0], np.uint64), np.array([92, 50, 0], np.uint64)
    rio._check_chunk_table("f", ok_off, ok_cnt, 150)  # exactly to the end of the file; an absent chunk is fine
    for off, cnt in (([8, 100], [92, 51]), ([8, 2**63], [92, 2**63]), ([151], [1]), ([0], [2**64 - 1])):
        with pytest.raises(rio.RasterError, match="outside the file"):
            rio._check_chunk_table("f", np.array(off, np.uint64), np.array(cnt, np.uint64), 150)
    assert rio._block_rows(1000, 128, 777, 4, 1 << 20) == 256 and rio._block_rows(1, 128, 330, 4, 100_000) == 1
    assert rio._block_rows(40000, 5, 40000, 4, 256 << 20) % 5 == 0


def test_device_codec_selection_asks_the_library(tmp_path):
    """pipeline_files(decode="auto", encode="auto") takes the device codec exactly when libdtb200 says it can"""
    a = _rand((300, 300), "float32", seed=3)
    cases = [(dict(compress="lzw", predictor=3, tiled=True, blockxsize=128, blockysize=128), True, True),
             (dict(compress="none", blockysize=8), True, True),
             (dict(compress="deflate", tiled=True, blockxsize=128, blockysize=128), True, False),  # decodes, is not written
             (dict(compress="lzw", blockysize=300), True, True),
             (dict(compress="lzw", tiled=True, blockxsize=1024, blockysize=512), False, True)]  # 2 MiB chunks: decode needs <= 1 MiB
    for kw, dec, enc in cases:
        p = tmp_path / "s.tif"
        with rio.open(p, "w", width=300, height=300, dtype="float32", **kw) as w:
            assert rio.device_encode_supported(w) == enc, kw
            w.write(a)
        with rio.open(p) as r:
            assert rio.device_decode_supported(r) == dec, kw
    from PIL import Image

    Image.fromarray(a).save(str(tmp_path / "pb.tif"), compression="packbits")
    assert rio.device_decode_supported(rio.open(tmp_path / "pb.tif"))
    # decode="auto" keeps Deflate and PackBits on the host codec until their kernels have run on a device
    assert rio._AUTO_DEVICE_COMPRESSIONS == ("none", "lzw")
    with pytest.raises(rio.RasterError, match="decode must be"):
        rio.read_to_device(tmp_path / "pb.tif", decode="gpu")


def test_damaged_headers_come_back_as_errors(tmp_path):
    """a file may claim anything: absurd chunk sizes and truncated data are reported, no exception crosses the C ABI"""
    def tiff(entries, data=b"\x80\x00\x40\x40"):
        ifd = struct.pack("<H", len(entries))
        for tag, typ, cnt, val in entries:
            ifd += struct.pack("<HHI", tag, typ, cnt) + (struct.pack("<HH", val, 0) if typ == 3 else struct.pack("<I", val))
        return b"II" + struct.pack("<HI", 42, 8 + len(data)) + data + ifd + struct.pack("<I", 0)

    p = tmp_path / "bad.tif"
    p.write_bytes(tiff([(256, 4, 1, 70000), (257, 4, 1, 70000), (258, 3, 1, 32), (259, 3, 1, 5), (277, 3, 1, 1), (322, 4, 1, 1 << 30),
                        (323, 4, 1, 1 << 30), (324, 4, 1, 8), (325, 4, 1, 4), (339, 3, 1, 3)]))
    with pytest.raises(rio.RasterError, match="2 GiB"):
        rio.open(p)
    p.write_bytes(tiff([(256, 4, 1, 8000), (257, 4, 1, 8000), (258, 3, 1, 32), (259, 3, 1, 5), (277, 3, 1, 1), (273, 4, 1, 8),
                        (278, 4, 1, 8000), (279, 4, 1, 4), (339, 3, 1, 3)]))
    with rio.open(p) as r:  # one 256 MB strip, four bytes of data
        with pytest.raises(rio.RasterError, match="decodes short"):
            r.read_rows(0, 2, threads=2)
    p.write_bytes(tiff([(256, 4, 1, 64), (257, 4, 1, 64), (258, 3, 1, 8), (259, 3, 1, 5), (277, 3, 1, 1), (273, 4, 1, 4000),
                        (278, 4, 1, 64), (279, 4, 1, 100)]))
    with rio.open(p) as r:
        with pytest.raises(rio.RasterError, match="outside the file"):
            r.read(1)


@pytest.mark.gpu
def test_file_to_device_and_back(tmp_path):
    import torch

    a = _rand((1000, 777), "float32", seed=6)
    p = tmp_path / "in.tif"
    with rio.open(p, "w", width=777, height=1000, dtype="float32", compress="lzw", tiled=True, blockxsize=128, blockysize=128, nodata=-100) as dst:
        dst.write(a)
    t = rio.read_to_device(p, block_bytes=1 << 20)  # 1 MiB blocks: 3 x 256 rows + a ragged one, both staging buffers reused
    torch.cuda.synchronize()
    assert t.is_cuda and t.dtype == torch.float32
    np.testing.assert_array_equal(t.cpu().numpy(), a)
    t2 = rio.read_to_device(p)  # single block
    np.testing.assert_array_equal(t2.cpu().numpy(), a)
    q = tmp_path / "out.tif"
    n = rio.write_from_device(q, t * 2, block_bytes=1 << 20, compress="deflate", predictor=3, tiled=True, blockxsize=128, blockysize=128,
                              **{k: v for k, v in rio.open(p).meta.items() if k in ("crs", "transform", "nodata")})
    assert 0 < n <= os.path.getsize(q)
    assert rio.open(q).transform == rio.open(p).transform and rio.open(q).nodata == -100
    np.testing.assert_array_equal(rio.open(q).read(1), a * 2)
    s = tmp_path / "strips.tif"
    rio.write_from_device(s, (t > 0).to(torch.uint8), block_bytes=100_000)
    np.testing.assert_array_equal(_pil_read(s), (a > 0).astype(np.uint8))


@pytest.mark.gpu
def test_pipeline_from_file_to_files(tmp_path):
    """GeoTIFF DEM in, one GeoTIFF per descriptor out == the array pipeline on the same DEM"""
    import oracle
    from descriptools_b200 import pipeline

    dem = oracle.conditioned_dem(300, 420, seed=11)
    hole = np.zeros(dem.shape, bool)
    hole[40:70, 100:160] = True
    stored = np.where(hole, np.float32(-3.4028230607370965e38), dem)  # the file carries GDAL's nodata, not -100
    crs = rio.GeoKeys((1, 1, 0, 1, 3072, 0, 1, 32722))
    p = tmp_path / "dem.tif"
    with rio.open(p, "w", width=420, height=300, dtype="float32", compress="lzw", tiled=True, blockxsize=128, blockysize=128,
                  nodata=-3.4028230607370965e38, crs=crs, transform=rio.Affine(12.5, 0, 1000.0, 0, -12.5, 9000.0)) as dst:
        dst.write(stored)
    want = pipeline.pipeline(np.where(hole, np.float32(-100), dem), 12.5, 300)
    for where in ("host", "device", "auto"):
        paths = pipeline.pipeline_files(p, tmp_path / ("out_" + where), river_threshold=300, block_bytes=200_000, decode=where, encode=where)
        assert sorted(paths) == sorted(pipeline.STAGE_OUTPUTS)
        for name, path in paths.items():
            with rio.open(path) as src:
                assert src.crs == crs and src.res == (12.5, 12.5) and src.nodata == (0 if name == "d8" else -100)
                assert src.compression == "lzw" and src.block_shapes == [(256, 256)]
                np.testing.assert_array_equal(src.read(1), want[name], err_msg=f"{name} ({where})")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,layout,compress,predictor", [("float32", "tiles", "lzw", 1), ("float32", "tiles", "lzw", 3), ("int16", "strips", "lzw", 2),
                                                             ("uint8", "tiles", "lzw", 1), ("int32", "tiles", "none", 1), ("float64", "strips", "none", 1),
                                                             ("int64", "tiles", "lzw", 2),
                                                             # Deflate (zlib streams written by this library's host codec = zlib itself)
                                                             ("float32", "tiles", "deflate", 1), ("float32", "tiles", "deflate", 3),
                                                             ("int16", "strips", "deflate", 2), ("uint8", "tiles", "deflate", 1),
                                                             ("float64", "strips", "deflate", 3), ("int32", "tiles", "deflate", 2)])
def test_tiles_decoded_on_the_device(tmp_path, dtype, layout, compress, predictor):
    import torch

    a = _rand((1000, 777), dtype, seed=12)
    p = tmp_path / "in.tif"
    kw = dict(tiled=True, blockxsize=128, blockysize=128) if layout == "tiles" else dict(blockysize=16)
    with rio.open(p, "w", width=777, height=1000, dtype=dtype, compress=compress, predictor=predictor, **kw) as dst:
        dst.write(a)
    from descriptools_b200 import _lib

    before = _lib.launch_count()
    t = rio.read_to_device(p, decode="device", group_chunks=14 if layout == "tiles" else 9)  # many spans: both staging buffers are reused
    torch.cuda.synchronize()
    assert _lib.launch_count() > before
    np.testing.assert_array_equal(t.cpu().numpy(), a)
    t = rio.read_to_device(p, decode="device")  # one span
    np.testing.assert_array_equal(t.cpu().numpy(), a)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["uint8", "uint16", "int32", "float32"])
def test_packbits_and_noise_decoded_on_the_device(tmp_path, dtype):
    """the device PackBits kernel on strips as libtiff (Pillow) writes them -- literal runs and long repeats -- and the
    device Deflate kernel on incompressible data (stored / near-stored blocks, literal-only streams) and on long matches"""
    import torch
    from PIL import Image

    p = str(tmp_path / "pb.tif")
    for a in (_rand((301, 333), dtype, seed=5), np.repeat(_rand((301, 9), dtype, seed=6, smooth=False), 37, axis=1)):
        Image.fromarray(a).save(p, compression="packbits")
        assert rio.open(p).compression == "packbits"
        t = rio.read_to_device(p, decode="device")
        torch.cuda.synchronize()
        np.testing.assert_array_equal(t.cpu().numpy(), a)
        t = rio.read_to_device(p, decode="device", rows=(100, 211))
        np.testing.assert_array_equal(t.cpu().numpy(), a[100:211])
    q = tmp_path / "z.tif"
    for smooth, block in ((False, 256), (True, 256), (True, 64)):
        a = _rand((700, 900), dtype, seed=41, smooth=smooth)
        if smooth:
            a[100:300] = a[100]  # long matches across rows
        with rio.open(q, "w", width=900, height=700, dtype=dtype, compress="deflate", tiled=True, blockxsize=block, blockysize=block) as dst:
            dst.write(a)
        t = rio.read_to_device(q, decode="device", group_chunks=5)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(t.cpu().numpy(), a)
    # a long literal-only LZW stream (noise): the lock-step decoder's table fills and resets many times
    a = _rand((1024, 1024), "uint8", seed=9, smooth=False)
    with rio.open(q, "w", width=1024, height=1024, dtype="uint8", compress="lzw", tiled=True, blockxsize=512, blockysize=512) as dst:
        dst.write(a)
    np.testing.assert_array_equal(rio.read_to_device(q, decode="device").cpu().numpy(), a)


@pytest.mark.gpu
def test_device_decoder_reports_damage_and_refuses_what_it_cannot_do(tmp_path):
    a = _rand((300, 300), "uint8", seed=13, smooth=False)
    p = tmp_path / "d.tif"
    with rio.open(p, "w", width=2048, height=600, dtype="uint8", compress="lzw", tiled=True, blockxsize=2048, blockysize=1024) as dst:
        dst.write(np.zeros((600, 2048), np.uint8))  # 2 MiB tiles: more than the device decoder's string table addresses
    with pytest.raises(rio.RasterError, match="1 MiB"):
        rio.read_to_device(p, decode="device")
    q = tmp_path / "l.tif"
    with rio.open(q, "w", width=300, height=300, dtype="uint8", compress="lzw", tiled=True, blockxsize=64, blockysize=64) as dst:
        dst.write(a)
    raw = bytearray(q.read_bytes())
    with rio.open(q) as r:
        _, _, off, cnt = rio.chunk_table(r)
    raw[int(off[3]) + 2:int(off[3]) + int(cnt[3])] = b"\xff" * (int(cnt[3]) - 2)  # codes far beyond the table
    q.write_bytes(bytes(raw))
    with pytest.raises(rio.RasterError, match="chunk 3"):
        rio.read_to_device(q, decode="device")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,layout,compress,predictor", [("float32", "tiles", "lzw", 3), ("float32", "tiles", "lzw", 1), ("int32", "tiles", "lzw", 2),
                                                             ("uint8", "strips", "lzw", 1), ("int16", "tiles", "none", 1), ("float64", "strips", "lzw", 3)])
def test_tiles_encoded_on_the_device(tmp_path, dtype, layout, compress, predictor):
    import torch

    from descriptools_b200 import _lib

    a = _rand((1000, 777), dtype, seed=14)
    t = torch.from_numpy(a).cuda()
    p = tmp_path / "out.tif"
    kw = dict(tiled=True, blockxsize=128, blockysize=128) if layout == "tiles" else dict(blockysize=16)
    before = _lib.launch_count()
    n = rio.write_from_device(p, t, encode="device", group_chunks=14 if layout == "tiles" else 9, compress=compress, predictor=predictor, nodata=-100,
                              transform=rio.Affine(2.0, 0, 10.0, 0, -2.0, 99.0), **kw)   # several groups: both slot buffers are reused
    assert _lib.launch_count() >= before + 2 and 0 < n <= os.path.getsize(p)
    with rio.open(p) as src:
        assert src.compression == compress and src.res == (2.0, 2.0) and src.nodata == -100
        np.testing.assert_array_equal(src.read(1), a)
    if dtype in PIL_MODES:
        np.testing.assert_array_equal(_pil_read(p), a)
    np.testing.assert_array_equal(rio.read_to_device(p, decode="device").cpu().numpy(), a)
    rio.write_from_device(p, t, encode="device", compress=compress, predictor=predictor, **kw)  # one group
    np.testing.assert_array_equal(rio.open(p).read(1), a)
    with pytest.raises(rio.RasterError, match="encode='host'"):
        rio.write_from_device(p, t, encode="device", compress="deflate")
    assert not os.path.exists(p)


@pytest.mark.gpu
def test_device_encoded_groups_are_written_in_pieces(tmp_path, monkeypatch):
    """a small block_bytes cuts every group into pieces of whole chunks (both pinned buffers reused): the file is byte
    for byte the one a single append per group gives"""
    import torch

    a = _rand((1000, 777), "float32", seed=15)
    t = torch.from_numpy(a).cuda()
    kw = dict(encode="device", compress="lzw", predictor=3, tiled=True, blockxsize=128, blockysize=128)
    one, many = tmp_path / "one.tif", tmp_path / "many.tif"
    rio.write_from_device(one, t, **kw)  # one group, one piece
    writes, real = [], rio.DatasetWriter.write_encoded

    def counted(self, first_chunk, *args, **kwargs):
        writes.append(first_chunk)
        return real(self, first_chunk, *args, **kwargs)

    monkeypatch.setattr(rio.DatasetWriter, "write_encoded", counted)
    rio.write_from_device(many, t, block_bytes=100_000, **kw)  # two groups of 28 chunks, pieces of about 100 kB
    assert len(writes) > 4 and writes == sorted(writes)
    assert one.read_bytes() == many.read_bytes()
    np.testing.assert_array_equal(rio.open(many).read(1), a)


@pytest.mark.gpu
@pytest.mark.parametrize("encode", ["host", "device"])
def test_failed_write_from_device_closes_once_and_leaves_no_file(tmp_path, monkeypatch, encode):
    import torch

    calls = _count_closes(monkeypatch)
    real_close = rio.DatasetWriter.close

    def close_then_fail(self):
        real_close(self)
        raise rio.RasterError("injected close failure")

    monkeypatch.setattr(rio.DatasetWriter, "close", close_then_fail)
    t = torch.from_numpy(_rand((300, 200), "float32", seed=2)).cuda()
    p = tmp_path / "f.tif"
    with pytest.raises(rio.RasterError, match="injected"):
        rio.write_from_device(p, t, encode=encode, compress="lzw", tiled=True, blockxsize=64, blockysize=64)
    assert list(calls.values()) == [1]
    assert not os.path.exists(p)


@pytest.mark.gpu
@pytest.mark.parametrize("decode", ["host", "device"])
def test_row_bands_from_a_file(tmp_path, decode):
    """read_to_device(rows=...) and BandRunner.load_file: every band decodes its own rows; the band run on the file
    equals the single-raster run on the array, bit for bit"""
    import oracle
    import torch

    from descriptools_b200 import bands, pipeline

    dem = oracle.conditioned_dem(640, 330, seed=17)
    hole = np.zeros(dem.shape, bool)
    hole[100:140, 40:90] = True  # stored with the file's own nodata value, normalised to -100 by load_file
    p = tmp_path / "dem.tif"
    with rio.open(p, "w", width=330, height=640, dtype="float32", compress="lzw", predictor=3, tiled=True, blockxsize=128, blockysize=128,
                  nodata=-9999.0) as dst:
        dst.write(np.where(hole, np.float32(-9999.0), dem))
    for band in ((0, 640), (64, 320), (320, 640), (130, 131)):  # seams inside tiles
        t = rio.read_to_device(p, rows=band, decode=decode, group_chunks=3 if decode == "device" else None, block_bytes=100_000)
        np.testing.assert_array_equal(t.cpu().numpy(), np.where(hole, np.float32(-9999.0), dem)[band[0]:band[1]], err_msg=str(band))
    clean = np.where(hole, np.float32(-100), dem)
    ref = pipeline.run_device(torch.from_numpy(clean).cuda(), 12.5, 300)
    runner = bands.BandRunner(640, 330, 12.5, 300, 0.4, 0.1, nbands=2)
    runner.load_file(p, decode=decode)
    runner.step()
    torch.cuda.synchronize()
    outs = runner.outputs()
    for name in ("slope", "d8", "acc", "idx", "fdist", "hand", "gfi"):
        got = torch.cat([o[name] for o in outs], 0).cpu().numpy()
        np.testing.assert_array_equal(got, ref[name].cpu().numpy(), err_msg=name)


@pytest.mark.gpu
def test_unconditioned_dem_file_is_conditioned_on_the_device(tmp_path):
    """SURVEY 8 f4: flowhand.fill_depressions == the oracle's priority flood; pipeline_files(condition=True) on a raw DEM
    file == the array pipeline on the conditioned DEM"""
    import oracle
    import descriptools_b200.flowhand as flowhand
    from descriptools_b200 import pipeline

    raw = oracle.synth_dem(300, 420, 0, 77)
    raw[120:150, 200:260] = -100
    want = oracle.priority_flood_eps(raw)
    assert (want != raw).sum() > 50  # there were pits
    np.testing.assert_array_equal(flowhand.fill_depressions(raw), want)
    np.testing.assert_array_equal(flowhand.fill_depressions(want), want)  # a fixed point
    p = tmp_path / "raw.tif"
    with rio.open(p, "w", width=420, height=300, dtype="float32", compress="lzw", predictor=3, tiled=True, blockxsize=128, blockysize=128,
                  nodata=-100) as dst:
        dst.write(raw)
    paths = pipeline.pipeline_files(p, tmp_path / "out", river_threshold=300, px=12.5, condition=True)
    ref = pipeline.pipeline(want, 12.5, 300)
    for name, path in paths.items():
        np.testing.assert_array_equal(rio.open(path).read(1), ref[name], err_msg=name)
