"""Row bands written straight into GeoTIFFs (bands.write_raster, BandRunner.write_files): every band encodes its own chunks
and writes them into one shared file, byte for byte the file one writer produces from the whole raster.

CPU: the encoder's lane code over a row window (dtb_selftest_tiff_encode_host), the host library's part writers and
chunk placement (dtbio_open_part / dtbio_write_encoded_at / dtbio_place_chunks), and the whole protocol over gloo and
LocalExchange with the lane code as the encoder.  GPU: the device encoder over a window, k logical bands from a raw DEM
file to seven files compared with pipeline_files, downslope, and two processes over NCCL where two GPUs are visible."""
import ctypes
import filecmp
import functools
import os
import socket
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import descriptools_b200.raster as rio

PX = 12.5
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rand(shape, dtype, seed):
    rng = np.random.default_rng(seed)
    dt = np.dtype(dtype)
    r = np.arange(shape[0])[:, None]
    c = np.arange(shape[1])[None, :]
    smooth = 40 * np.sin(r / 17.0) + 30 * np.cos(c / 11.0) + rng.integers(0, 4, shape)
    if dt.kind == "f":
        return (smooth + rng.random(shape)).astype(dt)
    if dt.kind == "u":
        return (smooth + 80).astype(dt)
    return smooth.astype(dt)


# ---- the encoders: lane code on the CPU ------------------------------------------------------------------------
def _selftest_encode(lay, a: np.ndarray, c0: int, c1: int):
    """chunks [c0, c1) of `a` (rows [lay.row_lo, lay.row_hi) of the raster, or all of it) -> (enc slots, sizes)"""
    from descriptools_b200 import _lib

    bound = _lib.lib.dtb_tiff_encode_bound(ctypes.byref(lay))
    assert bound > 0
    enc = np.zeros(max(1, c1 - c0) * bound, np.uint8)
    sizes = np.zeros(max(1, c1 - c0), np.int64)
    a = np.ascontiguousarray(a)
    rc = _lib.lib.dtb_selftest_tiff_encode_host(ctypes.byref(lay), a.ctypes.data, c0, c1 - c0, enc.ctypes.data, sizes.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"dtb_selftest_tiff_encode_host: {rc}")
    return enc, sizes[:c1 - c0], bound


def _pack(enc, sizes, bound):
    aligned = (sizes + 1) & ~1
    offs = np.cumsum(aligned) - aligned
    blob = np.zeros(int(aligned.sum()), np.uint8)
    for i, n in enumerate(sizes):
        blob[offs[i]:offs[i] + n] = enc[i * bound:i * bound + n]
    return blob, offs


def lane_encoder(lay, raster, c0, c1):
    """write_raster's encoder interface over the kernel's lane code: CPU tensors in, packed streams out"""
    enc, sizes, bound = _selftest_encode(lay, raster.numpy(), c0, c1)
    return _pack(enc, sizes, bound)[0], sizes


def _single_writer_file(path, a, meta):
    """what write_from_device(encode="device") writes: the streams of every chunk appended in chunk order"""
    w = rio.open(path, "w", width=a.shape[1], height=a.shape[0], dtype=a.dtype.name, **meta)
    lay, _, n = w.chunk_layout()
    enc, sizes, bound = _selftest_encode(lay, a, 0, n)
    blob, offs = _pack(enc, sizes, bound)
    w.write_encoded(0, blob, offs, sizes)
    w.close()
    return sizes


def _window(lay, lo, hi):
    from descriptools_b200 import _lib

    w = _lib.TiffLayout.from_buffer_copy(lay)
    w.row_lo, w.row_hi = lo, hi
    return w


# ---- CPU: the lane code over a row window ----------------------------------------------------------------------
@pytest.mark.parametrize("dtype,compress,predictor", [("uint8", "none", 1), ("int16", "lzw", 2), ("float32", "lzw", 3),
                                                      ("float64", "lzw", 1), ("int32", "lzw", 2)])
@pytest.mark.parametrize("layout", ["tiles", "strips"])
def test_lane_code_over_a_window_gives_the_whole_raster_streams(tmp_path, dtype, compress, predictor, layout):
    a = _rand((300, 203), dtype, seed=3)
    kw = dict(tiled=True, blockxsize=48, blockysize=64) if layout == "tiles" else dict(blockysize=40)
    w = rio.open(tmp_path / "x.tif", "w", width=203, height=300, dtype=dtype, compress=compress, predictor=predictor, **kw)
    lay, across, n = w.chunk_layout()
    w.abort()
    ch = lay.chunk_rows
    enc, sizes, bound = _selftest_encode(lay, a, 0, n)
    last = -(-300 // ch) - 1
    # windows on chunk boundaries, one that ends at the raster end (a partial last chunk-row), one wider than its chunks
    for lo, hi, k0, k1 in ((0, ch, 0, 1), (ch, 3 * ch, 1, 3), (last * ch, 300, last, last + 1), (ch, 300, 1, last + 1),
                           (ch - 5, 3 * ch + 7, 1, 3), (0, 300, 0, last + 1)):
        e, s, _ = _selftest_encode(_window(lay, lo, hi), a[lo:hi], k0 * across, k1 * across)
        np.testing.assert_array_equal(s, sizes[k0 * across:k1 * across], err_msg=str((lo, hi)))
        for i in range(len(s)):
            c = k0 * across + i
            assert bytes(e[i * bound:i * bound + s[i]]) == bytes(enc[c * bound:c * bound + sizes[c]]), (lo, hi, c)


def test_encoder_refuses_chunks_outside_the_window_without_a_device():
    from descriptools_b200 import _lib

    L = _lib.lib
    lay = _lib.TiffLayout(rows=300, cols=200, bps=4, predictor=3, compression=5, tiled=1, chunk_rows=64, chunk_cols=64, big_endian=0)
    across = 4
    ws = L.dtb_tiff_encode_workspace_bytes(ctypes.byref(lay), 8)
    assert L.dtb_tiff_encode_bound(ctypes.byref(_window(lay, 64, 128))) == L.dtb_tiff_encode_bound(ctypes.byref(lay))
    assert L.dtb_tiff_encode_workspace_bytes(ctypes.byref(_window(lay, 64, 128)), 8) == ws

    def call(lo, hi, c0, n):
        return L.dtb_tiff_encode_chunks(ctypes.byref(_window(lay, lo, hi)), 1, c0, n, 1, 1, 1, ws, None)

    def host(lo, hi, c0, n):
        return L.dtb_selftest_tiff_encode_host(ctypes.byref(_window(lay, lo, hi)), 1, c0, n, 1, 1)

    for f in (call, host):
        assert f(64, 128, 0, across) == -1           # chunk-row 0 starts above the window
        assert f(64, 128, across, 2 * across) == -1  # chunk-row 2 ends below it
        assert f(64, 127, across, across) == -1      # chunk-row 1 is cut
        assert f(256, 299, 4 * across, across) == -1  # the last chunk-row must reach the raster's last row
        assert f(-1, 64, 0, across) == -1 and f(64, 64, across, across) == -1 and f(0, 301, 0, across) == -1  # bad windows
        assert f(128, 64, 0, 0) == -1
        assert f(64, 128, across, across + 1) == -1 and f(0, 300, 5 * across - 1, 2) == -1
    assert host(0, 0, 0, 5 * across + 1) == -1  # whole raster: the range must lie in it


# ---- CPU: the host library's writers ------------------------------------------------------------------------------
_META = dict(compress="lzw", predictor=3, tiled=True, blockxsize=64, blockysize=64, nodata=-100,
             transform=rio.Affine(12.5, 0, 1000.0, 0, -12.5, 5000.0))


def _encoded(a, meta, path):
    """(chunks, encode slots of every chunk, sizes, slot bytes, file offsets of the single-writer layout)"""
    w = rio.open(path, "w", width=a.shape[1], height=a.shape[0], dtype=a.dtype.name, **meta)
    lay, _, n = w.chunk_layout()
    w.abort()
    enc, sizes, bound = _selftest_encode(lay, a, 0, n)
    aligned = (sizes + 1) & ~1
    return n, enc, sizes, bound, 16 + np.cumsum(aligned) - aligned


def _write_range(w, enc, sizes, bound, offs, c0, c1):
    blob, rel = _pack(enc[c0 * bound:c1 * bound], sizes[c0:c1], bound)
    w.write_encoded(c0, blob, rel, sizes[c0:c1], at=int(offs[c0]))


def _part_process(path, a_path, meta, c0, c1):
    a = np.load(a_path)
    n, enc, sizes, bound, offs = _encoded(a, meta, path + ".scratch")
    with rio.DatasetWriter(path, width=a.shape[1], height=a.shape[0], dtype=a.dtype.name, part=True, **meta) as p:
        _write_range(p, enc, sizes, bound, offs, c0, c1)


@pytest.mark.parametrize("processes", [1, 2])
def test_main_and_part_writers_give_the_single_writer_file(tmp_path, processes):
    from PIL import Image

    a = _rand((300, 203), "float32", seed=8)
    ref, got = str(tmp_path / "ref.tif"), str(tmp_path / "got.tif")
    _single_writer_file(ref, a, _META)
    n, enc, sizes, bound, offs = _encoded(a, _META, str(tmp_path / "s.tif"))
    main = rio.open(got, "w", width=203, height=300, dtype="float32", **_META)
    split = 2 * 4  # chunk-rows 0-1 by the main writer, 2-4 by the part writer
    _write_range(main, enc, sizes, bound, offs, 0, split)
    if processes == 1:
        with rio.DatasetWriter(got, width=203, height=300, dtype="float32", part=True, **_META) as p:
            _write_range(p, enc, sizes, bound, offs, split, n)
    else:
        np.save(tmp_path / "a.npy", a)
        code = (f"import sys; sys.path[:0] = [{REPO!r}, {os.path.join(REPO, 'tests')!r}]; import test_band_files as t; "
                f"t._part_process({got!r}, {str(tmp_path / 'a.npy')!r}, t._META, {split}, {n})")
        subprocess.run([sys.executable, "-c", code], check=True, cwd=REPO)
    assert os.path.getsize(got) > 16
    main.place_chunks(split, offs[split:], sizes[split:])
    main.close()
    assert filecmp.cmp(ref, got, shallow=False)
    with rio.open(got) as src:
        np.testing.assert_array_equal(src.read(1), a)
        assert src.nodata == -100 and src.res == (12.5, 12.5)
    Image.MAX_IMAGE_PIXELS = None
    np.testing.assert_array_equal(np.asarray(Image.open(got)), a)


def test_placement_is_checked_and_a_missing_chunk_removes_the_file(tmp_path):
    a = _rand((300, 203), "float32", seed=9)
    p = str(tmp_path / "p.tif")
    n, enc, sizes, bound, offs = _encoded(a, _META, str(tmp_path / "s.tif"))
    w = rio.open(p, "w", width=203, height=300, dtype="float32", **_META)
    blob, rel = _pack(enc[:4 * bound], sizes[:4], bound)
    with pytest.raises(rio.RasterError, match="even"):
        w.write_encoded(0, blob, rel, sizes[:4], at=17)
    with pytest.raises(rio.RasterError, match="header"):
        w.write_encoded(0, blob, rel, sizes[:4], at=8)
    with pytest.raises(rio.RasterError, match="overlap"):
        w.write_encoded(0, blob, np.zeros(4, np.int64), np.full(4, 2, np.int64), at=16)  # four chunks on one spot
    w.write_encoded(0, blob, rel, sizes[:4], at=16)
    with pytest.raises(rio.RasterError, match="twice"):
        w.place_chunks(3, [int(offs[10])], [int(sizes[3])])
    with pytest.raises(rio.RasterError, match="overlap"):
        w.place_chunks(4, [int(offs[3])], [int(sizes[4])])              # on top of chunk 3
    with pytest.raises(rio.RasterError, match="overlap"):
        w.place_chunks(4, [int(offs[4]), int(offs[4]) + 2], [int(sizes[4]), int(sizes[5])])  # on top of each other
    with pytest.raises(rio.RasterError, match="even"):
        w.place_chunks(4, [int(offs[4]) + 1], [int(sizes[4])])
    with pytest.raises(rio.RasterError, match="outside the raster"):
        w.place_chunks(n - 1, offs[-2:], sizes[-2:])
    w.place_chunks(4, offs[4:n - 1], sizes[4:n - 1])                      # every chunk but the last
    with pytest.raises(rio.RasterError, match="never written"):
        w.close()
    assert not os.path.exists(p)
    # a file takes its chunks either appended or at given offsets
    w = rio.open(p, "w", width=203, height=300, dtype="float32", **_META)
    w.write_encoded(0, blob, rel, sizes[:4])
    with pytest.raises(rio.RasterError, match="appended"):
        w.place_chunks(4, offs[4:5], sizes[4:5])
    w.abort()
    assert not os.path.exists(p)
    # a part writer takes chunks at offsets only, and leaves the file alone when it closes
    open(p, "wb").close()
    with rio.DatasetWriter(p, width=203, height=300, dtype="float32", part=True, **_META) as part:
        with pytest.raises(rio.RasterError, match="given offsets"):
            part.write_rows(0, a[:64])
    assert os.path.exists(p) and os.path.getsize(p) == 0
    with pytest.raises(rio.RasterError, match="predictor 3"):
        rio.DatasetWriter(p, width=203, height=300, dtype="int32", part=True, **_META)  # the checks of create
    with pytest.raises(rio.RasterError, match="cannot open"):
        rio.DatasetWriter(str(tmp_path / "absent.tif"), width=203, height=300, dtype="float32", part=True, **_META)


def test_a_classic_file_refuses_offsets_past_4gb(tmp_path):
    p = str(tmp_path / "c.tif")
    geo = dict(width=64, height=128, dtype="uint8", compress="none", tiled=True, blockxsize=64, blockysize=64)  # two chunks
    w = rio.open(p, "w", **geo)
    assert not w.bigtiff
    blob = np.zeros(4096, np.uint8)
    with pytest.raises(rio.RasterError, match="4 GB"):
        w.write_encoded(0, blob, [0], [4096], at=0xFFFFF000)
    with pytest.raises(rio.RasterError, match="4 GB"):
        w.place_chunks(0, [0xFFFFF000], [4096])
    w.abort()
    assert not os.path.exists(p)
    b = rio.open(p, "w", bigtiff=True, **geo)
    b.place_chunks(0, [0xFFFFF000], [4096])  # a BigTIFF takes it (only the table is written to: no 4 GB file)
    b.abort()  # chunk 1 is missing: no IFD is written
    assert not os.path.exists(p)


# ---- CPU: the protocol with the lane code ----------------------------------------------------------------------------
CASES = {
    # seams inside 256-row tiles; with 4 bands band 2 lies inside chunk-row 1; a partial last chunk-row
    "tiles": ((600, 203), "float32", dict(compress="lzw", predictor=3, tiled=True, blockxsize=96, blockysize=256, nodata=-100)),
    # seams on chunk-row boundaries: no hand-off
    "tiles64": ((448, 150), "int32", dict(compress="lzw", predictor=2, tiled=True, blockxsize=64, blockysize=64, nodata=-100)),
    # strips of 48 rows: every seam inside one; a stored file
    "strips": ((500, 131), "uint8", dict(compress="none", blockysize=48, nodata=0)),
}


@functools.lru_cache(maxsize=None)
def _case(name, tmp):
    shape, dtype, meta = CASES[name]
    a = _rand(shape, dtype, seed=len(name))
    ref = os.path.join(tmp, f"ref_{name}.tif")
    _single_writer_file(ref, a, meta)
    return a, ref


def _stand_ins(a, edges, indices):
    from descriptools_b200 import bands

    rows, cols = a.shape
    bs = [SimpleNamespace(index=i, grows=rows, cols=cols, dev=torch.device("cpu")) for i in indices]
    return bs, [torch.from_numpy(a[edges[i]:edges[i + 1]].copy()) for i in indices]


def _failing_encoder(bad_index):
    def enc(lay, raster, c0, c1):
        if lay.row_lo <= bad_index < lay.row_hi:
            raise RuntimeError("injected encoder failure")
        return lane_encoder(lay, raster, c0, c1)

    return enc


@pytest.mark.parametrize("k", [1, 2, 3, 4])
@pytest.mark.parametrize("name", sorted(CASES))
def test_write_raster_local_bands_give_the_single_writer_file(tmp_path_factory, tmp_path, name, k):
    from descriptools_b200 import bands

    a, ref = _case(name, str(tmp_path_factory.getbasetemp()))
    rows = a.shape[0]
    edges = bands.band_edges(rows, k)
    bs, ts = _stand_ins(a, edges, range(k))
    got = tmp_path / "got.tif"
    total = bands.write_raster(bs, bands.LocalExchange(k), got, ts, CASES[name][2], encoder=lane_encoder, piece_bytes=3000)
    assert filecmp.cmp(ref, got, shallow=False)
    assert total <= os.path.getsize(got)
    np.testing.assert_array_equal(rio.open(got).read(1), a)


def test_write_plan_covers_every_chunk_row_once():
    from descriptools_b200 import bands

    own, sends = bands.write_plan([0, 192, 320, 512, 700], 256, 700)
    assert own == [(0, 0, 0), (1, 1, 1), (2, 2, None), (2, 3, None)]
    assert sends == [(1, 0, 192, 256), (2, 1, 320, 512)]  # band 2 lies inside chunk-row 1: it owns nothing, sends everything
    for rows, k, ch in ((600, 4, 256), (700, 4, 256), (1000, 7, 48), (64 * 9, 9, 512), (130, 2, 16)):
        edges = bands.band_edges(rows, k)
        own, sends = bands.write_plan(edges, ch, rows)
        covered = []
        for k0, k1, s in own:
            covered += list(range(k0, k1)) + ([s] if s is not None else [])
        assert sorted(covered) == list(range(-(-rows // ch)))
        for src, dst, a, e in sends:  # every row of a straddled chunk-row arrives exactly once
            assert edges[src] == a and a < e <= edges[src + 1] and own[dst][2] == a // ch


def _gloo_worker(rank, world, port, tmp, names, bad, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        import torch.distributed as dist

        dist.init_process_group("gloo", rank=rank, world_size=world)
        from descriptools_b200 import bands

        x = bands.DistExchange()
        out = {}
        for name in names:
            shape, dtype, meta = CASES[name]
            a = _rand(shape, dtype, seed=len(name))
            edges = bands.band_edges(shape[0], world)
            bs, ts = _stand_ins(a, edges, [rank])
            path = os.path.join(tmp, f"{name}_{world}.tif")
            enc = lane_encoder if bad is None else _failing_encoder(bad)
            try:
                bands.write_raster(bs, x, path, ts, meta, encoder=enc, piece_bytes=5000)
                out[name] = "ok"
            except rio.RasterError as e:
                out[name] = "raised: " + str(e)
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, "ok", out))
    except Exception:  # pragma: no cover
        import traceback

        q.put((rank, "fail", traceback.format_exc()))


def _run_gloo(world, tmp, names, bad=None):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, world, port, str(tmp), names, bad, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = sorted(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    for rank, status, info in results:
        assert status == "ok", f"rank {rank}: {info}"
    return [info for _, _, info in results]


@pytest.mark.parametrize("world", [2, 3])
def test_write_raster_over_gloo_gives_the_single_writer_file(tmp_path_factory, tmp_path, world):
    names = sorted(CASES)
    infos = _run_gloo(world, tmp_path, names)
    for name in names:
        assert all(info[name] == "ok" for info in infos), (name, infos)
        _, ref = _case(name, str(tmp_path_factory.getbasetemp()))
        assert filecmp.cmp(ref, tmp_path / f"{name}_{world}.tif", shallow=False), name


def test_an_encoder_failure_on_one_rank_raises_everywhere_and_leaves_no_file(tmp_path):
    from descriptools_b200 import bands

    infos = _run_gloo(3, tmp_path, ["tiles"], bad=550)  # 3 bands of 600 rows: 0, 192, 384, 600 -- rank 2 fails
    assert all(info["tiles"].startswith("raised: ") and "encoding failed on 1 rank" in info["tiles"] for info in infos), infos
    assert not os.path.exists(tmp_path / "tiles_3.tif")
    a = _rand((600, 203), "float32", seed=5)
    edges = bands.band_edges(600, 4)
    bs, ts = _stand_ins(a, edges, range(4))
    with pytest.raises(rio.RasterError, match="encoding failed"):
        bands.write_raster(bs, bands.LocalExchange(4), tmp_path / "l.tif", ts, CASES["tiles"][2], encoder=_failing_encoder(10))
    assert not os.path.exists(tmp_path / "l.tif")
    with pytest.raises(rio.RasterError, match="rows per strip"):
        bands.write_raster(bs, bands.LocalExchange(4), tmp_path / "l.tif", ts, dict(compress="lzw"), encoder=lane_encoder)
    with pytest.raises(rio.RasterError, match="contiguous"):
        bands.write_raster(bs, bands.LocalExchange(4), tmp_path / "l.tif", ts[::-1], CASES["tiles"][2], encoder=lane_encoder)
    assert not os.path.exists(tmp_path / "l.tif")


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype,compress,predictor,layout", [("float32", "lzw", 3, "tiles"), ("int32", "lzw", 2, "strips"),
                                                             ("uint8", "none", 1, "tiles")])
def test_device_encoder_over_a_window_gives_the_whole_raster_streams(tmp_path, dtype, compress, predictor, layout):
    from descriptools_b200 import _lib

    a = _rand((700, 530), dtype, seed=4)
    kw = dict(tiled=True, blockxsize=128, blockysize=128) if layout == "tiles" else dict(blockysize=40)
    w = rio.open(tmp_path / "x.tif", "w", width=530, height=700, dtype=dtype, compress=compress, predictor=predictor, **kw)
    lay, across, n = w.chunk_layout()
    w.abort()
    t = torch.from_numpy(a).cuda()
    bound = _lib.lib.dtb_tiff_encode_bound(ctypes.byref(lay))

    def encode(L, src, c0, c1):
        ws_bytes = _lib.lib.dtb_tiff_encode_workspace_bytes(ctypes.byref(L), c1 - c0)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        enc = torch.zeros((c1 - c0) * bound, dtype=torch.uint8, device="cuda")
        sizes = torch.zeros(c1 - c0, dtype=torch.int64, device="cuda")
        _lib.check(_lib.lib.dtb_tiff_encode_chunks(ctypes.byref(L), src.data_ptr(), c0, c1 - c0, enc.data_ptr(), sizes.data_ptr(),
                                                   ws.data_ptr(), ws_bytes, None), "dtb_tiff_encode_chunks")
        torch.cuda.synchronize()
        return enc.cpu().numpy(), sizes.cpu().numpy()

    whole_enc, whole = encode(lay, t, 0, n)
    ch = lay.chunk_rows
    last = -(-700 // ch) - 1
    for lo, hi, k0, k1 in ((ch, 3 * ch, 1, 3), (last * ch, 700, last, last + 1), (ch - 5, 700, 1, last + 1)):
        e, s = encode(_window(lay, lo, hi), t[lo:hi].contiguous(), k0 * across, k1 * across)
        np.testing.assert_array_equal(s, whole[k0 * across:k1 * across])
        for i in range(len(s)):
            c = k0 * across + i
            assert bytes(e[i * bound:i * bound + s[i]]) == bytes(whole_enc[c * bound:c * bound + whole[c]]), (lo, hi, c)
    with pytest.raises(_lib.DtbError):
        encode(_window(lay, ch, 3 * ch), t[ch:3 * ch].contiguous(), 0, across)


def _raw_dem_file(path):
    """a raw DEM (pits to fill) with nodata across the seams of 2 to 4 bands, stored with its own nodata value"""
    import oracle

    raw = oracle.synth_dem(700, 530, 0, 23)
    hole = np.zeros(raw.shape, bool)
    # seams: 2 bands 0, 320, 700; 3 bands 0, 256, 448, 700; 4 bands 0, 192, 320, 512, 700
    hole[170:215, 40:120] = True    # across 192
    hole[250:262, 300:380] = True   # across 256
    hole[319, 200:330] = True       # the row right above 320
    hole[440:460, 480:530] = True   # across 448, at the right edge
    hole[505:520, 100:140] = True   # across 512
    with rio.open(path, "w", width=530, height=700, dtype="float32", compress="lzw", predictor=3, tiled=True, blockxsize=128,
                  blockysize=128, nodata=-9999.0, transform=rio.Affine(PX, 0, 500000.0, 0, -PX, 7000000.0)) as dst:
        dst.write(np.where(hole, np.float32(-9999.0), raw))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 3, 4])
def test_band_files_equal_pipeline_files(tmp_path_factory, tmp_path, k):
    """raw DEM file -> load_file(condition=True) -> step() -> write_files(): the seven files are those pipeline_files
    writes on one GPU, byte for byte, and read back to the runner's outputs"""
    from descriptools_b200 import bands, pipeline

    base = tmp_path_factory.getbasetemp()
    dem = base / "raw_dem.tif"
    ref = base / "ref_out"
    if not ref.exists():
        _raw_dem_file(dem)
        pipeline.pipeline_files(dem, ref, river_threshold=300, px=PX, condition=True)
    runner = bands.BandRunner(700, 530, PX, 300, 0.4, 0.1, nbands=k)
    runner.load_file(dem, condition=True)
    runner.step()
    paths = runner.write_files(tmp_path / "out")
    assert sorted(paths) == sorted(pipeline.STAGE_OUTPUTS)
    outs = runner.outputs()
    for name, p in paths.items():
        assert filecmp.cmp(ref / f"{name}.tif", p, shallow=False), name
        got = rio.read_to_device(p, decode="device")
        np.testing.assert_array_equal(got.cpu().numpy(), torch.cat([o[name] for o in outs], 0).cpu().numpy(), err_msg=name)


@pytest.mark.gpu
def test_downslope_through_write_raster_equals_write_from_device(tmp_path):
    from descriptools_b200 import bands, device

    import oracle

    dem = oracle.conditioned_dem(640, 330, seed=31)
    runner = bands.BandRunner(640, 330, PX, 300, nbands=3)
    runner.load([torch.from_numpy(dem[a:b].copy()) for a, b in zip(runner.edges, runner.edges[1:])])
    runner.step()
    per_band = runner.downslope(5.0)
    meta = dict(compress="lzw", predictor=3, tiled=True, blockxsize=256, blockysize=256, nodata=-100)
    runner.write_raster(tmp_path / "bands.tif", per_band, **meta)
    t = torch.from_numpy(dem).cuda()
    d8 = torch.cat([b.d8 for b in runner.bands], 0)
    single = device.downslope(t, d8, PX, 5.0)
    rio.write_from_device(tmp_path / "one.tif", single, encode="device", **meta)
    assert filecmp.cmp(tmp_path / "one.tif", tmp_path / "bands.tif", shallow=False)


def _nccl_worker(rank, world, port, dem, out_dir, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        import torch.distributed as dist

        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
        from descriptools_b200 import bands

        runner = bands.BandRunner(700, 530, PX, 300, 0.4, 0.1)
        runner.load_file(dem, condition=True)
        runner.step()
        runner.write_files(out_dir)
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, "ok", None))
    except Exception:  # pragma: no cover
        import traceback

        q.put((rank, "fail", traceback.format_exc()))


@pytest.mark.gpu
def test_band_files_two_processes_nccl(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from descriptools_b200 import pipeline

    dem = tmp_path / "raw.tif"
    _raw_dem_file(dem)
    pipeline.pipeline_files(dem, tmp_path / "ref", river_threshold=300, px=PX, condition=True)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, str(dem), str(tmp_path / "out"), q)) for r in range(2)]
    for p in procs:
        p.start()
    results = sorted(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    for rank, status, info in results:
        assert status == "ok", f"rank {rank}: {info}"
    for name in pipeline.STAGE_OUTPUTS:
        assert filecmp.cmp(tmp_path / "ref" / f"{name}.tif", tmp_path / "out" / f"{name}.tif", shallow=False), name
