"""raster.py -- the GeoTIFF files either side of the descriptor path (SURVEY.md section 8 f3).

The reference does its raster I/O with rasterio (Example/example.py:33-39, :106, :201-217):

    dem  = rio.open('input/12_dem.tif').read(1)
    meta = rio.open('input/12_dem.tif').meta
    meta.update(dtype=rio.uint8); meta.update(nodata=0)
    with rio.open(out_file, "w", **meta) as dist:
        dist.write(class_map.astype(rio.uint8))

This module keeps that calling convention (`import descriptools_b200.raster as rio`) over the native
multi-threaded codec libdtb200_io.so (include/dtb200_io.h, csrc/geotiff.cpp) and adds what a 40 000 x 40 000
raster needs: row blocks decoded straight into pinned host memory while the previous block is on its way to
the device (`read_to_device`), and the mirror image for results (`write_from_device`).  torch only owns the
pinned / device buffers and the copy stream.  Single-band rasters only (all the reference uses).
"""
from __future__ import annotations

import ctypes
import os
from collections import namedtuple
from ctypes import POINTER, Structure, byref, c_char_p, c_double, c_int, c_int32, c_int64, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdtb200_io.so")

# rasterio exposes dtype names as module attributes (example.py:205, :217)
uint8, int8, uint16, int16, uint32, int32 = "uint8", "int8", "uint16", "int16", "uint32", "int32"
uint64, int64, float32, float64 = "uint64", "int64", "float32", "float64"

_DTYPES = ("uint8", "int8", "uint16", "int16", "uint32", "int32", "uint64", "int64", "float32", "float64")
_COMPRESSION = {"none": 1, "lzw": 5, "deflate": 8, "packbits": 32773}
_COMPRESSION_NAME = {v: k for k, v in _COMPRESSION.items()}
# TIFF field types used for the georeferencing tags
_T_ASCII, _T_SHORT, _T_DOUBLE = 2, 3, 12
_TAG_GDAL_METADATA, _TAG_GDAL_NODATA = 42112, 42113


class RasterError(RuntimeError):
    pass


class _Info(Structure):
    _fields_ = [("rows", c_int64), ("cols", c_int64), ("dtype", c_int32), ("compression", c_int32), ("predictor", c_int32),
                ("tile_rows", c_int32), ("tile_cols", c_int32), ("rows_per_strip", c_int32), ("bigtiff", c_int32),
                ("big_endian", c_int32), ("has_nodata", c_int32), ("has_georef", c_int32), ("nodata", c_double),
                ("pixel_scale", c_double * 3), ("tiepoint", c_double * 6)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: run `python __graft_entry__.py` (or make -C descriptools_b200/csrc) first")
    lib = ctypes.CDLL(LIB_PATH)
    lib.dtbio_abi_version.restype = c_int
    lib.dtbio_error_string.restype = c_char_p
    lib.dtbio_error_string.argtypes = [c_int]
    lib.dtbio_last_error.restype = c_char_p
    lib.dtbio_dtype_size.restype = c_int64
    lib.dtbio_dtype_size.argtypes = [c_int]
    lib.dtbio_open.argtypes = [c_char_p, POINTER(c_void_p)]
    lib.dtbio_get_info.argtypes = [c_void_p, POINTER(_Info)]
    lib.dtbio_get_tag.argtypes = [c_void_p, c_int, POINTER(c_int), POINTER(c_int64), POINTER(c_void_p)]
    lib.dtbio_read_rows.argtypes = [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int]
    lib.dtbio_create.argtypes = [c_char_p, POINTER(_Info), POINTER(c_void_p)]
    lib.dtbio_writer_info.argtypes = [c_void_p, POINTER(_Info)]
    lib.dtbio_set_tag.argtypes = [c_void_p, c_int, c_int, c_int64, c_void_p]
    lib.dtbio_write_rows.argtypes = [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int]
    lib.dtbio_write_encoded.argtypes = [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p]
    lib.dtbio_open_part.argtypes = [c_char_p, POINTER(_Info), POINTER(c_void_p)]
    lib.dtbio_write_encoded_at.argtypes = [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int64]
    lib.dtbio_place_chunks.argtypes = [c_void_p, c_int64, c_int64, c_void_p, c_void_p]
    lib.dtbio_bytes_written.restype = c_int64
    lib.dtbio_bytes_written.argtypes = [c_void_p]
    lib.dtbio_close_reader.argtypes = [c_void_p]
    lib.dtbio_close_writer.argtypes = [c_void_p]
    if lib.dtbio_abi_version() != 1:
        raise ImportError("libdtb200_io.so has an unexpected ABI version")
    return lib


lib = _load()


def _check(rc: int, what: str) -> None:
    if rc != 0:
        detail = lib.dtbio_last_error().decode("utf-8", "replace")
        raise RasterError(f"{what}: {lib.dtbio_error_string(rc).decode()}" + (f" ({detail})" if detail else ""))


class Affine(namedtuple("Affine", "a b c d e f")):
    """x = a*col + b*row + c, y = d*col + e*row + f (the six numbers rasterio's `transform` carries)"""
    __slots__ = ()

    def __mul__(self, colrow):
        col, row = colrow
        return (self.a * col + self.b * row + self.c, self.d * col + self.e * row + self.f)


_IDENTITY = Affine(1.0, 0.0, 0.0, 0.0, 1.0, 0.0)  # what a raster without georeferencing reports (rasterio does the same)


class GeoKeys:
    """Coordinate reference system as stored in the file: the GeoKey directory (tag 34735) with its double
    and ASCII parameter tags, carried verbatim from a source raster to the rasters derived from it."""

    def __init__(self, directory=(), doubles=(), ascii_params=""):
        self.directory = tuple(int(v) for v in directory)
        self.doubles = tuple(float(v) for v in doubles)
        self.ascii_params = str(ascii_params)

    def __eq__(self, other):
        return isinstance(other, GeoKeys) and (self.directory, self.doubles, self.ascii_params) == (other.directory, other.doubles, other.ascii_params)

    def __hash__(self):
        return hash((self.directory, self.doubles, self.ascii_params))

    def __bool__(self):
        return bool(self.directory)

    def key(self, key_id: int):
        """value of one GeoKey (e.g. 3072 ProjectedCSTypeGeoKey -> EPSG code), None if absent"""
        d = self.directory
        for i in range(4, len(d) - 3, 4):
            if d[i] == key_id:
                loc, cnt, off = d[i + 1], d[i + 2], d[i + 3]
                if loc == 0:
                    return off
                if loc == 34736:
                    return self.doubles[off] if cnt == 1 else self.doubles[off:off + cnt]
                if loc == 34737:
                    return self.ascii_params[off:off + cnt].rstrip("|")
        return None

    def to_epsg(self):
        return self.key(3072) or self.key(2048)

    def __repr__(self):
        cite = self.key(1026) or self.key(3073) or self.key(2049) or ""
        return f"GeoKeys({len(self.directory) // 4 - 1} keys{', ' + repr(cite[:60]) if cite else ''})"


def _format_nodata(v, dtype: str) -> str:
    if v is None:
        return ""
    if np.dtype(dtype).kind in "iu" and float(v) == int(v):
        return str(int(v))
    return repr(float(v))


def _only_band_one(indexes) -> None:
    if indexes in (1, None):
        return
    if isinstance(indexes, int) or list(indexes) != [1]:
        raise RasterError("single-band raster: only band 1 exists")


class DatasetReader:
    """`rio.open(path)`: `.read(1)`, `.meta`, `.profile`, and row-block reads into caller-owned memory."""

    mode = "r"

    def __init__(self, path):
        self.name = os.fspath(path)
        h = c_void_p()
        _check(lib.dtbio_open(self.name.encode(), byref(h)), f"open {self.name}")
        self._h = h
        info = _Info()
        _check(lib.dtbio_get_info(self._h, byref(info)), "dtbio_get_info")
        self._info = info
        self.height, self.width, self.count = int(info.rows), int(info.cols), 1
        self.shape = (self.height, self.width)
        self.dtypes = (_DTYPES[info.dtype],)
        self.indexes = (1,)
        self.nodata = float(info.nodata) if info.has_nodata else None
        self.nodatavals = (self.nodata,)
        self.compression = _COMPRESSION_NAME.get(int(info.compression), str(int(info.compression)))
        self.is_tiled = info.tile_rows > 0
        self.block_shapes = [(int(info.tile_rows), int(info.tile_cols)) if self.is_tiled else (int(info.rows_per_strip), self.width)]
        self.closed = False

    # -- metadata -------------------------------------------------------------------------------------
    def tag(self, tag_id: int):
        """raw TIFF tag of the first IFD: tuple of numbers, or str for ASCII; None if absent"""
        t, n, p = c_int(), c_int64(), c_void_p()
        if lib.dtbio_get_tag(self._h, tag_id, byref(t), byref(n), byref(p)) != 0:
            return None
        np_t = {1: np.uint8, 2: None, 3: np.uint16, 4: np.uint32, 6: np.int8, 7: np.uint8, 8: np.int16, 9: np.int32, 11: np.float32,
                12: np.float64, 16: np.uint64, 17: np.int64, 5: np.uint32, 10: np.int32, 13: np.uint32, 18: np.uint64}[t.value]
        if np_t is None:
            return ctypes.string_at(p.value, n.value).split(b"\0")[0].decode("latin-1")
        k = n.value * (2 if t.value in (5, 10) else 1)
        if k == 0:
            return ()
        arr = np.frombuffer(ctypes.string_at(p.value, k * np.dtype(np_t).itemsize), dtype=np_t)
        return tuple(arr.tolist())

    @property
    def transform(self) -> Affine:
        m = self.tag(34264)
        if m and len(m) >= 16:
            return Affine(m[0], m[1], m[3], m[4], m[5], m[7])
        if not self._info.has_georef:
            return _IDENTITY
        s, t = self._info.pixel_scale, self._info.tiepoint
        return Affine(s[0], 0.0, t[3] - t[0] * s[0], 0.0, -s[1], t[4] + t[1] * s[1])

    @property
    def res(self):
        tr = self.transform
        return (abs(tr.a), abs(tr.e))

    @property
    def crs(self):
        d = self.tag(34735)
        if not d:
            return None
        return GeoKeys(d, self.tag(34736) or (), self.tag(34737) or "")

    @property
    def meta(self) -> dict:
        """the dictionary example.py:202-206 copies from the DEM to the class map"""
        return dict(driver="GTiff", dtype=self.dtypes[0], nodata=self.nodata, width=self.width, height=self.height, count=1,
                    crs=self.crs, transform=self.transform)

    @property
    def profile(self) -> dict:
        p = self.meta
        if self.is_tiled:
            p.update(tiled=True, blockysize=int(self._info.tile_rows), blockxsize=int(self._info.tile_cols))
        else:
            p.update(tiled=False, blockysize=int(self._info.rows_per_strip))
        p.update(compress=self.compression, predictor=int(self._info.predictor), bigtiff=bool(self._info.bigtiff), interleave="band")
        md = self.tag(_TAG_GDAL_METADATA)
        if md:
            p["gdal_metadata"] = md
        return p

    # -- pixels ---------------------------------------------------------------------------------------
    def read_rows(self, row0: int, nrows: int, out=None, threads: int = 0):
        """rows [row0, row0+nrows) into `out` (a C-contiguous-by-row NumPy array or a CPU torch tensor -- pinned
        for the device path -- of the file's dtype and at least (nrows, width)); returns it"""
        dt = np.dtype(self.dtypes[0])
        if out is None:
            out = np.empty((nrows, self.width), dtype=dt)
        if hasattr(out, "data_ptr"):  # torch CPU tensor
            if out.is_cuda:
                raise RasterError("read_rows decodes into host memory; use read_to_device for a CUDA tensor")
            ptr, stride, ok = out.data_ptr(), out.stride(0) * out.element_size(), out.stride(1) == 1 and out.element_size() == dt.itemsize
            rows_ok = out.shape[0] >= nrows and out.shape[1] >= self.width
        else:
            ptr, stride = out.ctypes.data, out.strides[0]
            ok = out.ndim == 2 and out.strides[1] == dt.itemsize and out.dtype.itemsize == dt.itemsize and out.flags.writeable
            rows_ok = out.shape[0] >= nrows and out.shape[1] >= self.width
        if not ok or not rows_ok:
            raise RasterError("read_rows: `out` must be 2-D, unit column stride, element size of the file's dtype and large enough")
        _check(lib.dtbio_read_rows(self._h, row0, nrows, c_void_p(ptr), stride, threads), f"read {self.name}")
        return out

    def read(self, indexes=None, out=None, threads: int = 0):
        """band 1 as a 2-D array (`read(1)`, example.py:33) or a (1, rows, cols) array (`read()` / `read([1])`)"""
        _only_band_one(indexes)
        a = self.read_rows(0, self.height, out, threads)
        return a if indexes == 1 else a.reshape((1,) + tuple(a.shape))

    def close(self):
        if not self.closed:
            lib.dtbio_close_reader(self._h)
            self.closed = True

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DatasetWriter:
    """`rio.open(path, "w", **meta)`: `.write(array)` (example.py:216-217) or ordered row blocks.

    part=True opens a file another writer created with the same `meta` (a row-band run: every rank writes the chunks it
    encoded with `write_encoded(..., at=)`); it writes no header, IFD or tags, and closing it leaves the file to the
    writer that created it."""

    mode = "w"

    def __init__(self, path, driver="GTiff", width=None, height=None, count=1, dtype=None, crs=None, transform=None, nodata=None,
                 compress=None, predictor=1, tiled=False, blockxsize=256, blockysize=None, bigtiff=False, gdal_metadata=None,
                 threads: int = 0, part: bool = False, **ignored):
        if driver not in ("GTiff", None):
            raise RasterError("only the GTiff driver is written")
        if count != 1:
            raise RasterError("single-band rasters only")
        if width is None or height is None or dtype is None:
            raise RasterError("width, height and dtype are required to create a raster")
        self.name = os.fspath(path)
        self.width, self.height, self.count = int(width), int(height), 1
        self.shape = (self.height, self.width)
        dtype = np.dtype(dtype).name
        if dtype not in _DTYPES:
            raise RasterError(f"dtype {dtype} cannot be stored")
        self.dtypes = (dtype,)
        comp = _COMPRESSION[(compress or "none").lower()] if isinstance(compress, (str, type(None))) else int(compress)
        info = _Info()
        info.rows, info.cols, info.dtype = self.height, self.width, _DTYPES.index(dtype)
        info.compression, info.predictor = comp, int(predictor)
        if tiled:
            info.tile_rows, info.tile_cols = int(blockysize or 256), int(blockxsize)
        else:
            info.rows_per_strip = int(blockysize or 0)
        bt = str(bigtiff).upper()
        info.bigtiff = 1 if bt in ("TRUE", "YES", "1") else 0
        h = c_void_p()
        if part:
            _check(lib.dtbio_open_part(self.name.encode(), byref(info), byref(h)), f"open {self.name} for its chunks")
        else:
            _check(lib.dtbio_create(self.name.encode(), byref(info), byref(h)), f"create {self.name}")
        self._h, self._threads, self.closed, self.part = h, threads, False, part
        _check(lib.dtbio_writer_info(self._h, byref(info)), "dtbio_writer_info")
        self.is_tiled, self.bigtiff = info.tile_rows > 0, bool(info.bigtiff)
        self._compression, self._predictor, self._tile_cols = int(info.compression), int(info.predictor), int(info.tile_cols)
        # row blocks handed to write_rows start and end on multiples of this (or on the last row)
        self.chunk_rows = int(info.tile_rows) if self.is_tiled else int(info.rows_per_strip)
        self.nodata, self.crs, self.transform = nodata, crs, transform
        if part:
            return
        try:
            if transform is not None and tuple(transform)[:6] != _IDENTITY:
                a, b, c, d, e, f = [float(v) for v in tuple(transform)[:6]]
                if b == 0.0 and d == 0.0:
                    self._set(33550, _T_DOUBLE, np.array([a, -e, 0.0]))
                    self._set(33922, _T_DOUBLE, np.array([0.0, 0.0, 0.0, c, f, 0.0]))
                else:
                    self._set(34264, _T_DOUBLE, np.array([a, b, 0, c, d, e, 0, f, 0, 0, 0, 0, 0, 0, 0, 1.0]))
            if crs:
                if not isinstance(crs, GeoKeys):
                    raise RasterError("crs must be the GeoKeys object of a raster opened with this module")
                self._set(34735, _T_SHORT, np.array(crs.directory, dtype=np.uint16))
                if crs.doubles:
                    self._set(34736, _T_DOUBLE, np.array(crs.doubles))
                if crs.ascii_params:
                    self._set(34737, _T_ASCII, crs.ascii_params)
            if nodata is not None:
                self._set(_TAG_GDAL_NODATA, _T_ASCII, _format_nodata(nodata, dtype))
            if gdal_metadata:
                self._set(_TAG_GDAL_METADATA, _T_ASCII, gdal_metadata)
        except Exception:
            self.closed = True
            lib.dtbio_close_writer(self._h)  # no chunks yet: the library removes the file
            raise

    def _set(self, tag, ttype, value):
        if ttype == _T_ASCII:
            raw = value.encode("latin-1") + b"\0"
            _check(lib.dtbio_set_tag(self._h, tag, ttype, len(raw), ctypes.c_char_p(raw)), "dtbio_set_tag")
        else:
            arr = np.ascontiguousarray(value, dtype=np.uint16 if ttype == _T_SHORT else np.float64)
            _check(lib.dtbio_set_tag(self._h, tag, ttype, arr.size, c_void_p(arr.ctypes.data)), "dtbio_set_tag")

    def write_rows(self, row0: int, block, threads: int | None = None):
        """rows [row0, row0+len(block)) from a NumPy array or CPU torch tensor of the raster's dtype; row0 and
        the end of the block must fall on chunk boundaries (multiples of `blockysize`) or on the last row"""
        dt = np.dtype(self.dtypes[0])
        if hasattr(block, "data_ptr"):
            if block.is_cuda:
                raise RasterError("write_rows encodes from host memory; use write_from_device for a CUDA tensor")
            ok = block.dim() == 2 and block.stride(1) == 1 and block.element_size() == dt.itemsize and block.shape[1] == self.width
            ptr, stride, n = block.data_ptr(), block.stride(0) * block.element_size(), block.shape[0]
        else:
            block = np.asarray(block)
            if block.ndim == 2 and block.dtype != dt:
                block = block.astype(dt)
            ok = block.ndim == 2 and block.strides[1] == dt.itemsize and block.shape[1] == self.width
            ptr, stride, n = block.ctypes.data, block.strides[0], block.shape[0]
        if not ok:
            raise RasterError("write_rows: block must be 2-D with the raster's width and unit column stride")
        _check(lib.dtbio_write_rows(self._h, row0, n, c_void_p(ptr), stride, self._threads if threads is None else threads), f"write {self.name}")

    def chunk_layout(self):
        """(layout, chunks across, chunks in all) for dtb_tiff_encode_chunks (include/dtb200.h)"""
        from ._lib import TiffLayout

        lay = TiffLayout()
        lay.rows, lay.cols, lay.bps = self.height, self.width, np.dtype(self.dtypes[0]).itemsize
        lay.predictor, lay.compression, lay.big_endian = self._predictor, self._compression, 0
        lay.tiled, lay.chunk_rows = (1 if self.is_tiled else 0), self.chunk_rows
        lay.chunk_cols = self._tile_cols if self.is_tiled else self.width
        across = -(-self.width // lay.chunk_cols) if self.is_tiled else 1
        return lay, across, across * -(-self.height // lay.chunk_rows)

    def write_encoded(self, first_chunk: int, blob, offsets, sizes, at: int | None = None):
        """chunks encoded on the device: `blob` (uint8 NumPy array or CPU tensor) holds chunk first_chunk + i at
        offsets[i] .. offsets[i] + sizes[i]; one file write for the whole group.  The blob goes to the end of the file,
        or with `at=` to that file offset (dtbio_write_encoded_at: even, past the 16 header bytes)."""
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        sizes = np.ascontiguousarray(sizes, dtype=np.int64)
        if hasattr(blob, "data_ptr"):
            ptr, nbytes = blob.data_ptr(), blob.numel() * blob.element_size()
        else:
            blob = np.ascontiguousarray(blob)
            ptr, nbytes = blob.ctypes.data, blob.nbytes
        if at is None:
            _check(lib.dtbio_write_encoded(self._h, first_chunk, sizes.size, c_void_p(ptr), nbytes, c_void_p(offsets.ctypes.data),
                                           c_void_p(sizes.ctypes.data)), f"write {self.name}")
        else:
            _check(lib.dtbio_write_encoded_at(self._h, first_chunk, sizes.size, c_void_p(ptr), nbytes, c_void_p(offsets.ctypes.data),
                                              c_void_p(sizes.ctypes.data), int(at)), f"write {self.name}")

    def place_chunks(self, first_chunk: int, file_offsets, sizes):
        """record chunks first_chunk + i that another writer put at file_offsets[i] (sizes[i] bytes) in this file"""
        file_offsets = np.ascontiguousarray(file_offsets, dtype=np.int64)
        sizes = np.ascontiguousarray(sizes, dtype=np.int64)
        if file_offsets.shape != sizes.shape:
            raise RasterError("place_chunks: one offset per size")
        _check(lib.dtbio_place_chunks(self._h, first_chunk, sizes.size, c_void_p(file_offsets.ctypes.data), c_void_p(sizes.ctypes.data)),
               f"place chunks in {self.name}")

    def abort(self):
        """close without finishing: the file is removed (a part writer only closes its descriptor)"""
        if not self.closed:
            self.closed = True
            lib.dtbio_close_writer(self._h)  # removes the file if a chunk is missing
        if not self.part and os.path.exists(self.name):
            os.unlink(self.name)

    def write(self, arr, indexes=None):
        a = np.asarray(arr)
        if a.ndim == 3:
            if a.shape[0] != 1:
                raise RasterError("single-band rasters only")
            a = a[0]
        if a.shape != self.shape:
            raise RasterError(f"array shape {a.shape} does not match the raster {self.shape}")
        _only_band_one(indexes)
        self.write_rows(0, np.ascontiguousarray(a, dtype=self.dtypes[0]))

    @property
    def bytes_written(self) -> int:
        return int(lib.dtbio_bytes_written(self._h))

    def close(self):
        if not self.closed:
            self.closed = True
            _check(lib.dtbio_close_writer(self._h), f"close {self.name}")

    def __enter__(self):
        return self

    def __exit__(self, exc_type, *exc):
        if exc_type is None:
            self.close()
        elif not self.closed:
            # leave no half-written file behind; the library unlinks it when chunks are missing
            self.closed = True
            lib.dtbio_close_writer(self._h)
        return False

    def __del__(self):
        if not getattr(self, "closed", True):
            self.closed = True
            lib.dtbio_close_writer(self._h)


def open(path, mode: str = "r", **kwargs):  # noqa: A001  (rasterio's name)
    """`rio.open(path)` -> DatasetReader; `rio.open(path, "w", **meta)` -> DatasetWriter (example.py:33, :216)"""
    if mode == "r":
        if kwargs:
            raise RasterError("unexpected keyword arguments for read mode: " + ", ".join(kwargs))
        return DatasetReader(path)
    if mode == "w":
        return DatasetWriter(path, **kwargs)
    raise RasterError(f"mode {mode!r} is not supported (use 'r' or 'w')")


# ---------------------------------------------------------------------------------------------------------
# file <-> device streaming
# ---------------------------------------------------------------------------------------------------------
def _block_rows(src_rows: int, chunk_rows: int, cols: int, itemsize: int, target_bytes: int) -> int:
    """rows per streamed block: about `target_bytes`, a multiple of the file's chunk height"""
    want = max(1, target_bytes // max(1, cols * itemsize))
    chunk_rows = max(1, chunk_rows)
    return min(max(chunk_rows, want // chunk_rows * chunk_rows), max(src_rows, 1))


def _rows(buf, k: int, br: int, rows: int, cols: int, dtype):
    """block k of `rows` rows streamed `br` at a time: (its first row, its rows as an (n, cols) `dtype` view of `buf`)"""
    n = min(br, rows - k * br)
    return k * br, buf[:n * cols * dtype.itemsize].view(dtype).view(n, cols)


def _to_device(count: int, cap: int, fill, send, copy) -> None:
    """Host -> device through min(2, count) pinned uint8 buffers of `cap` bytes: fill(k, buf) writes piece k on the host
    while piece k-1 is sent, then send(k, buf) enqueues on `copy` what reads the buffer.  Returns when all has run."""
    import torch

    stage = [torch.empty(cap, dtype=torch.uint8, pin_memory=True) for _ in range(min(2, count))]
    copy.wait_stream(torch.cuda.current_stream(copy.device))  # the destination may reuse memory the current stream still works on
    for k in range(count):
        fill(k, stage[k % len(stage)])
        copy.synchronize()  # piece k-1 is sent: its buffer takes piece k+1
        with torch.cuda.stream(copy):
            send(k, stage[k % len(stage)])
    copy.synchronize()


def _from_device(count: int, cap: int, fetch, drain, copy, ready) -> None:
    """Device -> host through min(2, count) pinned uint8 buffers of `cap` bytes: fetch(k, buf) enqueues the copy of piece
    k on `copy` (after the work on `ready`), drain(k, buf) consumes it on the host while piece k+1 is copied."""
    import torch

    stage = [torch.empty(cap, dtype=torch.uint8, pin_memory=True) for _ in range(min(2, count))]

    def enqueue(k):
        with torch.cuda.stream(copy):
            fetch(k, stage[k % len(stage)])

    copy.wait_stream(ready)
    if count:
        enqueue(0)
    for k in range(count):
        copy.synchronize()  # piece k has landed: nothing is enqueued behind it
        if k + 1 < count:
            enqueue(k + 1)  # into the other buffer, drained already
        drain(k, stage[k % len(stage)])


_WARPS_IN_FLIGHT = 148 * 8 * 4  # the codec kernels keep one chunk per resident warp (csrc/tiffcodec.cu)


def _chunks_per_group(n: int, across: int, chunk_raw: int, block_bytes: int) -> int:
    """chunks handed to one codec launch: whole chunk-rows, about `block_bytes` of decoded data but never fewer than fill
    the device (one warp per chunk) while leaving two groups to overlap with the copies, and at most 4 GiB decoded"""
    by_bytes = block_bytes // max(1, chunk_raw)
    fill = min(_WARPS_IN_FLIGHT, -(-n // 2))
    want = min(max(by_bytes, fill, 1), max(1, (4 << 30) // max(1, chunk_raw)))
    return min(n, max(1, -(-want // across)) * across)


def chunk_table(reader: "DatasetReader"):
    """(layout, offsets, byte counts) of a raster's chunks: what dtb_tiff_decode_chunks (include/dtb200.h) needs.
    offsets / counts are uint64 arrays in chunk order (tiles row-major, or strips top to bottom)."""
    from ._lib import TiffLayout

    info = reader._info
    lay = TiffLayout()
    lay.rows, lay.cols, lay.bps = reader.height, reader.width, np.dtype(reader.dtypes[0]).itemsize
    lay.predictor, lay.compression, lay.big_endian = int(info.predictor), int(info.compression), int(info.big_endian)
    lay.tiled = 1 if reader.is_tiled else 0
    lay.chunk_rows = int(info.tile_rows if reader.is_tiled else info.rows_per_strip)
    lay.chunk_cols = int(info.tile_cols) if reader.is_tiled else reader.width
    across = -(-reader.width // lay.chunk_cols) if reader.is_tiled else 1
    n = across * -(-reader.height // lay.chunk_rows)
    off = np.array(reader.tag(324 if reader.is_tiled else 273), dtype=np.uint64)[:n]
    cnt = reader.tag(325 if reader.is_tiled else 279)
    if cnt is None:  # uncompressed files may omit the byte counts
        rows_in = np.minimum(lay.chunk_rows, reader.height - (np.arange(n) // across) * lay.chunk_rows)
        cnt = rows_in * lay.chunk_cols * lay.bps
    cnt = np.array(cnt, dtype=np.uint64)[:n]
    cnt[off == 0] = 0
    return lay, across, off, cnt


# what decode="auto" hands to the device: the codecs whose kernels win there on a B200.  LZW does (profiles/r1z_*,
# r2zf_raster_codecs_*: 4.7-4.8 GB/s against 3.3-3.7 from 16 host threads at 16384 x 16384).  The Deflate kernel is correct on
# the device (tests/test_raster_io.py) but a draw -- 4.0-4.3 GB/s against 3.6-4.6 -- so Deflate and PackBits files take the
# host team unless the caller asks for decode="device".
_AUTO_DEVICE_COMPRESSIONS = ("none", "lzw")


def device_decode_supported(reader: "DatasetReader") -> bool:
    """can dtb_tiff_decode_chunks take this file?  (stored, LZW, Deflate or PackBits chunks of at most 1 MiB; the library decides)"""
    from ._lib import lib as cuda_lib

    lay = chunk_table(reader)[0]
    return int(cuda_lib.dtb_tiff_decode_workspace_bytes(ctypes.byref(lay), 1)) > 0


def device_encode_supported(writer: "DatasetWriter") -> bool:
    """can dtb_tiff_encode_chunks produce this file's chunks?  (stored or LZW; the library decides)"""
    from ._lib import lib as cuda_lib

    lay = writer.chunk_layout()[0]
    return int(cuda_lib.dtb_tiff_encode_bound(ctypes.byref(lay))) > 0


def _band_chunks(row_lo: int, row_hi: int, chunk_rows: int, across: int) -> tuple:
    """[first, last) of the chunks that hold raster rows [row_lo, row_hi)"""
    return (row_lo // chunk_rows) * across, -(-row_hi // chunk_rows) * across


def _check_chunk_table(name: str, off: np.ndarray, cnt: np.ndarray, file_size: int) -> None:
    """every chunk must lie inside the file: the device decoder reads exactly the bytes the table names, and a damaged
    table must neither size the staging buffers nor send a warp past the end of the compressed data"""
    size = np.uint64(file_size)
    bad = (cnt > size) | (off > size - np.minimum(cnt, size))
    if bool(bad[cnt > 0].any()):
        raise RasterError(f"{name}: chunk table points outside the file")


def _read_to_device_chunks(reader, out, block_bytes: int, copy, group_chunks=None, rows=None):
    """read_to_device(decode="device"): the compressed chunks go over PCIe as they lie in the file and are decoded
    by dtb_tiff_decode_chunks, one warp per chunk.  File spans are staged through pinned memory (_to_device); reading
    span k+1 overlaps the copy and decode of span k on `copy`."""
    import torch

    from ._lib import check
    from ._lib import lib as cuda_lib

    lay, across, off, cnt = chunk_table(reader)
    if not device_decode_supported(reader):
        raise RasterError(f"decode='device' handles stored, LZW, Deflate and PackBits chunks of at most 1 MiB, not this file ({reader.compression}, "
                          f"{reader.block_shapes[0]} chunks); use decode='host'")
    dev = out.device
    c_lo, c_hi = 0, off.size
    if rows is not None:  # a row band: `out` holds rows [rows[0], rows[1]) and the kernel stores only those
        lay.row_lo, lay.row_hi = int(rows[0]), int(rows[1])
        c_lo, c_hi = _band_chunks(lay.row_lo, lay.row_hi, lay.chunk_rows, across)
    n = c_hi - c_lo
    chunk_raw = lay.chunk_rows * lay.chunk_cols * lay.bps
    per_group = group_chunks or _chunks_per_group(n, across, chunk_raw, block_bytes)
    groups = [(g0, min(c_hi, g0 + per_group)) for g0 in range(c_lo, c_hi, per_group)]
    spans = []
    _check_chunk_table(reader.name, off[c_lo:c_hi], cnt[c_lo:c_hi], os.path.getsize(reader.name))
    for g0, g1 in groups:
        live = cnt[g0:g1] > 0
        lo = int(off[g0:g1][live].min()) if live.any() else 0
        hi = int((off[g0:g1] + cnt[g0:g1])[live].max()) if live.any() else 0
        spans.append((lo, hi))
    biggest = max(1, max(hi - lo for lo, hi in spans))
    comp = [torch.empty(biggest, dtype=torch.uint8, device=dev) for _ in range(min(2, len(groups)))]  # reused in order on `copy`
    ws_bytes = int(cuda_lib.dtb_tiff_decode_workspace_bytes(ctypes.byref(lay), per_group))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    status = torch.zeros(1, dtype=torch.int64, device=dev)

    def fill(k, buf):
        lo, hi = spans[k]
        view = memoryview(buf.numpy())[:hi - lo]
        got = 0
        while got < hi - lo:
            m = os.preadv(fd, [view[got:]], lo + got)
            if m <= 0:
                raise RasterError(f"{reader.name}: file ends inside a chunk")
            got += m

    def send(k, buf):
        (g0, g1), (lo, hi), c = groups[k], spans[k], comp[k % len(comp)]
        rel = off[g0:g1] - np.uint64(lo)
        rel[cnt[g0:g1] == 0] = 0
        table = torch.from_numpy(np.concatenate([rel, cnt[g0:g1]]).view(np.int64))
        c[:hi - lo].copy_(buf[:hi - lo], non_blocking=True)
        table_d = table.to(dev)  # small and pageable: synchronous with respect to the host, ordered on `copy`
        check(cuda_lib.dtb_tiff_decode_chunks(ctypes.byref(lay), c.data_ptr(), table_d.data_ptr(), table_d.data_ptr() + 8 * (g1 - g0),
                                              g0, g1 - g0, out.data_ptr(), ws.data_ptr(), ws_bytes, status.data_ptr(), copy.cuda_stream),
              "dtb_tiff_decode_chunks")

    fd = os.open(reader.name, os.O_RDONLY)
    try:
        _to_device(len(groups), biggest, fill, send, copy)
    finally:
        os.close(fd)
    code = int(status.item())
    if code:
        reason = {1: "corrupt compressed stream", 2: "pre-6.0 LZW", 3: "chunk decodes short"}.get(code & 7, "decode error")
        raise RasterError(f"{reader.name}: chunk {(code >> 3) - 1}: {reason}")
    torch.cuda.current_stream(dev).wait_stream(copy)
    return out


def read_to_device(src, device=None, out=None, block_bytes: int = 256 << 20, threads: int = 0, stream=None, decode: str = "host",
                   group_chunks: int | None = None, rows: tuple | None = None):
    """Decode a raster into a CUDA tensor.  Returns the tensor (dtype of the file); the current stream waits for
    the last copy.  `src` is a path or a DatasetReader.

    decode="host": two pinned staging blocks; while block k is copied to the device on `stream` (default: a private
    copy stream) the codec's thread team decodes block k+1.
    decode="device": the compressed chunks are copied instead and decoded on the device (stored, LZW and Deflate files;
    anything else raises -- nothing falls back silently); `group_chunks` overrides the number of chunks per launch.
    decode="auto": "device" for stored and LZW files the device decoder can take, else "host".
    rows=(r0, r1): only that row band of the raster (the tensor has r1 - r0 rows) -- what one rank of a row-band run
    loads (bands.BandRunner.load_file)."""
    import torch

    from . import device as _device

    if decode not in ("host", "device", "auto"):
        raise RasterError("decode must be 'host', 'device' or 'auto'")
    dev = torch.device(device) if device is not None else _device.require_cuda()
    reader = src if isinstance(src, DatasetReader) else DatasetReader(src)
    try:
        if decode == "auto":  # the device codec when it can take the file: an explicit choice between two complete paths
            on_device = reader.compression in _AUTO_DEVICE_COMPRESSIONS and device_decode_supported(reader)
            decode = "device" if on_device and (out is None or out.is_contiguous()) else "host"
        first, last = (0, reader.height) if rows is None else (int(rows[0]), int(rows[1]))
        if not 0 <= first < last <= reader.height:
            raise RasterError(f"read_to_device: rows {rows} outside the raster")
        shape = (last - first, reader.width)
        tdt = getattr(torch, reader.dtypes[0])
        if decode == "device":
            if out is None:
                out = torch.empty(shape, dtype=tdt, device=dev)
            elif tuple(out.shape) != shape or out.dtype != tdt or not out.is_cuda or not out.is_contiguous():
                raise RasterError("read_to_device: `out` must be a contiguous CUDA tensor of the (band of the) raster's shape and dtype")
            return _read_to_device_chunks(reader, out, block_bytes, stream if stream is not None else torch.cuda.Stream(device=out.device),
                                          group_chunks, None if rows is None else (first, last))
        nrows, cols = shape
        if out is None:
            out = torch.empty(shape, dtype=tdt, device=dev)
        elif tuple(out.shape) != shape or out.dtype != tdt or not out.is_cuda:
            raise RasterError("read_to_device: `out` must be a CUDA tensor of the (band of the) raster's shape and dtype")
        br = _block_rows(nrows, reader.block_shapes[0][0], cols, out.element_size(), block_bytes)

        def fill(k, buf):
            r0, rows_k = _rows(buf, k, br, nrows, cols, tdt)
            reader.read_rows(first + r0, rows_k.shape[0], rows_k, threads)

        def send(k, buf):
            r0, rows_k = _rows(buf, k, br, nrows, cols, tdt)
            out[r0:r0 + rows_k.shape[0]].copy_(rows_k, non_blocking=True)

        copy = stream if stream is not None else torch.cuda.Stream(device=out.device)
        _to_device(-(-nrows // br), br * cols * out.element_size(), fill, send, copy)
        torch.cuda.current_stream(out.device).wait_stream(copy)
        return out
    finally:
        if reader is not src:
            reader.close()


def encode_groups(lay, tensor, c_lo: int, c_hi: int, block_bytes: int = 256 << 20, group_chunks=None):
    """Encode chunks [c_lo, c_hi) of the layout `lay` on the tensor's device, in groups of whole chunk-rows: each group
    is encoded by dtb_tiff_encode_chunks (one warp per chunk) while the group before it is packed by dtb_tiff_pack_chunks.
    `tensor` is the contiguous raster, or with lay.row_lo / row_hi set the rows [row_lo, row_hi) of it (every chunk must
    lie inside them).

    Yields (g0, g1, blob, sizes, stream) per group, in chunk order: `blob` (device uint8) holds the group's streams back
    to back, each padded with a zero byte to even length -- the layout of the file, what write_packed takes -- and is
    ready on `stream`.  It is reused for a later group once the caller asks for the next one, so the caller copies it out
    first."""
    import torch

    from ._lib import check
    from ._lib import lib as cuda_lib

    bound = int(cuda_lib.dtb_tiff_encode_bound(ctypes.byref(lay)))
    if bound == 0:
        raise RasterError("encode='device' writes stored or LZW chunks (predictor 1-3, little-endian); use encode='host' for the rest")
    dev = tensor.device
    across = -(-lay.cols // lay.chunk_cols) if lay.tiled else 1
    chunk_raw = lay.chunk_rows * lay.chunk_cols * lay.bps
    n = c_hi - c_lo
    if n <= 0:
        return
    per_group = group_chunks or _chunks_per_group(n, across, chunk_raw, block_bytes)
    groups = [(g0, min(c_hi, g0 + per_group)) for g0 in range(c_lo, c_hi, per_group)]
    nbuf = min(2, len(groups))
    ws_bytes = int(cuda_lib.dtb_tiff_encode_workspace_bytes(ctypes.byref(lay), per_group))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)  # one workspace: the encode kernels run in order on one stream
    enc = [torch.empty(per_group * bound, dtype=torch.uint8, device=dev) for _ in range(nbuf)]
    sizes_d = [torch.empty(per_group, dtype=torch.int64, device=dev) for _ in range(nbuf)]
    blob = None  # packed streams of one group; grown to what the data needs
    work, io = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    work.wait_stream(torch.cuda.current_stream(dev))
    encoded, reusable = [None] * len(groups), [None] * nbuf

    def launch(k):
        g0, g1 = groups[k]
        b = k % nbuf
        if reusable[b] is not None:
            work.wait_event(reusable[b])  # the pack kernel that read this slot buffer has run
        check(cuda_lib.dtb_tiff_encode_chunks(ctypes.byref(lay), tensor.data_ptr(), g0, g1 - g0, enc[b].data_ptr(), sizes_d[b].data_ptr(),
                                              ws.data_ptr(), ws_bytes, work.cuda_stream), "dtb_tiff_encode_chunks")
        encoded[k] = torch.cuda.Event()
        encoded[k].record(work)

    launch(0)
    for k, (g0, g1) in enumerate(groups):
        b = k % nbuf
        if k + 1 < len(groups):
            launch(k + 1)
        io.wait_event(encoded[k])
        with torch.cuda.stream(io):
            sizes = sizes_d[b][:g1 - g0].cpu().numpy()  # synchronises `io`: the group is encoded
            if (sizes <= 0).any():
                raise RasterError("a chunk did not fit its encode slot")
            aligned = (sizes + 1) & ~1
            offsets = np.cumsum(aligned) - aligned
            total = int(aligned.sum())
            offsets_d = torch.from_numpy(offsets).to(dev)
            if blob is None or blob.numel() < total:
                blob = torch.empty(min(per_group * bound, total + total // 4 + 4096), dtype=torch.uint8, device=dev)
            blob[:total].zero_()  # the pad bytes
            check(cuda_lib.dtb_tiff_pack_chunks(enc[b].data_ptr(), bound, sizes_d[b].data_ptr(), offsets_d.data_ptr(), g1 - g0,
                                                blob.data_ptr(), io.cuda_stream), "dtb_tiff_pack_chunks")
            reusable[b] = torch.cuda.Event()
            reusable[b].record(io)
        yield g0, g1, blob[:total], sizes, io
    io.synchronize()
    torch.cuda.current_stream(dev).wait_stream(work)


def write_packed(w: "DatasetWriter", first_chunk: int, packed, sizes, piece_bytes: int, offsets=None, ready=None) -> None:
    """Write chunks first_chunk + i (sizes[i] bytes each), packed back to back in `packed` as encode_groups packs them, in
    chunk order and in pieces of whole chunks of about `piece_bytes`: appended (the same bytes as one append of the whole
    blob), or with `offsets` at file offset offsets[i] (a row band's chunks).  A device blob is staged through pinned
    memory after the work on `ready` (default: the current stream), the next piece copied while this one is written; a
    host blob (NumPy array or CPU tensor) is written as it lies."""
    import torch

    sizes = np.asarray(sizes, dtype=np.int64)
    aligned = (sizes + 1) & ~1
    rel = np.cumsum(aligned) - aligned
    pieces, a = [], 0  # (first, end) chunk of each piece, its bytes [lo, hi) in `packed`
    while a < len(sizes):
        b = min(len(sizes), max(a + 1, int(np.searchsorted(rel, rel[a] + piece_bytes, side="right"))))
        pieces.append((a, b, int(rel[a]), int(rel[b - 1] + aligned[b - 1])))
        a = b

    def put(j, buf):  # piece j, which starts at buf[0]
        a, b, lo, hi = pieces[j]
        w.write_encoded(first_chunk + a, buf[:hi - lo], rel[a:b] - lo, sizes[a:b], at=None if offsets is None else int(offsets[a]))

    if not getattr(packed, "is_cuda", False):
        host = packed.numpy() if hasattr(packed, "numpy") else packed
        for j, p in enumerate(pieces):
            put(j, host[p[2]:])
        return

    def fetch(j, buf):
        _, _, lo, hi = pieces[j]
        buf[:hi - lo].copy_(packed[lo:hi], non_blocking=True)

    _from_device(len(pieces), max(hi - lo for _, _, lo, hi in pieces), fetch, put, torch.cuda.Stream(device=packed.device),
                 ready if ready is not None else torch.cuda.current_stream(packed.device))


def layout_of(meta: dict):
    """(layout, chunks across, chunks in all) of the file `open(path, "w", **meta)` writes -- for the ranks of a row-band
    run, which encode their chunks before the file exists.  Strips need an explicit `blockysize`."""
    from ._lib import TiffLayout

    compress = meta.get("compress")
    comp = _COMPRESSION[(compress or "none").lower()] if isinstance(compress, (str, type(None))) else int(compress)
    lay = TiffLayout()
    lay.rows, lay.cols = int(meta["height"]), int(meta["width"])
    lay.bps = np.dtype(meta["dtype"]).itemsize
    lay.compression, lay.big_endian = comp, 0
    lay.predictor = 1 if comp == 1 else int(meta.get("predictor", 1) or 1)
    if meta.get("tiled"):
        lay.tiled, lay.chunk_rows, lay.chunk_cols = 1, int(meta.get("blockysize") or 256), int(meta.get("blockxsize", 256))
    else:
        if not meta.get("blockysize"):
            raise RasterError("give blockysize (rows per strip) for a striped file written by several writers")
        lay.tiled, lay.chunk_rows, lay.chunk_cols = 0, int(meta["blockysize"]), lay.cols
    across = -(-lay.cols // lay.chunk_cols) if lay.tiled else 1
    return lay, across, across * -(-lay.rows // lay.chunk_rows)


def write_from_device(path, tensor, block_bytes: int = 256 << 20, threads: int = 0, encode: str = "host",
                      group_chunks: int | None = None, **meta):
    """Mirror of read_to_device: a 2-D CUDA tensor goes to a GeoTIFF.  `meta` as for `open(path, "w", ...)`
    (width / height / dtype default to the tensor's).  Returns the number of bytes written.

    encode="host": row blocks; block k+1 is copied to its pinned staging buffer while the thread team encodes block k.
    encode="device": the chunks are encoded on the device and only the compressed bytes cross PCIe, in pieces of about
    `block_bytes` (write_packed) (stored and LZW files; anything else raises -- nothing falls back silently).
    encode="auto": "device" when device_encode_supported(writer), else "host".
    A failed call leaves no file."""
    import torch

    if encode not in ("host", "device", "auto"):
        raise RasterError("encode must be 'host', 'device' or 'auto'")
    if not tensor.is_cuda or tensor.dim() != 2:
        raise RasterError("write_from_device needs a 2-D CUDA tensor")
    rows, cols = tensor.shape
    meta = dict(meta)
    meta.setdefault("width", cols)
    meta.setdefault("height", rows)
    meta.setdefault("dtype", str(tensor.dtype).replace("torch.", ""))
    if np.dtype(meta["dtype"]).name != str(tensor.dtype).replace("torch.", ""):
        raise RasterError("write_from_device: dtype of the file must be the tensor's (convert on the device first)")
    w = DatasetWriter(path, threads=threads, **meta)
    try:
        if encode == "auto":
            encode = "device" if device_encode_supported(w) and tensor.is_contiguous() else "host"
        if encode == "device":
            if not tensor.is_contiguous():
                raise RasterError("write_from_device(encode='device') needs a contiguous tensor")
            lay, _, n = w.chunk_layout()
            for g0, _, blob, sizes, io in encode_groups(lay, tensor, 0, n, block_bytes, group_chunks):
                write_packed(w, g0, blob, sizes, block_bytes, ready=io)
        else:
            br = _block_rows(rows, w.chunk_rows, cols, tensor.element_size(), block_bytes)

            def fetch(k, buf):
                r0, rows_k = _rows(buf, k, br, rows, cols, tensor.dtype)
                rows_k.copy_(tensor[r0:r0 + rows_k.shape[0]], non_blocking=True)

            def drain(k, buf):
                w.write_rows(*_rows(buf, k, br, rows, cols, tensor.dtype))

            _from_device(-(-rows // br), br * cols * tensor.element_size(), fetch, drain, torch.cuda.Stream(device=tensor.device),
                         torch.cuda.current_stream(tensor.device))
        total = w.bytes_written
        w.close()
        return total
    except Exception:
        w.abort()
        raise
