"""ctypes binding of libdtb200.so (C ABI: include/dtb200.h).

There is no fallback: if the shared library is missing or a call fails, an exception is
raised.  PyTorch is used only to own device buffers and streams.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint32, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DTB_LIB_PATH") or os.path.join(_HERE, "libdtb200.so")  # override: debugging builds only

DTB_F32, DTB_I16 = 0, 1
DTB_I32, DTB_I64 = 0, 1
DTB_FA_FULL, DTB_FA_SUMMARY, DTB_FA_FINISH = 0, 1, 2
DTB_HAND_FULL, DTB_HAND_SUMMARY, DTB_HAND_FINISH = 0, 1, 2
DTB_FILL_INIT, DTB_FILL_SOLVE = 0, 1


class DtbError(RuntimeError):
    pass


class HandSeam(Structure):
    _fields_ = [
        ("halo", c_void_p),
        ("sum_state", c_void_p),
        ("sum_idx", c_void_p),
        ("sum_z", c_void_p),
        ("sum_acc", c_void_p),
        ("res_state", c_void_p),
        ("res_idx", c_void_p),
        ("res_z", c_void_p),
        ("res_acc", c_void_p),
    ]


class HandBand(Structure):
    _fields_ = [("mode", c_int), ("row_offset", c_int64), ("above", HandSeam), ("below", HandSeam)]


class HandArgs(Structure):
    _fields_ = [
        ("fdr", c_void_p),
        ("river", c_void_p),
        ("acc", c_void_p),
        ("acc_dtype", c_int),
        ("river_threshold", c_int64),
        ("dem", c_void_p),
        ("dem_dtype", c_int),
        ("rows", c_int64),
        ("cols", c_int64),
        ("px", c_double),
        ("max_moves", c_int64),
        ("fdist", c_void_p),
        ("idx", c_void_p),
        ("idx_dtype", c_int),
        ("hand", c_void_p),
        ("gfi", c_void_p),
        ("gfi_n", c_double),
        ("gfi_b", c_double),
        ("gfi_size", c_double),
        ("band", POINTER(HandBand)),
        ("entry_done", c_int),
    ]


class TiffLayout(Structure):
    _fields_ = [("rows", c_int64), ("cols", c_int64), ("bps", c_int32), ("predictor", c_int32), ("compression", c_int32),
                ("tiled", c_int32), ("chunk_rows", c_int32), ("chunk_cols", c_int32), ("big_endian", c_int32),
                ("row_lo", c_int64), ("row_hi", c_int64)]


class FlowaccArgs(Structure):
    _fields_ = [
        ("d8", c_void_p),
        ("rows", c_int64),
        ("cols", c_int64),
        ("halo_above", c_void_p),
        ("halo_below", c_void_p),
        ("inflow_above", c_void_p),
        ("inflow_below", c_void_p),
        ("acc", c_void_p),
        ("acc_dtype", c_int),
        ("nodata_fill", c_int64),
        ("exit_above", c_void_p),
        ("exit_below", c_void_p),
        ("term_above", c_void_p),
        ("term_below", c_void_p),
        ("mode", c_int),
        ("unfinalised_host", POINTER(c_int64)),
        ("hand_ws", c_void_p),
        ("hand_ws_bytes", c_size_t),
        ("hand_river_threshold", c_int64),
    ]


# name -> (restype, argtypes); mirrors include/dtb200.h one to one
SIGNATURES = {
    "dtb_abi_version": (c_int, []),
    "dtb_error_string": (c_char_p, [c_int]),
    "dtb_last_cuda_error": (c_char_p, []),
    "dtb_launch_count": (c_int64, []),
    "dtb_reset_launch_count": (None, []),
    "dtb_profile_enable": (None, [c_int]),
    "dtb_profile_collect": (c_int64, [c_char_p, c_int64]),
    "dtb_slope_d8": (c_int, [c_void_p, c_int, c_int64, c_int64, c_int64, c_int64, c_double, c_void_p, c_void_p, c_void_p]),
    "dtb_flowacc_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "dtb_flowacc": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int, c_int64, c_void_p, c_size_t,
                            POINTER(c_int64), c_void_p]),
    "dtb_flowacc_band": (c_int, [POINTER(FlowaccArgs), c_void_p, c_size_t, c_void_p]),
    "dtb_flowacc_boundary_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "dtb_flowacc_boundary_solve": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dtb_forest_workspace_bytes": (c_size_t, [c_int64]),
    "dtb_forest_accumulate": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dtb_hand_boundary_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "dtb_hand_boundary_solve": (c_int, [c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dtb_hand_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "dtb_hand": (c_int, [POINTER(HandArgs), c_void_p, c_size_t, c_void_p]),
    "dtb_chain_check": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int64,
                                c_void_p, c_void_p]),
    "dtb_nodata_to_sentinel_f32": (c_int, [c_void_p, c_int64, ctypes.c_float, c_int, c_void_p]),
    "dtb_hand_from_index": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p]),
    "dtb_downslope": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_int64, c_double, c_double, c_int64, c_void_p, c_void_p]),
    "dtb_downslope_window": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_int64, c_int64, c_int64, c_double, c_double, c_int64,
                                     c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "dtb_downslope_rows": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_int64, c_int64, c_int64, c_double, c_double, c_int64,
                                   c_void_p, c_void_p]),
    "dtb_river_accumulation": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p]),
    "dtb_gfi": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64, c_double, c_double, c_double, c_void_p, c_void_p]),
    "dtb_lnhlh": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64, c_double, c_double, c_double, c_void_p, c_void_p]),
    "dtb_ti_mti": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_double, c_double, c_void_p, c_void_p, c_void_p]),
    "dtb_slope_to_radians": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "dtb_eval_counts": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_double, POINTER(c_double), c_int, c_int, POINTER(c_int64),
                                c_void_p, c_size_t, c_void_p]),
    "dtb_eval_class_map": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_double, c_double, c_int, c_void_p, c_void_p, c_void_p]),
    "dtb_minmax_scale": (c_int, [c_void_p, c_int, c_int64, c_double, c_double, c_double, c_void_p, c_void_p]),
    "dtb_tiff_decode_workspace_bytes": (c_size_t, [POINTER(TiffLayout), c_int64]),
    "dtb_tiff_decode_chunks": (c_int, [POINTER(TiffLayout), c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p,
                                       c_size_t, c_void_p, c_void_p]),
    "dtb_selftest_tiff_decode_host": (c_int, [POINTER(TiffLayout), c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p,
                                              c_void_p]),
    "dtb_tiff_encode_bound": (c_size_t, [POINTER(TiffLayout)]),
    "dtb_tiff_encode_workspace_bytes": (c_size_t, [POINTER(TiffLayout), c_int64]),
    "dtb_tiff_encode_chunks": (c_int, [POINTER(TiffLayout), c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_size_t,
                                       c_void_p]),
    "dtb_tiff_pack_chunks": (c_int, [c_void_p, c_size_t, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "dtb_selftest_tiff_encode_host": (c_int, [POINTER(TiffLayout), c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "dtb_synth_dem_f32": (c_int, [c_int64, c_int64, c_int64, c_uint32, POINTER(c_float), c_float, c_float, c_float,
                                  c_float, c_void_p, c_void_p]),
    "dtb_fill_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "dtb_fill_depressions_f32": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_size_t, POINTER(c_int), c_void_p]),
    "dtb_fill_band_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "dtb_fill_band_f32": (c_int, [c_void_p, c_int64, c_int64, c_int, c_int, c_int, c_void_p, c_size_t, POINTER(c_int), POINTER(c_int),
                                  c_void_p]),
}


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise DtbError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C descriptools_b200/csrc).  descriptools_b200 has no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.dtb_abi_version() != 1:
        raise DtbError("libdtb200.so ABI version mismatch")
    return lib


lib = _load()


def check(code: int, what: str = "") -> None:
    if code != 0:
        msg = lib.dtb_error_string(code).decode()
        detail = lib.dtb_last_cuda_error().decode()
        raise DtbError(f"{what or 'libdtb200'} failed: {msg}" + (f" [{detail}]" if detail and code == -2 else ""))


def launch_count() -> int:
    return int(lib.dtb_launch_count())


def reset_launch_count() -> None:
    lib.dtb_reset_launch_count()


def profile_enable(on: bool = True) -> None:
    lib.dtb_profile_enable(1 if on else 0)


def profile_collect() -> dict:
    """{kernel name: (total ms, launches)} since profile_enable / the last collect"""
    buf = ctypes.create_string_buffer(1 << 16)
    lib.dtb_profile_collect(buf, len(buf))
    out = {}
    for line in buf.value.decode().splitlines():
        name, ms, n = line.rsplit(" ", 2)
        out[name] = (float(ms), int(n))
    return out
