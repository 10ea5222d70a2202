"""ctypes binding of libbgdebias_b200.so -- one entry per symbol of include/bgdebias.h.

The library is loaded on first use and the load fails loudly: a missing or unloadable .so is an
error, never a reason to compute on the CPU.
"""
from __future__ import annotations

import ctypes
import os
import pathlib
import threading

_PKG = pathlib.Path(__file__).resolve().parent
LIB_PATH = _PKG / "libbgdebias_b200.so"

BGD_OK, BGD_ERR_INVALID, BGD_ERR_CUDA, BGD_ERR_UNSUPPORTED, BGD_ERR_NO_DEVICE = range(5)
LAYOUT_NTCHW, LAYOUT_NCTHW = 0, 1
MEDIAN_AUTO, MEDIAN_SWAR, MEDIAN_BITSLICED, MEDIAN_COLPLANE, MEDIAN_LDSM = 0, 1, 2, 3, 4
LAYOUTS = {"NTCHW": LAYOUT_NTCHW, "NCTHW": LAYOUT_NCTHW}
LAYOUT_NTHWC = 2
OUT_LAYOUTS = {**LAYOUTS, "NTHWC": LAYOUT_NTHWC}        # layouts of the *_out blend entry points
OUT_F32, OUT_BF16, OUT_F16 = 0, 1, 2

_c = ctypes
_f32p, _i64p = _c.POINTER(_c.c_float), _c.POINTER(_c.c_int64)
_vp = _c.c_void_p
_blend_common = [_vp, _c.c_int64, _c.c_int64, _c.c_int64, _c.c_int64,       # fg, B, T, H, W
                 _vp, _c.c_int64, _c.c_int64, _c.c_int64,                   # pool, P, Hb, Wb
                 _vp, _vp, _vp, _vp, _vp,                                   # bg_idx, top, left, apply, lut
                 _f32p, _f32p, _c.c_double, _c.c_int, _vp]                  # mean, std, alpha, layout, out

class RaggedSlot(_c.Structure):
    """``bgd_ragged_slot`` of include/bgdebias.h (40 bytes)."""
    _fields_ = [("offset", _c.c_int64), ("h", _c.c_int32), ("w", _c.c_int32), ("Hb", _c.c_int32), ("Wb", _c.c_int32),
                ("xtab", _c.c_int32), ("ytab", _c.c_int32), ("kx", _c.c_int32), ("ky", _c.c_int32)]


class CropDesc(_c.Structure):
    """``bgd_crop_desc`` of include/bgdebias.h (48 bytes)."""
    _fields_ = [("offset", _c.c_int64), ("H", _c.c_int32), ("W", _c.c_int32), ("top", _c.c_int32), ("left", _c.c_int32),
                ("h", _c.c_int32), ("w", _c.c_int32), ("xtab", _c.c_int32), ("ytab", _c.c_int32), ("kx", _c.c_int32),
                ("ky", _c.c_int32)]


_ragged_common = [_c.c_int64, _c.c_int64, _c.c_int64, _c.c_int64,            # B, T, H, W
                  _vp, _vp, _c.c_int64, _vp,                                 # pool, slots, P, tables
                  _vp, _vp, _vp, _vp]                                        # bg_idx, top, left, apply

# name -> (restype, argtypes): the declarations of include/bgdebias.h, in header order
SIGNATURES = {
    "bgd_abi_version": (_c.c_int, []),
    "bgd_last_error": (_c.c_char_p, []),
    "bgd_device_info": (_c.c_int, [_c.c_int, _c.POINTER(_c.c_int), _c.POINTER(_c.c_int), _c.POINTER(_c.c_int),
                                   _i64p, _i64p]),
    "bgd_kernel_launch_count": (_c.c_int64, []),
    "bgd_median_set_variant": (_c.c_int, [_c.c_int]),
    "bgd_median_get_variant": (_c.c_int, []),
    "bgd_temporal_median_u8": (_c.c_int, [_vp, _c.c_int64, _c.c_int64, _vp, _vp]),
    "bgd_temporal_median_varlen_u8": (_c.c_int, [_vp, _i64p, _c.c_int64, _c.c_int64, _vp, _vp]),
    "bgd_temporal_median_u8_host": (_c.c_int, [_c.POINTER(_vp), _c.c_int64, _c.c_int64, _vp, _c.c_int]),
    "bgd_temporal_median_varlen_u8_host": (_c.c_int, [_vp, _i64p, _c.c_int64, _c.c_int64, _vp, _c.c_int]),
    "bgd_nan_temporal_reduce_f32": (_c.c_int, [_vp, _c.c_int64, _c.c_int64, _c.c_int, _c.c_int, _vp, _vp, _vp]),
    "bgd_nan_temporal_reduce_varlen_f32": (_c.c_int, [_vp, _i64p, _c.c_int64, _c.c_int64, _c.c_int, _c.c_int, _vp, _vp, _vp]),
    "bgd_actor_cut_mix_u8": (_c.c_int, [_vp, _vp, _vp, _c.c_int64, _vp, _vp, _vp]),
    "bgd_bgmix_blend_f32": (_c.c_int, _blend_common + [_vp]),
    "bgd_bgmix_blend_out": (_c.c_int, [_vp, _c.c_int64, _c.c_int64, _c.c_int64, _c.c_int64,
                                       _vp, _c.c_int, _c.c_int64, _c.c_int64, _c.c_int64,
                                       _vp, _vp, _vp, _vp, _vp, _f32p, _f32p, _c.c_double, _c.c_int, _c.c_int, _vp, _vp]),
    "bgd_bgmix_blend_normfg_f32": (_c.c_int, [_vp, _c.c_int64, _c.c_int64, _c.c_int64, _c.c_int64,
                                              _vp, _c.c_int, _c.c_int64, _c.c_int64, _c.c_int64,
                                              _vp, _vp, _vp, _vp, _f32p, _f32p, _c.c_double, _c.c_int, _vp, _vp]),
    "bgd_bgmix_blend_f32_host": (_c.c_int, _blend_common + [_c.POINTER(_c.c_double), _c.c_int]),
    "bgd_aa_resize_table": (_c.c_int, [_c.c_int64, _c.c_int64, _c.POINTER(_c.c_int32), _vp, _c.c_int64]),
    "bgd_aa_resize_u8_f32": (_c.c_int, [_vp, _c.POINTER(RaggedSlot), _vp, _vp, _vp]),
    "bgd_bgmix_blend_ragged_f32": (_c.c_int, [_vp] + _ragged_common + [_vp, _f32p, _f32p, _c.c_double, _c.c_int, _vp, _vp]),
    "bgd_bgmix_blend_ragged_out": (_c.c_int, [_vp] + _ragged_common + [_vp, _f32p, _f32p, _c.c_double, _c.c_int, _c.c_int,
                                                                       _vp, _vp]),
    "bgd_resized_crop_aa_u8_f32": (_c.c_int, [_vp, _c.c_int64, _vp, _c.c_int64, _vp, _c.c_int64, _c.c_int64, _c.c_int64,
                                              _vp, _vp]),
    "bgd_resize_bilinear_u8": (_c.c_int, [_vp, _c.c_int64, _i64p, _c.c_int64, _c.c_int64, _c.c_int64, _c.c_int64, _vp, _vp]),
    "bgd_bgmix_resize_blend_f32_host": (_c.c_int, [_vp, _c.c_int64, _i64p, _c.c_int64, _c.c_int64, _c.c_int64, _c.c_int64,
                                                   _vp, _c.c_int64, _c.c_int64, _c.c_int64, _vp, _vp, _vp, _vp, _vp,
                                                   _f32p, _f32p, _c.c_double, _c.c_int, _vp, _c.POINTER(_c.c_double), _c.c_int]),
    "bgd_bgmix_resize_blend_f32": (_c.c_int, [_vp, _c.c_int64, _i64p, _c.c_int64, _c.c_int64, _c.c_int64, _c.c_int64,
                                              _vp, _c.c_int, _c.c_int64, _c.c_int64, _c.c_int64,
                                              _vp, _vp, _vp, _vp, _vp, _f32p, _f32p, _c.c_double, _c.c_int, _vp, _vp]),
    "bgd_bgmix_resize_blend_out": (_c.c_int, [_vp, _c.c_int64, _i64p, _c.c_int64, _c.c_int64, _c.c_int64, _c.c_int64,
                                              _vp, _c.c_int, _c.c_int64, _c.c_int64, _c.c_int64,
                                              _vp, _vp, _vp, _vp, _vp, _f32p, _f32p, _c.c_double, _c.c_int, _c.c_int, _vp,
                                              _vp]),
    "bgd_resize_bilinear_cols_u8": (_c.c_int, [_vp, _c.c_int64, _i64p, _c.c_int, _c.c_int64, _c.c_int64, _c.c_int64, _c.c_int64,
                                               _vp, _vp]),
    "bgd_bgmix_resize_blend_cols_out": (_c.c_int, [_vp, _c.c_int64, _i64p, _c.c_int, _c.c_int64, _c.c_int64, _c.c_int64,
                                                   _c.c_int64, _vp, _c.c_int, _c.c_int64, _c.c_int64, _c.c_int64,
                                                   _vp, _vp, _vp, _vp, _vp, _f32p, _f32p, _c.c_double, _c.c_int, _c.c_int,
                                                   _vp, _vp]),
    "bgd_resize_crop_normalize_out": (_c.c_int, [_vp, _c.c_int64, _i64p, _c.c_int64, _c.c_int64, _c.c_int64, _c.c_int64,
                                                 _vp, _c.c_int, _c.c_int, _vp, _vp]),
    "bgd_ragged_pack_u8": (_c.c_int, [_vp, _c.c_int64, _i64p, _c.c_int64, _vp, _c.c_int64, _vp]),
    "bgd_ragged_gather_u8": (_c.c_int, [_vp, _i64p, _c.c_int64, _i64p, _c.c_int64, _vp, _c.c_int64, _vp]),
    "bgd_ipc_export": (_c.c_int, [_vp, _c.c_char_p, _i64p]),
    "bgd_ipc_open": (_c.c_int, [_c.c_char_p, _c.c_int, _c.POINTER(_vp)]),
    "bgd_ipc_close": (_c.c_int, [_vp]),
}

_lib = None
_lock = threading.Lock()


class BgdError(RuntimeError):
    """A non-zero bgd_status other than BGD_ERR_INVALID (which maps to ValueError)."""

    def __init__(self, status: int, message: str):
        super().__init__(f"libbgdebias_b200: {message} (status {status})")
        self.status = status


def lib() -> ctypes.CDLL:
    """Load (once) and return the library; raises if it is absent -- there is no fallback."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                path = pathlib.Path(os.environ.get("BGD_LIB_PATH", LIB_PATH))
                if not path.exists():
                    raise ImportError(
                        f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(nvcc, sm_100a).  bgdebias_b200 has no CPU fallback.")
                L = ctypes.CDLL(str(path))
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(L, name)           # AttributeError if the .so lacks a declared symbol
                    fn.restype, fn.argtypes = res, args
                if L.bgd_abi_version() != 1:
                    raise ImportError("libbgdebias_b200.so ABI version mismatch")
                _lib = L
    return _lib


def check(status: int) -> None:
    if status != BGD_OK:
        msg = lib().bgd_last_error().decode("utf-8", "replace")
        if status == BGD_ERR_INVALID:
            raise ValueError(f"libbgdebias_b200: {msg}")
        raise BgdError(status, msg)


def device_info(device: int = 0) -> dict:
    sm, ma, mi = _c.c_int(), _c.c_int(), _c.c_int()
    smem, mem = _c.c_int64(), _c.c_int64()
    check(lib().bgd_device_info(device, sm, ma, mi, smem, mem))
    return dict(sm_count=sm.value, cc=(ma.value, mi.value), smem_optin=smem.value, total_mem=mem.value)


def kernel_launch_count() -> int:
    return int(lib().bgd_kernel_launch_count())


def set_median_variant(variant: int) -> None:
    check(lib().bgd_median_set_variant(int(variant)))


def get_median_variant() -> int:
    return int(lib().bgd_median_get_variant())


def f32x3(values):
    vals = [float(v) for v in values]
    if len(vals) != 3:
        raise ValueError("expected 3 per-channel values")
    return (_c.c_float * 3)(*vals)


def i64_array(values):
    vals = [int(v) for v in values]
    return (_c.c_int64 * len(vals))(*vals)
