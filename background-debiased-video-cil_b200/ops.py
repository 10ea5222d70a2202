"""``torch.ops.bgdebias.*`` -- the CUDA kernels of libbgdebias_b200.so as torch.library custom ops.

PyTorch is plumbing here: it owns the device buffers and the stream; every op hands raw
pointers, sizes and the current ``cudaStream_t`` to the C ABI (include/bgdebias.h).  The ops are
registered for CUDA tensors only -- CPU tensors raise ``NotImplementedError`` -- and need the
built library (``ImportError`` otherwise).  Ops are stream-ordered and never synchronise.

    bgdebias::temporal_median(Tensor frames) -> Tensor
        frames uint8 [T, ...] -> uint8 [...]; np.median(frames, 0).astype(uint8), bit-exact
        (cil_tools/extract_background.py:73).
    bgdebias::temporal_median_varlen(Tensor frames, Tensor offsets) -> Tensor
        frames uint8 [sum T, ...], offsets int64/int32 CPU tensor [V+1] -> uint8 [V, ...]
        (what extract_background.py:102-109 does video by video).
    bgdebias::bgmix_blend(Tensor fg, Tensor bg_pool, Tensor bg_idx, Tensor top, Tensor left,
                          Tensor apply, Tensor fg_lut, Tensor bg_mean, Tensor bg_std,
                          float alpha, str layout, ScalarType? out_dtype=None) -> Tensor
        the batched form of BackgroundMixDataset._mix_background (libs/loader/comix_loader.py:138-145).
        ``layout`` "NTCHW", "NCTHW" or "NTHWC" (contiguous [B, T, H, W, 3], channels-last storage of both others);
        ``out_dtype`` float32 (None), bfloat16 or float16: the fp32 result rounded once, equal to its ``.to(out_dtype)``.
        bgmix_blend_ragged and bgmix_resize_blend take the same two arguments.
    bgdebias::bgmix_blend_ragged(Tensor fg, Tensor pool_bytes, Tensor slots, Tensor tables, <bgmix_blend arguments>) -> Tensor
        the same blend over a ragged uint8 pool (images of any sizes, or the random frames of comix_loader.py:133-136),
        with Resize(bg_resize) (comix_loader.py:72; torchvision's antialiased bilinear, bit-exact) inside the launch.
    bgdebias::resize_bilinear(Tensor src, Tensor geom, int T, int H, int W) -> Tensor
    bgdebias::bgmix_resize_blend(Tensor src, Tensor geom, int T, int H, int W, <bgmix_blend arguments>) -> Tensor
        the pipeline's Resize((W, H), keep_ratio=False) (config ..._bgmix_plus_randAug.py:136; cv2 INTER_LINEAR, bit-exact)
        on packed uint8 crops, alone or fused with the blend.
    bgdebias::ragged_pack(Tensor pool_bytes, Tensor segments, int out_bytes) -> Tensor
        one launch that gathers whole images of a ragged uint8 pool into one buffer (segments int64 [n, 3] = {source
        offset, destination offset, bytes}, 16-byte aligned): the owner side of pool.ShardedPool.fetch.
    bgdebias::ragged_gather(Tensor bases, Tensor base_bytes, Tensor segments, int out_bytes) -> Tensor
        the same one-launch gather from many sources (bases: device int64 [W] of base pointers, peer mappings included;
        segments int64 [n, 4] = {source, source offset, destination offset, bytes}): pool.PeerPool.gather.
    bgdebias::resized_crop_aa(Tensor src, Tensor desc, Tensor tables, int out_h, int out_w) -> Tensor
        RandomResizedCrop(100)(read_image(f).float()).permute(1, 2, 0) of many frames of any sizes, for host-made draws
        (cil_tools/extract_background.py:81,89-90; torchvision's antialiased bilinear, bit-exact).
"""
from __future__ import annotations

import ctypes
import math
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _cabi


def _stream_ptr(device: torch.device) -> int:
    return int(torch.cuda.current_stream(device).cuda_stream)


def _require(cond: bool, msg: str) -> None:
    if not cond:
        raise ValueError(msg)


# --------------------------------------------------------------------------- #
# temporal median
# --------------------------------------------------------------------------- #
@torch.library.custom_op("bgdebias::temporal_median", mutates_args=(), device_types="cuda")
def temporal_median(frames: torch.Tensor) -> torch.Tensor:
    _require(frames.dtype == torch.uint8, "temporal_median: frames must be uint8")
    _require(frames.dim() >= 1, "temporal_median: frames must be [T, ...]")
    T = frames.shape[0]
    _require(T > 0, "temporal_median: zero frames (the reference fails here too: median of nothing)")
    frames = frames.contiguous()
    out = torch.empty(frames.shape[1:], dtype=torch.uint8, device=frames.device)
    N = out.numel()
    with torch.cuda.device(frames.device):
        _cabi.check(_cabi.lib().bgd_temporal_median_u8(frames.data_ptr(), T, N, out.data_ptr(),
                                                       _stream_ptr(frames.device)))
    return out


@temporal_median.register_fake
def _(frames):
    return frames.new_empty(frames.shape[1:])


@torch.library.custom_op("bgdebias::temporal_median_varlen", mutates_args=(), device_types="cuda")
def temporal_median_varlen(frames: torch.Tensor, offsets: torch.Tensor) -> torch.Tensor:
    _require(frames.dtype == torch.uint8, "temporal_median_varlen: frames must be uint8")
    _require(frames.dim() >= 1, "temporal_median_varlen: frames must be [sum T, ...]")
    _require(offsets.dim() == 1 and offsets.numel() >= 1, "temporal_median_varlen: offsets must be [V+1]")
    _require(offsets.dtype in (torch.int64, torch.int32), "temporal_median_varlen: offsets must be int32/int64")
    offs = offsets.detach().to("cpu", torch.int64).contiguous()          # the planner runs on the host
    V = offs.numel() - 1
    _require(int(offs[0]) >= 0 and int(offs[-1]) <= frames.shape[0], "temporal_median_varlen: offsets out of range")
    frames = frames.contiguous()
    out = torch.empty((V,) + tuple(frames.shape[1:]), dtype=torch.uint8, device=frames.device)
    N = math.prod(frames.shape[1:])
    optr = ctypes.cast(offs.data_ptr(), ctypes.POINTER(ctypes.c_int64))
    with torch.cuda.device(frames.device):
        _cabi.check(_cabi.lib().bgd_temporal_median_varlen_u8(frames.data_ptr(), optr, V, N, out.data_ptr(),
                                                              _stream_ptr(frames.device)))
    return out


@temporal_median_varlen.register_fake
def _(frames, offsets):
    return frames.new_empty((offsets.shape[0] - 1,) + tuple(frames.shape[1:]))


# --------------------------------------------------------------------------- #
# NaN-masked temporal median / mean (sim_cam extraction, extract_background.py:91-98)
# --------------------------------------------------------------------------- #
def _nan_reduce(frames: torch.Tensor, avg_method: int, zero_is_missing: bool, as_float: bool) -> torch.Tensor:
    _require(frames.dtype == torch.float32, "nan_temporal_reduce: frames must be float32")
    _require(frames.dim() >= 1 and frames.shape[0] > 0, "nan_temporal_reduce: frames must be [T, ...] with T > 0 "
             "(the reference fails here too: nanmedian of nothing)")
    _require(avg_method in (0, 1), "nan_temporal_reduce: avg_method must be 0 (median) or 1 (mean)")
    frames = frames.contiguous()
    out = torch.empty(frames.shape[1:], dtype=torch.float32 if as_float else torch.uint8, device=frames.device)
    with torch.cuda.device(frames.device):
        _cabi.check(_cabi.lib().bgd_nan_temporal_reduce_f32(
            frames.data_ptr(), frames.shape[0], out.numel(), int(avg_method), int(bool(zero_is_missing)),
            None if as_float else out.data_ptr(), out.data_ptr() if as_float else None, _stream_ptr(frames.device)))
    return out


@torch.library.custom_op("bgdebias::nan_temporal_reduce", mutates_args=(), device_types="cuda")
def nan_temporal_reduce(frames: torch.Tensor, avg_method: int, zero_is_missing: bool) -> torch.Tensor:
    """uint8 ``[...]``: ``np.nanmedian`` / ``np.nanmean`` over axis 0, ``.astype(uint8)``."""
    return _nan_reduce(frames, avg_method, zero_is_missing, False)


@nan_temporal_reduce.register_fake
def _(frames, avg_method, zero_is_missing):
    return frames.new_empty(frames.shape[1:], dtype=torch.uint8)


@torch.library.custom_op("bgdebias::nan_temporal_reduce_varlen", mutates_args=(), device_types="cuda")
def nan_temporal_reduce_varlen(frames: torch.Tensor, offsets: torch.Tensor, avg_method: int, zero_is_missing: bool) -> torch.Tensor:
    """V frame folders concatenated along T (``offsets`` [V+1], host or device int64) -> uint8 ``[V, ...]``."""
    _require(frames.dtype == torch.float32 and frames.dim() >= 1, "nan_temporal_reduce_varlen: frames must be float32 [sum T, ...]")
    _require(offsets.dim() == 1 and offsets.numel() >= 1, "nan_temporal_reduce_varlen: offsets must be [V+1]")
    _require(avg_method in (0, 1), "nan_temporal_reduce_varlen: avg_method must be 0 (median) or 1 (mean)")
    offs = offsets.detach().to("cpu", torch.int64).contiguous()
    V = offs.numel() - 1
    _require(int(offs[0]) >= 0 and int(offs[-1]) <= frames.shape[0], "nan_temporal_reduce_varlen: offsets out of range")
    frames = frames.contiguous()
    out = torch.empty((V,) + tuple(frames.shape[1:]), dtype=torch.uint8, device=frames.device)
    optr = ctypes.cast(offs.data_ptr(), ctypes.POINTER(ctypes.c_int64))
    with torch.cuda.device(frames.device):
        _cabi.check(_cabi.lib().bgd_nan_temporal_reduce_varlen_f32(
            frames.data_ptr(), optr, V, math.prod(frames.shape[1:]), int(avg_method), int(bool(zero_is_missing)),
            out.data_ptr(), None, _stream_ptr(frames.device)))
    return out


@nan_temporal_reduce_varlen.register_fake
def _(frames, offsets, avg_method, zero_is_missing):
    return frames.new_empty((offsets.shape[0] - 1,) + tuple(frames.shape[1:]), dtype=torch.uint8)


@torch.library.custom_op("bgdebias::nan_temporal_reduce_f32", mutates_args=(), device_types="cuda")
def nan_temporal_reduce_f32(frames: torch.Tensor, avg_method: int, zero_is_missing: bool) -> torch.Tensor:
    """The float32 reduction before the uint8 cast (NaN where no frame is valid)."""
    return _nan_reduce(frames, avg_method, zero_is_missing, True)


@nan_temporal_reduce_f32.register_fake
def _(frames, avg_method, zero_is_missing):
    return frames.new_empty(frames.shape[1:])


# --------------------------------------------------------------------------- #
# RandomResizedCrop of many frames (sim_cam extraction, extract_background.py:81,89-90)
# --------------------------------------------------------------------------- #
CROP_DESC_FIELDS = ("offset", "H", "W", "top", "left", "h", "w", "xtab", "ytab", "kx", "ky")
_CROP_DESC_DTYPE = [(n, "<i8" if n == "offset" else "<i4") for n in CROP_DESC_FIELDS]     # bgd_crop_desc, 48 bytes


@torch.library.custom_op("bgdebias::resized_crop_aa", mutates_args=(), device_types="cuda")
def resized_crop_aa(src: torch.Tensor, desc: torch.Tensor, tables: torch.Tensor, out_h: int, out_w: int) -> torch.Tensor:
    """Frames planar uint8 ``[3, H, W]`` at byte offsets of the flat buffer ``src`` -> float32 ``[n, out_h, out_w, 3]``:
    frame k is ``resized_crop(frame, top, left, h, w, (out_h, out_w), antialias=True).permute(1, 2, 0)``, bit-exact.
    ``desc``: int64 ``[n, 11]`` (host or device) with the columns of :data:`CROP_DESC_FIELDS`; ``tables``: int32 weight
    tables on the device (``pool.AATables``; xtab / ytab = -1 where the crop size equals the output size)."""
    _require(src.dtype == torch.uint8 and src.dim() == 1, "resized_crop_aa: src must be a flat uint8 buffer")
    _require(desc.dim() == 2 and desc.shape[1] == len(CROP_DESC_FIELDS) and desc.dtype in (torch.int64, torch.int32),
             f"resized_crop_aa: desc must be int64 [n, {len(CROP_DESC_FIELDS)}]")
    _require(tables.dtype == torch.int32 and tables.dim() == 1, "resized_crop_aa: tables must be a flat int32 tensor")
    _require(tables.device == src.device, f"resized_crop_aa: tables must be on {src.device}")
    _require(out_h > 0 and out_w > 0, "resized_crop_aa: the output size must be positive")
    d = desc.detach().to("cpu", torch.int64).contiguous().numpy()
    _require(bool((d[:, 1:] >= -(1 << 31)).all() and (d[:, 1:] < (1 << 31)).all()), "resized_crop_aa: desc values out of int32 range")
    h_desc = np.empty(d.shape[0], dtype=_CROP_DESC_DTYPE)
    for k, name in enumerate(CROP_DESC_FIELDS):
        h_desc[name] = d[:, k]
    src, tables = src.contiguous(), tables.contiguous()
    out = torch.empty((d.shape[0], out_h, out_w, 3), dtype=torch.float32, device=src.device)
    with torch.cuda.device(src.device):
        _cabi.check(_cabi.lib().bgd_resized_crop_aa_u8_f32(src.data_ptr(), src.numel(), h_desc.ctypes.data, d.shape[0],
                                                           tables.data_ptr(), tables.numel(), out_h, out_w, out.data_ptr(),
                                                           _stream_ptr(src.device)))
    return out


@resized_crop_aa.register_fake
def _(src, desc, tables, out_h, out_w):
    return src.new_empty((desc.shape[0], out_h, out_w, 3), dtype=torch.float32)


# --------------------------------------------------------------------------- #
# batched ragged gather (owner side of pool.ShardedPool.fetch, replaces comix_loader.py:126-131 per owned image)
# --------------------------------------------------------------------------- #
@torch.library.custom_op("bgdebias::ragged_pack", mutates_args=(), device_types="cuda")
def ragged_pack(pool_bytes: torch.Tensor, segments: torch.Tensor, out_bytes: int) -> torch.Tensor:
    """uint8 ``[out_bytes]`` whose bytes ``[dst, dst + bytes)`` are ``pool_bytes[src:src + bytes]`` for every row
    ``{src, dst, bytes}`` of ``segments`` (int64 ``[n, 3]``, host or device; offsets 16-byte aligned).  Bytes outside every
    segment are left uninitialised."""
    _require(pool_bytes.dtype == torch.uint8 and pool_bytes.dim() == 1, "ragged_pack: pool_bytes must be a flat uint8 buffer")
    _require(segments.dim() == 2 and segments.shape[1] == 3 and segments.dtype in (torch.int64, torch.int32),
             "ragged_pack: segments must be int64 [n, 3]")
    _require(out_bytes >= 0, "ragged_pack: out_bytes must be >= 0")
    seg = segments.detach().to("cpu", torch.int64).contiguous()
    pool_bytes = pool_bytes.contiguous()
    out = torch.empty(out_bytes, dtype=torch.uint8, device=pool_bytes.device)
    with torch.cuda.device(pool_bytes.device):
        _cabi.check(_cabi.lib().bgd_ragged_pack_u8(pool_bytes.data_ptr(), pool_bytes.numel(),
                                                   ctypes.cast(seg.data_ptr(), ctypes.POINTER(ctypes.c_int64)), seg.shape[0],
                                                   out.data_ptr(), out_bytes, _stream_ptr(pool_bytes.device)))
    return out


@ragged_pack.register_fake
def _(pool_bytes, segments, out_bytes):
    return pool_bytes.new_empty((out_bytes,))


@torch.library.custom_op("bgdebias::ragged_gather", mutates_args=(), device_types="cuda")
def ragged_gather(bases: torch.Tensor, base_bytes: torch.Tensor, segments: torch.Tensor, out_bytes: int) -> torch.Tensor:
    """uint8 ``[out_bytes]`` whose bytes ``[dst, dst + bytes)`` are the bytes ``[src, src + bytes)`` of source ``r`` for every row
    ``{r, src, dst, bytes}`` of ``segments`` (int64 ``[n, 4]``, host or device; offsets 16-byte aligned).  ``bases``: device
    int64 ``[W]``, the 16-byte aligned base address of every source (this process's memory or a peer mapping of
    ``bgd_ipc_open``); ``base_bytes``: int64 ``[W]`` (host), the readable bytes from each base.  Every segment is checked
    against these sizes before the launch.  Bytes outside every segment are left uninitialised."""
    _require(bases.dtype == torch.int64 and bases.dim() == 1 and bases.is_cuda, "ragged_gather: bases must be device int64 [W]")
    _require(base_bytes.dim() == 1 and base_bytes.numel() == bases.numel() and not base_bytes.is_floating_point(),
             "ragged_gather: base_bytes must be int64 [W], one size per base")
    _require(segments.dim() == 2 and segments.shape[1] == 4 and segments.dtype in (torch.int64, torch.int32),
             "ragged_gather: segments must be int64 [n, 4]")
    _require(out_bytes >= 0, "ragged_gather: out_bytes must be >= 0")
    seg = segments.detach().to("cpu", torch.int64).contiguous()
    sizes = base_bytes.detach().to("cpu", torch.int64).contiguous()
    bases = bases.contiguous()
    out = torch.empty(out_bytes, dtype=torch.uint8, device=bases.device)
    i64p = ctypes.POINTER(ctypes.c_int64)
    with torch.cuda.device(bases.device):
        _cabi.check(_cabi.lib().bgd_ragged_gather_u8(bases.data_ptr(), ctypes.cast(sizes.data_ptr(), i64p), sizes.numel(),
                                                     ctypes.cast(seg.data_ptr(), i64p), seg.shape[0], out.data_ptr(), out_bytes,
                                                     _stream_ptr(bases.device)))
    return out


@ragged_gather.register_fake
def _(bases, base_bytes, segments, out_bytes):
    return bases.new_empty((out_bytes,), dtype=torch.uint8)


# --------------------------------------------------------------------------- #
# ActorCutMix blend (actor_cut_mix_loader.py:143-163)
# --------------------------------------------------------------------------- #
@torch.library.custom_op("bgdebias::actor_cut_mix", mutates_args=(), device_types="cuda")
def actor_cut_mix(actor: torch.Tensor, mask: torch.Tensor, scene: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """uint8 ``[T,H,W,3]`` x3 -> (``actor * mask + scene * (1 - mask)`` uint8, int64 scalar = sum of the mask's channel 0)."""
    for name, t in (("actor", actor), ("mask", mask), ("scene", scene)):
        _require(t.dtype == torch.uint8, f"actor_cut_mix: {name} must be uint8")
    _require(actor.shape == mask.shape == scene.shape, "actor_cut_mix: actor, mask and scene must have one shape")
    _require(actor.dim() >= 1 and actor.shape[-1] == 3, "actor_cut_mix: channel-last [..., 3] frames expected")
    actor, mask, scene = actor.contiguous(), mask.contiguous(), scene.contiguous()
    out = torch.empty_like(actor)
    total = torch.zeros((), dtype=torch.int64, device=actor.device)
    with torch.cuda.device(actor.device):
        _cabi.check(_cabi.lib().bgd_actor_cut_mix_u8(actor.data_ptr(), mask.data_ptr(), scene.data_ptr(), actor.numel(),
                                                     out.data_ptr(), total.data_ptr(), _stream_ptr(actor.device)))
    return out, total


@actor_cut_mix.register_fake
def _(actor, mask, scene):
    return torch.empty_like(actor), actor.new_empty((), dtype=torch.int64)


# --------------------------------------------------------------------------- #
# BG-mix blend
# --------------------------------------------------------------------------- #
def _host3(t: torch.Tensor, name: str):
    _require(t.numel() == 3, f"bgmix_blend: {name} must have 3 values")
    return _cabi.f32x3(t.detach().to("cpu", torch.float32).tolist())


_OUT_DTYPES = {torch.float32: _cabi.OUT_F32, torch.bfloat16: _cabi.OUT_BF16, torch.float16: _cabi.OUT_F16}


def _out_spec(name: str, layout: str, out_dtype: Optional[torch.dtype]) -> torch.dtype:
    """Validates the output arguments of the uint8-foreground blends; returns the output dtype."""
    _require(layout in _cabi.OUT_LAYOUTS, f"{name}: layout must be one of {sorted(_cabi.OUT_LAYOUTS)}")
    dt = torch.float32 if out_dtype is None else out_dtype
    _require(dt in _OUT_DTYPES, f"{name}: out_dtype must be float32, bfloat16 or float16 (got {dt})")
    return dt


def _out_shape(B: int, T: int, H: int, W: int, layout: str) -> tuple:
    return {"NTCHW": (B, T, 3, H, W), "NCTHW": (B, 3, T, H, W), "NTHWC": (B, T, H, W, 3)}[layout]


@torch.library.custom_op("bgdebias::bgmix_blend", mutates_args=(), device_types="cuda")
def bgmix_blend(fg: torch.Tensor, bg_pool: torch.Tensor, bg_idx: torch.Tensor, top: torch.Tensor,
                left: torch.Tensor, apply: torch.Tensor, fg_lut: torch.Tensor, bg_mean: torch.Tensor,
                bg_std: torch.Tensor, alpha: float, layout: str, out_dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    _require(fg.dtype == torch.uint8 and fg.dim() == 5 and fg.shape[-1] == 3,
             "bgmix_blend: fg must be uint8 [B, T, H, W, 3]")
    _require(bg_pool.dim() == 4 and bg_pool.shape[1] == 3 and bg_pool.dtype in (torch.float32, torch.uint8),
             "bgmix_blend: bg_pool must be float32 or uint8 [P, 3, Hb, Wb]")
    out_dt = _out_spec("bgmix_blend", layout, out_dtype)
    B, T, H, W, _ = fg.shape
    P, _, Hb, Wb = bg_pool.shape
    dev = fg.device
    for name, t, dt in (("bg_idx", bg_idx, torch.int32), ("top", top, torch.int32), ("left", left, torch.int32),
                        ("apply", apply, torch.uint8)):
        _require(t.dtype == dt and t.dim() == 1 and t.shape[0] == B, f"bgmix_blend: {name} must be {dt} [B]")
        _require(t.device == dev, f"bgmix_blend: {name} must be on {dev}")
    _require(fg_lut.dtype == torch.float32 and tuple(fg_lut.shape) == (3, 256) and fg_lut.device == dev,
             "bgmix_blend: fg_lut must be float32 [3, 256] on the device")
    _require(bg_pool.device == dev, "bgmix_blend: bg_pool must be on the same device as fg")
    fg, bg_pool = fg.contiguous(), bg_pool.contiguous()
    bg_idx, top, left, apply, fg_lut = (x.contiguous() for x in (bg_idx, top, left, apply, fg_lut))
    out = torch.empty(_out_shape(B, T, H, W, layout), dtype=out_dt, device=dev)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().bgd_bgmix_blend_out(
            fg.data_ptr(), B, T, H, W, bg_pool.data_ptr(), int(bg_pool.dtype == torch.uint8), P, Hb, Wb, bg_idx.data_ptr(),
            top.data_ptr(), left.data_ptr(), apply.data_ptr(), fg_lut.data_ptr(), _host3(bg_mean, "bg_mean"),
            _host3(bg_std, "bg_std"), float(alpha), _cabi.OUT_LAYOUTS[layout], _OUT_DTYPES[out_dt], out.data_ptr(),
            _stream_ptr(dev)))
    return out


@bgmix_blend.register_fake
def _(fg, bg_pool, bg_idx, top, left, apply, fg_lut, bg_mean, bg_std, alpha, layout, out_dtype=None):
    B, T, H, W, _ = fg.shape
    return fg.new_empty(_out_shape(B, T, H, W, layout), dtype=_out_spec("bgmix_blend", layout, out_dtype))


# --------------------------------------------------------------------------- #
# BG-mix over a ragged uint8 pool (pool.RaggedPool): Resize + RandomCrop + Normalize + blend in one launch
# --------------------------------------------------------------------------- #
def _check_ragged(name, B, dev, pool_bytes, slots, tables, bg_idx, top, left, apply):
    _require(pool_bytes.dtype == torch.uint8 and pool_bytes.dim() == 1, f"{name}: pool_bytes must be a flat uint8 buffer")
    _require(slots.dtype == torch.uint8 and slots.dim() == 1 and slots.numel() % 40 == 0 and slots.numel() > 0,
             f"{name}: slots must be the uint8 view of a bgd_ragged_slot table (40 bytes per image)")
    _require(tables.dtype == torch.int32 and tables.dim() == 1, f"{name}: tables must be int32")
    for nm, t, dt in (("bg_idx", bg_idx, torch.int32), ("top", top, torch.int32), ("left", left, torch.int32),
                      ("apply", apply, torch.uint8)):
        _require(t.dtype == dt and t.dim() == 1 and t.shape[0] == B and t.device == dev, f"{name}: {nm} must be {dt} [B] on {dev}")
    for nm, t in (("pool_bytes", pool_bytes), ("slots", slots), ("tables", tables)):
        _require(t.device == dev, f"{name}: {nm} must be on {dev}")
    _require(slots.data_ptr() % 8 == 0, f"{name}: slots must be 8-byte aligned")


@torch.library.custom_op("bgdebias::bgmix_blend_ragged", mutates_args=(), device_types="cuda")
def bgmix_blend_ragged(fg: torch.Tensor, pool_bytes: torch.Tensor, slots: torch.Tensor, tables: torch.Tensor,
                       bg_idx: torch.Tensor, top: torch.Tensor, left: torch.Tensor, apply: torch.Tensor,
                       fg_lut: torch.Tensor, bg_mean: torch.Tensor, bg_std: torch.Tensor, alpha: float, layout: str,
                       out_dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    _require(fg.dtype == torch.uint8 and fg.dim() == 5 and fg.shape[-1] == 3, "bgmix_blend_ragged: fg must be uint8 [B, T, H, W, 3]")
    out_dt = _out_spec("bgmix_blend_ragged", layout, out_dtype)
    B, T, H, W, _ = fg.shape
    dev = fg.device
    _check_ragged("bgmix_blend_ragged", B, dev, pool_bytes, slots, tables, bg_idx, top, left, apply)
    _require(fg_lut.dtype == torch.float32 and tuple(fg_lut.shape) == (3, 256) and fg_lut.device == dev,
             "bgmix_blend_ragged: fg_lut must be float32 [3, 256] on the device")
    fg = fg.contiguous()
    bg_idx, top, left, apply, fg_lut, pool_bytes, slots, tables = (x.contiguous() for x in (bg_idx, top, left, apply, fg_lut, pool_bytes, slots, tables))
    out = torch.empty(_out_shape(B, T, H, W, layout), dtype=out_dt, device=dev)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().bgd_bgmix_blend_ragged_out(
            fg.data_ptr(), B, T, H, W, pool_bytes.data_ptr(), slots.data_ptr(), slots.numel() // 40, tables.data_ptr(),
            bg_idx.data_ptr(), top.data_ptr(), left.data_ptr(), apply.data_ptr(), fg_lut.data_ptr(), _host3(bg_mean, "bg_mean"),
            _host3(bg_std, "bg_std"), float(alpha), _cabi.OUT_LAYOUTS[layout], _OUT_DTYPES[out_dt], out.data_ptr(), _stream_ptr(dev)))
    return out


@bgmix_blend_ragged.register_fake
def _(fg, pool_bytes, slots, tables, bg_idx, top, left, apply, fg_lut, bg_mean, bg_std, alpha, layout, out_dtype=None):
    B, T, H, W, _ = fg.shape
    return fg.new_empty(_out_shape(B, T, H, W, layout), dtype=_out_spec("bgmix_blend_ragged", layout, out_dtype))


@torch.library.custom_op("bgdebias::bgmix_blend_ragged_normfg", mutates_args=(), device_types="cuda")
def bgmix_blend_ragged_normfg(fg_norm: torch.Tensor, pool_bytes: torch.Tensor, slots: torch.Tensor, tables: torch.Tensor,
                              bg_idx: torch.Tensor, top: torch.Tensor, left: torch.Tensor, apply: torch.Tensor,
                              bg_mean: torch.Tensor, bg_std: torch.Tensor, alpha: float, layout: str) -> torch.Tensor:
    """Ragged-pool blend for a foreground that is already normalised (fp32 ``[B, T, 3, H, W]``)."""
    _require(fg_norm.dtype == torch.float32 and fg_norm.dim() == 5 and fg_norm.shape[2] == 3,
             "bgmix_blend_ragged_normfg: fg_norm must be float32 [B, T, 3, H, W]")
    _require(layout in _cabi.LAYOUTS, f"bgmix_blend_ragged_normfg: layout must be one of {sorted(_cabi.LAYOUTS)}")
    B, T, _, H, W = fg_norm.shape
    dev = fg_norm.device
    _check_ragged("bgmix_blend_ragged_normfg", B, dev, pool_bytes, slots, tables, bg_idx, top, left, apply)
    fg_norm = fg_norm.contiguous()
    bg_idx, top, left, apply, pool_bytes, slots, tables = (x.contiguous() for x in (bg_idx, top, left, apply, pool_bytes, slots, tables))
    out = torch.empty((B, T, 3, H, W) if layout == "NTCHW" else (B, 3, T, H, W), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().bgd_bgmix_blend_ragged_normfg_f32(
            fg_norm.data_ptr(), B, T, H, W, pool_bytes.data_ptr(), slots.data_ptr(), slots.numel() // 40, tables.data_ptr(),
            bg_idx.data_ptr(), top.data_ptr(), left.data_ptr(), apply.data_ptr(), _host3(bg_mean, "bg_mean"),
            _host3(bg_std, "bg_std"), float(alpha), _cabi.LAYOUTS[layout], out.data_ptr(), _stream_ptr(dev)))
    return out


@bgmix_blend_ragged_normfg.register_fake
def _(fg_norm, pool_bytes, slots, tables, bg_idx, top, left, apply, bg_mean, bg_std, alpha, layout):
    B, T, _, H, W = fg_norm.shape
    return fg_norm.new_empty((B, T, 3, H, W) if layout == "NTCHW" else (B, 3, T, H, W))


# --------------------------------------------------------------------------- #
# foreground pipeline tail: Resize (cv2 INTER_LINEAR, bit-exact) [-> Normalize -> FormatShape -> blend]
# --------------------------------------------------------------------------- #
def pack_clips(clips, pin: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
    """Host helper: uint8 clips ``[T, h_i, w_i, 3]`` of different crop sizes -> (flat uint8 buffer, int64 ``[B, 5]`` geometry
    ``{offset, h, w, row stride, frame stride}``) in the form ``resize_bilinear`` / ``bgmix_resize_blend`` take.  Pure CPU."""
    clips = [torch.as_tensor(c) for c in clips]
    T = clips[0].shape[0] if clips else 0
    geom = torch.empty((len(clips), 5), dtype=torch.int64)
    total = 0
    for i, c in enumerate(clips):
        _require(c.dtype == torch.uint8 and c.dim() == 4 and c.shape[3] == 3, "pack_clips: clips must be uint8 [T, h, w, 3]")
        _require(c.shape[0] == T, "pack_clips: every clip needs the same number of frames")
        h, w = int(c.shape[1]), int(c.shape[2])
        geom[i] = torch.tensor([total, h, w, w * 3, h * w * 3])
        total += T * h * w * 3
    size = total + 4 + (-total) % 4                       # 32-bit loads: multiple of 4, slack for one-column crops
    buf = torch.zeros(size, dtype=torch.uint8, pin_memory=pin)
    for i, c in enumerate(clips):
        o = int(geom[i, 0])
        buf[o:o + c.numel()] = c.reshape(-1)
    return buf, geom


def _check_packed(name: str, src: torch.Tensor, geom: torch.Tensor):
    _require(src.dtype == torch.uint8 and src.dim() == 1, f"{name}: src must be a flat uint8 buffer")
    _require(geom.dim() == 2 and geom.shape[1] == 5, f"{name}: geom must be int64 [B, 5]")
    _require(src.numel() % 4 == 0, f"{name}: src must be a multiple of 4 bytes long (ops.pack_clips pads)")
    g = geom.detach().to("cpu", torch.int64).contiguous()
    return src.contiguous(), g, ctypes.cast(g.data_ptr(), ctypes.POINTER(ctypes.c_int64))


@torch.library.custom_op("bgdebias::resize_bilinear", mutates_args=(), device_types="cuda")
def resize_bilinear(src: torch.Tensor, geom: torch.Tensor, T: int, H: int, W: int) -> torch.Tensor:
    """Packed uint8 crops (see :func:`pack_clips`) -> uint8 ``[B, T, H, W, 3]``; every frame equals
    ``cv2.resize(frame, (W, H), interpolation=cv2.INTER_LINEAR)``, the arithmetic of mmaction's ``Resize``."""
    src, g, gptr = _check_packed("resize_bilinear", src, geom)
    out = torch.empty((g.shape[0], T, H, W, 3), dtype=torch.uint8, device=src.device)
    with torch.cuda.device(src.device):
        _cabi.check(_cabi.lib().bgd_resize_bilinear_u8(src.data_ptr(), src.numel(), gptr, g.shape[0], T, H, W, out.data_ptr(),
                                                       _stream_ptr(src.device)))
    return out


@resize_bilinear.register_fake
def _(src, geom, T, H, W):
    return src.new_empty((geom.shape[0], T, H, W, 3))


@torch.library.custom_op("bgdebias::bgmix_resize_blend", mutates_args=(), device_types="cuda")
def bgmix_resize_blend(src: torch.Tensor, geom: torch.Tensor, T: int, H: int, W: int, bg_pool: torch.Tensor,
                       bg_idx: torch.Tensor, top: torch.Tensor, left: torch.Tensor, apply: torch.Tensor, fg_lut: torch.Tensor,
                       bg_mean: torch.Tensor, bg_std: torch.Tensor, alpha: float, layout: str,
                       out_dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """``bgmix_blend(resize_bilinear(src, geom, T, H, W), ...)`` in one launch (the resized uint8 batch never exists)."""
    src, g, gptr = _check_packed("bgmix_resize_blend", src, geom)
    B = g.shape[0]
    _require(bg_pool.dim() == 4 and bg_pool.shape[1] == 3 and bg_pool.dtype in (torch.float32, torch.uint8),
             "bgmix_resize_blend: bg_pool must be float32 or uint8 [P, 3, Hb, Wb]")
    out_dt = _out_spec("bgmix_resize_blend", layout, out_dtype)
    P, _, Hb, Wb = bg_pool.shape
    dev = src.device
    for name, t, dt in (("bg_idx", bg_idx, torch.int32), ("top", top, torch.int32), ("left", left, torch.int32),
                        ("apply", apply, torch.uint8)):
        _require(t.dtype == dt and t.dim() == 1 and t.shape[0] == B and t.device == dev,
                 f"bgmix_resize_blend: {name} must be {dt} [B] on {dev}")
    _require(fg_lut.dtype == torch.float32 and tuple(fg_lut.shape) == (3, 256) and fg_lut.device == dev,
             "bgmix_resize_blend: fg_lut must be float32 [3, 256] on the device")
    _require(bg_pool.device == dev, "bgmix_resize_blend: bg_pool must be on the same device as src")
    bg_pool = bg_pool.contiguous()
    bg_idx, top, left, apply, fg_lut = (x.contiguous() for x in (bg_idx, top, left, apply, fg_lut))
    out = torch.empty(_out_shape(B, T, H, W, layout), dtype=out_dt, device=dev)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().bgd_bgmix_resize_blend_out(
            src.data_ptr(), src.numel(), gptr, B, T, H, W, bg_pool.data_ptr(), int(bg_pool.dtype == torch.uint8), P, Hb, Wb,
            bg_idx.data_ptr(), top.data_ptr(), left.data_ptr(), apply.data_ptr(), fg_lut.data_ptr(), _host3(bg_mean, "bg_mean"),
            _host3(bg_std, "bg_std"), float(alpha), _cabi.OUT_LAYOUTS[layout], _OUT_DTYPES[out_dt], out.data_ptr(), _stream_ptr(dev)))
    return out


@bgmix_resize_blend.register_fake
def _(src, geom, T, H, W, bg_pool, bg_idx, top, left, apply, fg_lut, bg_mean, bg_std, alpha, layout, out_dtype=None):
    B = geom.shape[0]
    return src.new_empty(_out_shape(B, T, H, W, layout), dtype=_out_spec("bgmix_resize_blend", layout, out_dtype))


# --------------------------------------------------------------------------- #
# host-side table for the foreground normalisation
# --------------------------------------------------------------------------- #
def make_fg_lut(mean: Sequence[float], std: Sequence[float], device=None) -> torch.Tensor:
    """[3, 256] fp32 table of mmaction ``Normalize`` (mmcv.imnormalize_) outputs per uint8 level.

    mmcv evaluates ``cv2.subtract(img_f32, float64(mean)); cv2.multiply(img_f32, 1/float64(std))``,
    i.e. ``f32(f64(f32(x) - f32(mean)) * (1 / f64(std)))``: an fp32 subtract, then a multiply whose
    scale is a double.  Built once per (mean, std) on the host in exactly that precision.
    """
    mean64 = torch.tensor([float(m) for m in mean], dtype=torch.float64)
    std64 = torch.tensor([float(s) for s in std], dtype=torch.float64)
    x = torch.arange(256, dtype=torch.float32)
    d32 = x[None, :] - mean64.to(torch.float32)[:, None]
    lut = (d32.to(torch.float64) * (1.0 / std64)[:, None]).to(torch.float32)
    return lut.to(device) if device is not None else lut


@torch.library.custom_op("bgdebias::bgmix_blend_normfg", mutates_args=(), device_types="cuda")
def bgmix_blend_normfg(fg_norm: torch.Tensor, bg_pool: torch.Tensor, bg_idx: torch.Tensor, top: torch.Tensor,
                       left: torch.Tensor, apply: torch.Tensor, bg_mean: torch.Tensor, bg_std: torch.Tensor,
                       alpha: float, layout: str) -> torch.Tensor:
    """Blend for a foreground that is already normalised: fp32 [B, T, 3, H, W] (the ``imgs`` the
    reference's pipeline produces, libs/loader/comix_loader.py:142)."""
    _require(fg_norm.dtype == torch.float32 and fg_norm.dim() == 5 and fg_norm.shape[2] == 3,
             "bgmix_blend_normfg: fg_norm must be float32 [B, T, 3, H, W]")
    _require(bg_pool.dim() == 4 and bg_pool.shape[1] == 3 and bg_pool.dtype in (torch.float32, torch.uint8),
             "bgmix_blend_normfg: bg_pool must be float32 or uint8 [P, 3, Hb, Wb]")
    _require(layout in _cabi.LAYOUTS, f"bgmix_blend_normfg: layout must be one of {sorted(_cabi.LAYOUTS)}")
    B, T, _, H, W = fg_norm.shape
    P, _, Hb, Wb = bg_pool.shape
    dev = fg_norm.device
    for name, t, dt in (("bg_idx", bg_idx, torch.int32), ("top", top, torch.int32), ("left", left, torch.int32),
                        ("apply", apply, torch.uint8)):
        _require(t.dtype == dt and t.dim() == 1 and t.shape[0] == B and t.device == dev,
                 f"bgmix_blend_normfg: {name} must be {dt} [B] on {dev}")
    _require(bg_pool.device == dev, "bgmix_blend_normfg: bg_pool must be on the same device as fg_norm")
    fg_norm, bg_pool = fg_norm.contiguous(), bg_pool.contiguous()
    bg_idx, top, left, apply = (x.contiguous() for x in (bg_idx, top, left, apply))
    shape = (B, T, 3, H, W) if layout == "NTCHW" else (B, 3, T, H, W)
    out = torch.empty(shape, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().bgd_bgmix_blend_normfg_f32(
            fg_norm.data_ptr(), B, T, H, W, bg_pool.data_ptr(), int(bg_pool.dtype == torch.uint8), P, Hb, Wb,
            bg_idx.data_ptr(), top.data_ptr(), left.data_ptr(), apply.data_ptr(), _host3(bg_mean, "bg_mean"),
            _host3(bg_std, "bg_std"), float(alpha), _cabi.LAYOUTS[layout], out.data_ptr(), _stream_ptr(dev)))
    return out


@bgmix_blend_normfg.register_fake
def _(fg_norm, bg_pool, bg_idx, top, left, apply, bg_mean, bg_std, alpha, layout):
    B, T, _, H, W = fg_norm.shape
    shape = (B, T, 3, H, W) if layout == "NTCHW" else (B, 3, T, H, W)
    return fg_norm.new_empty(shape)
