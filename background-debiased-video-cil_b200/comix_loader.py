"""Drop-in for ``libs/loader/comix_loader.py`` of the reference: ``BackgroundMixDataset`` (same
constructor kwargs, attributes, methods and returned dict), a ``BackgroundMix`` pipeline transform,
and the batch-level GPU blend the B200 path is built around.

What runs where
---------------
* RNG draws, gating, pool bookkeeping: host, in exactly the reference's order
  (``random.random()`` gate -> ``torch.randint(len(bg_files))`` -> RandomCrop's top then left).
* Pixels: ``torch.ops.bgdebias.bgmix_blend`` / ``bgmix_blend_normfg`` (CUDA).  No CPU blend exists.

Two ways to use the dataset
---------------------------
``device_mix=False`` (default, the reference's contract): ``prepare_train_frames`` returns
``imgs`` fp32 ``[T,3,H,W]`` already blended, ``bg_idx`` as in the reference.  ``imgs`` from the
pipeline (already normalised, comix_loader.py:107) is moved to the GPU, blended there and returned
on its original device.  Works with ``num_workers=0`` or CUDA-capable workers.

``device_mix=True`` (the fast path): the pipeline stops before ``Normalize`` and yields uint8 frames
``[T,H,W,3]``; ``prepare_train_frames`` only draws the parameters (``bg_idx``, ``bg_top``,
``bg_left``, ``bg_apply``) and ``BackgroundMixDataset.gpu_collate`` / ``mix_batch_on_device`` turns a
collated uint8 batch into the fp32 training tensor ``[B,T,3,H,W]`` with one kernel launch.  With DataLoader
worker processes use ``collate_fn=dataset.host_collate`` (host tensors only, safe after ``fork``) and call
``dataset.device_finish(batch)`` in the training process: the batch crosses PCIe as uint8, a quarter of the
reference's fp32 bytes.  The pipeline may also stop before its last ``Resize((224, 224), keep_ratio=False)``: crops of
mixed sizes are packed by ``host_collate`` and resized (cv2 INTER_LINEAR, bit for bit) inside the blend launch.
``device_finish(batch, dtype=torch.bfloat16, memory_format=torch.channels_last)`` hands a bf16-autocast model its input
directly: the blend's fp32 result rounded once to bf16, stored channels-last by the same launch.

Evaluation datasets (``test_mode=True``: val, test, the herding feature pass, the NME class means) never mix.  With
``device_mix=True`` their pipeline stops after ``RawFrameDecode`` and ``device_test_pipeline`` takes the steps it no longer
runs -- ``Resize(scale=(-1, S))``, ``CenterCrop`` or ``ThreeCrop``, ``Normalize`` and ``FormatShape('NCHW')``, see
:class:`EvalPipeline` -- which ``device_finish`` runs on the native-size uint8 frames in one launch.

Training datasets without a host-only step between decode and crop (no ``RandAugment``) can stop after ``RawFrameDecode``
as well: ``device_train_pipeline`` takes ``Resize(scale=(-1, S))``, ``MultiScaleCrop``, the final ``Resize``,
``Normalize`` and ``FormatShape('NCHW')`` (see :class:`TrainPipeline`); the worker draws the crop where MultiScaleCrop
would, and ``device_finish`` runs both resizes inside the blend launch.
"""
from __future__ import annotations

import os
import os.path as osp
import pathlib
import random
from concurrent.futures import ThreadPoolExecutor
from typing import Callable, List, Optional, Sequence

import numpy as np
import torch

from . import ops
from .pool import (AATables, BackgroundPool, BackgroundStore, PeerPool, RaggedPool, ShardedPool, resize_like_reference,
                   resized_hw)

try:  # mmaction is optional: register into its registries when it is importable
    from mmaction.datasets import RawframeDataset as _MMRawframeDataset
    from mmaction.datasets.builder import DATASETS as _DATASETS, PIPELINES as _PIPELINES
    _HAVE_MMACTION = True
except Exception:  # pragma: no cover - depends on the environment
    _MMRawframeDataset, _DATASETS, _PIPELINES, _HAVE_MMACTION = None, None, None, False


def _register(registry):
    def deco(cls):
        if registry is not None:
            try:
                registry.register_module()(cls)
            except Exception:
                pass
        return cls
    return deco


class _RawframeBase:
    """Minimal stand-in for ``mmaction.datasets.RawframeDataset`` when mmaction is absent.

    ``ann_file``: a list of dicts (``frame_dir``, ``total_frames``, ``label``) or a text file with
    ``<frame_dir> <total_frames> <label>`` per line (mmaction's rawframe annotation format).
    ``pipeline``: a callable ``dict -> dict`` or a list of such callables.
    """

    def __init__(self, ann_file, pipeline, data_prefix=None, test_mode=False, filename_tmpl='img_{:05}.jpg',
                 with_offset=False, multi_class=False, num_classes=None, start_index=1, modality='RGB',
                 sample_by_class=False, power=0., dynamic_length=False, **kwargs):
        self.ann_file = ann_file
        self.data_prefix = osp.realpath(data_prefix) if data_prefix is not None and osp.isdir(data_prefix) else data_prefix
        self.test_mode = test_mode
        self.filename_tmpl = filename_tmpl
        self.start_index = start_index
        self.modality = modality
        if callable(pipeline):
            self.pipeline = pipeline
        else:
            steps = list(pipeline)
            if any(isinstance(s, dict) for s in steps):
                raise TypeError("dict pipeline configs need mmaction; pass callables instead")

            def _compose(results, _steps=steps):
                for s in _steps:
                    results = s(results)
                    if results is None:
                        return None
                return results
            self.pipeline = _compose
        self.video_infos = self.load_annotations()

    def load_annotations(self):
        if isinstance(self.ann_file, (list, tuple)):
            return [dict(v) for v in self.ann_file]
        infos = []
        with open(self.ann_file) as f:
            for line in f:
                parts = line.split()
                if not parts:
                    continue
                frame_dir = parts[0]
                if self.data_prefix is not None:
                    frame_dir = osp.join(self.data_prefix, frame_dir)
                infos.append(dict(frame_dir=frame_dir, total_frames=int(parts[1]), label=int(parts[2])))
        return infos

    def __len__(self):
        return len(self.video_infos)

    def prepare_train_frames(self, idx):
        import copy
        results = copy.deepcopy(self.video_infos[idx])
        results['filename_tmpl'] = self.filename_tmpl
        results['modality'] = self.modality
        results['start_index'] = self.start_index
        return self.pipeline(results)

    def prepare_test_frames(self, idx):
        # the pipeline alone, as mmaction's RawframeDataset.prepare_test_frames: never a subclass's training-time mix
        return _RawframeBase.prepare_train_frames(self, idx)

    def __getitem__(self, idx):
        return self.prepare_test_frames(idx) if self.test_mode else self.prepare_train_frames(idx)


_Base = _MMRawframeDataset if _HAVE_MMACTION else _RawframeBase


def _read_image(path: str, reader: Optional[Callable] = None) -> torch.Tensor:
    """``reader(path)``, or ``torchvision.io.read_image(mode=RGB)`` as the reference decodes a background (comix_loader.py:130)."""
    if reader is not None:
        return torch.as_tensor(reader(path))
    from torchvision.io import ImageReadMode, read_image
    return read_image(path, mode=ImageReadMode.RGB)


def _blend_clip(imgs: torch.Tensor, bg: torch.Tensor, top: int, left: int, mean, std, alpha: float, device) -> torch.Tensor:
    """One normalised clip fp32 ``[T,3,H,W]`` blended on ``device`` with the crop at (top, left) of one resized background
    ``[3,Hb,Wb]`` (comix_loader.py:138-145); returned on the clip's device."""
    i32 = lambda v: torch.tensor([v], dtype=torch.int32, device=device)   # noqa: E731
    out = torch.ops.bgdebias.bgmix_blend_normfg(
        imgs.to(device, torch.float32).unsqueeze(0), bg.unsqueeze(0).to(device), i32(0), i32(top), i32(left),
        torch.ones(1, dtype=torch.uint8, device=device), torch.tensor(mean), torch.tensor(std), float(alpha), "NTCHW")[0]
    return out.to(imgs.device)


def draw_crop(h: int, w: int, crop) -> tuple:
    """``RandomCrop.get_params`` (torchvision): nothing drawn when the image already has the crop
    size, else top then left from torch's global generator."""
    th, tw = crop
    if h < th or w < tw:
        raise ValueError(f"Required crop size {(th, tw)} is larger than input image size {(h, w)}")
    if w == tw and h == th:
        return 0, 0
    top = int(torch.randint(0, h - th + 1, size=(1,)).item())
    left = int(torch.randint(0, w - tw + 1, size=(1,)).item())
    return top, left


def _steps_in_order(who: str, steps: Sequence[dict], expected: tuple) -> List[dict]:
    """The step dicts, checked to be of the ``expected`` types (a tuple of alternatives per position), in that order."""
    steps = [dict(s) for s in steps]
    for i, step in enumerate(steps):
        if i >= len(expected) or step.get('type') not in expected[i]:
            raise ValueError(f"{who}: step {i}, {step.get('type')!r}, has no device form (expected "
                             f"{', '.join(' or '.join(e) for e in expected)}, in this order)")
    if len(steps) < len(expected):
        raise ValueError(f"{who}: the {' or '.join(expected[len(steps)])} step is missing")
    return steps


def _only(step: dict, **allowed) -> None:
    """Keys other than ``type`` must be in ``allowed``; those with a non-None value there must equal it."""
    for k, v in step.items():
        if k == 'type':
            continue
        if k not in allowed or (allowed[k] is not None and v != allowed[k]):
            raise ValueError(f"{step['type']}: {k}={v!r} has no device form")


def _short_side(resize: dict) -> int:
    """S of a ``Resize(scale=(-1, S))`` (or ``(S, -1)``) step, keep_ratio and bilinear."""
    _only(resize, scale=None, keep_ratio=True, interpolation='bilinear', lazy=False)
    scale = resize.get('scale')
    if not (isinstance(scale, (tuple, list)) and len(scale) == 2 and min(scale) == -1 and max(scale) > 0
            and all(isinstance(v, int) for v in scale)):
        raise ValueError(f"Resize: only scale=(-1, S) or (S, -1) has a device form (got scale={scale!r})")
    return int(max(scale))


def rescale_short_side(h: int, w: int, short_side: int) -> tuple:
    """``(Hr, Wr)`` of mmaction's ``Resize(scale=(-1, S))`` for an ``h x w`` frame: ``mmcv.rescale_size((w, h), (inf, S))``,
    ``f = S / min(h, w)``, ``(int(w * f + 0.5), int(h * f + 0.5))``."""
    f = short_side / min(h, w)
    return int(h * f + 0.5), int(w * f + 0.5)


def _size_hw(step: dict, key: str) -> tuple:
    """``(h, w)`` of a size given as an int or mmaction's ``(w, h)`` pair."""
    v = step.get(key)
    w, h = (v, v) if isinstance(v, int) else tuple(v) if isinstance(v, (tuple, list)) and len(v) == 2 else (None, None)
    if not (isinstance(w, int) and isinstance(h, int) and w > 0 and h > 0):
        raise ValueError(f"{step['type']}: {key} must be a positive int or (w, h) (got {v!r})")
    return h, w


def _normalize(norm: dict) -> tuple:
    _only(norm, mean=None, std=None, to_bgr=False, adjust_magnitude=False)
    if len(norm.get('mean', ())) != 3 or len(norm.get('std', ())) != 3:
        raise ValueError("Normalize: mean and std must have 3 values (RGB)")
    return tuple(float(m) for m in norm['mean']), tuple(float(v) for v in norm['std'])


def _format_nchw(fmt: dict) -> None:
    _only(fmt, input_format=None, collapse=False)
    if fmt.get('input_format') != 'NCHW':
        raise ValueError(f"FormatShape: only input_format='NCHW' has a device form (got {fmt.get('input_format')!r})")


class EvalPipeline:
    """The tail of an evaluation pipeline that the device runs on decoded uint8 frames (``resize_crop_normalize``):

        Resize(scale=(-1, S)) -> CenterCrop(c) | ThreeCrop(c) -> Normalize(mean, std) -> FormatShape('NCHW')

    ``steps`` are the mmaction step dicts of these four, in this order, moved verbatim out of ``test_pipeline``.  Any other
    step, or another form of these (``keep_ratio=False``, another interpolation, ``to_bgr=True``, ``TenCrop``, NCTHW, ...),
    raises ``ValueError`` naming the step; such a config keeps its CPU pipeline.

    The rules restate mmaction2 0.x ``mmaction/datasets/pipelines/augmentations.py`` (``Resize``, ``CenterCrop``,
    ``ThreeCrop``, ``Normalize``) and ``formating.py`` (``FormatShape``), and mmcv 1.x ``mmcv/image/geometric.py``
    (``rescale_size``, ``_scale_size``, ``imresize``); neither package is a dependency:

    * Resize, ``keep_ratio=True``, bilinear: ``scale=(-1, S)`` or ``(S, -1)`` becomes ``(inf, S)``, and
      ``mmcv.rescale_size((w, h), (inf, S))`` gives ``f = S / min(h, w)``, ``(Wr, Hr) = (int(w * f + 0.5), int(h * f + 0.5))``;
      pixels are ``cv2.resize(img, (Wr, Hr), interpolation=cv2.INTER_LINEAR)``.  240x320 -> 256x341, 320x240 -> 341x256.
    * CenterCrop: ``left = (Wr - cw) // 2``, ``top = (Hr - ch) // 2``.
    * ThreeCrop: needs ``ch == Hr`` or ``cw == Wr`` (mmaction asserts it).  If ``ch == Hr``: ``step = (Wr - cw) // 2`` and the
      windows start at left 0, ``2 * step``, ``step`` in that order (so 85 pixels of slack give a right crop at 84); else the
      same vertically.  The output is crop-major: crop k's frames follow crop k-1's.
    * ``crop_size``: an int or ``(cw, ch)`` (mmaction's ``_pair`` order).  A crop larger than the resized frame raises.
    * Normalize, ``to_bgr=False``: :func:`ops.make_fg_lut` of ``(mean, std)``, as the training path normalises.
    * FormatShape('NCHW'): ``[K * T, 3, ch, cw]`` per clip.
    """

    def __init__(self, steps: Sequence[dict]):
        resize, crop, norm, fmt = _steps_in_order('device_test_pipeline', steps,
                                                  (('Resize',), ('CenterCrop', 'ThreeCrop'), ('Normalize',), ('FormatShape',)))
        self.short_side = _short_side(resize)
        _only(crop, crop_size=None, lazy=False)
        self.three, self.crop_hw = crop['type'] == 'ThreeCrop', _size_hw(crop, 'crop_size')
        self.mean, self.std = _normalize(norm)
        _format_nchw(fmt)

    @property
    def n_crops(self) -> int:
        return 3 if self.three else 1

    def windows(self, h: int, w: int) -> tuple:
        """``(Hr, Wr, [(top, left), ...])`` for a native ``h x w`` frame: the resized size and every crop's window."""
        Hr, Wr = rescale_short_side(h, w, self.short_side)
        ch, cw = self.crop_hw
        if not self.three:
            if ch > Hr or cw > Wr:
                raise ValueError(f"CenterCrop: crop {ch}x{cw} is larger than the resized frame {Hr}x{Wr}")
            return Hr, Wr, [((Hr - ch) // 2, (Wr - cw) // 2)]
        if ch == Hr and cw <= Wr:
            step = (Wr - cw) // 2
            return Hr, Wr, [(0, 0), (0, 2 * step), (0, step)]
        if cw == Wr and ch <= Hr:
            step = (Hr - ch) // 2
            return Hr, Wr, [(0, 0), (2 * step, 0), (step, 0)]
        raise ValueError(f"ThreeCrop: crop {ch}x{cw} must span the height or the width of the resized frame {Hr}x{Wr}")

    def geometry(self, fg_geom: torch.Tensor) -> torch.Tensor:
        """int64 ``[B * K, 9]`` for ``resize_crop_normalize`` from the ``[B, 5]`` geometry of ``ops.pack_clips``: clip-major,
        then crop, so that the ``[B * K, T, 3, ch, cw]`` output is ``[B, K * T, 3, ch, cw]``."""
        rows = []
        for q in fg_geom.tolist():
            Hr, Wr, wins = self.windows(int(q[1]), int(q[2]))
            rows += [q[:5] + [Hr, Wr, top, left] for top, left in wins]
        return torch.tensor(rows, dtype=torch.int64).reshape(-1, 9)


class TrainPipeline:
    """The geometric tail of a training pipeline that the device runs on decoded uint8 frames, fused with the BG-mix blend:

        Resize(scale=(-1, S)) -> MultiScaleCrop(...) -> Resize(scale=(W, H), keep_ratio=False) -> Normalize -> FormatShape('NCHW')

    ``steps`` are the mmaction step dicts of these five, in this order, moved verbatim out of ``train_pipeline``.  Any other
    step, or another form of these (``lazy=True``, another interpolation, ``to_bgr=True``, NCTHW, ...), raises
    ``ValueError`` naming the step; such a config keeps its CPU pipeline.  A pipeline with a host-only step between
    ``RawFrameDecode`` and ``MultiScaleCrop`` (``RandAugment``) cannot use this route.

    The rules restate mmaction2 0.x ``mmaction/datasets/pipelines/augmentations.py`` (``Resize``, ``MultiScaleCrop``,
    ``Normalize``) and mmcv 1.x ``rescale_size`` / ``imresize``; neither package is a dependency:

    * Resize(scale=(-1, S)): :func:`rescale_short_side`, as :class:`EvalPipeline`; pixels ``cv2.resize(img, (Wr, Hr),
      interpolation=cv2.INTER_LINEAR)``.
    * MultiScaleCrop(input_size, scales=(1,), max_wh_scale_gap=1, random_crop=False, num_fixed_crops=5), on the Hr x Wr
      frame: ``base = min(Hr, Wr)``, ``crop_sizes = [int(base * s) for s in scales]``; the candidates are ``[w, h]`` for
      every ``(i, h)``, ``(j, w)`` of ``enumerate(crop_sizes)`` (h outer, w inner) with ``abs(i - j) <= max_wh_scale_gap``;
      ``crop_size = random.choice(candidates)`` (Python's ``random``); each side with ``abs(side - input_size[k]) < 3``
      becomes ``input_size[k]`` (``input_size`` an int or ``(w, h)``, mmaction's ``_pair``).  The offset: with
      ``random_crop``, ``x0 = random.randint(0, Wr - cw)`` then ``y0 = random.randint(0, Hr - ch)``; otherwise, with
      ``w_step = (Wr - cw) // 4`` and ``h_step = (Hr - ch) // 4``, ``(x0, y0) = random.choice`` of the (x, y) offsets
      ``(0, 0), (4w, 0), (0, 4h), (4w, 4h), (2w, 2h)`` and, for ``num_fixed_crops=13``, then ``(0, 2h), (4w, 2h), (2w, 4h),
      (2w, 0), (w, h), (3w, h), (w, 3h), (3w, 3h)`` (w = w_step, h = h_step).  The crop is ``img[y0:y0 + ch, x0:x0 + cw]``.
    * Resize(scale=(W, H), keep_ratio=False): ``cv2.resize(crop, (W, H), interpolation=cv2.INTER_LINEAR)``.
    * Normalize, ``to_bgr=False``: :func:`ops.make_fg_lut` of ``(mean, std)``.  FormatShape('NCHW'): ``[T, 3, H, W]``.

    The draws happen on the host (:meth:`draw`, in the worker, where the CPU pipeline would make them); the pixels of all
    three geometric steps are one launch with the blend (``ops.TWO_STAGE_COLS``).
    """

    def __init__(self, steps: Sequence[dict]):
        resize, msc, final, norm, fmt = _steps_in_order(
            'device_train_pipeline', steps, (('Resize',), ('MultiScaleCrop',), ('Resize',), ('Normalize',), ('FormatShape',)))
        self.short_side = _short_side(resize)
        _only(msc, input_size=None, scales=None, max_wh_scale_gap=None, random_crop=None, num_fixed_crops=None, lazy=False)
        self.input_hw = _size_hw(msc, 'input_size')
        scales = msc.get('scales', (1,))
        if not (isinstance(scales, (tuple, list)) and scales and all(isinstance(v, (int, float)) and 0 < v for v in scales)):
            raise ValueError(f"MultiScaleCrop: scales must be a non-empty tuple of positive numbers (got {scales!r})")
        self.scales = tuple(scales)
        self.max_wh_scale_gap = msc.get('max_wh_scale_gap', 1)
        if not isinstance(self.max_wh_scale_gap, int) or self.max_wh_scale_gap < 0:
            raise ValueError(f"MultiScaleCrop: max_wh_scale_gap must be an int >= 0 (got {self.max_wh_scale_gap!r})")
        self.random_crop = msc.get('random_crop', False)
        if not isinstance(self.random_crop, bool):
            raise ValueError(f"MultiScaleCrop: random_crop must be a bool (got {self.random_crop!r})")
        self.num_fixed_crops = msc.get('num_fixed_crops', 5)
        if self.num_fixed_crops not in (5, 13):
            raise ValueError(f"MultiScaleCrop: num_fixed_crops must be 5 or 13 (got {self.num_fixed_crops!r})")
        _only(final, scale=None, keep_ratio=False, interpolation='bilinear', lazy=False)
        if final.get('keep_ratio', True) is not False:
            raise ValueError("Resize: keep_ratio must be False in the Resize after MultiScaleCrop")
        self.out_hw = _size_hw(final, 'scale')
        self.mean, self.std = _normalize(norm)
        _format_nchw(fmt)

    def draw(self, h: int, w: int) -> tuple:
        """``(Hr, Wr, y0, x0, ch, cw)`` for a native ``h x w`` frame, drawn from Python's ``random`` as MultiScaleCrop draws."""
        Hr, Wr = rescale_short_side(h, w, self.short_side)
        base = min(Hr, Wr)
        crop_sizes = [int(base * s) for s in self.scales]
        candidates = [[cw, ch] for i, ch in enumerate(crop_sizes) for j, cw in enumerate(crop_sizes)
                      if abs(i - j) <= self.max_wh_scale_gap]
        size = random.choice(candidates)
        in_wh = (self.input_hw[1], self.input_hw[0])
        for k in range(2):
            if abs(size[k] - in_wh[k]) < 3:
                size[k] = in_wh[k]
        cw, ch = size
        if ch > Hr or cw > Wr or ch < 1 or cw < 1:
            raise ValueError(f"MultiScaleCrop: crop {ch}x{cw} does not fit the resized frame {Hr}x{Wr}")
        if self.random_crop:
            x0 = random.randint(0, Wr - cw)
            y0 = random.randint(0, Hr - ch)
        else:
            ws, hs = (Wr - cw) // 4, (Hr - ch) // 4
            offsets = [(0, 0), (4 * ws, 0), (0, 4 * hs), (4 * ws, 4 * hs), (2 * ws, 2 * hs)]
            if self.num_fixed_crops == 13:
                offsets += [(0, 2 * hs), (4 * ws, 2 * hs), (2 * ws, 4 * hs), (2 * ws, 0), (ws, hs), (3 * ws, hs), (ws, 3 * hs),
                            (3 * ws, 3 * hs)]
            x0, y0 = random.choice(offsets)
        return Hr, Wr, y0, x0, ch, cw


@_register(_DATASETS)
class BackgroundMixDataset(_Base):
    """Same signature as the reference class (libs/loader/comix_loader.py:16-45) plus four
    keyword-only extensions: ``device`` (CUDA device of the pool and the blend), ``device_mix``
    (see module docstring), ``bg_reader`` (callable ``path -> uint8 [3,h,w]``, defaults to
    ``torchvision.io.read_image(mode=RGB)`` as in the reference), ``device_test_pipeline`` (the
    step dicts of :class:`EvalPipeline`, required by ``device_mix=True`` with ``test_mode=True``) and
    ``device_train_pipeline`` (the step dicts of :class:`TrainPipeline`, for ``device_mix=True`` training
    datasets whose pipeline then stops after ``RawFrameDecode``)."""

    def __init__(self,
                 ann_file,
                 pipeline,
                 bg_dir: str,
                 extract_bg_if_not_found=True,      # extract background with TMF if not found
                 back_ground_from_bg_dir=True,      # find background in folders
                 map_bg_to_video=True,              # each video associated with a background (same prefix)
                 merge_bg_files=True,
                 bg_image_extension='.jpg',
                 bg_resize=256,
                 bg_crop_size=(224, 224),
                 bg_mean=[123.675, 116.28, 103.53],
                 bg_std=[58.395, 57.12, 57.375],
                 alpha=0.5,
                 prob=0.25,
                 with_randAug=False,
                 data_prefix=None,
                 test_mode=False,
                 filename_tmpl='img_{:05}.jpg',
                 with_offset=False,
                 multi_class=False,
                 num_classes=None,
                 start_index=1,
                 modality='RGB',
                 sample_by_class=False,
                 power=0.,
                 dynamic_length=False,
                 device='cuda',
                 device_mix=False,
                 bg_reader: Optional[Callable] = None,
                 device_test_pipeline: Optional[Sequence[dict]] = None,
                 device_train_pipeline: Optional[Sequence[dict]] = None,
                 **kwargs):
        if device_train_pipeline is not None:
            if device_test_pipeline is not None:
                raise ValueError("device_train_pipeline and device_test_pipeline are exclusive: a dataset trains or evaluates")
            if not device_mix or test_mode:
                raise ValueError("device_train_pipeline is the training tail of device_mix=True with test_mode=False")
            if with_randAug:
                raise ValueError("device_train_pipeline cannot run with with_randAug=True: the gate reads the flag RandAugment "
                                 "sets, and RandAugment runs on the host between RawFrameDecode and MultiScaleCrop")
        if device_test_pipeline is not None and not (device_mix and test_mode):
            raise ValueError("device_test_pipeline is the evaluation tail of device_mix=True with test_mode=True")
        if device_mix and test_mode and device_test_pipeline is None:
            raise ValueError("device_mix=True with test_mode=True needs device_test_pipeline: the Resize, crop, Normalize "
                             "and FormatShape steps moved out of test_pipeline")
        self._eval = EvalPipeline(device_test_pipeline) if device_test_pipeline is not None else None
        self._train = TrainPipeline(device_train_pipeline) if device_train_pipeline is not None else None
        super().__init__(ann_file, pipeline, data_prefix, test_mode, filename_tmpl, with_offset, multi_class,
                         num_classes, start_index, modality, sample_by_class, power, dynamic_length, **kwargs)
        bg_dir = osp.realpath(bg_dir)                 # same reason as the reference, comix_loader.py:61-68
        self.bg_dir = pathlib.Path(bg_dir)
        self.bg_image_extension = bg_image_extension
        self.bg_dir.mkdir(exist_ok=True, parents=True)
        self.bg_resize = bg_resize
        self.bg_crop_size = tuple(bg_crop_size) if not isinstance(bg_crop_size, int) else (bg_crop_size, bg_crop_size)
        if self._train is not None and self._train.out_hw != self.bg_crop_size:
            raise ValueError(f"device_train_pipeline: the final Resize gives {self._train.out_hw} (h, w), bg_crop_size is "
                             f"{self.bg_crop_size}; the blend needs them equal")
        self.bg_mean = [float(m) for m in bg_mean]
        self.bg_std = [float(s) for s in bg_std]
        self.alpha = alpha
        self.prob = prob
        self.with_randAug = with_randAug
        self.extract_bg_if_not_found = extract_bg_if_not_found
        self.back_ground_from_bg_dir = back_ground_from_bg_dir
        self.map_bg_to_video = map_bg_to_video
        self.merge_bg_files = merge_bg_files
        self.device = torch.device(device)
        self.device_mix = device_mix
        self._bg_reader = bg_reader
        self._attach(self.device)
        self._resized_cache = {}                          # path -> size after Resize, for forked DataLoader workers
        self._aa: Optional[AATables] = None
        self._luts: dict = {}                             # (mean, std) -> foreground LUT on self.device

        # pool assembly: the three modes of comix_loader.py:84-103
        if self.back_ground_from_bg_dir:
            if map_bg_to_video:
                self.bg_files = []
                for info in self.video_infos:
                    data_path = pathlib.Path(info['frame_dir'])
                    bg_image_file = (self.bg_dir / data_path.name).with_suffix(self.bg_image_extension)
                    if bg_image_file.exists():
                        self.bg_files.append(str(bg_image_file))
                    elif self.extract_bg_if_not_found:
                        # The reference appends str(ndarray) here (comix_loader.py:96-98), which poisons
                        # the pool; the evident intent -- extract, write, remember the PATH -- is what runs.
                        bg_extraction_tmf(data_path, bg_image_file, device=self.device)
                        self.bg_files.append(str(bg_image_file))
            else:
                self.bg_files = [str(p) for p in self.bg_dir.glob("*")]
        else:
            self.bg_files = []

    # ---- background access -------------------------------------------------------------------
    def _read_bg(self, path: str) -> torch.Tensor:
        return _read_image(path, self._bg_reader)

    def _random_frame(self) -> torch.Tensor:
        """A random frame of a random video (comix_loader.py:133-136): ``random.choice``, then ``random.randint``."""
        video = random.choice(self.video_infos)
        frame_index = random.randint(self.start_index, video['total_frames'] - 1 + self.start_index)
        return self._read_bg(osp.join(video['frame_dir'], self.filename_tmpl.format(frame_index)))

    def _get_bg_image(self):
        """Same draws and return value as the reference (comix_loader.py:126-136): a float ``[3,h,w]``
        RGB image (values 0..255) and its pool index (-2 in random-frame mode)."""
        if self.back_ground_from_bg_dir:
            bg_idx = torch.randint(len(self.bg_files), (1,)).item()
            return self._read_bg(self.bg_files[bg_idx]).float(), bg_idx
        return self._random_frame().float(), -2      # to pass sanity check

    def device_pool(self) -> BackgroundPool:
        """The pool for the current ``bg_files``, index i = ``bg_files[i]``.  Every path is decoded + resized
        once per dataset object and stays on ``self.device`` (:class:`BackgroundStore`); when the caller
        replaces or mutates ``bg_files`` -- the CIL trainer does between tasks (libs/cil/cil.py:150-160,
        193-195,390-393: unions and extensions of path lists) -- only paths not seen before are decoded and
        the new pool is a new slot table over the same pixels."""
        key = tuple(self.bg_files)
        if self._pool is None or key != self._pool_key:
            if self._store is None:
                self._store = BackgroundStore(self.bg_resize, self.device)
            self._store.ensure(self.bg_files, self._read_bg)
            self._pool = self._store.view(list(self.bg_files))
            self._pool_key = key
        return self._pool

    def attach_pool(self, paths: Sequence[str], ragged: RaggedPool) -> None:
        """Use backgrounds that are already on the device -- the result of ``pool.gather_extracted_backgrounds`` after a
        sharded extraction -- instead of decoding ``bg_files`` again: ``paths[i]`` is image ``i`` of ``ragged``.  Paths
        are matched after ``realpath`` like ``bg_dir`` (comix_loader.py:61-68); files of ``bg_files`` that are not among
        them are decoded on demand as usual."""
        store = BackgroundStore(self.bg_resize, ragged.device)
        store.adopt([osp.realpath(p) for p in paths], ragged)
        self._attach(ragged.device, store=store)

    def attach_sharded_pool(self, paths: Sequence[str], sharded: ShardedPool) -> None:
        """Mix from a pool sharded across the ranks of a process group (``pool.shard_extracted_backgrounds``): ``paths[i]`` names
        global image ``i`` of ``sharded``.  Each rank keeps only its own images; :meth:`device_finish` fetches the images a
        batch drew from their owners (one ``all_to_all_single``) and blends them, bit-equal to :meth:`attach_pool` with the
        replicated pool.  ``bg_files`` may list any of these names, in any order and with repeats -- the CIL pool operations
        stay inside the extracted set; a name outside it raises ``ValueError``, nothing is decoded on demand.  Sizes come from
        the index, so DataLoader workers forked after this call draw crops without reading a file.

        Every rank of the pool's group must call :meth:`device_finish` (or :meth:`mix_batch_on_device`) once per batch, in
        lockstep: see :meth:`pool.ShardedPool.fetch`."""
        if [str(p) for p in paths] != sharded.names:
            raise ValueError("paths must be the names of the sharded pool's images, in index order")
        self._attach(sharded.device, sharded=sharded, fetch=sharded.fetch)

    def attach_peer_pool(self, paths: Sequence[str], peer: PeerPool) -> None:
        """The twin of :meth:`attach_sharded_pool` for a pool whose shards are mapped into every rank of one node
        (``pool.PeerPool.open``): the same names, the same ``ValueError`` for a name outside the index, the same draws and
        bits; but :meth:`device_finish` reads the images a batch drew straight from their owners' memory with one local
        launch (:meth:`pool.PeerPool.gather`) -- no collective, so ranks need not call it in lockstep, and the host does
        not wait for the device.  Attaching a pool of any other kind detaches this one."""
        self.attach_sharded_pool(paths, peer.sharded)
        self._fetch = peer.gather

    def _attach(self, device, store: Optional[BackgroundStore] = None, sharded: Optional[ShardedPool] = None,
                fetch: Optional[Callable] = None) -> None:
        """Mix from one pool, detaching any other: the replica ``store`` (``None``: built from ``bg_files`` on demand), or a
        ``sharded`` pool with ``fetch(bg_idx, apply) -> (batch pool, slot)`` that brings a batch's images to this rank."""
        self._store, self._pool, self._pool_key = store, None, None
        self._sharded, self._fetch, self._shard_rows = sharded, fetch, None
        self.device = device

    def _sharded_rows(self) -> np.ndarray:
        """Global index of every entry of the current ``bg_files`` (cached per list)."""
        key = tuple(self.bg_files)
        if self._shard_rows is None or key != self._shard_rows[0]:
            self._shard_rows = (key, self._sharded.rows_of(self.bg_files))
        return self._shard_rows[1]

    # ---- per-sample API (reference contract) ---------------------------------------------------
    def prepare_train_frames(self, idx):
        """Prepare the frames for training given the index (comix_loader.py:105-124)."""
        result = super().prepare_train_frames(idx)
        if self._train is not None:
            # MultiScaleCrop's draws, where the CPU pipeline makes them: before the gate's random.random()
            imgs = result['imgs']
            h, w = (imgs[0].shape[0], imgs[0].shape[1]) if isinstance(imgs, (list, tuple)) else tuple(imgs.shape[1:3])
            result['fg_window'] = self._train.draw(int(h), int(w))
        result['bg_idx'] = -1
        if self.device_mix:
            result['bg_top'], result['bg_left'], result['bg_apply'] = 0, 0, 0

        # when randAug is in the pipeline, only apply BGMix when randAug is not applied
        if self.with_randAug:
            if not result['randAug']:
                result = self._mix_background(result)
        elif random.random() < self.prob:
            result = self._mix_background(result)

        # sanity check
        if self.with_randAug:
            if result['randAug']:
                assert result['bg_idx'] == -1
            else:
                assert result['bg_idx'] != -1
        return result

    def _mix_background(self, result):
        """comix_loader.py:138-145.  ``device_mix=False``: blends ``result['imgs']`` (fp32 [T,3,H,W],
        already normalised) on the GPU and returns it on its original device.  ``device_mix=True``:
        only draws ``bg_idx`` / crop offsets; pixels are mixed per batch by :meth:`gpu_collate`."""
        th, tw = self.bg_crop_size
        if self.device_mix:
            if self.back_ground_from_bg_dir:
                bg_idx = torch.randint(len(self.bg_files), (1,)).item()
                h, w = self._bg_hw(bg_idx)                # RandomCrop sees the DRAWN image after Resize (:72-73,139-140)
            else:
                # random frame of a random video (:133-136): same draws, the decoded uint8 frame travels with the sample
                img = self._random_frame()
                h, w = self._resized_hw(int(img.shape[1]), int(img.shape[2]))
                result['bg_img'] = img.to(torch.uint8)
                bg_idx = -2                               # to pass sanity check
            top, left = draw_crop(h, w, (th, tw))
            result['bg_idx'], result['bg_top'], result['bg_left'], result['bg_apply'] = bg_idx, top, left, 1
            return result

        if torch.cuda._is_in_bad_fork():
            raise RuntimeError(
                "BackgroundMixDataset(device_mix=False) blends on the GPU inside __getitem__, but this DataLoader worker "
                "was forked after CUDA was initialised and cannot use it.  Use device_mix=True with "
                "collate_fn=dataset.host_collate and dataset.device_finish(batch) in the training process (workers then "
                "never touch CUDA), or num_workers=0, or multiprocessing_context='spawn'.  There is no CPU blend.")
        bg_img, bg_idx = self._get_bg_image()
        bg_img = resize_like_reference(bg_img, self.bg_resize)           # Resize(bg_resize), :72
        top, left = draw_crop(bg_img.shape[1], bg_img.shape[2], (th, tw))   # RandomCrop, :73
        imgs = result['imgs']
        if imgs.dim() != 4 or imgs.shape[1] != 3 or tuple(imgs.shape[2:]) != (th, tw):
            raise ValueError(f"imgs must be [T, 3, {th}, {tw}] (got {tuple(imgs.shape)})")
        result['imgs'] = _blend_clip(imgs, bg_img, top, left, self.bg_mean, self.bg_std, self.alpha, self.device)
        result['bg_idx'] = bg_idx
        return result

    def _resized_hw(self, h: int, w: int) -> tuple:
        return (h, w) if self.bg_resize is None else resized_hw(h, w, self.bg_resize)

    def _bg_hw(self, bg_idx: int) -> tuple:
        """Size after Resize of ``bg_files[bg_idx]``: from the resident pool / store when they know the file; else a
        process that owns the GPU decodes the image into the store (once), and a forked DataLoader worker reads the image
        header (cached per path).  With a sharded pool the global index answers."""
        if self._sharded is not None:
            return self._sharded.hw(int(self._sharded.rows_of([self.bg_files[bg_idx]])[0]))
        if self._pool is not None and tuple(self.bg_files) == self._pool_key:
            return self._pool.hw_of(bg_idx)
        path = self.bg_files[bg_idx]
        if self._store is not None and path in self._store.slot_of:
            return self._store.hw_of(self._store.slot_of[path])
        if path in self._resized_cache:
            return self._resized_cache[path]
        if self.device.type == "cuda" and torch.cuda.is_available() and not torch.cuda._is_in_bad_fork():
            # a process that may use the GPU decodes the image once, into the store, and reads its size there
            if self._store is None:
                self._store = BackgroundStore(self.bg_resize, self.device)
            self._store.ensure([path], self._read_bg)
            return self._store.hw_of(self._store.slot_of[path])
        if self._bg_reader is not None:                   # DataLoader worker: size only, cached per path
            img = self._read_bg(path)
            h, w = int(img.shape[1]), int(img.shape[2])
        else:
            from PIL import Image
            with Image.open(path) as im:                  # header only
                w, h = im.size
        self._resized_cache[path] = self._resized_hw(h, w)
        return self._resized_cache[path]

    def _pool_hw(self) -> tuple:
        """Size after Resize of the first pool image (kept for callers that warm the size cache before forking)."""
        return self._bg_hw(0)

    # ---- batch API (device_mix=True) -------------------------------------------------------------
    def mix_batch_on_device(self, fg_u8: torch.Tensor, bg_idx, bg_top, bg_left, bg_apply,
                            img_mean: Optional[Sequence[float]] = None, img_std: Optional[Sequence[float]] = None,
                            layout: str = "NTCHW", fg_geom: Optional[torch.Tensor] = None,
                            fg_frames: Optional[int] = None, bg_imgs: Optional[Sequence[torch.Tensor]] = None,
                            bg_slot=None, dtype: torch.dtype = torch.float32,
                            memory_format: torch.memory_format = torch.contiguous_format) -> torch.Tensor:
        """uint8 ``[B,T,H,W,3]`` (host or device) + per-sample draws -> fp32 ``[B,T,3,H,W]`` on the device.
        ``img_mean``/``img_std`` are the foreground's ``Normalize`` parameters (default: the bg ones,
        as in every shipped config).

        The background of sample b is pool image ``bg_idx[b]`` -- from the dense fp32 cache when the pool has one
        image size and fits, else from the ragged uint8 store with ``Resize`` inside the launch; with a sharded pool
        (:meth:`attach_sharded_pool`) from the images fetched from their owners, a collective, or read from their owners'
        peer-mapped memory (:meth:`attach_peer_pool`), a local launch -- or, in random-frame
        mode (``back_ground_from_bg_dir=False``), ``bg_imgs[bg_slot[b]]``: the uint8 frames the batch drew.

        Clips whose size is not ``bg_crop_size`` -- a pipeline that stops before the final
        ``Resize((224, 224), keep_ratio=False)`` (config :136) -- are resized with cv2's INTER_LINEAR arithmetic, inside
        the blend launch for a dense pool: either a stacked batch of one other size, or packed crops of mixed sizes
        (``fg_u8`` flat, ``fg_geom`` int64 ``[B,5]``, ``fg_frames`` = T; see ``ops.pack_clips``).

        ``dtype`` float32, bfloat16 or float16: the fp32 blend rounded once to nearest even (equal to ``.to(dtype)`` of the
        float32 batch).  ``memory_format=torch.channels_last``: the launch writes ``[B,T,H,W,3]`` and the method returns
        its permuted view, logical ``[B,T,3,H,W]`` (whose ``flatten(0, 1)`` is ``channels_last``) for ``layout="NTCHW"``
        or ``[B,3,T,H,W]`` in ``channels_last_3d`` strides for ``layout="NCTHW"``."""
        if layout not in ("NTCHW", "NCTHW"):
            raise ValueError(f"layout must be 'NTCHW' or 'NCTHW' (got {layout!r})")
        if dtype not in (torch.float32, torch.bfloat16, torch.float16):
            raise ValueError(f"dtype must be torch.float32, torch.bfloat16 or torch.float16 (got {dtype})")
        if memory_format not in (torch.contiguous_format, torch.channels_last):
            raise ValueError(f"memory_format must be torch.contiguous_format or torch.channels_last (got {memory_format})")
        channels_last = memory_format == torch.channels_last
        op_layout = "NTHWC" if channels_last else layout
        dev = self.device
        mean = self.bg_mean if img_mean is None else img_mean
        std = self.bg_std if img_std is None else img_std
        lut = self._lut(tuple(mean), tuple(std))
        as_dev = lambda v, dt: torch.as_tensor(v, dtype=dt).to(dev, non_blocking=True)   # noqa: E731
        th, tw = self.bg_crop_size
        top, left, app = as_dev(bg_top, torch.int32), as_dev(bg_left, torch.int32), as_dev(bg_apply, torch.uint8)
        if bg_imgs is not None:
            batch_pool = RaggedPool(self.bg_resize, dev, tables=self._aa_tables())
            batch_pool.append(bg_imgs)
            ragged, dense, rows = batch_pool, None, as_dev(bg_slot, torch.int32)
        elif self._sharded is not None:
            # sharded pool: fetch the drawn images from their owners (a collective) or gather them from the peer mappings
            # (a local launch), then the random-frame route
            idx = torch.as_tensor(bg_idx).cpu().clamp(min=0, max=max(len(self.bg_files) - 1, 0))
            gidx = torch.from_numpy(self._sharded_rows())[idx] if len(self.bg_files) else idx
            batch_pool, slot = self._fetch(gidx, torch.as_tensor(bg_apply).cpu())
            if not len(batch_pool):                       # nothing mixed on this rank: a placeholder the blend never reads
                batch_pool.append([torch.zeros((3, th, tw), dtype=torch.uint8)])
            ragged, dense, rows = batch_pool, None, as_dev(slot, torch.int32)
        else:
            pool = self.device_pool()
            ragged, dense = pool.ragged, pool.tensor
            rows = pool.rows(as_dev(bg_idx, torch.int32).clamp(min=0))
        mean_t, std_t = torch.tensor(self.bg_mean), torch.tensor(self.bg_std)
        if fg_geom is None and tuple(fg_u8.shape[2:4]) != (th, tw):
            B, T, h, w, _ = fg_u8.shape
            frame = h * w * 3
            fg_geom = torch.tensor([[b * T * frame, h, w, w * 3, frame] for b in range(B)], dtype=torch.int64)
            flat = fg_u8.reshape(-1)
            fg_u8 = torch.cat([flat, flat.new_zeros(4 + (-flat.numel()) % 4)])
            fg_frames = T
        fg_u8 = fg_u8.to(dev, non_blocking=True)
        if fg_geom is not None and dense is not None:
            out = torch.ops.bgdebias.bgmix_resize_blend(fg_u8, fg_geom, int(fg_frames), th, tw, dense, rows, top, left, app, lut,
                                                        mean_t, std_t, float(self.alpha), op_layout, dtype)
        else:
            if fg_geom is not None:
                fg_u8 = torch.ops.bgdebias.resize_bilinear(fg_u8, fg_geom, int(fg_frames), th, tw)
            if dense is not None:
                out = torch.ops.bgdebias.bgmix_blend(fg_u8, dense, rows, top, left, app, lut, mean_t, std_t, float(self.alpha),
                                                     op_layout, dtype)
            else:
                out = torch.ops.bgdebias.bgmix_blend_ragged(fg_u8, ragged.data, ragged.slots_tensor, ragged.tables.tensor, rows,
                                                            top, left, app, lut, mean_t, std_t, float(self.alpha), op_layout, dtype)
        if channels_last:                                 # [B,T,H,W,3] -> logical [B,T,3,H,W] / [B,3,T,H,W]
            return out.permute(0, 1, 4, 2, 3) if layout == "NTCHW" else out.permute(0, 4, 1, 2, 3)
        return out

    def _aa_tables(self) -> AATables:
        if self._aa is None:
            self._aa = AATables(self.device)
        return self._aa

    def _lut(self, mean, std) -> torch.Tensor:
        if (mean, std) not in self._luts:
            self._luts[(mean, std)] = ops.make_fg_lut(mean, std, self.device)
        return self._luts[(mean, std)]

    @staticmethod
    def host_collate(samples: List[dict]) -> dict:
        """``collate_fn`` for ``device_mix=True`` that is safe in DataLoader worker processes (no CUDA): stacks
        the uint8 clips ``[B,T,H,W,3]`` and the per-sample draws into host tensors.  Pair it with
        :meth:`device_finish` in the training process; with ``pin_memory=True`` the batch travels as uint8,
        a quarter of the bytes of the reference's fp32 batch (libs/cil/cil.py:203-210).

        Samples of a ``device_train_pipeline`` dataset carry native-size frames: they are packed with ``ops.pack_clips``
        and ``fg_geom`` is the ``[B, 11]`` two-stage geometry (``ops.TWO_STAGE_COLS``) of their MultiScaleCrop draws.

        Samples without draws (``test_mode=True``) make an evaluation batch: the native-size uint8 frames packed with
        ``ops.pack_clips`` (sizes may differ per video) and ``label``, for the eval route of :meth:`device_finish`."""
        clips = [torch.as_tensor(np.stack(s['imgs']) if isinstance(s['imgs'], (list, tuple)) else s['imgs']) for s in samples]
        out = {}
        if 'fg_window' in samples[0]:
            # device_train_pipeline: native-size frames and each sample's (Hr, Wr, y0, x0, ch, cw), the two-stage geometry
            out['imgs'], g5 = ops.pack_clips(clips)
            out['fg_geom'] = torch.cat([g5, torch.tensor([s['fg_window'] for s in samples], dtype=torch.int64)], 1)
            out['fg_frames'] = int(clips[0].shape[0])
        elif 'bg_idx' not in samples[0]:
            out['imgs'], out['fg_geom'] = ops.pack_clips(clips)
            out['fg_frames'] = int(clips[0].shape[0])
            if 'label' in samples[0]:
                out['label'] = torch.stack([torch.as_tensor(s['label']) for s in samples])
            return out
        elif all(c.shape == clips[0].shape for c in clips):
            out['imgs'] = torch.stack(clips)
        else:
            # the pipeline stopped before Resize((224, 224), keep_ratio=False) (config :136): MultiScaleCrop's crops differ in
            # size per sample, so they travel packed and device_finish resizes them inside the blend launch
            out['imgs'], out['fg_geom'] = ops.pack_clips(clips)
            out['fg_frames'] = int(clips[0].shape[0])
        out.update({
            'bg_idx': torch.tensor([int(s['bg_idx']) for s in samples], dtype=torch.int64),
            'bg_top': torch.tensor([int(s['bg_top']) for s in samples], dtype=torch.int32),
            'bg_left': torch.tensor([int(s['bg_left']) for s in samples], dtype=torch.int32),
            'bg_apply': torch.tensor([int(s['bg_apply']) for s in samples], dtype=torch.uint8),
        })
        if any('bg_img' in s for s in samples):
            # random-frame mode: the frames the batch drew are its pool; unmixed samples point at frame 0 and are ignored
            out['bg_imgs'] = [torch.as_tensor(s['bg_img']) for s in samples if 'bg_img' in s]
            slot, nxt = [], 0
            for s in samples:
                slot.append(nxt if 'bg_img' in s else 0)
                nxt += 'bg_img' in s
            out['bg_slot'] = torch.tensor(slot, dtype=torch.int32)
        if 'label' in samples[0]:
            out['label'] = torch.stack([torch.as_tensor(s['label']) for s in samples])
        if 'randAug' in samples[0]:
            out['randAug'] = torch.tensor([bool(s['randAug']) for s in samples])
        return out

    def device_finish(self, batch: dict, layout: str = "NTCHW", dtype: torch.dtype = torch.float32,
                      memory_format: torch.memory_format = torch.contiguous_format) -> dict:
        """The GPU half of the ``device_mix=True`` path: turns a :meth:`host_collate` batch into the dict the
        reference's default_collate would hand the model (``imgs`` fp32 ``[B,T,3,H,W]`` on the device, ``label``,
        ``randAug``, ``bg_idx``) with one fused launch.  ``dtype`` / ``memory_format``: see :meth:`mix_batch_on_device`.

        An evaluation batch (no draws) runs the dataset's :class:`EvalPipeline` instead, in one launch that reads neither
        the background pool nor any file: ``imgs`` ``[B, K*T, 3, ch, cw]`` (K crops, crop-major, as mmaction's ThreeCrop and
        FormatShape('NCHW') yield after default_collate) and ``label``."""
        if 'bg_idx' not in batch:
            return self._finish_eval(batch, layout, dtype, memory_format)
        out = {k: v for k, v in batch.items()
               if k not in ('imgs', 'bg_top', 'bg_left', 'bg_apply', 'fg_geom', 'fg_frames', 'bg_imgs', 'bg_slot')}
        if not self.back_ground_from_bg_dir and 'bg_imgs' not in batch:
            # random-frame mode and no sample of the batch was mixed: a placeholder frame the blend never reads
            batch = dict(batch, bg_imgs=[torch.zeros((3, *self.bg_crop_size), dtype=torch.uint8)],
                         bg_slot=torch.zeros(len(batch['bg_idx']), dtype=torch.int32))
        fg_geom = batch.get('fg_geom')
        norm = {}
        if fg_geom is not None and fg_geom.shape[1] == len(ops.TWO_STAGE_COLS):
            if self._train is None:
                raise ValueError("a batch with the two-stage geometry needs a dataset built with device_train_pipeline")
            norm = dict(img_mean=self._train.mean, img_std=self._train.std)
        out['imgs'] = self.mix_batch_on_device(batch['imgs'], batch['bg_idx'], batch['bg_top'], batch['bg_left'],
                                               batch['bg_apply'], layout=layout, fg_geom=fg_geom, **norm,
                                               fg_frames=batch.get('fg_frames'), bg_imgs=batch.get('bg_imgs'),
                                               bg_slot=batch.get('bg_slot'), dtype=dtype, memory_format=memory_format)
        return out

    def _finish_eval(self, batch: dict, layout: str, dtype: torch.dtype, memory_format: torch.memory_format) -> dict:
        if self._eval is None:
            raise ValueError("an evaluation batch (no mix draws) needs a dataset built with device_test_pipeline")
        if layout != "NTCHW":
            raise ValueError(f"evaluation batches are FormatShape('NCHW'): layout must be 'NTCHW' (got {layout!r})")
        if memory_format not in (torch.contiguous_format, torch.channels_last):
            raise ValueError(f"memory_format must be torch.contiguous_format or torch.channels_last (got {memory_format})")
        ev, dev = self._eval, self.device
        geom = ev.geometry(batch['fg_geom'])
        B, K, T = batch['fg_geom'].shape[0], ev.n_crops, int(batch['fg_frames'])
        ch, cw = ev.crop_hw
        channels_last = memory_format == torch.channels_last
        src = batch['imgs'].to(dev, non_blocking=True)
        imgs = torch.ops.bgdebias.resize_crop_normalize(src, geom, T, ch, cw, self._lut(ev.mean, ev.std),
                                                        "NTHWC" if channels_last else "NTCHW", dtype)
        if channels_last:                                 # [B*K,T,H,W,3] -> logical [B,K*T,3,H,W]
            imgs = imgs.view(B, K * T, ch, cw, 3).permute(0, 1, 4, 2, 3)
        else:
            imgs = imgs.view(B, K * T, 3, ch, cw)
        out = {'imgs': imgs}
        if 'label' in batch:
            out['label'] = batch['label']
        return out

    def gpu_collate(self, samples: List[dict], dtype: torch.dtype = torch.float32,
                    memory_format: torch.memory_format = torch.contiguous_format) -> dict:
        """:meth:`host_collate` + :meth:`device_finish` in one call, for ``num_workers=0`` loaders."""
        return self.device_finish(self.host_collate(samples), dtype=dtype, memory_format=memory_format)


def bg_extraction_tmf(data_path, dest, from_video=False, device='cuda'):
    """Rawframes variant of the reference (libs/loader/comix_loader.py:148-164): temporal median of
    ALL images of a frame folder (no interval, no cap), written to ``dest``; returns the
    ``[H,W,3]`` uint8 BGR array.  ``from_video=True`` raises ``NotImplementedError`` like the reference."""
    import cv2
    if from_video:
        raise NotImplementedError
    data_path = pathlib.Path(data_path)
    files = [str(f) for f in data_path.glob('*')]
    # JPEG decode dominates this call: spread it over the host cores (cv2 releases the GIL; the median ignores order)
    with ThreadPoolExecutor(max_workers=min(16, len(os.sched_getaffinity(0)))) as ex:
        frames = list(ex.map(cv2.imread, files))
    frames = [f for f in frames if f is not None]
    if not frames:
        raise ValueError(f"no readable frames under {data_path}")     # reference: nan median -> imwrite raises
    stack = torch.from_numpy(np.stack(frames)).to(device, non_blocking=True)
    median_frame = torch.ops.bgdebias.temporal_median(stack).cpu().numpy()
    cv2.imwrite(str(dest), median_frame)
    return median_frame


@_register(_PIPELINES)
class BackgroundMix:
    """mmaction-style pipeline transform (``__call__(results) -> results``) doing what
    ``BackgroundMixDataset._mix_background`` does, for pipelines that mix inside ``Compose``.

    Place it after ``FormatShape``/``ToTensor`` (``results['imgs']``: fp32 ``[T,3,H,W]``, normalised).
    The gate follows the dataset's: with ``with_randAug`` it mixes iff ``results['randAug']`` is false,
    else with probability ``prob``.  Sets ``results['bg_idx']`` (-1 when not mixed).
    """

    def __init__(self, bg_files: Sequence[str], bg_resize=256, bg_crop_size=(224, 224),
                 bg_mean=(123.675, 116.28, 103.53), bg_std=(58.395, 57.12, 57.375), alpha=0.5, prob=0.25,
                 with_randAug=False, device='cuda', bg_reader: Optional[Callable] = None):
        self.bg_files = list(bg_files)
        self.bg_resize, self.bg_crop_size = bg_resize, tuple(bg_crop_size)
        self.bg_mean, self.bg_std = [float(m) for m in bg_mean], [float(s) for s in bg_std]
        self.alpha, self.prob, self.with_randAug = alpha, prob, with_randAug
        self.device = torch.device(device)
        self._bg_reader = bg_reader

    def _read(self, path):
        return _read_image(path, self._bg_reader)

    def __call__(self, results):
        results['bg_idx'] = -1
        mix = (not results['randAug']) if self.with_randAug else (random.random() < self.prob)
        if not mix:
            return results
        bg_idx = torch.randint(len(self.bg_files), (1,)).item()
        bg = resize_like_reference(self._read(self.bg_files[bg_idx]).float(), self.bg_resize)
        top, left = draw_crop(bg.shape[1], bg.shape[2], self.bg_crop_size)
        imgs = torch.as_tensor(results['imgs'])
        results['imgs'] = _blend_clip(imgs, bg, top, left, self.bg_mean, self.bg_std, self.alpha, self.device)
        results['bg_idx'] = bg_idx
        return results

    def __repr__(self):
        return (f"{self.__class__.__name__}(n_bg={len(self.bg_files)}, bg_resize={self.bg_resize}, "
                f"bg_crop_size={self.bg_crop_size}, alpha={self.alpha}, prob={self.prob}, "
                f"with_randAug={self.with_randAug})")
