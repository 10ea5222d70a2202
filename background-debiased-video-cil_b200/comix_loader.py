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
        return self.prepare_train_frames(idx)

    def __getitem__(self, idx):
        return self.prepare_test_frames(idx) if self.test_mode else self.prepare_train_frames(idx)


_Base = _MMRawframeDataset if _HAVE_MMACTION else _RawframeBase


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


@_register(_DATASETS)
class BackgroundMixDataset(_Base):
    """Same signature as the reference class (libs/loader/comix_loader.py:16-45) plus three
    keyword-only extensions: ``device`` (CUDA device of the pool and the blend), ``device_mix``
    (see module docstring) and ``bg_reader`` (callable ``path -> uint8 [3,h,w]``, defaults to
    ``torchvision.io.read_image(mode=RGB)`` as in the reference)."""

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
                 **kwargs):
        super().__init__(ann_file, pipeline, data_prefix, test_mode, filename_tmpl, with_offset, multi_class,
                         num_classes, start_index, modality, sample_by_class, power, dynamic_length, **kwargs)
        bg_dir = osp.realpath(bg_dir)                 # same reason as the reference, comix_loader.py:61-68
        self.bg_dir = pathlib.Path(bg_dir)
        self.bg_image_extension = bg_image_extension
        self.bg_dir.mkdir(exist_ok=True, parents=True)
        self.bg_resize = bg_resize
        self.bg_crop_size = tuple(bg_crop_size) if not isinstance(bg_crop_size, int) else (bg_crop_size, bg_crop_size)
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
        self._pool: Optional[BackgroundPool] = None
        self._pool_key = None
        self._store: Optional[BackgroundStore] = None
        self._sharded: Optional[ShardedPool] = None
        self._peer: Optional[PeerPool] = None             # set with _sharded: gather from peer mappings instead of fetch
        self._shard_of: dict = {}                         # name (and its realpath) -> global index of the sharded pool
        self._shard_rows_key, self._shard_rows = None, None
        self._resized_cache = {}

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
        if self._bg_reader is not None:
            return torch.as_tensor(self._bg_reader(path))
        from torchvision.io import ImageReadMode, read_image
        return read_image(path, mode=ImageReadMode.RGB)

    def _get_bg_image(self):
        """Same draws and return value as the reference (comix_loader.py:126-136): a float ``[3,h,w]``
        RGB image (values 0..255) and its pool index (-2 in random-frame mode)."""
        if self.back_ground_from_bg_dir:
            bg_idx = torch.randint(len(self.bg_files), (1,)).item()
            return self._read_bg(self.bg_files[bg_idx]).float(), bg_idx
        video = random.choice(self.video_infos)
        frame_index = random.randint(self.start_index, video['total_frames'] - 1 + self.start_index)
        path = osp.join(video['frame_dir'], self.filename_tmpl.format(frame_index))
        return self._read_bg(path).float(), -2      # to pass sanity check

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
        self._store, self._pool, self._pool_key = store, None, None
        self._sharded, self._peer = None, None
        self.device = ragged.device

    def attach_sharded_pool(self, paths: Sequence[str], sharded: ShardedPool) -> None:
        """Mix from a pool sharded across the ranks of a process group (``pool.shard_extracted_backgrounds``): ``paths[i]`` names
        global image ``i`` of ``sharded``.  Each rank keeps only its own images; :meth:`device_finish` fetches the images a
        batch drew from their owners (one ``all_to_all_single``) and blends them, bit-equal to :meth:`attach_pool` with the
        replicated pool.  ``bg_files`` may list any of these names, in any order and with repeats -- the CIL pool operations
        stay inside the extracted set; a name outside it raises ``ValueError``, nothing is decoded on demand.  Sizes come from
        the index, so DataLoader workers forked after this call draw crops without reading a file.

        Every rank of the pool's group must call :meth:`device_finish` (or :meth:`mix_batch_on_device`) once per batch, in
        lockstep: see :meth:`pool.ShardedPool.fetch`."""
        if len(paths) != len(sharded):
            raise ValueError("one path per image of the sharded pool")
        of: dict = {}
        for i, p in enumerate(paths):
            of.setdefault(str(p), i)
            of.setdefault(osp.realpath(p), i)             # bg_files are matched after realpath like bg_dir (:61-68)
        self._sharded, self._shard_of, self._peer = sharded, of, None
        self._shard_rows_key, self._shard_rows = None, None
        self._store, self._pool, self._pool_key = None, None, None
        self.device = sharded.device

    def attach_peer_pool(self, paths: Sequence[str], peer: PeerPool) -> None:
        """The twin of :meth:`attach_sharded_pool` for a pool whose shards are mapped into every rank of one node
        (``pool.PeerPool.open``): the same names, the same ``ValueError`` for a name outside the index, the same draws and
        bits; but :meth:`device_finish` reads the images a batch drew straight from their owners' memory with one local
        launch (:meth:`pool.PeerPool.gather`) -- no collective, so ranks need not call it in lockstep, and the host does
        not wait for the device.  Attaching a pool of any other kind detaches this one."""
        self.attach_sharded_pool(paths, peer.sharded)
        self._peer = peer

    def _shard_index(self, path: str) -> int:
        i = self._shard_of.get(path)
        if i is None:
            i = self._shard_of.get(osp.realpath(path))
        if i is None:
            raise ValueError(f"background {path!r} of bg_files is not in the sharded pool's index; a sharded pool mixes "
                             "only the extracted backgrounds it was built from")
        return i

    def _sharded_rows(self) -> np.ndarray:
        """Global index of every entry of the current ``bg_files`` (cached per list)."""
        key = tuple(self.bg_files)
        if self._shard_rows is None or key != self._shard_rows_key:
            self._shard_rows = np.array([self._shard_index(p) for p in self.bg_files], dtype=np.int64)
            self._shard_rows_key = key
        return self._shard_rows

    # ---- per-sample API (reference contract) ---------------------------------------------------
    def prepare_train_frames(self, idx):
        """Prepare the frames for training given the index (comix_loader.py:105-124)."""
        result = super().prepare_train_frames(idx)
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
                video = random.choice(self.video_infos)
                frame_index = random.randint(self.start_index, video['total_frames'] - 1 + self.start_index)
                img = self._read_bg(osp.join(video['frame_dir'], self.filename_tmpl.format(frame_index)))
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
        dev = self.device
        i32 = lambda v: torch.tensor([v], dtype=torch.int32, device=dev)   # noqa: E731
        blend = torch.ops.bgdebias.bgmix_blend_normfg(
            imgs.to(dev, torch.float32).unsqueeze(0), bg_img.unsqueeze(0).to(dev), i32(0), i32(top), i32(left),
            torch.ones(1, dtype=torch.uint8, device=dev), torch.tensor(self.bg_mean), torch.tensor(self.bg_std),
            float(self.alpha), "NTCHW")[0]
        result['imgs'] = blend.to(imgs.device)
        result['bg_idx'] = bg_idx
        return result

    def _resized_hw(self, h: int, w: int) -> tuple:
        return (h, w) if self.bg_resize is None else resized_hw(h, w, self.bg_resize)

    def _bg_hw(self, bg_idx: int) -> tuple:
        """Size after Resize of ``bg_files[bg_idx]``: from the resident pool / store when they know the file; else a
        process that owns the GPU decodes the image into the store (once), and a forked DataLoader worker reads the image
        header (cached per path).  With a sharded pool the global index answers."""
        if self._sharded is not None:
            return self._sharded.hw(self._shard_index(self.bg_files[bg_idx]))
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
            img = torch.as_tensor(self._bg_reader(path))
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
            get = self._peer.gather if self._peer is not None else self._sharded.fetch
            batch_pool, slot = get(gidx, torch.as_tensor(bg_apply).cpu())
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
        if "aa_tables" not in self._resized_cache:
            self._resized_cache["aa_tables"] = AATables(self.device)
        return self._resized_cache["aa_tables"]

    def _lut(self, mean, std) -> torch.Tensor:
        key = ("lut", mean, std)
        if key not in self._resized_cache:
            self._resized_cache[key] = ops.make_fg_lut(mean, std, self.device)
        return self._resized_cache[key]

    @staticmethod
    def host_collate(samples: List[dict]) -> dict:
        """``collate_fn`` for ``device_mix=True`` that is safe in DataLoader worker processes (no CUDA): stacks
        the uint8 clips ``[B,T,H,W,3]`` and the per-sample draws into host tensors.  Pair it with
        :meth:`device_finish` in the training process; with ``pin_memory=True`` the batch travels as uint8,
        a quarter of the bytes of the reference's fp32 batch (libs/cil/cil.py:203-210)."""
        clips = [torch.as_tensor(s['imgs']) for s in samples]
        out = {}
        if all(c.shape == clips[0].shape for c in clips):
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
        ``randAug``, ``bg_idx``) with one fused launch.  ``dtype`` / ``memory_format``: see :meth:`mix_batch_on_device`."""
        out = {k: v for k, v in batch.items()
               if k not in ('imgs', 'bg_top', 'bg_left', 'bg_apply', 'fg_geom', 'fg_frames', 'bg_imgs', 'bg_slot')}
        if self.back_ground_from_bg_dir or 'bg_imgs' in batch:
            out['imgs'] = self.mix_batch_on_device(batch['imgs'], batch['bg_idx'], batch['bg_top'], batch['bg_left'],
                                                   batch['bg_apply'], layout=layout, fg_geom=batch.get('fg_geom'),
                                                   fg_frames=batch.get('fg_frames'), bg_imgs=batch.get('bg_imgs'),
                                                   bg_slot=batch.get('bg_slot'), dtype=dtype, memory_format=memory_format)
        else:                                             # random-frame mode and no sample of the batch was mixed
            out['imgs'] = self.mix_batch_on_device(batch['imgs'], batch['bg_idx'], batch['bg_top'], batch['bg_left'],
                                                   batch['bg_apply'], layout=layout, fg_geom=batch.get('fg_geom'),
                                                   fg_frames=batch.get('fg_frames'),
                                                   bg_imgs=[torch.zeros((3, *self.bg_crop_size), dtype=torch.uint8)],
                                                   bg_slot=torch.zeros(len(batch['bg_idx']), dtype=torch.int32),
                                                   dtype=dtype, memory_format=memory_format)
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
        if self._bg_reader is not None:
            return torch.as_tensor(self._bg_reader(path))
        from torchvision.io import ImageReadMode, read_image
        return read_image(path, mode=ImageReadMode.RGB)

    def __call__(self, results):
        results['bg_idx'] = -1
        mix = (not results['randAug']) if self.with_randAug else (random.random() < self.prob)
        if not mix:
            return results
        bg_idx = torch.randint(len(self.bg_files), (1,)).item()
        bg = resize_like_reference(self._read(self.bg_files[bg_idx]).float(), self.bg_resize)
        top, left = draw_crop(bg.shape[1], bg.shape[2], self.bg_crop_size)
        imgs = torch.as_tensor(results['imgs'])
        dev = self.device
        i32 = lambda v: torch.tensor([v], dtype=torch.int32, device=dev)   # noqa: E731
        out = torch.ops.bgdebias.bgmix_blend_normfg(
            imgs.to(dev, torch.float32).unsqueeze(0), bg.unsqueeze(0).to(dev), i32(0), i32(top), i32(left),
            torch.ones(1, dtype=torch.uint8, device=dev), torch.tensor(self.bg_mean), torch.tensor(self.bg_std),
            float(self.alpha), "NTCHW")[0]
        results['imgs'] = out.to(imgs.device)
        results['bg_idx'] = bg_idx
        return results

    def __repr__(self):
        return (f"{self.__class__.__name__}(n_bg={len(self.bg_files)}, bg_resize={self.bg_resize}, "
                f"bg_crop_size={self.bg_crop_size}, alpha={self.alpha}, prob={self.prob}, "
                f"with_randAug={self.with_randAug})")
