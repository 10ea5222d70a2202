"""Video-to-GPU staging: pinned double buffer between the host decoder and the median kernel.

The reference keeps a Python list of decoded frames per video and calls ``np.median`` on it
(cil_tools/extract_background.py:48-73).  Here decoded frames are written straight into a pinned
slab that holds several whole videos back to back (``[sum T, N]`` uint8 plus the offsets table);
when a slab is full it is copied to the device on its own stream, reduced with one
``temporal_median_varlen`` launch, and the ``[V, N]`` backgrounds are copied back -- while the
decoder is already filling the other slab.

``add_video`` may be called from many decoder threads at once: a thread reserves its rows under a lock and
copies its frames into the slab outside it (numpy releases the GIL for the copy), so packing scales with the
decoder threads instead of serialising on the caller.

What a slab is reduced with is a parameter (``reduce=``): :class:`MedianReduce` (the default, tmf) or
``extract_background.SimCamReduce`` (RandomResizedCrop + NaN-masked median / mean, whose frames may differ in size).
"""
from __future__ import annotations

import threading
from typing import Callable, List, Optional, Sequence

import numpy as np
import torch

from . import ops as _ops  # noqa: F401  (registers torch.ops.bgdebias.*)


class _Slab:
    def __init__(self, nbytes: int, device: torch.device):
        with torch.cuda.device(device):
            self.host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
            self.dev = torch.empty(nbytes, dtype=torch.uint8, device=device)
            self.stream = torch.cuda.Stream(device)
            self.done = torch.cuda.Event()
        self.reset()

    def reset(self):
        self.used = 0
        self.N = None
        self.offsets: List[int] = [0]
        self.tags: list = []
        self.shapes: list = []             # result shape per video
        self.starts: List[int] = []        # first byte of each video in the slab
        self.metas: list = []              # per-video data for the reduction (add_video's `meta`)
        self.out_host: Optional[torch.Tensor] = None
        self.pending = False
        self.filling = 0                   # reservations whose frames are still being copied in


class MedianReduce:
    """The tmf reduction: per-pixel temporal median of every video of a slab, one ``temporal_median_varlen`` launch.
    All frames of a slab have one size."""
    mixed_sizes = False

    def result_shape(self, frame_shape: tuple) -> tuple:
        return frame_shape

    def __call__(self, data: torch.Tensor, slab: "_Slab") -> torch.Tensor:
        """``data``: the slab's bytes on the device; returns uint8 ``[V, N]`` on the current stream."""
        return torch.ops.bgdebias.temporal_median_varlen(data.view(slab.offsets[-1], slab.N),
                                                         torch.tensor(slab.offsets, dtype=torch.int64))


class FrameStager:
    """``add_video(frames, tag)`` queues one decoded video (list/array of uint8 frames);
    ``on_result(tag, background_ndarray)`` is called for every video once its reduction (``reduce``, by default the
    temporal median) is back on the host.  Call :meth:`flush` at the end."""

    def __init__(self, on_result: Callable, device="cuda", slab_mb: int = 512, reduce=None):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("FrameStager needs a CUDA device: there is no CPU path")
        self.on_result = on_result
        self.reduce = reduce if reduce is not None else MedianReduce()
        self.slab_bytes = int(slab_mb) << 20
        self.slabs: List[Optional[_Slab]] = [None, None]
        self.cur = 0
        self._cv = threading.Condition()

    def add_video(self, frames: Sequence[np.ndarray], tag, meta=None) -> None:
        """Thread-safe.  ``frames``: a list of uint8 frames (arrays or CPU tensors; of one shape unless the reduction
        takes mixed sizes) or one ``[T, ...]`` uint8 array, packed back to back.  ``meta`` goes to the reduction."""
        T = len(frames)
        if T == 0:
            # reference: np.median([]) -> nan -> cv2.imwrite raises (extract_background.py:73-74)
            raise ValueError(f"{tag}: no frames decoded")
        shape = tuple(frames[0].shape)
        stacked = isinstance(frames, np.ndarray)
        if stacked:
            if frames.dtype != np.uint8:
                raise ValueError(f"{tag}: frames must be uint8")
            sizes = None
        else:
            frames = [np.asarray(f) for f in frames]
            for t, f in enumerate(frames):
                if f.dtype != np.uint8 or (tuple(f.shape) != shape and not self.reduce.mixed_sizes):
                    raise ValueError(f"{tag}: frame {t} differs in shape or dtype")
            sizes = [f.size for f in frames]
        N = int(np.prod(shape))
        need = T * N if sizes is None else sum(sizes)
        with self._cv:
            slab = self._room_for(need, None if self.reduce.mixed_sizes else N)
            off = slab.used
            slab.N = None if self.reduce.mixed_sizes else N
            slab.used += need
            slab.offsets.append(slab.offsets[-1] + T)
            slab.tags.append(tag)
            slab.shapes.append(self.reduce.result_shape(shape))
            slab.starts.append(off)
            slab.metas.append(meta)
            slab.filling += 1
        try:
            if stacked:
                slab.host[off:off + need].view(T, N).numpy()[:] = frames.reshape(T, N)
            else:
                buf = slab.host[off:off + need].numpy()
                pos = 0
                for f, n in zip(frames, sizes):
                    buf[pos:pos + n] = f.reshape(-1)
                    pos += n
        finally:
            with self._cv:
                slab.filling -= 1
                self._cv.notify_all()

    def _room_for(self, need: int, N: int) -> _Slab:
        """The slab the next ``need`` bytes go to (lock held): submits the current one when it is full or holds
        frames of another size -- after every thread still copying into it has finished -- and moves to the other."""
        while True:
            i = self.cur
            slab = self.slabs[i]
            if slab is None:
                self.slabs[i] = slab = _Slab(max(self.slab_bytes, need), self.device)
                return slab
            if slab.pending:
                self._drain(i)
            if slab.used == 0 and slab.host.numel() < need:           # a video larger than the slab: grow it
                self.slabs[i] = slab = _Slab(need, self.device)
                return slab
            if slab.used + need <= slab.host.numel() and (slab.used == 0 or slab.N == N):
                return slab
            while slab.filling:
                self._cv.wait()
            if self.cur == i and self.slabs[i] is slab and slab.used and not slab.pending:    # nobody else did it meanwhile
                self._submit(i)
                self.cur ^= 1

    def _submit(self, i: int) -> None:
        slab = self.slabs[i]
        if slab is None or not slab.tags:
            return
        # decoder threads land here too: the current device is per thread
        with torch.cuda.device(self.device), torch.cuda.stream(slab.stream):
            slab.dev[:slab.used].copy_(slab.host[:slab.used], non_blocking=True)
            out = self.reduce(slab.dev[:slab.used], slab)
            slab.out_host = torch.empty(out.shape, dtype=torch.uint8, pin_memory=True)
            slab.out_host.copy_(out, non_blocking=True)
            slab.done.record(slab.stream)
        slab.pending = True

    def _drain(self, i: int) -> None:
        slab = self.slabs[i]
        if slab is None or not slab.pending:
            return
        slab.done.synchronize()
        res = slab.out_host.numpy()
        for v, (tag, shape) in enumerate(zip(slab.tags, slab.shapes)):
            self.on_result(tag, res[v].reshape(shape).copy())
        slab.reset()

    def flush(self) -> None:
        """Call after every ``add_video`` has returned."""
        with self._cv:
            while any(sl is not None and sl.filling for sl in self.slabs):
                self._cv.wait()
            self._submit(self.cur)
            for i in (self.cur ^ 1, self.cur):
                self._drain(i)
