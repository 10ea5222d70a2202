"""GPU-resident background pool for the BG-mix blend.

The reference keeps the pool as a list of JPEG paths (``BackgroundMixDataset.bg_files``,
libs/loader/comix_loader.py:84-103) and decodes + resizes one image per mixed sample inside a
DataLoader worker (:126-140).  Here the pool is decoded and resized ONCE, with the very ops the
reference uses (``torchvision.io.read_image`` and ``torchvision.transforms.Resize``), and kept on the
device as fp32 ``[P, 3, Hb, Wb]``; the blend kernel then crops, normalises and mixes.  Index ``i`` of
the pool is index ``i`` of ``bg_files`` -- the reference's ``bg_idx``.
"""
from __future__ import annotations

from typing import Dict, List, NamedTuple, Optional, Sequence, Tuple

import numpy as np
import torch

SLOT_DTYPE = np.dtype([("offset", "<i8"), ("h", "<i4"), ("w", "<i4"), ("Hb", "<i4"), ("Wb", "<i4"),
                       ("xtab", "<i4"), ("ytab", "<i4"), ("kx", "<i4"), ("ky", "<i4")])   # bgd_ragged_slot, 40 bytes


def resized_hw(h: int, w: int, size: int) -> tuple:
    """Output size of torchvision ``Resize(int)``: short edge -> ``size``, long edge truncated."""
    short, long = (w, h) if w <= h else (h, w)
    new_short, new_long = size, int(size * long / short)
    return (new_long, new_short) if w <= h else (new_short, new_long)


def resize_like_reference(img_chw: torch.Tensor, size: Optional[int]) -> torch.Tensor:
    """``Resize(size)`` exactly as bg_pipeline applies it (comix_loader.py:72): float CHW tensor,
    torchvision defaults.  ``size=None`` skips the resize."""
    img = img_chw.float()
    if size is None:
        return img
    from torchvision.transforms import Resize
    return Resize(size)(img)


def _map_in_order(fn, items, workers: Optional[int] = None) -> list:
    """``[fn(x) for x in items]`` on a small thread pool (JPEG decode and torch's resize release the GIL); a pool of
    13,320 UCF101 backgrounds takes ~50 s to decode + resize on one thread."""
    items = list(items)
    if workers is None:
        import os
        workers = max(1, min(16, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)))
    if workers <= 1 or len(items) < 8:
        return [fn(x) for x in items]
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(workers) as ex:
        return list(ex.map(fn, items))


class AATables:
    """Weight tables of torchvision's antialiased bilinear ``Resize`` (ATen's separable CPU kernel), one per distinct
    ``(in_size, out_size)``, evaluated on the host by ``bgd_aa_resize_table`` and kept in one int32 device tensor."""

    def __init__(self, device):
        self.device = torch.device(device)
        self._host: List[np.ndarray] = []
        self._where: Dict[Tuple[int, int], Tuple[int, int]] = {}
        self._words = 0
        self._dev: Optional[torch.Tensor] = None

    def lookup(self, in_size: int, out_size: int) -> Tuple[int, int]:
        """(word offset, taps) of the table for this axis; (-1, 0) when the size does not change (the pass is skipped)."""
        if in_size == out_size:
            return -1, 0
        key = (int(in_size), int(out_size))
        if key not in self._where:
            import ctypes
            from . import _cabi
            taps = ctypes.c_int32()
            _cabi.check(_cabi.lib().bgd_aa_resize_table(key[0], key[1], ctypes.byref(taps), None, 0))
            words = np.empty(key[1] * (2 + taps.value), dtype=np.int32)
            _cabi.check(_cabi.lib().bgd_aa_resize_table(key[0], key[1], ctypes.byref(taps), words.ctypes.data, words.size))
            self._where[key] = (self._words, int(taps.value))
            self._host.append(words)
            self._words += words.size
            self._dev = None
        return self._where[key]

    @property
    def tensor(self) -> torch.Tensor:
        if self._dev is None:
            host = np.concatenate(self._host) if self._host else np.zeros(1, np.int32)
            self._dev = torch.from_numpy(host).to(self.device)
        return self._dev

    def tensor_for(self, stream: torch.cuda.Stream) -> torch.Tensor:
        """:attr:`tensor` for a launch on ``stream``.  A new key replaces the device tensor, and the caching allocator
        would hand the old one's memory to the next allocation of the stream it was made on, while a launch on
        ``stream`` may still read it; marking the use on ``stream`` keeps that memory out of reuse until the work
        enqueued there so far has finished."""
        t = self.tensor
        t.record_stream(stream)
        return t


class RaggedPool:
    """Backgrounds of ANY sizes, uint8 at native size, in one device byte buffer plus a slot table -- the form
    ``bgdebias::bgmix_blend_ragged`` reads.  ``Resize(bg_resize)`` (comix_loader.py:72) happens inside the blend launch,
    so a pool costs ``3*h*w`` bytes per image (Sth-Sth-v2: ~68 GB instead of ~308 GB resized fp32) and images of
    different widths (HMDB51, Sth-Sth-v2) share one pool, each cropped at its own resized size as the reference does."""

    def __init__(self, bg_resize: Optional[int] = 256, device="cuda", tables: Optional[AATables] = None):
        self.bg_resize = bg_resize
        self.device = torch.device(device)
        self.tables = tables if tables is not None else AATables(self.device)
        self.data: Optional[torch.Tensor] = None          # uint8 [capacity] on the device
        self.used = 0                                     # bytes in use
        self.slots = np.zeros(0, dtype=SLOT_DTYPE)        # host copy of the slot table
        self._slots_dev: Optional[torch.Tensor] = None

    def __len__(self) -> int:
        return int(self.slots.shape[0])

    def make_slot(self, offset: int, h: int, w: int) -> np.void:
        Hb, Wb = (h, w) if self.bg_resize is None else resized_hw(h, w, self.bg_resize)
        xtab, kx = self.tables.lookup(w, Wb)
        ytab, ky = self.tables.lookup(h, Hb)
        return np.array([(offset, h, w, Hb, Wb, xtab, ytab, kx, ky)], dtype=SLOT_DTYPE)[0]

    def append(self, images: Sequence) -> None:
        """``images``: uint8 ``[3, h, w]`` arrays / tensors (what ``read_image(mode=RGB)`` returns), any sizes."""
        imgs = []
        for im in images:
            t = torch.as_tensor(im)
            if t.dim() != 3 or t.shape[0] != 3 or t.dtype != torch.uint8:
                raise ValueError("background images must be uint8 [3, h, w]")
            imgs.append(t.contiguous())
        if not imgs:
            return
        sizes = [int(t.numel()) for t in imgs]
        starts = [(o + 15) & ~15 for o in np.cumsum([0] + [(n + 15) & ~15 for n in sizes[:-1]]).tolist()]
        total = starts[-1] + sizes[-1]
        base = (self.used + 15) & ~15
        need = base + total
        if self.data is None or need > self.data.numel():
            cap = max(need, 2 * (self.data.numel() if self.data is not None else 0))
            grown = torch.empty(cap, dtype=torch.uint8, device=self.device)
            if self.data is not None and self.used:
                grown[:self.used].copy_(self.data[:self.used])
            self.data = grown
        staging = torch.empty(total, dtype=torch.uint8, pin_memory=self.device.type == "cuda")
        for t, o in zip(imgs, starts):
            staging[o:o + t.numel()] = t.reshape(-1)
        self.data[base:base + total].copy_(staging, non_blocking=True)
        new = np.zeros(len(imgs), dtype=SLOT_DTYPE)
        for i, (t, o) in enumerate(zip(imgs, starts)):
            new[i] = self.make_slot(base + o, int(t.shape[1]), int(t.shape[2]))
        self.slots = np.concatenate([self.slots, new])
        self.used = need
        self._slots_dev = None

    @classmethod
    def from_uniform_buffer(cls, data: torch.Tensor, n: int, h: int, w: int, bg_resize: Optional[int] = 256) -> "RaggedPool":
        """``n`` images of one size already resident back to back in ``data`` (uint8, ``n * 3 * h * w`` bytes, planar
        ``[3][h][w]`` each): adopt the buffer as a pool without copying -- e.g. the all-gathered backgrounds of a
        dataset of one resolution kept as uint8 (Sth-Sth-v2: 220,847 x 240 x 427 x 3 = 67.9 GB)."""
        if data.dtype != torch.uint8 or data.dim() != 1 or data.numel() < n * 3 * h * w:
            raise ValueError("data must be a flat uint8 buffer of at least n * 3 * h * w bytes")
        pool = cls(bg_resize, data.device)
        pool.data, pool.used = data, n * 3 * h * w
        one = pool.make_slot(0, h, w)
        slots = np.repeat(np.array([one], dtype=SLOT_DTYPE), n)
        slots["offset"] = np.arange(n, dtype=np.int64) * (3 * h * w)
        pool.slots = slots
        return pool

    @property
    def slots_tensor(self) -> torch.Tensor:
        """The slot table as a uint8 device tensor (``len(self) * 40`` bytes)."""
        if self._slots_dev is None:
            raw = np.ascontiguousarray(self.slots).view(np.uint8).reshape(-1)
            self._slots_dev = torch.from_numpy(raw.copy()).to(self.device)
        return self._slots_dev

    def hw(self, slot: int) -> Tuple[int, int]:
        """Size of image ``slot`` after Resize -- what RandomCrop draws its offsets from."""
        s = self.slots[slot]
        return int(s["Hb"]), int(s["Wb"])

    def uniform_hw(self) -> Optional[Tuple[int, int, int, int]]:
        """(h, w, Hb, Wb) if every image has the same size, else None."""
        if not len(self):
            return None
        s0 = self.slots[0]
        same = (self.slots["h"] == s0["h"]).all() and (self.slots["w"] == s0["w"]).all()
        return (int(s0["h"]), int(s0["w"]), int(s0["Hb"]), int(s0["Wb"])) if same else None

    def resized(self, slot: int) -> torch.Tensor:
        """fp32 ``[3, Hb, Wb]``: ``Resize(bg_resize)(read_image(...).float())`` of one image, computed on the device."""
        import ctypes
        from . import _cabi
        s = self.slots[slot]
        out = torch.empty((3, int(s["Hb"]), int(s["Wb"])), dtype=torch.float32, device=self.device)
        c_slot = _cabi.RaggedSlot(*[int(s[k]) for k in SLOT_DTYPE.names])
        with torch.cuda.device(self.device):
            _cabi.check(_cabi.lib().bgd_aa_resize_u8_f32(self.data.data_ptr(), ctypes.byref(c_slot), self.tables.tensor.data_ptr(),
                                                         out.data_ptr(), int(torch.cuda.current_stream(self.device).cuda_stream)))
        return out


class BackgroundPool:
    """Backgrounds after ``Resize``, resident on one device.

    ``tensor``: fp32 (or uint8 when built with ``keep_uint8=True`` and no resize) ``[P, 3, Hb, Wb]``, or ``None`` for a
    pool that only exists in ragged form (images of several sizes, or too large to keep resized).
    ``ragged``: the :class:`RaggedPool` behind a :class:`BackgroundStore` view.
    ``names``:  one label per slot (file path or video name), same order as ``bg_files``.
    """

    def __init__(self, tensor: Optional[torch.Tensor], names: Sequence[str], ragged: Optional["RaggedPool"] = None):
        if tensor is None and ragged is None:
            raise ValueError("a pool needs a dense tensor or a ragged store")
        if tensor is not None:
            if tensor.dim() != 4 or tensor.shape[1] != 3:
                raise ValueError("pool tensor must be [P, 3, Hb, Wb]")
            if len(names) != tensor.shape[0]:
                raise ValueError("one name per pool slot")
        self.tensor = tensor                              # dense form, or None: blend from `ragged`
        self.ragged = ragged                              # uint8 images of any sizes (a store view always has it)
        self._slots_host: Optional[List[int]] = None
        self.names: List[str] = list(names)
        self.index_names: List[str] = self.names          # pool index i -> name (differs from `names` for a store view)
        self.slots: Optional[torch.Tensor] = None         # int32 [len(index_names)]: pool index -> row of `tensor`; None = identity

    def __len__(self) -> int:
        return len(self.index_names)

    @property
    def hw(self) -> tuple:
        """(Hb, Wb) of a pool whose images all resize to one shape."""
        if self.tensor is not None:
            return int(self.tensor.shape[2]), int(self.tensor.shape[3])
        u = self.ragged.uniform_hw()
        if u is None:
            raise ValueError("backgrounds of several sizes: ask hw_of(bg_idx)")
        return u[2], u[3]

    def hw_of(self, bg_idx: int) -> tuple:
        """Size after Resize of the image pool index ``bg_idx`` draws -- what RandomCrop.get_params sees
        (comix_loader.py:73 applied to that image)."""
        if self.ragged is None:
            return self.hw
        slot = self._slots_host[bg_idx] if self._slots_host is not None else bg_idx
        return self.ragged.hw(slot)

    def rows(self, bg_idx: torch.Tensor) -> torch.Tensor:
        """Rows of ``tensor`` for pool indices ``bg_idx`` (int32, on the pool's device)."""
        if self.slots is None:
            return bg_idx
        return self.slots[bg_idx.clamp(min=0, max=len(self.index_names) - 1).long()]

    @classmethod
    def from_images(cls, images: Sequence, names: Optional[Sequence[str]] = None, bg_resize: Optional[int] = 256,
                    device="cuda", keep_uint8: bool = False, ragged: Optional[bool] = None) -> "BackgroundPool":
        """``images``: uint8 RGB arrays/tensors ``[3, h, w]`` (what ``read_image(mode=RGB)`` returns).

        Images of one size give a dense pool (resized with torchvision itself on the host); images of several sizes --
        or ``ragged=True`` -- give a ragged uint8 pool that is resized inside the blend launch."""
        if len(images) == 0:
            raise ValueError("empty background pool")     # reference: torch.randint(0, ...) raises at draw time
        tens = []
        for im in images:
            t = torch.as_tensor(im)
            if t.dim() != 3 or t.shape[0] != 3:
                raise ValueError("background images must be [3, h, w]")
            tens.append(t)
        names = list(names) if names is not None else [str(i) for i in range(len(tens))]
        if ragged is None:
            ragged = len({tuple(t.shape) for t in tens}) != 1
        if ragged:
            rp = RaggedPool(bg_resize, device)
            rp.append([t.to(torch.uint8) for t in tens])
            return cls(None, names, ragged=rp)
        prepare = lambda t: t.to(torch.uint8) if (keep_uint8 and bg_resize is None) else resize_like_reference(t, bg_resize)  # noqa: E731
        pool = torch.stack(_map_in_order(prepare, tens)).contiguous()
        return cls(pool.to(device, non_blocking=True), names)

    @classmethod
    def from_files(cls, bg_files: Sequence[str], bg_resize: Optional[int] = 256, device="cuda") -> "BackgroundPool":
        """Decode with ``torchvision.io.read_image(mode=RGB)`` like ``_get_bg_image`` (comix_loader.py:130)."""
        from torchvision.io import ImageReadMode, read_image
        imgs = _map_in_order(lambda f: read_image(str(f), mode=ImageReadMode.RGB), bg_files)
        return cls.from_images(imgs, [str(f) for f in bg_files], bg_resize, device)

    @classmethod
    def from_index(cls, bg_dir, bg_resize: Optional[int] = 256, device="cuda") -> "BackgroundPool":
        """Rebuild the pool from the index the extraction CLI writes beside its JPEG folder
        (``extract_background.write_background_index``, ``<bg_dir>.bg_index.json``): same order on every rank,
        no video is read."""
        import json
        import pathlib
        bg_dir = pathlib.Path(bg_dir)
        index = bg_dir.parent / (bg_dir.name + ".bg_index.json")
        entries = json.loads(index.read_text())
        if not entries:
            raise ValueError(f"{index} lists no backgrounds")
        return cls.from_files([str(bg_dir / e["file"]) for e in entries], bg_resize, device)

    @staticmethod
    def all_gather_index(local_names: Sequence[str], group=None) -> list:
        """Index-only form of :meth:`all_gather` for pools too large to replicate (Sth-Sth-v2: ~68 GB of uint8
        backgrounds): every rank learns ``[(name, owner_rank, slot_on_owner), ...]`` in rank order -- the global
        pool index -- while the pixels stay sharded where they were extracted."""
        import torch.distributed as dist
        world = dist.get_world_size(group)
        names_per_rank: List[Optional[list]] = [None] * world
        dist.all_gather_object(names_per_rank, list(local_names), group=group)
        return [(n, r, i) for r, per in enumerate(names_per_rank) for i, n in enumerate(per)]

    # ---- one collective: assemble the pool from per-rank shards (SURVEY.md section 8e) ----------
    @staticmethod
    def all_gather(local_names: Sequence[str], local_bgs: torch.Tensor, group=None, events=None):
        """All-gather per-rank backgrounds ``[P_r, ...]`` (uint8 or fp32, any device the backend
        supports) and their names.  Returns ``(names, tensor)`` in rank order, identical on every
        rank -- the index the single-process run would have produced for the rank-ordered list.

        The pixels are gathered IN PLACE: every rank's shard lands at its final position of the result, no padded
        staging copy and no concatenation.  Shards of equal size (and the contiguous ceil split of
        extract_background.py:128-133, where only the last shard is shorter) need nothing else; for any other
        mix of sizes one compacting copy follows.  ``events``: optional pair of CUDA events recorded around the pixel
        collective alone (the name exchange before it is host work)."""
        import torch.distributed as dist
        world = dist.get_world_size(group)
        names_per_rank: List[Optional[list]] = [None] * world
        dist.all_gather_object(names_per_rank, list(local_names), group=group)
        counts = [len(n) for n in names_per_rank]
        if local_bgs.shape[0] != len(local_names):
            raise ValueError("one name per local background")
        max_n = max(counts) if counts else 0
        item_shape = tuple(local_bgs.shape[1:])
        names = [n for per in names_per_rank for n in per]
        if max_n == 0:
            return names, local_bgs.new_empty((0,) + item_shape)
        send = local_bgs.contiguous()
        if send.shape[0] < max_n:                          # a short shard sends a padded copy (only its own, small, side)
            send = torch.cat([send, send.new_zeros((max_n - send.shape[0],) + item_shape)])
        gathered = local_bgs.new_empty((world * max_n,) + item_shape)
        if events is not None:
            events[0].record()
        dist.all_gather_into_tensor(gathered, send, group=group)
        if events is not None:
            events[1].record()
        total = sum(counts)
        if all(c == max_n for c in counts[:-1]):           # gaps only after the last shard: the result is a prefix view
            return names, gathered[:total]
        # any other mix of shard sizes (not produced by the extraction's split): one compacting copy
        return names, torch.cat([gathered[r * max_n:r * max_n + c] for r, c in enumerate(counts)], 0)


def all_gather_ragged(local_names: Sequence[str], local: "RaggedPool", group=None):
    """The same collective for backgrounds of mixed sizes: every rank contributes the byte buffer of its
    :class:`RaggedPool` (the decoded JPEGs it extracted) and the image sizes; the gathered ``[world, max_bytes]``
    buffer IS the pool of the result -- the slot table carries each image's offset, so nothing is moved or padded
    after the collective.  Returns ``(names, RaggedPool)`` in rank order, identical on every rank."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    meta = [(str(n), int(s["offset"]), int(s["h"]), int(s["w"])) for n, s in zip(local_names, local.slots)]
    if len(meta) != len(local):
        raise ValueError("one name per local background")
    metas: List[Optional[list]] = [None] * world
    dist.all_gather_object(metas, (int(local.used), meta), group=group)
    max_bytes = (max(u for u, _ in metas) + 15) & ~15
    out = RaggedPool(local.bg_resize, local.device)
    if max_bytes == 0:
        return [], out
    send = torch.zeros(max_bytes, dtype=torch.uint8, device=local.device)
    if local.used:
        send[:local.used].copy_(local.data[:local.used])
    out.data = torch.empty(world * max_bytes, dtype=torch.uint8, device=local.device)
    dist.all_gather_into_tensor(out.data, send, group=group)
    out.used = world * max_bytes
    names, slots = [], []
    for r, (_, per) in enumerate(metas):
        for n, off, h, w in per:
            names.append(n)
            slots.append(out.make_slot(r * max_bytes + off, h, w))
    out.slots = np.array(slots, dtype=SLOT_DTYPE) if slots else np.zeros(0, dtype=SLOT_DTYPE)
    return names, out


def gather_extracted_backgrounds(output_dir, image_suffix: str = ".jpg", bg_resize: Optional[int] = 256, device="cuda",
                                 group=None):
    """After a sharded extraction (``extract_background`` under torchrun: one rank = one GPU = one contiguous slice of
    the sorted video list, extract_background.py:128-133) every rank holds the JPEGs it wrote.  This is the path's one
    collective: each rank decodes ITS files with ``torchvision.io.read_image(mode=RGB)`` -- the JPEG round trip is part
    of what the reference mixes (libs/loader/comix_loader.py:130), so the raw medians are not gathered -- and the
    pixels + names are all-gathered over NCCL / NVLink into a pool resident on every GPU.  Returns
    ``(paths, RaggedPool)``: the same index and pixels as decoding the whole directory on one rank."""
    import pathlib
    import torch.distributed as dist
    from torchvision.io import ImageReadMode, read_image
    from .shard import contiguous_splits
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    files = sorted(str(f) for f in pathlib.Path(output_dir).glob("*" + image_suffix))
    mine = contiguous_splits(files, world)[rank] if files else []
    local = RaggedPool(bg_resize, device)
    local.append(_map_in_order(lambda f: read_image(f, mode=ImageReadMode.RGB), mine))
    return all_gather_ragged(mine, local, group)


def _pad16(n):
    return (n + 15) & ~15


class ShardRoute(NamedTuple):
    """What one rank does in one exchange of :meth:`ShardedPool.fetch` (see :func:`route_requests`)."""
    segments: np.ndarray        # int64 [n, 3] {source offset in the local pool, offset in the send buffer, bytes}
    send_splits: List[int]      # bytes of the send buffer for each destination rank
    recv_splits: List[int]      # bytes of the receive buffer from each source rank
    recv_offsets: np.ndarray    # int64, offset in the receive buffer of each of this rank's requests, in request order


def route_requests(requests: Sequence[Sequence[int]], owner: np.ndarray, slot: np.ndarray, nbytes: np.ndarray, rank: int,
                   local_offsets: np.ndarray) -> ShardRoute:
    """Routing of one exchange, the same pure function on every rank.  ``requests[r]``: the global pool indices rank r asks for
    (deduplicated, in its request order); ``owner`` / ``slot`` / ``nbytes``: owning rank, slot on the owner and native size
    ``3*h*w`` of every global index; ``local_offsets``: byte offset of every slot of THIS rank's pool.

    The send buffer holds, for destination d = 0, 1, ..., the images d requested that this rank owns, in d's request order;
    so the chunk rank r receives from source s holds r's requests owned by s in r's order, and the receiver computes its
    offsets without asking the sender.  Every image starts on a 16-byte boundary (its size is padded), so every chunk is a
    multiple of 16 bytes and every offset of both buffers is 16-byte aligned."""
    world = len(requests)
    owner, slot, nbytes = np.asarray(owner), np.asarray(slot), np.asarray(nbytes, dtype=np.int64)
    segs, send_splits, at = [], [], 0
    for d in range(world):
        start = at
        for g in requests[d]:
            if owner[g] == rank:
                b = int(nbytes[g])
                segs.append((int(local_offsets[slot[g]]), at, b))
                at += _pad16(b)
        send_splits.append(at - start)
    mine = [int(g) for g in requests[rank]]
    recv_splits = [0] * world
    for g in mine:
        recv_splits[int(owner[g])] += _pad16(int(nbytes[g]))
    chunk_at = np.concatenate([[0], np.cumsum(recv_splits)[:-1]]).astype(np.int64) if world else np.zeros(0, np.int64)
    fill = list(chunk_at)
    recv_offsets = np.empty(len(mine), dtype=np.int64)
    for k, g in enumerate(mine):
        r = int(owner[g])
        recv_offsets[k] = fill[r]
        fill[r] += _pad16(int(nbytes[g]))
    segments = np.array(segs, dtype=np.int64).reshape(-1, 3)
    return ShardRoute(segments, send_splits, recv_splits, recv_offsets)


def peer_segments(requests: Sequence[int], owner: np.ndarray, src_offset: np.ndarray,
                  nbytes: np.ndarray) -> Tuple[np.ndarray, np.ndarray, int]:
    """Host side of :meth:`PeerPool.gather`, a pure function.  ``requests``: this rank's global pool indices (deduplicated, in
    request order, :meth:`ShardedPool.requests_of`); ``owner`` / ``src_offset`` / ``nbytes``: owning rank, byte offset in the
    owner's pool buffer and native size ``3*h*w`` of every global index.

    Returns ``(segments, dst, total)``: int64 ``[n, 4]`` rows ``{owner, source offset, destination offset, bytes}`` for
    ``ragged_gather``, the destination offset of every request, and the size of the per-batch buffer.  Image ``k`` of the
    batch is ``requests[k]``; every image starts on a 16-byte boundary (sizes are padded), as :meth:`RaggedPool.append` lays
    a pool out."""
    req = np.asarray(requests, dtype=np.int64).reshape(-1)
    b = np.asarray(nbytes, dtype=np.int64)[req]
    padded = (b + 15) & ~15
    dst = np.concatenate([[0], np.cumsum(padded)[:-1]]).astype(np.int64) if req.size else np.zeros(0, np.int64)
    segments = np.stack([np.asarray(owner, dtype=np.int64)[req], np.asarray(src_offset, dtype=np.int64)[req], dst, b], 1)
    return segments.reshape(-1, 4), dst, int(padded.sum())


class ShardedPool:
    """A background pool sharded across the ranks of a process group: each rank keeps only the images it owns (a
    :class:`RaggedPool`, ~1/world of the replica: Sth-Sth-v2 67.9 GB -> ~8.5 GB per GPU on 8), plus the global index that
    every rank holds identically -- ``names[P]``, ``owner[P]``, ``slot[P]`` and the native ``h[P]``, ``w[P]`` -- and one
    :class:`AATables` with the resize tables of every size in the index.  Index ``i`` is what
    ``BackgroundPool.all_gather_index`` calls ``i``: ranks in order, each rank's images in its order.

    :meth:`fetch` brings the images a batch drew to the rank that mixes it, as whole native images, and returns them as a
    per-batch :class:`RaggedPool` -- the form ``bgmix_blend_ragged`` reads, bit-equal to blending from the replica.

    ``group``: the process group the index was gathered over (``None``: the default group); ``rank`` / ``world`` are this
    process's rank in it and its size, and :meth:`fetch` runs its collectives on it, so the routing and the exchange can
    never use different groups."""

    def __init__(self, local: RaggedPool, names: Sequence[str], owner, slot, h, w, rank: int, world: int, group=None):
        self.local = local
        self.names: List[str] = list(names)
        self.owner = np.asarray(owner, dtype=np.int64)
        self.slot = np.asarray(slot, dtype=np.int64)
        self.h = np.asarray(h, dtype=np.int64)
        self.w = np.asarray(w, dtype=np.int64)
        self.rank, self.world = int(rank), int(world)
        self.group = group
        self.bg_resize = local.bg_resize
        self.device = local.device
        self.tables = local.tables
        if not (len(self.names) == len(self.owner) == len(self.slot) == len(self.h) == len(self.w)):
            raise ValueError("one owner, slot and size per index entry")
        if int((self.owner == self.rank).sum()) != len(local):
            raise ValueError("the local pool must hold exactly the images the index assigns to this rank")
        misaligned = np.flatnonzero(local.slots["offset"] % 16) if len(local) else np.zeros(0, np.int64)
        if misaligned.size:
            # ragged_pack reads whole images with 16-byte vectors; RaggedPool.append aligns every image, a pool adopted with
            # from_uniform_buffer only when 3*h*w is a multiple of 16
            raise ValueError(f"local image {int(misaligned[0])} starts at byte {int(local.slots['offset'][misaligned[0]])}, "
                             "not a multiple of 16: a sharded pool needs 16-byte aligned images (build it with "
                             "RaggedPool.append)")
        self.nbytes = 3 * self.h * self.w
        self._hw: Dict[Tuple[int, int], Tuple[int, int]] = {}      # native -> resized size; fills the tables for every size
        for hw in set(zip(self.h.tolist(), self.w.tolist())):
            s = local.make_slot(0, *hw)
            self._hw[hw] = (int(s["Hb"]), int(s["Wb"]))

    def __len__(self) -> int:
        return len(self.names)

    @classmethod
    def from_local(cls, names: Sequence[str], ragged: RaggedPool, group=None) -> "ShardedPool":
        """Collective: one ``all_gather_object`` of ``(name, h, w)`` per local image -- the index of ``all_gather_index``
        plus the native sizes.  ``names[i]`` is image ``i`` of ``ragged``; no pixel leaves its rank."""
        import torch.distributed as dist
        if len(names) != len(ragged):
            raise ValueError("one name per local background")
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        meta = [(str(n), int(s["h"]), int(s["w"])) for n, s in zip(names, ragged.slots)]
        metas: List[Optional[list]] = [None] * world
        dist.all_gather_object(metas, meta, group=group)
        rows = [(n, r, i, hh, ww) for r, per in enumerate(metas) for i, (n, hh, ww) in enumerate(per)]
        cols = list(zip(*rows)) if rows else [[]] * 5
        return cls(ragged, cols[0], cols[1], cols[2], cols[3], cols[4], rank, world, group)

    def index(self) -> list:
        """``[(name, owner_rank, slot_on_owner), ...]``: what ``BackgroundPool.all_gather_index`` returns."""
        return [(n, int(r), int(i)) for n, r, i in zip(self.names, self.owner, self.slot)]

    def hw(self, i: int) -> Tuple[int, int]:
        """Size after Resize of global image ``i`` -- what RandomCrop draws its offsets from."""
        return self._hw[(int(self.h[i]), int(self.w[i]))]

    @property
    def resident_bytes(self) -> int:
        """Bytes of the local pool buffer on this rank's device."""
        return int(self.local.data.numel()) if self.local.data is not None else 0

    @staticmethod
    def requests_of(bg_idx, apply) -> List[int]:
        """The global indices a batch asks for: those of the applied samples, deduplicated, in sample order."""
        idx = torch.as_tensor(bg_idx).tolist()
        app = torch.as_tensor(apply).tolist()
        return list(dict.fromkeys(int(g) for g, a in zip(idx, app) if a))

    def route(self, requests: Sequence[Sequence[int]]) -> ShardRoute:
        """:func:`route_requests` for this rank."""
        for r, req in enumerate(requests):
            bad = [g for g in req if not 0 <= g < len(self)]
            if bad:
                raise ValueError(f"rank {r} requests background {bad[0]}, outside the {len(self)}-image index")
        return route_requests(requests, self.owner, self.slot, self.nbytes, self.rank, self.local.slots["offset"])

    def pack(self, route: ShardRoute) -> torch.Tensor:
        """The send buffer of ``route``: one ``ragged_pack`` launch over the local pool."""
        total = int(sum(route.send_splits))
        src = self.local.data if self.local.data is not None else torch.empty(0, dtype=torch.uint8, device=self.device)
        return torch.ops.bgdebias.ragged_pack(src, torch.from_numpy(route.segments), total)

    def assemble(self, recv: torch.Tensor, requests: Sequence[int], route: ShardRoute) -> RaggedPool:
        """The per-batch pool over the receive buffer: image ``k`` is ``requests[k]`` (this rank's requests)."""
        batch = RaggedPool(self.bg_resize, self.device, tables=self.tables)
        batch.data, batch.used = recv, int(recv.numel())
        slots = [self.local.make_slot(int(o), int(self.h[g]), int(self.w[g])) for o, g in zip(route.recv_offsets, requests)]
        batch.slots = np.array(slots, dtype=SLOT_DTYPE) if slots else np.zeros(0, dtype=SLOT_DTYPE)
        return batch

    def fetch(self, bg_idx, apply) -> Tuple[RaggedPool, torch.Tensor]:
        """Collective.  ``bg_idx`` / ``apply`` ([B], host or device): the global pool index and the mix flag of every sample
        of this rank's batch.  Returns ``(batch pool, slot)``: a :class:`RaggedPool` holding the drawn images and the int32
        ``[B]`` slot of each sample in it (0 for a sample that is not mixed; the blend ignores it).

        EVERY rank of the pool's group must call ``fetch`` once per batch, in the same order -- also at world size 1 and
        for a batch that mixes nothing -- because the call is two collectives on that group: an ``all_gather_object`` of
        every rank's requests (after which every rank knows the whole request matrix and computes its send segments, its
        receive splits and the receive offsets with :func:`route_requests`, no further exchange), then one ``ragged_pack``
        launch and one ``all_to_all_single`` of bytes on the current stream.  The self-chunk carries the rank's own images,
        so local and remote images take the same path.  A DDP training step, which mixes one batch per rank per step, meets
        this.

        The host waits here: the split sizes of ``all_to_all_single`` must be known on the host, and on an NCCL group
        ``all_gather_object`` reads the gathered sizes back from the device, so the call returns only after the work already
        queued on the current stream (e.g. the previous step's backward) has finished.  The replicated pool never waits."""
        import torch.distributed as dist
        mine = self.requests_of(bg_idx, apply)
        requests: List[Optional[list]] = [None] * self.world
        dist.all_gather_object(requests, mine, group=self.group)
        route = self.route(requests)
        recv = torch.empty(int(sum(route.recv_splits)), dtype=torch.uint8, device=self.device)
        if any(requests):                                  # every rank sees the same matrix: all skip or none does
            send = self.pack(route)
            dist.all_to_all_single(recv, send, route.recv_splits, route.send_splits, group=self.group)
        return self.assemble(recv, mine, route), self.sample_slots(bg_idx, apply, mine)

    @staticmethod
    def sample_slots(bg_idx, apply, requests: Sequence[int]) -> torch.Tensor:
        """int32 ``[B]``: the image of the batch pool each sample blends (0 for a sample that is not mixed)."""
        where = {g: k for k, g in enumerate(requests)}
        app = torch.as_tensor(apply).tolist()
        return torch.tensor([where[int(g)] if a else 0 for g, a in zip(torch.as_tensor(bg_idx).tolist(), app)],
                            dtype=torch.int32)


_USE_FETCH = ("mix from this pool with BackgroundMixDataset.attach_sharded_pool (ShardedPool.fetch, an exchange over the "
              "process group) instead")


def check_peer_meta(metas: Sequence[dict]) -> None:
    """The refusals of :meth:`PeerPool.open` that every rank decides alike from the gathered metadata, a pure function.
    ``metas[r]``: ``host`` (host id), ``uuid`` (device), ``handle`` (64 bytes, or ``None`` for an empty shard), ``offset``,
    ``bytes`` and ``error`` (why the shard could not be exported, or ``None``) of rank ``r``.  Raises ``ValueError`` when the
    ranks do not all run on one host, or when a rank could not export its shard."""
    for r, m in enumerate(metas):
        if m["host"] != metas[0]["host"]:
            raise ValueError(f"ranks 0 and {r} run on different hosts ({metas[0]['host']!r}, {m['host']!r}): a PeerPool maps "
                             f"GPU memory between the processes of one node; {_USE_FETCH}")
    for r, m in enumerate(metas):
        if m["error"] is not None:
            raise ValueError(f"rank {r} cannot export its shard for peer mapping: {m['error']}; {_USE_FETCH}")
        if m["handle"] is not None and (len(m["handle"]) != 64 or m["offset"] % 16):
            raise ValueError(f"rank {r} exported a malformed handle or an unaligned buffer (offset {m['offset']}); {_USE_FETCH}")


def _host_id() -> str:
    """Host name plus the kernel's boot id: two machines that share a host name still differ."""
    import socket
    try:
        with open("/proc/sys/kernel/random/boot_id") as f:
            boot = f.read().strip()
    except OSError:
        boot = ""
    return f"{socket.gethostname()}/{boot}"


class PeerPool:
    """A :class:`ShardedPool` whose shards are mapped into every rank of one node, so a rank reads the images its batch drew
    straight from their owners' HBM (over NVLink between GPUs) instead of exchanging them.  Built by :meth:`open`, a
    collective; after it :meth:`gather` is local: one ``ragged_gather`` launch per batch, no collective, no lockstep between
    ranks and no host synchronisation.  The result is bit-equal to the replica, as for :meth:`ShardedPool.fetch`.

    ``bases`` (device int64 ``[W]``) holds, for every rank, the address of its pool buffer in this process -- this rank's own
    buffer, or a peer mapping -- and ``base_bytes`` (host int64 ``[W]``) the bytes in use there; ``src_offset[i]`` is the byte
    offset of global image ``i`` in its owner's buffer.  The pool keeps ``sharded`` -- and with it the local buffer that peers
    read -- alive.  Lifetime rule: :meth:`close` (collective) before any rank drops, grows or appends to its shard."""

    def __init__(self, sharded: ShardedPool, bases: Sequence[int], base_bytes: Sequence[int], src_offset,
                 mapped: Optional[Dict[int, int]] = None):
        if not (len(bases) == len(base_bytes) == sharded.world):
            raise ValueError("one base address and size per rank")
        if any(int(b) % 16 for b in bases):
            raise ValueError("ragged_gather reads 16-byte vectors: every base address must be 16-byte aligned")
        self.sharded = sharded
        self.device = sharded.device
        self.bases: Optional[torch.Tensor] = torch.tensor([int(b) for b in bases], dtype=torch.int64, device=self.device)
        self.base_bytes = torch.tensor([int(b) for b in base_bytes], dtype=torch.int64)
        self.src_offset = np.asarray(src_offset, dtype=np.int64)
        if len(self.src_offset) != len(sharded):
            raise ValueError("one source offset per index entry")
        self._mapped: Dict[int, int] = dict(mapped or {})          # rank -> base returned by bgd_ipc_open
        local = sharded.local
        self._local_state = self._state(local)

    @staticmethod
    def _state(local: RaggedPool) -> tuple:
        return (id(local.data), local.data.data_ptr() if local.data is not None else 0, local.used, len(local))

    def __len__(self) -> int:
        return len(self.sharded)

    @classmethod
    def open(cls, sharded: ShardedPool) -> "PeerPool":
        """Collective on ``sharded.group``: map every rank's shard into every other rank.  Each rank synchronises its device
        (its shard is fully written), exports its buffer (``bgd_ipc_export``), and one ``all_gather_object`` shares
        ``(host id, device UUID, handle, offset, bytes)`` and the slot offsets; each rank then opens every other rank's handle
        (its own buffer is used directly: a handle cannot be opened in the process that exported it), and a second gather of
        the outcomes makes every rank raise together.  ``ValueError`` -- pointing at ``attach_sharded_pool`` / ``fetch`` --
        when the ranks are on different hosts, when a buffer cannot be exported (``expandable_segments``, the
        ``cudaMallocAsync`` backend) or when a peer cannot be mapped."""
        import ctypes
        import torch.distributed as dist
        from . import _cabi
        local, rank, group = sharded.local, sharded.rank, sharded.group
        dev = sharded.device if sharded.device.index is not None else torch.device("cuda", torch.cuda.current_device())
        torch.cuda.synchronize(dev)
        meta = dict(host=_host_id(), uuid=str(torch.cuda.get_device_properties(dev).uuid), handle=None, offset=0,
                    bytes=int(local.used), error=None, offsets=np.asarray(local.slots["offset"], dtype=np.int64))
        if local.used:
            handle = ctypes.create_string_buffer(64)
            off = ctypes.c_int64()
            try:
                with torch.cuda.device(dev):
                    _cabi.check(_cabi.lib().bgd_ipc_export(local.data.data_ptr(), handle, ctypes.byref(off)))
                meta.update(handle=handle.raw, offset=int(off.value))
            except (ValueError, _cabi.BgdError) as e:
                meta["error"] = str(e)
        metas: List[Optional[dict]] = [None] * sharded.world
        dist.all_gather_object(metas, meta, group=group)
        check_peer_meta(metas)
        mapped: Dict[int, int] = {}
        error = None
        for r, m in enumerate(metas):
            if r == rank or m["handle"] is None:
                continue
            base = ctypes.c_void_p()
            try:
                _cabi.check(_cabi.lib().bgd_ipc_open(m["handle"], dev.index, ctypes.byref(base)))
            except (ValueError, _cabi.BgdError) as e:
                error = f"rank {rank} (device {meta['uuid']}) cannot map the shard of rank {r} (device {m['uuid']}): {e}"
                break
            mapped[r] = int(base.value)
        errors: List[Optional[str]] = [None] * sharded.world
        dist.all_gather_object(errors, error, group=group)
        failed = [e for e in errors if e is not None]
        if failed:
            _close_mappings(mapped, dev)
            raise ValueError(f"{failed[0]}; {_USE_FETCH}")
        bases = [local.data.data_ptr() if r == rank and local.used else
                 (mapped[r] + m["offset"] if r in mapped else 0) for r, m in enumerate(metas)]
        src_offset = np.zeros(len(sharded), dtype=np.int64)
        for r, m in enumerate(metas):
            own = sharded.owner == r
            src_offset[own] = m["offsets"][sharded.slot[own]]
        return cls(sharded, bases, [m["bytes"] for m in metas], src_offset, mapped)

    def gather(self, bg_idx, apply) -> Tuple[RaggedPool, torch.Tensor]:
        """Local.  ``bg_idx`` / ``apply`` ([B], host or device): the global pool index and the mix flag of every sample of this
        rank's batch.  Returns ``(batch pool, slot)`` as :meth:`ShardedPool.fetch` does -- the same deduplicated request order,
        every image on a 16-byte boundary, the int32 ``[B]`` slot of each sample (0 for a sample that is not mixed) -- from one
        ``ragged_gather`` launch on the current stream.  Ranks call it independently, as many times as they like; the host
        never waits for the device (the slot table travels from pinned memory, and ``slot`` is returned pinned)."""
        if self.bases is None:
            raise RuntimeError("PeerPool.gather after close()")
        sp = self.sharded
        if self._state(sp.local) != self._local_state:
            raise RuntimeError("the local shard was reallocated or appended to after PeerPool.open: peers would read a stale "
                               "mapping; close() the PeerPool before changing a shard, then open a new one")
        mine = sp.requests_of(bg_idx, apply)
        bad = [g for g in mine if not 0 <= g < len(sp)]
        if bad:
            raise ValueError(f"background {bad[0]} is outside the {len(sp)}-image index")
        segments, dst, total = peer_segments(mine, sp.owner, self.src_offset, sp.nbytes)
        batch = RaggedPool(sp.bg_resize, self.device, tables=sp.tables)
        batch.data = torch.ops.bgdebias.ragged_gather(self.bases, self.base_bytes, torch.from_numpy(segments), total)
        batch.used = total
        if mine:
            batch.slots = np.array([sp.local.make_slot(int(o), int(sp.h[g]), int(sp.w[g])) for o, g in zip(dst, mine)],
                                   dtype=SLOT_DTYPE)
            raw = torch.from_numpy(batch.slots.view(np.uint8).reshape(-1))
            batch._slots_dev = raw.pin_memory().to(self.device, non_blocking=True)
        return batch, sp.sample_slots(bg_idx, apply, mine).pin_memory()     # pinned: its upload does not wait either

    def close(self) -> None:
        """Collective on the pool's group: each rank synchronises its device (its gathers have finished reading), all ranks
        meet at a barrier, then each unmaps its peers' shards.  Call it before any rank drops or changes its shard."""
        import torch.distributed as dist
        if self.bases is None:
            return
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.sharded.group)
        _close_mappings(self._mapped, self.device)
        self._mapped, self.bases = {}, None


def _close_mappings(mapped: Dict[int, int], device) -> None:
    from . import _cabi
    with torch.cuda.device(device):
        for base in mapped.values():
            _cabi.check(_cabi.lib().bgd_ipc_close(base))
    mapped.clear()


def shard_extracted_backgrounds(output_dir, image_suffix: str = ".jpg", bg_resize: Optional[int] = 256, device="cuda",
                                group=None):
    """The sharded twin of :func:`gather_extracted_backgrounds`: the same contiguous split of the sorted JPEGs, each rank
    decodes its own files with ``torchvision.io.read_image(mode=RGB)`` and KEEPS them; only names and sizes are all-gathered.
    Returns ``(paths, ShardedPool)`` with ``paths[i]`` the file of global index ``i`` (the same list, in the same order, as
    :func:`gather_extracted_backgrounds` returns)."""
    import pathlib
    import torch.distributed as dist
    from torchvision.io import ImageReadMode, read_image
    from .shard import contiguous_splits
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    files = sorted(str(f) for f in pathlib.Path(output_dir).glob("*" + image_suffix))
    mine = contiguous_splits(files, world)[rank] if files else []
    local = RaggedPool(bg_resize, device)
    local.append(_map_in_order(lambda f: read_image(f, mode=ImageReadMode.RGB), mine))
    sharded = ShardedPool.from_local(mine, local, group)
    return list(sharded.names), sharded


class BackgroundStore:
    """Backgrounds resident on one device across pool changes (SURVEY.md section 8f, row 3).

    The reference's trainer rewrites ``dataset.bg_files`` between CIL tasks -- ``keep_all_backgrounds``
    (libs/cil/cil.py:193-195,690-694), ``cbf_full_bg`` (:146-160) and ``merge_bg_files`` (:390-393) are
    unions / extensions of path lists -- and every sample then decodes its background again.  Here each
    path is decoded once and stays on the device as uint8 at its native size (:class:`RaggedPool`: any mix of
    sizes, ``Resize`` evaluated inside the blend launch); a pool is an int32 slot table over the store, so set
    operations on the path lists never copy or re-decode pixels, and duplicates in ``bg_files`` (``extend``
    creates them) share a slot and keep their draw probability.

    When every image has the same size and the resized fp32 copy fits ``dense_budget_bytes`` (default: a quarter
    of the device's memory), :attr:`tensor` additionally caches ``Resize(bg_resize)`` of every image as fp32
    ``[n, 3, Hb, Wb]`` -- computed on the device by the same arithmetic -- and the blend reads that instead
    (one load per value instead of a 2x2..3x3 tap window).  Both forms give identical bits.
    """

    def __init__(self, bg_resize: Optional[int] = 256, device="cuda", keep_uint8: bool = False,
                 dense_budget_bytes: Optional[int] = None):
        self.bg_resize = bg_resize
        self.device = torch.device(device)
        self.keep_uint8 = keep_uint8                      # dense cache as uint8 (only without a resize)
        self.ragged = RaggedPool(bg_resize, self.device)
        self.slot_of: dict = {}                           # name -> slot
        self.decoded = 0                                  # images decoded so far (what a rebuild would repeat)
        self.dense_budget_bytes = dense_budget_bytes
        self._dense: Optional[torch.Tensor] = None        # [capacity, 3, Hb, Wb]
        self._dense_rows = 0

    def __len__(self) -> int:
        return len(self.slot_of)

    @property
    def hw(self) -> tuple:
        """(Hb, Wb) of a store whose images all have one size."""
        u = self.ragged.uniform_hw()
        if u is None:
            raise ValueError("empty background store" if not len(self) else
                             "backgrounds of several sizes: ask hw_of(slot)")
        return u[2], u[3]

    def hw_of(self, slot: int) -> tuple:
        return self.ragged.hw(slot)

    def ensure(self, names: Sequence[str], reader) -> None:
        """Make every name resident; ``reader(name) -> uint8 [3, h, w]`` is called for new names only."""
        new = [n for n in dict.fromkeys(names) if n not in self.slot_of]
        if not new:
            return
        def prepare(n):
            t = torch.as_tensor(reader(n))
            if t.dim() != 3 or t.shape[0] != 3:
                raise ValueError("background images must be [3, h, w]")
            return t.to(torch.uint8)

        imgs = _map_in_order(prepare, new)
        used = len(self.slot_of)
        self.ragged.append(imgs)
        for i, n in enumerate(new):
            self.slot_of[n] = used + i
        self.decoded += len(new)

    def adopt(self, names: Sequence[str], ragged: "RaggedPool") -> None:
        """Start from an already resident pool (``gather_extracted_backgrounds``): ``names[i]`` is image ``i`` of
        ``ragged``; nothing is decoded.  Only for an empty store."""
        if len(self.slot_of):
            raise ValueError("adopt() needs an empty store")
        if len(names) != len(ragged) or ragged.bg_resize != self.bg_resize:
            raise ValueError("one name per image, same bg_resize")
        self.ragged = ragged
        self.device = ragged.device
        self.slot_of = {}
        for i, n in enumerate(names):
            self.slot_of.setdefault(n, i)                # a repeated name keeps its first image

    def _budget(self) -> int:
        if self.dense_budget_bytes is not None:
            return int(self.dense_budget_bytes)
        if self.device.type == "cuda":
            return int(torch.cuda.get_device_properties(self.device).total_memory // 4)
        return 1 << 34

    @property
    def tensor(self) -> Optional[torch.Tensor]:
        """Dense cache ``[len(self), 3, Hb, Wb]`` (fp32 after Resize, or uint8 with ``keep_uint8`` and no resize) for a
        store of one image size within the budget, else ``None`` (the blend then reads the ragged store)."""
        n = len(self)
        u = self.ragged.uniform_hw()
        if u is None or n == 0:
            self._dense, self._dense_rows = None, 0
            return None
        h, w, Hb, Wb = u
        as_u8 = self.keep_uint8 and self.bg_resize is None
        if n * 3 * Hb * Wb * (1 if as_u8 else 4) > self._budget():
            self._dense, self._dense_rows = None, 0
            return None
        if self._dense is None or self._dense.shape[0] < n:
            cap = max(n, 2 * (self._dense.shape[0] if self._dense is not None else 0))
            grown = torch.empty((cap, 3, Hb, Wb), dtype=torch.uint8 if as_u8 else torch.float32, device=self.device)
            if self._dense is not None and self._dense_rows:
                grown[:self._dense_rows].copy_(self._dense[:self._dense_rows])
            self._dense = grown
        for slot in range(self._dense_rows, n):
            s = self.ragged.slots[slot]
            if (h, w) == (Hb, Wb) or self.device.type != "cuda":
                raw = self.ragged.data[int(s["offset"]):int(s["offset"]) + 3 * h * w].view(3, h, w)
                self._dense[slot].copy_(raw if as_u8 else resize_like_reference(raw, None if (h, w) == (Hb, Wb) else self.bg_resize))
            else:
                self._dense[slot].copy_(self.ragged.resized(slot))
        self._dense_rows = n
        return self._dense[:n]

    def view(self, names: Sequence[str]) -> "BackgroundPool":
        """The pool whose index ``i`` is ``names[i]`` (the reference's ``bg_idx``): shares this store's
        pixels; ``slots`` maps pool index -> store slot."""
        if len(names) == 0:
            raise ValueError("empty background pool")
        missing = [n for n in names if n not in self.slot_of]
        if missing:
            raise KeyError(f"{len(missing)} backgrounds are not resident (first: {missing[0]}); call ensure() first")
        pool = BackgroundPool(self.tensor, list(self.slot_of), ragged=self.ragged)
        pool.index_names = list(names)
        pool.slots = torch.tensor([self.slot_of[n] for n in names], dtype=torch.int32, device=self.device)
        pool._slots_host = [self.slot_of[n] for n in names]
        return pool
