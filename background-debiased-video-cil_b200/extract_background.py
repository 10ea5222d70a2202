"""Drop-in for ``cil_tools/extract_background.py`` of the reference: same CLI flags, same function
signatures, same output files (``<output_dir>/<video name>.jpg``); the per-pixel temporal median
runs on the GPU (``torch.ops.bgdebias.temporal_median*``), everything else stays on the host.

    python -m bgdebias_b200.extract_background --video_dir D --output_dir O --from_video \
        [--glob_pattern '*'] [--num_workers 4] [--image_suffix .jpg] [--interval 1] \
        [--max_frames 500] [--size 256] [--method tmf] [--avg_method median]

``--num_workers`` keeps its meaning "number of parallel shards of the video list"; every shard is
one process bound to one GPU (shard i -> GPU i mod #GPUs).  Additional, optional flags:
``--decode_threads`` (host decoder threads per shard) and ``--slab_mb`` (pinned staging slab size).

Behaviour kept from the reference on purpose
* frames are kept while ``len(frames) <= max_frames``: up to ``max_frames + 1`` frames (:52);
* a frame is kept when ``count % interval == 0`` where ``count`` counts decoded frames (:54-60);
* ``--size`` is accepted and unused, backgrounds are written at native resolution (:27,57);
* videos whose output already exists are skipped (:119-126).
Behaviour NOT kept: the image-folder branch of the reference raises ``ValueError`` on the first
readable image (``if img:`` on an ndarray, :67-68); here it reads the images as evidently intended.
"""
from __future__ import annotations

import argparse
import json
import os
import pathlib
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from typing import List

import cv2
import numpy as np
import torch

from . import shard as _shard
from .staging import FrameStager


def parse_args(argv=None):
    parser = argparse.ArgumentParser()
    parser.add_argument('--video_dir', required=True)
    parser.add_argument('--glob_pattern', default='*')
    parser.add_argument('--output_dir', required=True)
    parser.add_argument('--num_workers', type=int, default=4)
    parser.add_argument('--from_video', action='store_true')
    parser.add_argument('--image_suffix', default='.jpg')
    parser.add_argument('--interval', type=int, default=1)
    parser.add_argument('--max_frames', type=int, default=500)
    parser.add_argument('--size', type=int, default=256)
    parser.add_argument('--method', default='tmf')
    parser.add_argument('--avg_method', default='median')
    # extensions
    parser.add_argument('--decode_threads', type=int, default=0, help='host decoder threads per shard; 0 = the host cores divided by the shards')
    parser.add_argument('--slab_mb', type=int, default=512)
    parser.add_argument('--gather_pool', action='store_true',
                        help='under torchrun: after the extraction, all-gather the decoded backgrounds into a mix pool '
                             'resident on every GPU (main() returns (paths, RaggedPool))')
    parser.add_argument('--gather_pool_resize', action='store_true',
                        help='with --gather_pool: set the pool up for Resize(--size) inside the blend (the reference\'s bg_resize)')
    return parser.parse_args(argv)


def read_frames(data_path: pathlib.Path, from_video: bool, interval: int, max_frames: int) -> List[np.ndarray]:
    """The frame-collection loops of the reference (extract_background.py:48-71)."""
    frames = []
    count = 0
    if from_video:
        cap = cv2.VideoCapture(str(data_path))
        while cap.isOpened() and len(frames) <= max_frames:
            ret, frame_ = cap.read()
            if count % interval == 0:
                if ret:
                    frames.append(frame_)
                else:
                    break
            elif not ret:
                break              # end of stream on a skipped position: the next kept read would fail too
            count += 1
        cap.release()
    else:
        for img_f in sorted(pathlib.Path(data_path).glob('*')):
            if len(frames) > max_frames:
                break
            if count % interval == 0:
                img = cv2.imread(str(img_f))
                if img is not None:
                    frames.append(img)
            count += 1
    return frames


_scratch = threading.local()


def read_frames_packed(data_path: pathlib.Path, from_video: bool, interval: int, max_frames: int) -> np.ndarray:
    """:func:`read_frames` for the batched path: the same frames as one ``[T, H, W, 3]`` uint8 array that lives in a
    scratch buffer of the calling thread (valid until the thread's next call).  The decoder writes each kept frame
    straight into the scratch, so a decoder thread allocates nothing per frame."""
    if not from_video:
        frames = read_frames(data_path, from_video, interval, max_frames)
        return np.stack(frames) if frames else np.empty((0,), np.uint8)
    cap = cv2.VideoCapture(str(data_path))
    n, count, buf = 0, 0, getattr(_scratch, "buf", None)
    try:
        while cap.isOpened() and n <= max_frames:
            keep = count % interval == 0
            if not keep:
                if not cap.grab():                                 # skipped position: advance without converting
                    break
                count += 1
                continue
            dst = buf[n] if (buf is not None and n < len(buf)) else None
            ret, frame = cap.read(dst) if dst is not None else cap.read()
            if not ret:
                break
            if keep:
                if buf is None or buf.shape[1:] != frame.shape or n >= len(buf):
                    grown = np.empty((max(max_frames + 1, n + 1),) + frame.shape, np.uint8)      # pages are touched on use
                    if buf is not None and buf.shape[1:] == frame.shape:
                        grown[:n] = buf[:n]
                    _scratch.buf = buf = grown
                if frame is not dst and not (dst is not None and np.shares_memory(frame, dst)):
                    buf[n] = frame                                 # first frame of a size, or cv2 returned its own array
                n += 1
            count += 1
    finally:
        cap.release()
    return buf[:n] if buf is not None else np.empty((0,), np.uint8)


def temporal_median_frames(frames: List[np.ndarray], device=0) -> np.ndarray:
    """``np.median(frames, axis=0).astype(np.uint8)`` on the GPU for a list of host frames, through the
    host-buffer entry point of the C ABI (gathers the separately allocated frames into pinned memory)."""
    import ctypes
    from . import _cabi
    if len(frames) == 0:
        raise ValueError("median of zero frames")        # reference: nan median, cv2.imwrite raises
    shape = frames[0].shape
    arrs = [np.ascontiguousarray(f, dtype=np.uint8) for f in frames]
    for a in arrs:
        if a.shape != shape:
            raise ValueError("all frames must have the same shape")
    N = int(np.prod(shape))
    ptrs = (ctypes.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
    out = np.empty(shape, np.uint8)
    dev = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
    index = dev.index if dev.index is not None else torch.cuda.current_device()      # 'cuda' = the current device
    _cabi.check(_cabi.lib().bgd_temporal_median_u8_host(ptrs, len(arrs), N, out.ctypes.data, index))
    return out


def bg_extraction_tmf(data_path: pathlib.Path, dest: pathlib.Path,
                      from_video: bool, interval: int, max_frames: int, *args, **kwargs):
    """extract background using median temporal filtering -- same signature and return value as
    the reference (extract_background.py:42-75): writes ``dest`` and returns the ``[H,W,3]`` uint8
    median frame.  ``device=`` (keyword) selects the GPU."""
    frames = read_frames(pathlib.Path(data_path), from_video, interval, max_frames)
    median_frame = temporal_median_frames(frames, kwargs.get('device', 0))
    cv2.imwrite(str(dest), median_frame)
    return median_frame


SIM_CAM_CROP = 100


def sim_cam_files(data_path: pathlib.Path, interval: int, max_frames: int) -> List[pathlib.Path]:
    """The frames the reference's loop reads (extract_background.py:82-88): every ``interval``-th file of the sorted
    folder except the last, at most ``max_frames`` of them."""
    return sorted(pathlib.Path(data_path).glob('*'))[:-1:interval][:max_frames]


def read_sim_cam_frames(data_path: pathlib.Path, interval: int, max_frames: int) -> List[torch.Tensor]:
    """The decoded frames of a folder, uint8 ``[3, H, W]`` each: ``torchvision.io.read_image`` as the reference decodes
    them (:89).  An empty folder, an unreadable file and an image without exactly 3 channels raise ``ValueError`` (the
    reference fails on them too: nanmedian of nothing, read_image's error, cvtColor(BGR2RGB) on :99)."""
    from torchvision.io import read_image
    frames = []
    for f in sim_cam_files(data_path, interval, max_frames):
        try:
            img = read_image(str(f))
        except RuntimeError as e:
            raise ValueError(f"{f}: cannot decode ({e})") from e
        if img.dim() != 3 or img.shape[0] != 3:
            raise ValueError(f"{f}: {tuple(img.shape)} is not a 3-channel image")
        frames.append(img)
    if not frames:
        raise ValueError(f"no frames under {data_path}")
    return frames


def crop_draws(sizes) -> List[tuple]:
    """``(top, left, h, w)`` per frame of frame sizes ``(H, W)`` in order: the draws ``RandomResizedCrop(100)`` makes
    for those frames (:81,90) -- ``get_params`` with torchvision's default scale and ratio on the global torch RNG,
    which depends on the frame size only.  Call it on one thread, in the reference's frame order."""
    from torchvision.transforms import RandomResizedCrop
    rrc = RandomResizedCrop(SIM_CAM_CROP)
    return [tuple(int(v) for v in rrc.get_params(torch.empty(1, 1, 1).expand(3, int(H), int(W)), rrc.scale, rrc.ratio))
            for H, W in sizes]


def crop_descriptors(frames, draws, tables) -> torch.Tensor:
    """int64 ``[n, 11]`` descriptors of ``torch.ops.bgdebias.resized_crop_aa`` for ``frames`` = ``(byte offset, H, W)``
    and ``draws`` = ``(top, left, h, w)``; ``tables`` (:class:`pool.AATables`) gains the weight tables they need."""
    rows = []
    for (off, H, W), (i, j, h, w) in zip(frames, draws):
        xtab, kx = tables.lookup(w, SIM_CAM_CROP)
        ytab, ky = tables.lookup(h, SIM_CAM_CROP)
        rows.append((off, H, W, i, j, h, w, xtab, ytab, kx, ky))
    return torch.tensor(rows, dtype=torch.int64).reshape(-1, 11)


def _frame_layout(start: int, frames) -> list:
    """``(byte offset, H, W)`` of ``[3, H, W]`` frames packed back to back from ``start``."""
    out, off = [], start
    for f in frames:
        H, W = int(f.shape[1]), int(f.shape[2])
        out.append((off, H, W))
        off += 3 * H * W
    return out


class SimCamReduce:
    """The sim_cam reduction of a staged slab (``staging.FrameStager(reduce=...)``): one ``resized_crop_aa`` launch over
    every frame of the slab (frames of any sizes), then one ``nan_temporal_reduce_varlen`` launch (zeros are missing,
    :91) -> uint8 ``[V, 100, 100, 3]``.  ``add_video``'s ``meta`` is the folder's ``[(byte offset from the folder's
    first byte, H, W)]`` and its draws."""
    mixed_sizes = True

    def __init__(self, device, avg_method: int):
        from .pool import AATables
        self.tables = AATables(device)
        self.avg_method = int(avg_method)

    def result_shape(self, frame_shape: tuple) -> tuple:
        return (SIM_CAM_CROP, SIM_CAM_CROP, 3)

    def __call__(self, data: torch.Tensor, slab) -> torch.Tensor:
        frames, draws = [], []
        for start, (layout, d) in zip(slab.starts, slab.metas):
            frames += [(start + off, H, W) for off, H, W in layout]
            draws += d
        desc = crop_descriptors(frames, draws, self.tables)
        crops = torch.ops.bgdebias.resized_crop_aa(data, desc, self.tables.tensor_for(torch.cuda.current_stream(data.device)),
                                                   SIM_CAM_CROP, SIM_CAM_CROP)
        return torch.ops.bgdebias.nan_temporal_reduce_varlen(crops, torch.tensor(slab.offsets, dtype=torch.int64),
                                                             self.avg_method, True)


def sim_cam_background(data_path: pathlib.Path, interval: int, max_frames: int, avg_method: int, device=0) -> np.ndarray:
    """uint8 ``[100,100,3]``: the ``ave_frame`` of extract_background.py:94-98.  The frames are decoded on the host;
    the crops (one launch for the folder, draws from the torch RNG as the reference makes them) and the NaN-masked
    median (``avg_method`` 0) or mean (1) over them, zeros counting as missing (:91), run on the GPU."""
    from . import ops as _ops  # noqa: F401  (registers torch.ops.bgdebias.*)
    from .pool import AATables
    dev = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
    frames = read_sim_cam_frames(data_path, interval, max_frames)
    draws = crop_draws([f.shape[1:] for f in frames])
    layout = _frame_layout(0, frames)
    host = torch.empty(sum(3 * H * W for _, H, W in layout), dtype=torch.uint8, pin_memory=True)
    for f, (off, H, W) in zip(frames, layout):
        host[off:off + 3 * H * W] = f.reshape(-1)
    tables = AATables(dev)
    desc = crop_descriptors(layout, draws, tables)
    with torch.cuda.device(dev):
        crops = torch.ops.bgdebias.resized_crop_aa(host.to(dev, non_blocking=True), desc, tables.tensor, SIM_CAM_CROP,
                                                   SIM_CAM_CROP)
        return torch.ops.bgdebias.nan_temporal_reduce(crops, int(avg_method), True).cpu().numpy()


def sim_cam_motion_bg_extract(data_path, dest, from_video, interval, max_frames, avg_method, device=0):
    """Simulated-camera-motion extraction, same signature and side effect as the reference
    (extract_background.py:78-99): reads the image folder ``data_path`` (``from_video`` is ignored there
    too), writes ``dest`` and returns ``None``."""
    ave_frame = sim_cam_background(pathlib.Path(data_path), interval, max_frames, avg_method, device)
    cv2.imwrite(str(dest), cv2.cvtColor(ave_frame, cv2.COLOR_BGR2RGB))


def in_submission_order(pool, fn, items, window: int):
    """``fn(item)`` for every item on the executor ``pool``, at most ``window`` in flight, results yielded in the order
    of ``items`` -- whatever order the threads finish in."""
    pending, it = [], iter(items)
    while True:
        while len(pending) < window:
            nxt = next(it, None)
            if nxt is None:
                break
            pending.append(pool.submit(fn, nxt))
        if not pending:
            return
        yield pending.pop(0).result()


def bg_extract_multiple(paths: List[pathlib.Path], output_dir: pathlib.Path, from_video: bool,
                        interval: int, max_frames: int, process_id: int, method, avg_method: int,
                        device=None, decode_threads: int = 4, slab_mb: int = 512):
    """Same role and leading arguments as the reference (extract_background.py:102-109).  For the ``tmf`` and
    ``sim_cam`` methods the videos / frame folders of this shard are decoded by a thread pool into a pinned slab and
    reduced many-per-launch; any other ``method`` callable is invoked video by video like the reference.  Returns
    the failures, ``[(path, reason)]``; the other videos still finish."""
    output_dir = pathlib.Path(output_dir)
    if method is not bg_extraction_tmf and method is not sim_cam_motion_bg_extract:
        for data_path in paths:
            method(data_path, (output_dir / data_path.name).with_suffix('.jpg'), from_video, interval, max_frames, avg_method)
        return []
    if device is None:
        device = _shard.device_for(process_id, torch.cuda.device_count())
    dev = torch.device(f"cuda:{device}" if isinstance(device, int) else device)
    torch.cuda.set_device(dev)
    sim_cam = method is sim_cam_motion_bg_extract

    os.environ.setdefault("OPENCV_FFMPEG_THREADS", "1")     # many videos in flight: one FFmpeg thread per capture, no oversubscription
    n_dec = max(1, decode_threads)
    # JPEGs are encoded by their own small pool, so a background reaches the disk as soon as its slab is reduced: the
    # skip-if-exists resume (and a kill mid-shard) then find the finished part, and host memory holds the backgrounds of
    # a few slabs instead of the whole shard.  Decodes are submitted in a sliding window for the same reason.
    with ThreadPoolExecutor(max_workers=n_dec) as pool, ThreadPoolExecutor(max_workers=max(1, min(4, n_dec // 4))) as writers:
        writes = []

        def write(tag, bg):                                  # JPEG encoding off the staging path
            if sim_cam:                                      # the reference's channel swap before imwrite (:99)
                writes.append(writers.submit(lambda t, b: cv2.imwrite(str(t), cv2.cvtColor(b, cv2.COLOR_BGR2RGB)), tag, bg))
            else:
                writes.append(writers.submit(cv2.imwrite, str(tag), bg))

        stager = FrameStager(write, dev, slab_mb, reduce=SimCamReduce(dev, avg_method) if sim_cam else None)

        def decode(p):
            # tmf: decode into this thread's scratch frames, then pack them into the pinned slab from this thread
            try:
                if sim_cam:
                    return p, read_sim_cam_frames(p, interval, max_frames)
                frames = read_frames_packed(p, from_video, interval, max_frames)
                if not len(frames):
                    return p, "no frames decoded"
                stager.add_video(frames, (output_dir / p.name).with_suffix('.jpg'))
                return p, None
            except Exception as e:  # keep going, report at the end
                return p, repr(e)

        failures = []
        for p, r in in_submission_order(pool, decode, paths, 4 * n_dec):
            if isinstance(r, list):
                # sim_cam: the crop draws of a folder are made here, on one thread in the order of `paths` -- the order
                # the reference's worker draws them in, whatever order the decoder threads finish in
                stager.add_video(r, (output_dir / p.name).with_suffix('.jpg'),
                                 (_frame_layout(0, r), crop_draws([f.shape[1:] for f in r])))
            elif r is not None:
                failures.append((str(p), r))
            while writes and writes[0].done():
                writes.pop(0).result()                       # surface write errors early, keep the list short
        stager.flush()
        for w in writes:
            w.result()
    return failures


def _shard_entry(rank, shard_paths, output_dir, from_video, interval, max_frames, method_name, avg_method,
                 decode_threads, slab_mb):
    method = bg_extraction_tmf if method_name == 'tmf' else sim_cam_motion_bg_extract
    failures = bg_extract_multiple(shard_paths, pathlib.Path(output_dir), from_video, interval, max_frames, rank,
                                   method, avg_method, None, decode_threads, slab_mb)
    if failures:
        raise RuntimeError(f"{len(failures)} videos failed in shard {rank}: {failures[:5]}")


def main(argv=None):
    args = parse_args(argv)
    output_dir = pathlib.Path(args.output_dir)
    output_dir.mkdir(exist_ok=True)
    video_dir = pathlib.Path(args.video_dir)

    # check duplicated background (extract_background.py:118-126)
    video_paths = set(video_dir.glob(args.glob_pattern))
    extracted = [p_ for p_ in video_paths if (output_dir / p_.name).with_suffix(args.image_suffix).exists()]
    video_paths = sorted(video_paths.difference(extracted))
    print('Found {} backgrounds'.format(len(extracted)))
    print('Extracting background from {} videos'.format(len(video_paths)))

    if args.method not in ('tmf', 'sim_cam'):
        raise ValueError
    if args.avg_method == 'median':
        avg_method = 0
    elif args.avg_method == 'mean':
        avg_method = 1
    else:
        raise ValueError

    if _under_torchrun():
        return _main_torchrun(args, output_dir, video_paths, len(extracted), avg_method)

    splits = _shard.contiguous_splits(video_paths, args.num_workers)
    if args.decode_threads <= 0:
        args.decode_threads = max(1, min(32, len(os.sched_getaffinity(0)) // max(1, sum(1 for s_ in splits if len(s_)))))
    t0 = time.perf_counter()
    _shard.run_shards(_shard_entry, splits, str(output_dir), args.from_video, args.interval, args.max_frames,
                      args.method, avg_method, args.decode_threads, args.slab_mb)
    seconds = time.perf_counter() - t0
    index = write_background_index(output_dir, args.image_suffix)
    # one line of run metrics (the reference reports nothing for this path)
    print(json.dumps({"extracted": len(video_paths), "skipped_existing": len(extracted), "backgrounds_indexed": len(index),
                      "seconds": round(seconds, 3), "videos_per_s": round(len(video_paths) / seconds, 2) if seconds > 0 else None,
                      "shards": sum(1 for s_ in splits if len(s_)), "method": args.method}))


def _under_torchrun() -> bool:
    return int(os.environ.get("WORLD_SIZE", "1")) >= 1 and "RANK" in os.environ and "MASTER_ADDR" in os.environ


def _main_torchrun(args, output_dir, video_paths, n_skipped, avg_method):
    """``torchrun --nproc-per-node N -m bgdebias_b200.extract_background ...``: one rank = one process = one GPU = one
    contiguous slice of the sorted video list (the reference's split, extract_background.py:128-133, over ranks
    instead of forked workers); no collective on the extraction itself.  With ``--gather_pool`` the ranks then run the
    path's one collective (``pool.gather_extracted_backgrounds``) and return the device-resident mix pool."""
    import torch.distributed as dist
    world, rank = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    device = local_rank % max(1, torch.cuda.device_count())
    torch.cuda.set_device(device)
    own_group = not dist.is_initialized()
    if own_group:
        dist.init_process_group("nccl", device_id=torch.device("cuda", device))
    mine = _shard.contiguous_splits(video_paths, world)[rank]
    if args.decode_threads <= 0:
        args.decode_threads = max(1, min(32, len(os.sched_getaffinity(0)) // world))
    method = bg_extraction_tmf if args.method == 'tmf' else sim_cam_motion_bg_extract
    t0 = time.perf_counter()
    failures = bg_extract_multiple(mine, output_dir, args.from_video, args.interval, args.max_frames, rank, method, avg_method,
                                   device, args.decode_threads, args.slab_mb)
    counts = [None] * world
    dist.all_gather_object(counts, (len(mine), [f[0] for f in failures]))     # also the barrier: every JPEG is on disk
    seconds = time.perf_counter() - t0
    if rank == 0:
        index = write_background_index(output_dir, args.image_suffix)
        print(json.dumps({"extracted": len(video_paths), "skipped_existing": n_skipped, "backgrounds_indexed": len(index),
                          "seconds": round(seconds, 3), "videos_per_s": round(len(video_paths) / seconds, 2) if seconds > 0 else None,
                          "shards": world, "launcher": "torchrun", "method": args.method}))
    failed = [f for _, fs in counts for f in fs]
    pool = None
    if not failed and args.gather_pool:
        from .pool import gather_extracted_backgrounds
        dist.barrier()                                                          # the index / directory listing is complete
        pool = gather_extracted_backgrounds(output_dir, args.image_suffix, args.size if args.gather_pool_resize else None,
                                            torch.device("cuda", device))
    if own_group:
        dist.barrier()
        dist.destroy_process_group()
    if failed:
        raise RuntimeError(f"{len(failed)} videos failed: {failed[:5]}")
    return pool


INDEX_SUFFIX = ".bg_index.json"


def index_path(output_dir: pathlib.Path) -> pathlib.Path:
    """``<output_dir>.bg_index.json`` BESIDE the directory, not in it: the reference's Places365-style pools take
    every file of ``bg_dir`` as a background (``glob('*')``, comix_loader.py:100-101), so nothing else may live there."""
    output_dir = pathlib.Path(output_dir)
    return output_dir.parent / (output_dir.name + INDEX_SUFFIX)


def write_background_index(output_dir: pathlib.Path, image_suffix: str = '.jpg') -> list:
    """Persist the background index beside the JPEG folder: ``[{"name", "file", "height", "width"}, ...]`` sorted by
    name -- the pool order ``BackgroundMixDataset(map_bg_to_video=False)`` and ``BackgroundPool.from_index`` use, so
    a mix pool can be rebuilt (and all-gathered by name) without touching the videos again.  Rewritten from the
    directory listing on every run, so it also covers backgrounds kept by the skip-if-exists resume."""
    output_dir = pathlib.Path(output_dir)
    entries = []
    for f in sorted(output_dir.glob('*' + image_suffix)):
        ok, w, h = _image_size(f)
        if ok:
            entries.append({"name": f.stem, "file": f.name, "height": h, "width": w})
    dest = index_path(output_dir)
    tmp = dest.with_name(dest.name + ".tmp")
    tmp.write_text(json.dumps(entries))
    tmp.replace(dest)                               # atomic: a crashed run never leaves half an index
    return entries


def _image_size(path: pathlib.Path):
    img = cv2.imread(str(path), cv2.IMREAD_UNCHANGED)
    if img is None:
        return False, 0, 0
    return True, int(img.shape[1]), int(img.shape[0])


if __name__ == '__main__':
    main(sys.argv[1:])
