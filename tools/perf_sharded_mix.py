"""Step time of BG-mix from a sharded pool against the replicated pool, under ``torchrun --nproc-per-node W``.

Workload: configs[4] batches (64 clips x 8 x 224 x 224 per rank, mix probability 0.25) over a Sth-Sth-v2-sized pool of
220,847 uint8 backgrounds of 240x427 (67.9 GB).  Every rank holds its 1/W shard (the sharded mode) AND a full replica (the
mode it replaces), both filled with the same seeded pixels, and alternates in one run:

  sharded: ShardedPool.fetch (all_gather_object of the requests, ragged_pack, all_to_all_single) + bgmix_blend_ragged
           over the fetched images
  replica: bgmix_blend_ragged over the resident replica

Each step is bracketed by torch.cuda.synchronize() and a host clock (fetch includes host work and a collective); the
fetch is also timed alone inside the sharded step.  Outputs of both modes are compared bit for bit on every step.

    torchrun --nproc-per-node 8 tools/perf_sharded_mix.py --steps 40 --warmup 5
"""
from __future__ import annotations

import argparse
import json
import os
import pathlib
import sys
import time

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=220_847)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--prob", type=float, default=0.25)
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=dev)
    import bgdebias_b200.ops as ops
    from bgdebias_b200 import pool
    from bgdebias_b200.shard import contiguous_splits

    H, W, P = 240, 427, args.images
    img = 3 * H * W
    # replica: every image i holds bytes generated from seed i's chunk; the shard is the same bytes for its images
    replica_buf = torch.empty(P * img, dtype=torch.uint8, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(7)
    step_imgs = 4096
    for a in range(0, P, step_imgs):
        b = min(P, a + step_imgs)
        replica_buf[a * img:b * img] = torch.randint(0, 256, ((b - a) * img,), dtype=torch.uint8, device=dev, generator=gen)
    replica = pool.RaggedPool.from_uniform_buffer(replica_buf, P, H, W, 256)
    mine = contiguous_splits(list(range(P)), world)[rank]
    lo, n_local = (mine[0] if mine else 0), len(mine)
    local_buf = replica_buf[lo * img:(lo + n_local) * img].clone()
    local = pool.RaggedPool.from_uniform_buffer(local_buf, n_local, H, W, 256)
    sharded = pool.ShardedPool.from_local([f"bg{i}" for i in mine], local)
    Hb, Wb = sharded.hw(0)
    torch.cuda.synchronize()

    B, T, th, tw = args.batch, 8, 224, 224
    g = torch.Generator(device=dev)
    g.manual_seed(100 + rank)
    fg = torch.randint(0, 256, (B, T, th, tw, 3), dtype=torch.uint8, device=dev, generator=g)
    lut = ops.make_fg_lut((123.675, 116.28, 103.53), (58.395, 57.12, 57.375), dev)
    mean_t, std_t = torch.tensor((123.675, 116.28, 103.53)), torch.tensor((58.395, 57.12, 57.375))
    rng = np.random.default_rng(1000 + rank)

    def draws():
        idx = torch.from_numpy(rng.integers(0, P, B))
        app = torch.from_numpy((rng.random(B) < args.prob).astype(np.uint8))
        top = torch.from_numpy(rng.integers(0, Hb - th + 1, B).astype(np.int32))
        left = torch.from_numpy(rng.integers(0, Wb - tw + 1, B).astype(np.int32))
        return idx, app, top.to(dev), left.to(dev), app.to(dev)

    def blend(rp, rows, top, left, app_d):
        return torch.ops.bgdebias.bgmix_blend_ragged(fg, rp.data, rp.slots_tensor, rp.tables.tensor, rows, top, left, app_d,
                                                     lut, mean_t, std_t, 0.5, "NTCHW")

    t_sh, t_fetch, t_rep, mixed, equal = [], [], [], [], True
    for it in range(args.warmup + args.steps):
        idx, app, top, left, app_d = draws()
        # sharded
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        batch, slot = sharded.fetch(idx, app)
        if not len(batch):
            batch.append([torch.zeros((3, th, tw), dtype=torch.uint8)])
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        out_s = blend(batch, slot.to(dev), top, left, app_d)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        # replica
        t3 = time.perf_counter()
        out_r = blend(replica, idx.to(dev, torch.int32), top, left, app_d)
        torch.cuda.synchronize()
        t4 = time.perf_counter()
        equal &= bool(torch.equal(out_s.view(torch.int32), out_r.view(torch.int32)))
        if it >= args.warmup:
            t_sh.append(t2 - t0)
            t_fetch.append(t1 - t0)
            t_rep.append(t4 - t3)
            mixed.append(int(app.sum()))
    med = lambda v: float(np.median(v)) * 1e3                       # noqa: E731
    res = dict(rank=rank, local_images=n_local, resident_bytes=sharded.resident_bytes, replica_bytes=int(replica_buf.numel()),
               ms_sharded_step=med(t_sh), ms_fetch=med(t_fetch), ms_replica_step=med(t_rep),
               fetch_share=float(np.median(np.array(t_fetch) / np.array(t_sh))), mixed_per_step=float(np.mean(mixed)),
               bit_equal=equal)
    gathered = [None] * world
    dist.all_gather_object(gathered, res)
    if rank == 0:
        for r in gathered:
            print(json.dumps(r))
        pick = lambda k: [r[k] for r in gathered]                     # noqa: E731
        print(json.dumps(dict(
            world=world, images=P, image=f"{H}x{W}", batch=f"{B}x{T}x{th}x{tw}", prob=args.prob, steps=args.steps,
            pool_gb_per_gpu_sharded=round(max(pick("resident_bytes")) / 1e9, 2),
            pool_gb_per_gpu_replica=round(gathered[0]["replica_bytes"] / 1e9, 2),
            ms_sharded_step_median_of_ranks=round(float(np.median(pick("ms_sharded_step"))), 3),
            ms_sharded_step_max_rank=round(max(pick("ms_sharded_step")), 3),
            ms_fetch_median_of_ranks=round(float(np.median(pick("ms_fetch"))), 3),
            ms_replica_step_median_of_ranks=round(float(np.median(pick("ms_replica_step"))), 3),
            fetch_share_median_of_ranks=round(float(np.median(pick("fetch_share"))), 3),
            bit_equal_all_ranks=all(pick("bit_equal")))))
    dist.destroy_process_group()
    return 0 if all(r["bit_equal"] for r in gathered) else 1


if __name__ == "__main__":
    sys.exit(main())
