"""Step time of BG-mix from a peer-mapped sharded pool against ShardedPool.fetch and the replicated pool, under
``torchrun --nproc-per-node W`` (NCCL, one GPU per rank).

Workload: configs[4] batches (64 clips x 8 x 224 x 224 per rank, mix probability 0.25) over a Sth-Sth-v2-sized pool of
220,847 uint8 backgrounds of 240x427 (67.9 GB).  Every rank holds the whole pool once (the replica) and takes its 1/W shard
as a view of it, so the three modes read the same bytes; three datasets mix the same batch through ``device_finish``:

  replica: attach_pool            -- bgmix_blend_ragged over the resident replica
  fetch:   attach_sharded_pool    -- ShardedPool.fetch (all_gather_object, ragged_pack, all_to_all_single) + blend
  peer:    attach_peer_pool       -- PeerPool.gather (one ragged_gather launch from the peer mappings) + blend

Step time: torch.cuda.synchronize(), host clock, device_finish, torch.cuda.synchronize(), alternating the modes every step;
the outputs are compared bit for bit with the replica on every step.  Host wait: ~20 ms of device work
(torch.cuda._sleep) is queued in front of device_finish, and the host time spent inside the call is recorded together with
whether the stream was still busy when it returned (a mode that waits for the stream returns only after it drained).

    torchrun --nproc-per-node 8 tools/perf_peer_mix.py --steps 30 --warmup 5
"""
from __future__ import annotations

import argparse
import json
import os
import pathlib
import subprocess
import sys
import tempfile
import time

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

MODES = ("replica", "fetch", "peer")


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=220_847)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--prob", type=float, default=0.25)
    ap.add_argument("--sleep-ms", type=float, default=20.0)
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip()
        print(f"# {card}", flush=True)
    from bgdebias_b200 import comix_loader as cl, pool
    from bgdebias_b200.shard import contiguous_splits

    H, W, P = 240, 427, args.images
    img = 3 * H * W
    replica_buf = torch.empty(P * img, dtype=torch.uint8, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(7)
    for a in range(0, P, 4096):
        b = min(P, a + 4096)
        replica_buf[a * img:b * img] = torch.randint(0, 256, ((b - a) * img,), dtype=torch.uint8, device=dev, generator=gen)
    replica = pool.RaggedPool.from_uniform_buffer(replica_buf, P, H, W, 256)
    mine = contiguous_splits(list(range(P)), world)[rank]
    lo, n_local = (mine[0] if mine else 0), len(mine)
    local = pool.RaggedPool.from_uniform_buffer(replica_buf[lo * img:(lo + n_local) * img], n_local, H, W, 256)
    shared = [tempfile.mkdtemp(prefix="bgd_perf_peer_") if rank == 0 else None]
    dist.broadcast_object_list(shared, src=0)
    root = os.path.realpath(shared[0])                               # attach_pool matches names after realpath
    paths = [os.path.join(root, f"bg{i}.jpg") for i in range(P)]
    sharded = pool.ShardedPool.from_local(paths[lo:lo + n_local], local)
    peer = pool.PeerPool.open(sharded)
    Hb, Wb = sharded.hw(0)

    B, T, th, tw = args.batch, 8, 224, 224
    infos = [dict(frame_dir=f"/d/v{i}", total_frames=8, label=i) for i in range(B)]
    datasets = {}
    for mode in MODES:
        ds = cl.BackgroundMixDataset(infos, lambda r: r, bg_dir=shared[0], extract_bg_if_not_found=False, device_mix=True,
                                     prob=args.prob, device=dev)
        if mode == "replica":
            ds.attach_pool(paths, replica)
        elif mode == "fetch":
            ds.attach_sharded_pool(paths, sharded)
        else:
            ds.attach_peer_pool(paths, peer)
        ds.bg_files = list(paths)
        datasets[mode] = ds
    g = torch.Generator(device=dev)
    g.manual_seed(100 + rank)
    fg = torch.randint(0, 256, (B, T, th, tw, 3), dtype=torch.uint8, device=dev, generator=g)
    rng = np.random.default_rng(1000 + rank)

    def draws() -> dict:
        return dict(imgs=fg, bg_idx=torch.from_numpy(rng.integers(0, P, B)).pin_memory(),
                    bg_top=torch.from_numpy(rng.integers(0, Hb - th + 1, B).astype(np.int32)).pin_memory(),
                    bg_left=torch.from_numpy(rng.integers(0, Wb - tw + 1, B).astype(np.int32)).pin_memory(),
                    bg_apply=torch.from_numpy((rng.random(B) < args.prob).astype(np.uint8)).pin_memory())

    step_ms = {m: [] for m in MODES}
    host_ms = {m: [] for m in MODES}
    busy = {m: 0 for m in MODES}
    mixed, equal = [], True
    sleep_cycles = int(args.sleep_ms * 1e-3 * 1.9e9)
    for it in range(args.warmup + args.steps):
        batch = draws()
        outs = {}
        for mode in MODES:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            outs[mode] = datasets[mode].device_finish(batch)["imgs"]
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            gate = torch.cuda.Event()
            torch.cuda._sleep(sleep_cycles)
            gate.record()
            t2 = time.perf_counter()
            datasets[mode].device_finish(batch)
            t3 = time.perf_counter()
            still_busy = not gate.query()
            torch.cuda.synchronize()
            if it >= args.warmup:
                step_ms[mode].append((t1 - t0) * 1e3)
                host_ms[mode].append((t3 - t2) * 1e3)
                busy[mode] += still_busy
        for mode in ("fetch", "peer"):
            equal &= bool(torch.equal(outs[mode].view(torch.int32), outs["replica"].view(torch.int32)))
        if it >= args.warmup:
            mixed.append(int(batch["bg_apply"].sum()))
    med = lambda v: round(float(np.median(v)), 3)                      # noqa: E731
    res = dict(rank=rank, local_images=n_local, mapped_peers=sorted(peer._mapped), mixed_per_step=float(np.mean(mixed)),
               **{f"ms_step_{m}": med(step_ms[m]) for m in MODES},
               **{f"ms_host_in_device_finish_{m}": med(host_ms[m]) for m in MODES},
               **{f"returned_while_busy_{m}": f"{busy[m]}/{args.steps}" for m in MODES}, bit_equal=equal)
    peer.close()
    gathered = [None] * world
    dist.all_gather_object(gathered, res)
    if rank == 0:
        for r in gathered:
            print(json.dumps(r))
        pick = lambda k: [r[k] for r in gathered]                     # noqa: E731
        print(json.dumps(dict(
            world=world, images=P, image=f"{H}x{W}", batch=f"{B}x{T}x{th}x{tw}", prob=args.prob, steps=args.steps,
            sleep_ms=args.sleep_ms, pool_gb_per_gpu_sharded=round(n_local * img / 1e9, 2),
            **{f"ms_step_{m}_median_of_ranks": round(float(np.median(pick(f"ms_step_{m}"))), 3) for m in MODES},
            **{f"ms_host_in_device_finish_{m}_median_of_ranks": round(float(np.median(pick(f"ms_host_in_device_finish_{m}"))), 3)
               for m in MODES},
            bit_equal_all_ranks=all(pick("bit_equal")))))
    dist.barrier()
    if rank == 0:
        os.rmdir(shared[0])
    dist.destroy_process_group()
    return 0 if all(r["bit_equal"] for r in gathered) else 1


if __name__ == "__main__":
    sys.exit(main())
