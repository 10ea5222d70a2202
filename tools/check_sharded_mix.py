"""Multi-GPU check of the sharded background pool: under ``torchrun --nproc-per-node W`` every rank owns an uneven shard of a
pool of three image sizes (the last rank owns nothing), draws its own batches, and mixes them from the sharded pool; the same
batches are mixed from the replicated pool with ``attach_pool``, and every rank's output must be bit-equal.  Also reports the
pool bytes each rank keeps against the replica.

``--via fetch`` (default): ``BackgroundMixDataset.attach_sharded_pool``, the images of every batch exchanged with
``ShardedPool.fetch``; every rank mixes 4 batches in lockstep.
``--via peer``: every rank maps every other rank's shard with ``pool.PeerPool.open`` and mixes with ``attach_peer_pool``, reading
the images straight from their owners' memory; rank r mixes 2 + (r mod 3) batches, so the ranks are not in lockstep.  Then
``PeerPool.close``; each rank also reports the peers it mapped.

    torchrun --nproc-per-node 8 tools/check_sharded_mix.py                            # NCCL, one GPU per rank
    torchrun --nproc-per-node 8 tools/check_sharded_mix.py --backend gloo             # gloo, ranks may share GPUs
    torchrun --nproc-per-node 8 tools/check_sharded_mix.py --backend gloo --via peer

``--backend gloo`` runs the same collectives (for ``fetch`` the request ``all_gather_object`` and the ``all_to_all_single`` of
device bytes; for ``peer`` only the build and close collectives) through gloo, so the routing, the exchange and the peer
mappings can be checked with more ranks than GPUs: rank r uses GPU r mod (GPUs on the host), and processes sharing one GPU map
each other's allocations on it.
"""
from __future__ import annotations

import argparse
import json
import os
import pathlib
import random
import shutil
import sys
import tempfile

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

SIZES = [(240, 320), (240, 427), (256, 341)]


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--backend", choices=("nccl", "gloo"), default="nccl")
    ap.add_argument("--via", choices=("fetch", "peer"), default="fetch", help="how a rank reaches the other ranks' images")
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    dev = torch.device("cuda", local_rank % torch.cuda.device_count() if args.backend == "gloo" else local_rank)
    torch.cuda.set_device(dev)
    if args.backend == "nccl":
        dist.init_process_group("nccl", device_id=dev)
    else:
        dist.init_process_group("gloo")
    from bgdebias_b200 import comix_loader as cl, pool

    counts = [(3 * r + 5) % 7 + 1 for r in range(world)]          # uneven shards ...
    counts[-1] = 0                                                 # ... and an empty one
    P = sum(counts)
    rng = np.random.default_rng(1234)                              # the same pool on every rank
    imgs = [torch.from_numpy(rng.integers(0, 256, (3, *SIZES[i % 3]), dtype=np.uint8)) for i in range(P)]
    # one directory for every rank: the index names (and bg_files) must be the same strings everywhere
    shared = [tempfile.mkdtemp(prefix=f"bgd_{args.via}_check_") if rank == 0 else None]
    dist.broadcast_object_list(shared, src=0)
    tmp = pathlib.Path(shared[0])
    paths = [os.path.realpath(tmp / f"bg{i:04d}.jpg") for i in range(P)]
    first = sum(counts[:rank])
    local = pool.RaggedPool(256, dev)
    local.append(imgs[first:first + counts[rank]])
    sharded = pool.ShardedPool.from_local(paths[first:first + counts[rank]], local)
    assert sharded.names == paths, "the global index must list every image in rank order"
    peer = pool.PeerPool.open(sharded) if args.via == "peer" else None
    replica = pool.RaggedPool(256, dev)
    replica.append(imgs)

    B, T = 16, 4
    infos = [dict(frame_dir=f"/d/v{i}", total_frames=8, label=i) for i in range(B)]

    def pipe(r):
        g = np.random.default_rng(1000 * rank + int(r["label"]))
        return dict(r, imgs=torch.from_numpy(g.integers(0, 256, (T, 224, 224, 3), dtype=np.uint8)))

    def dataset(prob):
        return cl.BackgroundMixDataset(infos, pipe, bg_dir=str(tmp), extract_bg_if_not_found=False, device_mix=True,
                                       prob=prob, device=dev)

    bg_files = paths + paths[: P // 2]                             # a union with repeats, as the CIL trainer builds
    checked, mixed, mismatches = 0, 0, []
    # fetch: every rank mixes every batch in lockstep; peer: ranks mix different numbers of batches
    steps, empty_step = (4, 2) if args.via == "fetch" else (2 + rank % 3, 1)
    for step in range(steps):
        prob = 0.0 if (step == empty_step and rank == 0) else 0.5  # one rank mixes nothing on one step
        outs = {}
        for kind in ("replica", "sharded"):
            ds = dataset(prob)
            if kind == "replica":
                ds.attach_pool(paths, replica)
            elif peer is None:
                ds.attach_sharded_pool(paths, sharded)
            else:
                ds.attach_peer_pool(paths, peer)
            ds.bg_files = list(bg_files)
            random.seed(100 * step + rank)
            torch.manual_seed(100 * step + rank)
            batch = ds.host_collate([ds[i] for i in range(B)])
            forms = {}
            for dt, mf in [(torch.float32, torch.contiguous_format), (torch.bfloat16, torch.channels_last)]:
                forms[str(dt)] = ds.device_finish(batch, dtype=dt, memory_format=mf)["imgs"]
            outs[kind] = (batch, forms)
        rb, rf = outs["replica"]
        sb, sf = outs["sharded"]
        mixed += int(sb["bg_apply"].sum())
        if not torch.equal(rb["bg_idx"], sb["bg_idx"]):
            mismatches.append((step, "bg_idx"))
        for k in rf:
            a, b = rf[k].contiguous().cpu(), sf[k].contiguous().cpu()
            bits = torch.int32 if a.dtype == torch.float32 else torch.int16
            checked += 1
            if not torch.equal(a.view(bits), b.view(bits)):
                mismatches.append((step, k))
    res = dict(rank=rank, local_images=counts[rank], mixed_samples=mixed, forms_checked=checked, mismatches=mismatches,
               resident_bytes=sharded.resident_bytes, replica_bytes=int(replica.data.numel()))
    if peer is None:
        torch.cuda.synchronize()
    else:
        res.update(batches=steps, mapped_peers=sorted(peer._mapped))
        peer.close()
    gathered = [None] * world
    dist.all_gather_object(gathered, res)
    ok = all(not g["mismatches"] for g in gathered)
    if rank == 0:
        for g in gathered:
            print(json.dumps(g))
        rep = gathered[0]["replica_bytes"]
        print(json.dumps(dict(world=world, backend=args.backend, gpus=torch.cuda.device_count(), images=P, image_sizes=SIZES, bit_equal=ok,
                              resident_over_replica=[round(g["resident_bytes"] / rep, 4) for g in gathered],
                              mean_resident_over_replica=round(sum(g["resident_bytes"] for g in gathered) / world / rep, 4))))
    dist.barrier()
    if rank == 0:
        shutil.rmtree(tmp, ignore_errors=True)
    dist.destroy_process_group()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
