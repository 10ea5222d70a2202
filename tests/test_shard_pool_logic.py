"""CPU tests of the sharded background pool's host logic: the routing of one exchange (pool.route_requests), the index
ShardedPool.from_local all-gathers (gloo, world size 2), and the dataset's refusal of names outside that index."""
import os

import numpy as np
import pytest
import torch


def _index(rng, world, counts):
    owner = np.concatenate([np.full(c, r, np.int64) for r, c in enumerate(counts)])
    slot = np.concatenate([np.arange(c, dtype=np.int64) for c in counts])
    nbytes = 3 * rng.integers(1, 40, owner.size) * rng.integers(1, 40, owner.size)
    # local byte offsets as RaggedPool.append lays them out: 16-byte aligned, images back to back
    offsets = []
    for r, c in enumerate(counts):
        sizes = nbytes[owner == r]
        offsets.append(np.concatenate([[0], np.cumsum((sizes + 15) & ~15)[:-1]]).astype(np.int64) if c else np.zeros(0, np.int64))
    return owner, slot, nbytes, offsets


@pytest.mark.parametrize("world,counts", [(2, [5, 3]), (3, [4, 0, 7]), (4, [1, 1, 1, 9]), (1, [6])])
def test_routing_agrees_between_sender_and_receiver(world, counts):
    """Every rank computes its send segments and its receive offsets alone from the request matrix; the bytes rank s sends
    to rank d must land exactly where d expects each image, and the split sizes must match pairwise."""
    from bgdebias_b200.pool import route_requests
    rng = np.random.default_rng(world * 100 + sum(counts))
    owner, slot, nbytes, offsets = _index(rng, world, counts)
    P = owner.size
    requests = []
    for r in range(world):
        k = int(rng.integers(0, P + 1))
        drawn = rng.integers(0, P, k).tolist()
        requests.append(list(dict.fromkeys(drawn)))
    if world > 1:
        requests[-1] = []                                       # a rank that mixes nothing this step
    routes = [route_requests(requests, owner, slot, nbytes, r, offsets[r]) for r in range(world)]
    for s in range(world):
        seg = routes[s].segments
        assert seg.dtype == np.int64 and seg.shape[1] == 3
        assert (seg[:, :2] % 16 == 0).all()
        assert sum(routes[s].send_splits) == (int(((seg[:, 2] + 15) & ~15).sum()) if len(seg) else 0)
        for d in range(world):
            assert routes[s].send_splits[d] == routes[d].recv_splits[s]
    # emulate all_to_all_single: the receive buffer of d is the chunks for d of every source, in source order; check every
    # requested image's (source slot offset, size) lands at d's receive offset
    for d in range(world):
        placed = {}
        base = 0
        for s in range(world):
            seg = routes[s].segments
            lo = sum(routes[s].send_splits[:d])
            hi = lo + routes[s].send_splits[d]
            for so, do, b in seg:
                if lo <= do < hi:
                    placed[base + (do - lo)] = (s, so, b)
            base += routes[d].recv_splits[s]
        assert sum(routes[d].recv_splits) == base
        assert len(placed) == len(requests[d])
        for g, off in zip(requests[d], routes[d].recv_offsets):
            assert off % 16 == 0
            assert placed[int(off)] == (owner[g], offsets[owner[g]][slot[g]], nbytes[g])


def _index_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from bgdebias_b200.pool import BackgroundPool, RaggedPool, ShardedPool
    sizes = [[(30, 40), (30, 52), (44, 30)], []][rank] if world == 2 else []
    names = [f"r{rank}_{i}" for i in range(len(sizes))]
    local = RaggedPool(36, "cpu")
    local.append([torch.full((3, h, w), i, dtype=torch.uint8) for i, (h, w) in enumerate(sizes)])
    sp = ShardedPool.from_local(names, local)
    index = BackgroundPool.all_gather_index(names)
    q.put((rank, sp.index(), index, sp.h.tolist(), sp.w.tolist(), [sp.hw(i) for i in range(len(sp))],
           sp.resident_bytes, len(local)))
    dist.destroy_process_group()


def test_from_local_index_is_all_gather_index_plus_sizes():
    """World size 2 over gloo, rank 1 owns nothing: every rank gets the index of all_gather_index and the native and
    resized sizes of every image."""
    import multiprocessing as mp
    from bgdebias_b200.pool import resized_hw
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 35500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_index_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=180) for _ in procs], key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    sizes = [(30, 40), (30, 52), (44, 30)]
    for rank, index, ref, h, w, hw, resident, n_local in res:
        assert index == ref == [("r0_0", 0, 0), ("r0_1", 0, 1), ("r0_2", 0, 2)]
        assert list(zip(h, w)) == sizes
        assert hw == [resized_hw(a, b, 36) for a, b in sizes]
        assert n_local == (3 if rank == 0 else 0) and (resident > 0) == (rank == 0)


def test_dataset_rejects_a_name_outside_the_index(tmp_path):
    """bg_files may repeat and reorder index names; a name that is not in the index raises a ValueError naming it (no
    decode on demand), and sizes come from the index without reading any file."""
    from bgdebias_b200 import comix_loader as cl
    from bgdebias_b200.pool import RaggedPool, ShardedPool, resized_hw
    bg = tmp_path / "bg"
    bg.mkdir()
    local = RaggedPool(256, "cpu")
    local.append([torch.zeros((3, 240, 320), dtype=torch.uint8), torch.zeros((3, 240, 427), dtype=torch.uint8)])
    names = [str(bg / "a.jpg"), str(bg / "b.jpg"), str(bg / "c.jpg")]
    sp = ShardedPool(local, names, [0, 0, 1], [0, 1, 0], [240, 240, 256], [320, 427, 256], rank=0, world=2)
    infos = [dict(frame_dir=f"/d/{n}", total_frames=3, label=0) for n in ("a", "b")]
    ds = cl.BackgroundMixDataset(infos, lambda r: r, bg_dir=str(bg), extract_bg_if_not_found=False, device="cpu")
    ds.attach_sharded_pool(names, sp)
    ds.bg_files = [names[2], names[1], names[2], names[0]]     # a CIL union with a repeat
    assert [ds._bg_hw(i) for i in range(4)] == [(256, 256), resized_hw(240, 427, 256), (256, 256), resized_hw(240, 320, 256)]
    assert sp.rows_of(ds.bg_files).tolist() == [2, 1, 2, 0]
    missing = str(bg / "not_extracted.jpg")
    ds.bg_files = ds.bg_files + [missing]
    with pytest.raises(ValueError, match="not_extracted.jpg"):
        ds._bg_hw(4)
    with pytest.raises(ValueError, match="not_extracted.jpg"):
        sp.rows_of(ds.bg_files)
    with pytest.raises(ValueError, match="index order"):
        ds.attach_sharded_pool(names[::-1], sp)
    with pytest.raises(ValueError):
        ShardedPool(local, names, [0, 1, 1], [0, 0, 1], [240, 240, 256], [320, 427, 256], rank=0, world=2)   # 1 != 2 local
