"""CPU tests of ShardedPool's global index over three gloo ranks in which ranks above 0 own images (owner / slot numbering
and rank order), of the process group the pool keeps, and of the refusal of a local pool whose images are not 16-byte
aligned."""
import os

import numpy as np
import pytest
import torch

# rank -> native sizes of the images it owns: rank 1 owns none, rank 2 owns sizes rank 0 does not have
SHARDS = {0: [(30, 40), (44, 30)], 1: [], 2: [(26, 50), (30, 40), (52, 36)]}


def _index_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from bgdebias_b200.pool import BackgroundPool, RaggedPool, ShardedPool
    names = [f"r{rank}_{i}" for i in range(len(SHARDS[rank]))]
    local = RaggedPool(36, "cpu")
    local.append([torch.full((3, h, w), 10 * rank + i, dtype=torch.uint8) for i, (h, w) in enumerate(SHARDS[rank])])
    group = dist.new_group([0, 1, 2], backend="gloo")
    sp = ShardedPool.from_local(names, local, group)
    ref = BackgroundPool.all_gather_index(names)
    q.put((rank, sp.index(), ref, list(zip(sp.h.tolist(), sp.w.tolist())), [sp.hw(i) for i in range(len(sp))],
           sp.group is group, (sp.rank, sp.world), len(local)))
    dist.destroy_process_group()


def test_index_of_three_ranks_with_images_above_rank_zero():
    import multiprocessing as mp
    from bgdebias_b200.pool import resized_hw
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 37500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_index_worker, args=(r, 3, port, q)) for r in range(3)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=180) for _ in procs], key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    exp_index = [(f"r{r}_{i}", r, i) for r in range(3) for i in range(len(SHARDS[r]))]
    exp_sizes = [hw for r in range(3) for hw in SHARDS[r]]
    for rank, index, ref, sizes, hw, same_group, rank_world, n_local in res:
        assert index == ref == exp_index
        assert sizes == exp_sizes
        assert hw == [resized_hw(h, w, 36) for h, w in exp_sizes]
        assert same_group and rank_world == (rank, 3) and n_local == len(SHARDS[rank])


def test_unaligned_local_pool_is_refused_when_the_pool_is_built():
    """ragged_pack copies whole images with 16-byte vectors: a local pool adopted with from_uniform_buffer whose image size
    3*h*w is not a multiple of 16 is refused by the constructor, not at the first fetch."""
    from bgdebias_b200.pool import RaggedPool, ShardedPool
    bad = RaggedPool.from_uniform_buffer(torch.zeros(2 * 3 * 3 * 5, dtype=torch.uint8), 2, 3, 5, bg_resize=None)
    with pytest.raises(ValueError, match="16"):
        ShardedPool(bad, ["a", "b"], [0, 0], [0, 1], [3, 3], [5, 5], rank=0, world=1)
    good = RaggedPool.from_uniform_buffer(torch.zeros(2 * 3 * 4 * 4, dtype=torch.uint8), 2, 4, 4, bg_resize=None)
    sp = ShardedPool(good, ["a", "b"], [0, 0], [0, 1], [4, 4], [4, 4], rank=0, world=1)
    assert sp.group is None and np.array_equal(sp.local.slots["offset"], [0, 48])
