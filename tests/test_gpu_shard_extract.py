"""The sharded pool built from a directory of extracted JPEGs (pool.shard_extracted_backgrounds), and the multi-rank exchange
of ShardedPool.fetch.

* Over a world-size-1 NCCL group, shard_extracted_backgrounds returns the paths gather_extracted_backgrounds returns, keeps
  the same pixels, and remembers its group.
* Two ranks over gloo, sharing one GPU, each decode their slice of the directory and exchange the images their batches drew
  with fetch (all_gather_object + ragged_pack + all_to_all_single of device bytes): every blend from the fetched images
  equals the blend from the replicated pool (torchvision's decode of every file), bit for bit -- also on a step where one
  rank mixes nothing."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SIZES = [(240, 320), (240, 427), (256, 341), (240, 320), (250, 300)]
MEAN, STD = (123.675, 116.28, 103.53), (58.395, 57.12, 57.375)


def _write_jpegs(d, seed=5):
    import cv2
    rng = np.random.default_rng(seed)
    for i, (h, w) in enumerate(SIZES):
        cv2.imwrite(str(d / f"v{i:02d}.jpg"), rng.integers(0, 256, (h, w, 3), dtype=np.uint8))


def test_shard_extracted_backgrounds_equals_gather(tmp_path):
    import torch.distributed as dist
    from bgdebias_b200 import _cabi, pool
    _cabi.lib()
    _write_jpegs(tmp_path)
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", init_method=f"file://{tmp_path / 'pg'}", rank=0, world_size=1,
                            device_id=torch.device("cuda:0"))
    try:
        group = dist.new_group([0])
        paths_g, gathered = pool.gather_extracted_backgrounds(tmp_path, ".jpg", 256, "cuda", group)
        paths_s, sharded = pool.shard_extracted_backgrounds(tmp_path, ".jpg", 256, "cuda", group)
        assert paths_s == paths_g == sharded.names and len(paths_s) == len(SIZES)
        assert sharded.group is group and (sharded.rank, sharded.world) == (0, 1)
        local = sharded.local
        for field in ("offset", "h", "w", "Hb", "Wb"):
            assert np.array_equal(local.slots[field], gathered.slots[field]), field
        assert torch.equal(local.data[:local.used].cpu(), gathered.data[:local.used].cpu())
        assert sharded.resident_bytes == local.used
    finally:
        dist.destroy_process_group()


def _gloo_worker(rank, world, init, bg_dir, q):
    import torch.distributed as dist
    from torchvision.io import ImageReadMode, read_image
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", init_method=init, rank=rank, world_size=world)
    import bgdebias_b200.ops as ops
    from bgdebias_b200 import pool
    paths, sharded = pool.shard_extracted_backgrounds(bg_dir, ".jpg", 256, "cuda")
    replica = pool.RaggedPool(256, "cuda")
    replica.append([read_image(p, mode=ImageReadMode.RGB) for p in paths])
    lut = ops.make_fg_lut(MEAN, STD, "cuda")
    rng = np.random.default_rng(50 + rank)
    B, T, P = 12, 3, len(paths)
    checked, equal = 0, True
    for step in range(4):
        idx = torch.from_numpy(rng.integers(0, P, B))
        app = torch.from_numpy((rng.random(B) < (0.0 if (step == 1 and rank == 0) else 0.6)).astype(np.uint8))
        hw = [sharded.hw(int(i)) for i in idx]
        top = torch.tensor([int(rng.integers(0, h - 224 + 1)) for h, _ in hw], dtype=torch.int32, device="cuda")
        left = torch.tensor([int(rng.integers(0, w - 224 + 1)) for _, w in hw], dtype=torch.int32, device="cuda")
        fg = torch.from_numpy(rng.integers(0, 256, (B, T, 224, 224, 3), dtype=np.uint8)).cuda()
        batch, slot = sharded.fetch(idx, app)
        if not len(batch):
            batch.append([torch.zeros((3, 224, 224), dtype=torch.uint8)])
        app_d = app.to("cuda")
        for dt, layout in [(torch.float32, "NTCHW"), (torch.bfloat16, "NTHWC")]:
            got = torch.ops.bgdebias.bgmix_blend_ragged(fg, batch.data, batch.slots_tensor, batch.tables.tensor,
                                                        slot.to("cuda"), top, left, app_d, lut, torch.tensor(MEAN),
                                                        torch.tensor(STD), 0.5, layout, dt)
            exp = torch.ops.bgdebias.bgmix_blend_ragged(fg, replica.data, replica.slots_tensor, replica.tables.tensor,
                                                        idx.to("cuda", torch.int32), top, left, app_d, lut, torch.tensor(MEAN),
                                                        torch.tensor(STD), 0.5, layout, dt)
            bits = torch.int32 if dt == torch.float32 else torch.int16
            equal &= bool(torch.equal(got.cpu().view(bits), exp.cpu().view(bits)))
            checked += 1
    q.put((rank, len(sharded.local), sharded.names == paths, checked, equal))
    dist.destroy_process_group()


def test_fetch_over_two_gloo_ranks_equals_replica(tmp_path):
    import multiprocessing as mp
    bg = tmp_path / "bg"
    bg.mkdir()
    _write_jpegs(bg, seed=9)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    init = f"file://{tmp_path / 'pg'}"
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, init, str(bg), q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in procs], key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert [r[1] for r in res] == [3, 2]                       # the contiguous ceil split of 5 files over 2 ranks
    for rank, n_local, same_names, checked, equal in res:
        assert same_names and checked == 8 and equal, rank
