"""BG-mix from a sharded pool read through peer mappings (pool.PeerPool, BackgroundMixDataset.attach_peer_pool).

* ``ragged_gather`` (one launch from a table of source base pointers) equals torch slicing of 2-4 separate source tensors,
  passes opcheck, and rejects every kind of bad segment on the host, before anything is launched.
* Emulated peers -- the base table of each rank holds the W shards of one process -- give ``device_finish`` outputs bit-equal
  to ``attach_pool`` with the replicated pool, in every dtype, layout and memory format, for clips and packed crops, also
  for a batch that mixes nothing.
* ``device_finish`` through the peer pool does not wait for the work queued on the stream.
* Two spawned gloo ranks sharing one GPU map each other's shard with ``PeerPool.open`` (CUDA IPC); rank 0 mixes three batches
  and rank 1 one, with no lockstep, bit-equal to the replica; ``close()`` succeeds and both processes are joined."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

MEAN, STD = (123.675, 116.28, 103.53), (58.395, 57.12, 57.375)
SIZES = [(240, 320), (240, 427), (240, 352), (256, 256)]


@pytest.fixture(scope="module")
def env():
    import bgdebias_b200.ops as ops
    from bgdebias_b200 import _cabi, pool
    assert torch.cuda.is_available()
    _cabi.lib()
    return ops, _cabi, pool


def _bits(t: torch.Tensor) -> torch.Tensor:
    t = t.contiguous().cpu()
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)


def _images(rng, sizes):
    return [torch.from_numpy(rng.integers(0, 256, (3, h, w), dtype=np.uint8)) for h, w in sizes]


# ---- ragged_gather --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_src", [2, 3, 4])
def test_ragged_gather_equals_slicing_in_one_launch(env, n_src):
    ops, _cabi, pool = env
    rng = np.random.default_rng(n_src)
    sources = [torch.randint(0, 256, (int(rng.integers(1, 300)) * 16 + 4096,), dtype=torch.uint8, device="cuda")
               for _ in range(n_src)]
    sources.append(sources[0][:0])                                             # plus an empty source, never read
    bases = torch.tensor([s.data_ptr() for s in sources], dtype=torch.int64, device="cuda")
    sizes = torch.tensor([s.numel() for s in sources], dtype=torch.int64)
    segs, at = [], 0
    for k in range(40):
        r = k if k < n_src else int(rng.integers(0, n_src))                   # every non-empty source is read
        n = sources[r].numel()
        so = int(rng.integers(0, n // 16)) * 16
        b = int(rng.integers(1, n - so + 1)) if k < n_src or rng.random() < 0.9 else 0   # any size, some empty
        segs.append((r, so, at, b))
        at += (b + 15) & ~15
    seg = torch.tensor(segs, dtype=torch.int64)
    n0 = _cabi.kernel_launch_count()
    out = torch.ops.bgdebias.ragged_gather(bases, sizes, seg, at)
    torch.cuda.synchronize()
    assert _cabi.kernel_launch_count() - n0 == 1
    got = out.cpu()
    for r, so, do, b in segs:
        assert torch.equal(got[do:do + b], sources[r][so:so + b].cpu())
    n0 = _cabi.kernel_launch_count()
    empty = torch.ops.bgdebias.ragged_gather(bases, sizes, torch.zeros((0, 4), dtype=torch.int64), 0)
    assert empty.numel() == 0 and _cabi.kernel_launch_count() == n0


def test_ragged_gather_opcheck(env):
    a = torch.randint(0, 256, (4096,), dtype=torch.uint8, device="cuda")
    b = torch.randint(0, 256, (2048,), dtype=torch.uint8, device="cuda")
    bases = torch.tensor([a.data_ptr(), b.data_ptr()], dtype=torch.int64, device="cuda")
    sizes = torch.tensor([4096, 2048], dtype=torch.int64)
    seg = torch.tensor([[1, 1024, 0, 512], [0, 0, 512, 1024], [0, 2048, 1536, 2048]], dtype=torch.int64)   # all 3584 bytes
    torch.library.opcheck(torch.ops.bgdebias.ragged_gather, (bases, sizes, seg, 3584))


def test_ragged_gather_rejects_bad_segments_without_a_launch(env):
    ops, _cabi, pool = env
    a = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    b = torch.zeros(1024, dtype=torch.uint8, device="cuda")
    bases = torch.tensor([a.data_ptr(), b.data_ptr()], dtype=torch.int64, device="cuda")
    sizes = torch.tensor([4096, 1024], dtype=torch.int64)
    good = [0, 0, 0, 64]
    bad = {
        "source index out of range": [2, 0, 0, 64],
        "negative source index": [-1, 0, 0, 64],
        "misaligned source": [0, 8, 0, 64],
        "misaligned destination": [0, 0, 4, 64],
        "reads past its source": [1, 1008, 0, 32],
        "writes past the output": [0, 0, 1008, 32],
        "negative size": [0, 0, 0, -1],
    }
    for what, row in bad.items():
        n0 = _cabi.kernel_launch_count()
        with pytest.raises(ValueError, match="ragged_gather"):
            torch.ops.bgdebias.ragged_gather(bases, sizes, torch.tensor([good, row], dtype=torch.int64), 1024)
        assert _cabi.kernel_launch_count() == n0, what
    with pytest.raises(ValueError):
        torch.ops.bgdebias.ragged_gather(bases, sizes, torch.zeros((2, 3), dtype=torch.int64), 64)
    with pytest.raises(ValueError):
        torch.ops.bgdebias.ragged_gather(bases, sizes[:1], torch.tensor([good]), 64)


# ---- emulated peers: the W shards live in this process ------------------------------------------------------------------
def _peers(pool, imgs, counts, names=None, bg_resize=256):
    """The PeerPool every rank of a world of len(counts) would open, with its base table pointing at the W shards held here."""
    world = len(counts)
    owner = np.concatenate([np.full(c, r, np.int64) for r, c in enumerate(counts)])
    slot = np.concatenate([np.arange(c, dtype=np.int64) for c in counts])
    h, w = [int(t.shape[1]) for t in imgs], [int(t.shape[2]) for t in imgs]
    names = names or [f"bg{i}" for i in range(len(imgs))]
    shards, at = [], 0
    for r, c in enumerate(counts):
        local = pool.RaggedPool(bg_resize, "cuda")
        local.append(imgs[at:at + c])
        at += c
        shards.append(pool.ShardedPool(local, names, owner, slot, h, w, r, world))
    bases = [sp.local.data.data_ptr() if sp.local.used else 0 for sp in shards]
    sizes = [sp.local.used for sp in shards]
    src_offset = [int(shards[o].local.slots["offset"][s]) for o, s in zip(owner, slot)]
    return [pool.PeerPool(sp, bases, sizes, src_offset) for sp in shards], names


def _dataset(cl, bg_dir, clip_sizes, T, prob=0.6):
    infos = [dict(frame_dir=f"/d/v{i}", total_frames=8, label=i) for i in range(len(clip_sizes))]

    def pipe(r):
        i = int(r["label"])
        h, w = clip_sizes[i]
        g = np.random.default_rng(100 + i)
        return dict(r, imgs=torch.from_numpy(g.integers(0, 256, (T, h, w, 3), dtype=np.uint8)))

    return cl.BackgroundMixDataset(infos, pipe, bg_dir=str(bg_dir), extract_bg_if_not_found=False, device_mix=True,
                                   prob=prob, device="cuda")


FORMS = [(dt, mf, layout) for dt in (torch.float32, torch.bfloat16, torch.float16)
         for mf in (torch.contiguous_format, torch.channels_last) for layout in ("NTCHW", "NCTHW")]


@pytest.mark.parametrize("fg_form", ["clips", "packed_crops"])
@pytest.mark.parametrize("prob", [0.6, 0.0])
def test_device_finish_peer_equals_replicated(env, tmp_path, fg_form, prob):
    """Three ranks, one of them with an empty shard; every rank's batch from attach_peer_pool equals the same batch from
    attach_pool with the replica, in every form -- also when the batch mixes nothing."""
    import random
    ops, _cabi, pool = env
    from bgdebias_b200 import comix_loader as cl
    rng = np.random.default_rng(21)
    counts = [4, 0, 5]
    imgs = _images(rng, [SIZES[i % len(SIZES)] for i in range(sum(counts))])
    peers, names = _peers(pool, imgs, counts, [os.path.realpath(tmp_path / f"bg{i}.jpg") for i in range(len(imgs))])
    rep = pool.RaggedPool(256, "cuda")
    rep.append(imgs)
    B, T = 8, 3
    clip_sizes = [(224, 224)] * B if fg_form == "clips" else [(int(h), int(w)) for h, w in rng.integers(168, 257, (B, 2))]
    bg_files = [names[i] for i in (3, 1, 1, 8, 0, 5, 2, 7, 4, 6)]          # a reordered list with a repeat
    for rank, peer in enumerate(peers):
        results = {}
        for kind in ("replica", "peer"):
            ds = _dataset(cl, tmp_path, clip_sizes, T, prob)
            if kind == "replica":
                ds.attach_pool(names, rep)
            else:
                ds.attach_peer_pool(names, peer)
            ds.bg_files = list(bg_files)
            random.seed(5 + rank)
            torch.manual_seed(5 + rank)
            batch = ds.host_collate([ds[i] for i in range(B)])
            results[kind] = (batch, {f: ds.device_finish(batch, layout=f[2], dtype=f[0], memory_format=f[1]) for f in FORMS})
        (rb, ro), (pb, po) = results["replica"], results["peer"]
        assert torch.equal(rb["bg_idx"], pb["bg_idx"]) and torch.equal(rb["bg_apply"], pb["bg_apply"])
        assert (int(pb["bg_apply"].sum()) > 0) == (prob > 0)
        for f in FORMS:
            assert ro[f]["imgs"].shape == po[f]["imgs"].shape and ro[f]["imgs"].stride() == po[f]["imgs"].stride()
            assert torch.equal(_bits(po[f]["imgs"]), _bits(ro[f]["imgs"])), (rank, f)


def test_device_finish_reads_through_the_pool_attached_last(env, tmp_path):
    """device_finish brings a batch's images through the pool attached last: PeerPool.gather, ShardedPool.fetch, or neither
    (the replica of attach_pool)."""
    ops, _cabi, pool = env
    from bgdebias_b200 import comix_loader as cl
    imgs = _images(np.random.default_rng(1), SIZES[:2])
    peers, names = _peers(pool, imgs, [1, 1], [os.path.realpath(tmp_path / f"bg{i}.jpg") for i in range(2)])
    calls = []

    def counted(what, fn):
        def call(*args):
            calls.append(what)
            return fn(*args)
        return call

    for r, peer in enumerate(peers):
        gather = peer.gather
        peer.gather = counted(f"gather{r}", gather)
        peer.sharded.fetch = counted(f"fetch{r}", gather)     # the real fetch is a collective; gather returns the same batch

    ds = _dataset(cl, tmp_path, [(224, 224)], 2, prob=1.0)

    def finish():
        calls.clear()
        ds.bg_files = [names[0]]
        ds.device_finish(ds.host_collate([ds[0]]))
        return list(calls)

    ds.attach_peer_pool(names, peers[0])
    assert finish() == ["gather0"]
    ds.attach_sharded_pool(names, peers[0].sharded)
    assert finish() == ["fetch0"]
    ds.attach_peer_pool(names, peers[0])
    ds.attach_pool(names[:1], peers[0].sharded.local)
    assert finish() == []
    ds.attach_peer_pool(names, peers[1])
    assert finish() == ["gather1"]
    ds.bg_files = [names[1], str(tmp_path / "not_there.jpg")]
    assert ds._bg_hw(0) == peers[1].sharded.hw(1)
    with pytest.raises(ValueError, match="not_there.jpg"):
        ds._bg_hw(1)


def test_gather_refuses_a_changed_local_shard(env):
    ops, _cabi, pool = env
    imgs = _images(np.random.default_rng(2), SIZES[:3])
    peers, _ = _peers(pool, imgs, [2, 1])
    peers[0].gather(torch.tensor([0, 2]), torch.tensor([1, 1]))
    peers[0].sharded.local.append(_images(np.random.default_rng(3), [(16, 16)]))
    with pytest.raises(RuntimeError, match="stale"):
        peers[0].gather(torch.tensor([0, 2]), torch.tensor([1, 1]))


def test_device_finish_through_the_peer_pool_does_not_wait_for_the_stream(env, tmp_path):
    """With ~0.2 s of device work queued in front, device_finish of a peer-pool batch (pinned, as a DataLoader with
    pin_memory=True hands it over) returns before that work has finished -- fetch would wait for it."""
    import time
    ops, _cabi, pool = env
    from bgdebias_b200 import comix_loader as cl
    imgs = _images(np.random.default_rng(4), [SIZES[i % len(SIZES)] for i in range(6)])
    peers, names = _peers(pool, imgs, [2, 4])
    ds = _dataset(cl, tmp_path, [(224, 224)] * 6, 4, prob=0.9)
    ds.attach_peer_pool(names, peers[1])
    ds.bg_files = list(names)
    torch.manual_seed(0)
    batch = ds.host_collate([ds[i] for i in range(6)])
    assert int(batch["bg_apply"].sum()) > 0
    batch = {k: v.pin_memory() if isinstance(v, torch.Tensor) else v for k, v in batch.items()}
    ref = ds.device_finish(batch, dtype=torch.bfloat16)["imgs"]            # warm-up: LUT, resize tables, pinned blocks
    torch.cuda.synchronize()
    gate = torch.cuda.Event()
    torch.cuda._sleep(int(0.2 * 1.9e9))
    gate.record()
    t0 = time.perf_counter()
    out = ds.device_finish(batch, dtype=torch.bfloat16)["imgs"]
    host_s = time.perf_counter() - t0
    still_busy = not gate.query()
    torch.cuda.synchronize()
    assert still_busy, f"the host spent {host_s:.3f} s in device_finish and the stream had drained: it waited"
    assert host_s < 0.15
    assert torch.equal(_bits(out), _bits(ref))


# ---- two processes, CUDA IPC ----------------------------------------------------------------------------------------------
def _ipc_worker(rank, world, init, q):
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", init_method=init, rank=rank, world_size=world)
    try:
        import bgdebias_b200.ops as ops
        from bgdebias_b200 import pool
        counts = [3, 2]
        rng = np.random.default_rng(77)                                    # the same pool on both ranks
        imgs = _images(rng, [SIZES[i % len(SIZES)] for i in range(sum(counts))])
        first = sum(counts[:rank])
        local = pool.RaggedPool(256, "cuda")
        local.append(imgs[first:first + counts[rank]])
        sharded = pool.ShardedPool.from_local([f"bg{i}" for i in range(first, first + counts[rank])], local)
        peer = pool.PeerPool.open(sharded)
        mapped = len(peer._mapped)
        replica = pool.RaggedPool(256, "cuda")
        replica.append(imgs)
        lut = ops.make_fg_lut(MEAN, STD, "cuda")
        g = np.random.default_rng(500 + rank)
        B, T, P = 10, 2, sum(counts)
        equal, checked = True, 0
        for step in range(3 if rank == 0 else 1):                          # no lockstep: the ranks mix different counts
            idx = torch.from_numpy(g.integers(0, P, B))
            app = torch.from_numpy((g.random(B) < 0.7).astype(np.uint8))
            hw = [sharded.hw(int(i)) for i in idx]
            top = torch.tensor([int(g.integers(0, h - 224 + 1)) for h, _ in hw], dtype=torch.int32, device="cuda")
            left = torch.tensor([int(g.integers(0, w - 224 + 1)) for _, w in hw], dtype=torch.int32, device="cuda")
            fg = torch.from_numpy(g.integers(0, 256, (B, T, 224, 224, 3), dtype=np.uint8)).cuda()
            batch, slot = peer.gather(idx, app)
            app_d = app.to("cuda")
            for dt, layout in [(torch.float32, "NTCHW"), (torch.bfloat16, "NTHWC")]:
                got = torch.ops.bgdebias.bgmix_blend_ragged(fg, batch.data, batch.slots_tensor, batch.tables.tensor,
                                                            slot.to("cuda"), top, left, app_d, lut, torch.tensor(MEAN),
                                                            torch.tensor(STD), 0.5, layout, dt)
                exp = torch.ops.bgdebias.bgmix_blend_ragged(fg, replica.data, replica.slots_tensor, replica.tables.tensor,
                                                            idx.to("cuda", torch.int32), top, left, app_d, lut,
                                                            torch.tensor(MEAN), torch.tensor(STD), 0.5, layout, dt)
                equal &= bool(torch.equal(_bits(got), _bits(exp)))
                checked += 1
        peer.close()
        q.put((rank, mapped, checked, equal, None))
    except Exception as e:                                                 # reported to the parent, which fails the test
        q.put((rank, 0, 0, False, repr(e)))
    finally:
        dist.destroy_process_group()


def test_peer_pool_over_ipc_between_two_processes(tmp_path):
    import multiprocessing as mp
    import queue
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    init = f"file://{tmp_path / 'pg'}"
    procs = [ctx.Process(target=_ipc_worker, args=(r, 2, init, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = []
    try:
        for _ in procs:
            res.append(q.get(timeout=300))
    except queue.Empty:
        pass
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.kill()
                p.join()
    assert len(res) == 2, res
    for rank, mapped, checked, equal, err in sorted(res):
        assert err is None, (rank, err)
        assert mapped == 1 and equal and checked == (6 if rank == 0 else 2), rank
    assert all(p.exitcode == 0 for p in procs)
