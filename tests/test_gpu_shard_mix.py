"""BG-mix from a background pool sharded across ranks (pool.ShardedPool, BackgroundMixDataset.attach_sharded_pool).

* ``ragged_pack`` (the owner's one-launch gather) equals torch slicing, takes one launch, passes opcheck and rejects bad
  segment tables.
* One process holds 2-4 shards of a pool of mixed widths; the exchange is emulated by concatenating, for each receiving
  rank, the packed chunks of every source in rank order -- what ``all_to_all_single`` delivers -- and every blend from the
  fetched images equals ``bgmix_blend_ragged`` on the replicated pool, bit for bit, for every output dtype and layout, for
  resized clips and for packed crops.
* With a real NCCL group of world size 1, ``device_finish`` of a sharded dataset equals the same batch from ``attach_pool``
  with the replicated pool."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DTYPES = [torch.float32, torch.bfloat16, torch.float16]
LAYOUTS = ["NTCHW", "NCTHW", "NTHWC"]
MEAN, STD = (123.675, 116.28, 103.53), (58.395, 57.12, 57.375)


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


# ---- ragged_pack ----------------------------------------------------------------------------------------------------------
def _pack_case(env, rng, sizes, picks):
    ops, _cabi, pool = env
    rp = pool.RaggedPool(None, "cuda")
    imgs = _images(rng, sizes)
    rp.append(imgs)
    segs, at = [], 0
    for k in picks:
        b = int(imgs[k].numel())
        segs.append((int(rp.slots[k]["offset"]), at, b))
        at += (b + 15) & ~15
    seg = torch.tensor(segs, dtype=torch.int64).reshape(-1, 3)
    n0 = _cabi.kernel_launch_count()
    out = torch.ops.bgdebias.ragged_pack(rp.data, seg, at)
    torch.cuda.synchronize()
    launches = _cabi.kernel_launch_count() - n0
    got = out.cpu()
    for (so, do, b), k in zip(segs, picks):
        assert torch.equal(got[do:do + b], rp.data[so:so + b].cpu())
        assert torch.equal(got[do:do + b], imgs[k].reshape(-1))
    return launches, rp


@pytest.mark.parametrize("case", ["mixed", "one", "many", "empty", "zero_bytes"])
def test_ragged_pack_equals_slicing(env, case):
    rng = np.random.default_rng(len(case))
    if case == "mixed":
        sizes = [(240, 427), (240, 320), (17, 5), (1, 1), (256, 341), (3, 7)]
        picks = [4, 0, 2, 3, 0, 5, 1]                     # a repeat, odd sizes (byte tails), a 3-byte image
    elif case == "one":
        sizes, picks = [(240, 427)], [0]
    elif case == "many":
        sizes = [(int(h), int(w)) for h, w in rng.integers(1, 90, (300, 2))]
        picks = rng.permutation(300).tolist()
    else:
        sizes, picks = [(8, 8)], []
    if case == "zero_bytes":
        ops, _cabi, pool = env
        rp = pool.RaggedPool(None, "cuda")
        rp.append(_images(rng, [(8, 8)]))
        n0 = _cabi.kernel_launch_count()
        out = torch.ops.bgdebias.ragged_pack(rp.data, torch.tensor([[0, 0, 0], [16, 32, 0]]), 48)
        torch.cuda.synchronize()
        assert out.numel() == 48 and _cabi.kernel_launch_count() == n0
        return
    launches, _ = _pack_case(env, rng, sizes, picks)
    assert launches == (1 if picks else 0)


def test_ragged_pack_opcheck(env):
    ops, _cabi, pool = env
    src = torch.randint(0, 256, (4096,), dtype=torch.uint8, device="cuda")
    seg = torch.tensor([[1024, 0, 512], [0, 512, 1024], [2048, 1536, 2048]], dtype=torch.int64)   # covers all 3584 bytes
    torch.library.opcheck(torch.ops.bgdebias.ragged_pack, (src, seg, 3584))


def test_ragged_pack_rejects_bad_segments(env):
    src = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    bad = {
        "misaligned source": [[8, 0, 64]],
        "misaligned destination": [[0, 4, 64]],
        "source out of range": [[4080, 0, 32]],
        "destination out of range": [[0, 1008, 32]],
        "negative": [[0, 0, -1]],
    }
    for what, seg in bad.items():
        with pytest.raises(ValueError, match="ragged_pack"):
            torch.ops.bgdebias.ragged_pack(src, torch.tensor(seg, dtype=torch.int64), 1024)
    with pytest.raises(ValueError, match="16-byte aligned"):
        torch.ops.bgdebias.ragged_pack(src[1:], torch.tensor([[0, 0, 16]], dtype=torch.int64), 1024)
    with pytest.raises(ValueError):
        torch.ops.bgdebias.ragged_pack(src, torch.zeros((2, 2), dtype=torch.int64), 64)


# ---- emulated exchange between 2-4 shards ---------------------------------------------------------------------------------
SIZES = [(120, 160), (120, 214), (120, 176), (128, 128), (100, 180)]          # mixed widths, all >= the crop after Resize
BG_RESIZE, CROP = 128, (112, 112)
SIZES2 = [(240, 320), (240, 427), (240, 352), (256, 256)]                     # dataset tests: Resize(256), 224 crops


def _shards(pool, imgs, counts):
    """ShardedPool objects of every rank of a world of len(counts), built as from_local would (index in rank order)."""
    world = len(counts)
    owner = np.concatenate([np.full(c, r, np.int64) for r, c in enumerate(counts)])
    slot = np.concatenate([np.arange(c, dtype=np.int64) for c in counts])
    h = [int(t.shape[1]) for t in imgs]
    w = [int(t.shape[2]) for t in imgs]
    names = [f"bg{i}" for i in range(len(imgs))]
    out, at = [], 0
    for r, c in enumerate(counts):
        local = pool.RaggedPool(BG_RESIZE, "cuda")
        local.append(imgs[at:at + c])
        at += c
        out.append(pool.ShardedPool(local, names, owner, slot, h, w, r, world))
    return out


def _emulated_fetch(shards, batches):
    """fetch() of every rank with all_gather_object / all_to_all_single replaced by their results."""
    world = len(shards)
    requests = [shards[0].requests_of(b["idx"], b["app"]) for b in batches]
    routes = [sp.route(requests) for sp in shards]
    sends = [sp.pack(rt) for sp, rt in zip(shards, routes)]
    out = []
    for d in range(world):
        parts = []
        for s in range(world):
            lo = sum(routes[s].send_splits[:d])
            parts.append(sends[s][lo:lo + routes[s].send_splits[d]])
        recv = torch.cat(parts) if parts else torch.empty(0, dtype=torch.uint8, device="cuda")
        assert recv.numel() == sum(routes[d].recv_splits)
        batch = shards[d].assemble(recv, requests[d], routes[d])
        out.append((batch, shards[d].sample_slots(batches[d]["idx"], batches[d]["app"], requests[d])))
    return out


def _draws(rng, pool_hw, B, P):
    idx = rng.integers(0, P, B)
    app = (rng.random(B) < 0.7).astype(np.uint8)
    top = [int(rng.integers(0, pool_hw[i][0] - CROP[0] + 1)) for i in idx]
    left = [int(rng.integers(0, pool_hw[i][1] - CROP[1] + 1)) for i in idx]
    return dict(idx=torch.from_numpy(idx), app=torch.from_numpy(app), top=torch.tensor(top, dtype=torch.int32),
                left=torch.tensor(left, dtype=torch.int32))


@pytest.mark.parametrize("counts", [[7, 5], [1, 0, 11], [4, 4, 3, 1]])
@pytest.mark.parametrize("fg_form", ["clips", "packed_crops"])
def test_emulated_exchange_equals_replicated_pool(env, counts, fg_form):
    ops, _cabi, pool = env
    rng = np.random.default_rng(sum(counts) * 7 + len(counts))
    P = sum(counts)
    imgs = _images(rng, [SIZES[i % len(SIZES)] for i in rng.permutation(P)])
    rep = pool.RaggedPool(BG_RESIZE, "cuda")
    rep.append(imgs)
    shards = _shards(pool, imgs, counts)
    pool_hw = [rep.hw(i) for i in range(P)]
    for i in range(P):
        assert shards[0].hw(i) == pool_hw[i]
    B, T = 6, 3
    batches = [_draws(rng, pool_hw, B, P) for _ in counts]
    if len(counts) > 2:
        batches[-1]["app"][:] = 0                                            # a rank that mixes nothing
    fetched = _emulated_fetch(shards, batches)
    lut = ops.make_fg_lut(MEAN, STD, "cuda")
    mean_t, std_t = torch.tensor(MEAN), torch.tensor(STD)
    for d, (batch, slot) in enumerate(fetched):
        b = batches[d]
        if not len(batch):
            batch.append([torch.zeros((3, *CROP), dtype=torch.uint8)])
        if fg_form == "clips":
            fg = torch.from_numpy(rng.integers(0, 256, (B, T, *CROP, 3), dtype=np.uint8)).cuda()
        else:
            clips = [torch.from_numpy(rng.integers(0, 256, (T, int(h), int(w), 3), dtype=np.uint8))
                     for h, w in rng.integers(90, 150, (B, 2))]
            src, geom = ops.pack_clips(clips)
            fg = torch.ops.bgdebias.resize_bilinear(src.cuda(), geom, T, *CROP)
        dev = lambda x, dt: x.to("cuda", dt)                                  # noqa: E731
        top, left, app = dev(b["top"], torch.int32), dev(b["left"], torch.int32), dev(b["app"], torch.uint8)
        for dt in DTYPES:
            for layout in LAYOUTS:
                exp = torch.ops.bgdebias.bgmix_blend_ragged(fg, rep.data, rep.slots_tensor, rep.tables.tensor,
                                                            dev(b["idx"], torch.int32), top, left, app, lut, mean_t, std_t,
                                                            0.5, layout, dt)
                got = torch.ops.bgdebias.bgmix_blend_ragged(fg, batch.data, batch.slots_tensor, batch.tables.tensor,
                                                            dev(slot, torch.int32), top, left, app, lut, mean_t, std_t,
                                                            0.5, layout, dt)
                assert torch.equal(_bits(got), _bits(exp)), (d, dt, layout)


# ---- real NCCL group of world size 1 --------------------------------------------------------------------------------------
@pytest.fixture
def nccl_group(tmp_path):
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", init_method=f"file://{tmp_path / 'pg'}", rank=0, world_size=1,
                            device_id=torch.device("cuda:0"))
    yield
    dist.destroy_process_group()


def _dataset(cl, bg_dir, clip_sizes, T):
    infos = [dict(frame_dir=f"/d/v{i}", total_frames=8, label=i) for i in range(len(clip_sizes))]

    def pipe(r):
        i = int(r["label"])
        h, w = clip_sizes[i]
        g = np.random.default_rng(100 + i)
        return dict(r, imgs=torch.from_numpy(g.integers(0, 256, (T, h, w, 3), dtype=np.uint8)))

    return cl.BackgroundMixDataset(infos, pipe, bg_dir=str(bg_dir), extract_bg_if_not_found=False, device_mix=True,
                                   prob=0.6, device="cuda")


@pytest.mark.parametrize("pool_sizes", ["uniform", "mixed"])
@pytest.mark.parametrize("fg_form", ["clips", "packed_crops"])
def test_device_finish_sharded_equals_replicated(env, nccl_group, tmp_path, pool_sizes, fg_form):
    """A uniform pool takes the dense route on the replica (bgmix_blend / bgmix_resize_blend), a mixed one the ragged route;
    the sharded dataset always fetches and blends ragged, and every form must give the same bits."""
    import random
    import torch.distributed as dist
    ops, _cabi, pool = env
    from bgdebias_b200 import comix_loader as cl
    rng = np.random.default_rng(11)
    sizes = [(240, 320)] * 9 if pool_sizes == "uniform" else [SIZES2[i % len(SIZES2)] for i in range(9)]
    imgs = _images(rng, sizes)
    paths = [os.path.realpath(tmp_path / f"bg{i}.jpg") for i in range(len(imgs))]
    rep = pool.RaggedPool(256, "cuda")
    rep.append(imgs)
    local = pool.RaggedPool(256, "cuda")
    local.append(imgs)
    sharded = pool.ShardedPool.from_local(paths, local, dist.group.WORLD)
    assert sharded.index() == [(p, 0, i) for i, p in enumerate(paths)]
    B, T = 8, 4
    clip_sizes = [(224, 224)] * B if fg_form == "clips" else [(int(h), int(w)) for h, w in rng.integers(168, 257, (B, 2))]
    bg_files = [paths[i] for i in (3, 1, 1, 8, 0, 5, 2, 7, 4, 6)]           # a reordered list with a repeat
    results = {}
    for kind in ("replica", "sharded"):
        ds = _dataset(cl, tmp_path, clip_sizes, T)
        if kind == "replica":
            ds.attach_pool(paths, rep)
        else:
            ds.attach_sharded_pool(paths, sharded)
        ds.bg_files = list(bg_files)
        random.seed(3)
        torch.manual_seed(3)
        batch = ds.host_collate([ds[i] for i in range(B)])
        assert int(batch["bg_apply"].sum()) > 0
        outs = {}
        for dt, mf in [(torch.float32, torch.contiguous_format), (torch.bfloat16, torch.channels_last),
                       (torch.float16, torch.contiguous_format)]:
            for layout in ("NTCHW", "NCTHW"):
                outs[(dt, mf, layout)] = ds.device_finish(batch, layout=layout, dtype=dt, memory_format=mf)
        results[kind] = (batch, outs)
    rb, ro = results["replica"]
    sb, so = results["sharded"]
    assert torch.equal(rb["bg_idx"], sb["bg_idx"]) and torch.equal(rb["bg_top"], sb["bg_top"])
    assert torch.equal(rb["bg_left"], sb["bg_left"]) and torch.equal(rb["bg_apply"], sb["bg_apply"])
    for key in ro:
        assert set(ro[key]) == set(so[key])
        assert ro[key]["imgs"].shape == so[key]["imgs"].shape and ro[key]["imgs"].stride() == so[key]["imgs"].stride()
        assert torch.equal(_bits(so[key]["imgs"]), _bits(ro[key]["imgs"])), key
        assert torch.equal(so[key]["bg_idx"], ro[key]["bg_idx"])


def test_device_finish_sharded_with_no_mixed_sample(env, nccl_group, tmp_path):
    """A batch that mixes nothing still takes part in the exchange and returns the normalised clips."""
    import torch.distributed as dist
    ops, _cabi, pool = env
    from bgdebias_b200 import comix_loader as cl
    imgs = _images(np.random.default_rng(2), [(240, 320), (240, 427)])
    paths = [os.path.realpath(tmp_path / f"bg{i}.jpg") for i in range(2)]
    local = pool.RaggedPool(256, "cuda")
    local.append(imgs)
    ds = _dataset(cl, tmp_path, [(224, 224)] * 4, 2)
    ds.attach_sharded_pool(paths, pool.ShardedPool.from_local(paths, local, dist.group.WORLD))
    ds.bg_files = list(paths)
    ds.prob = 0.0
    batch = ds.host_collate([ds[i] for i in range(4)])
    out = ds.device_finish(batch)["imgs"]
    lut = ops.make_fg_lut(MEAN, STD)
    exp = torch.stack([lut[c][batch["imgs"][..., c].long()] for c in range(3)], 2)
    assert torch.equal(out.cpu(), exp)
