"""The training route on the GPU: the two-stage geometry of bgmix_resize_blend / resize_bilinear against cv2 (resize to
(Wr, Hr), slice the MultiScaleCrop window, resize to 224) and the BG-mix oracle, bit for bit; and the dataset's
``device_train_pipeline`` route (native frames, host_collate -> device_finish) against the crops route (a worker running
Resize + MultiScaleCrop on the host) for dense, ragged, random-frame and emulated peer pools."""
import os
import random

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")

from oracle import bgmix_oracle as bo                     # noqa: E402

MEAN, STD = bo.DEFAULT_MEAN, bo.DEFAULT_STD
SIZES = [(240, 320), (240, 427), (256, 340), (320, 240), (233, 301)]
SCALES = (1, 0.875, 0.75, 0.66)


@pytest.fixture(scope="module")
def env():
    import bgdebias_b200.ops as ops
    from bgdebias_b200 import _cabi, comix_loader
    assert torch.cuda.is_available()
    _cabi.lib()
    return ops, _cabi, comix_loader


def _steps(num_fixed_crops=13, random_crop=False):
    return [dict(type="Resize", scale=(-1, 256)),
            dict(type="MultiScaleCrop", input_size=224, scales=SCALES, random_crop=random_crop, max_wh_scale_gap=1,
                 num_fixed_crops=num_fixed_crops),
            dict(type="Resize", scale=(224, 224), keep_ratio=False),
            dict(type="Normalize", mean=list(MEAN), std=list(STD), to_bgr=False), dict(type="FormatShape", input_format="NCHW")]


def _bits(t: torch.Tensor) -> torch.Tensor:
    t = t.contiguous().cpu()
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)


def _two_stage_cv2(clip, Hr, Wr, y0, x0, ch, cw, H=224, W=224):
    return np.stack([cv2.resize(cv2.resize(f, (Wr, Hr), interpolation=cv2.INTER_LINEAR)[y0:y0 + ch, x0:x0 + cw], (W, H),
                                interpolation=cv2.INTER_LINEAR) for f in clip])


def _windows(rng, clips):
    """One row per (clip, candidate crop size of every scale pair) with a random offset: the 11-column geometry."""
    out = []
    for k, clip in enumerate(clips):
        from bgdebias_b200.comix_loader import rescale_short_side
        Hr, Wr = rescale_short_side(clip.shape[1], clip.shape[2], 256)
        sizes = [int(min(Hr, Wr) * s) for s in SCALES]
        snap = lambda v: 224 if abs(v - 224) < 3 else v                     # noqa: E731
        for i, ch in enumerate(sizes):
            for j, cw in enumerate(sizes):
                if abs(i - j) <= 1:
                    ch2, cw2 = snap(ch), snap(cw)
                    out.append((k, Hr, Wr, int(rng.integers(0, Hr - ch2 + 1)), int(rng.integers(0, Wr - cw2 + 1)), ch2, cw2))
    return out


@pytest.mark.parametrize("T", [1, 8, 16])
@pytest.mark.parametrize("apply_mode", ["none", "all", "mixed"])
def test_bit_exact_against_cv2_and_the_oracle(env, T, apply_mode):
    ops, cabi, _ = env
    rng = np.random.default_rng(T)
    clips = [rng.integers(0, 256, (T, h, w, 3), dtype=np.uint8) for h, w in SIZES]
    wins = _windows(rng, clips)
    buf, g5 = ops.pack_clips(clips)
    geom = torch.tensor([g5[k].tolist() + [Hr, Wr, y0, x0, ch, cw] for k, Hr, Wr, y0, x0, ch, cw in wins])
    B, H, W = len(wins), 224, 224
    dev = torch.device("cuda")
    pool = rng.uniform(0, 255, (4, 3, 256, 300)).astype(np.float32)
    idx = rng.integers(0, 4, B)
    top, left = rng.integers(0, 256 - H + 1, B), rng.integers(0, 300 - W + 1, B)
    app = {"none": np.zeros(B, np.int64), "all": np.ones(B, np.int64), "mixed": rng.integers(0, 2, B)}[apply_mode]
    fg = np.stack([_two_stage_cv2(clips[k], Hr, Wr, y0, x0, ch, cw) for k, Hr, Wr, y0, x0, ch, cw in wins])
    exp = bo.mix_batch(fg, pool, idx, top, left, app, crop=(H, W), alpha=0.5)
    t = lambda a, dt: torch.tensor(np.asarray(a), dtype=dt, device=dev)     # noqa: E731
    lut = ops.make_fg_lut(MEAN, STD, dev)
    src, d_pool = buf.to(dev), torch.from_numpy(pool).to(dev)
    draws = (t(idx, torch.int32), t(top, torch.int32), t(left, torch.int32), t(app, torch.uint8), lut, torch.tensor(MEAN),
             torch.tensor(STD), 0.5)

    n0 = cabi.kernel_launch_count()
    u8 = torch.ops.bgdebias.resize_bilinear(src, geom, T, H, W)
    assert cabi.kernel_launch_count() - n0 == 1
    assert np.array_equal(u8.cpu().numpy(), fg)
    n0 = cabi.kernel_launch_count()
    got = torch.ops.bgdebias.bgmix_resize_blend(src, geom, T, H, W, d_pool, *draws, "NTCHW")
    assert cabi.kernel_launch_count() - n0 == 1
    np.testing.assert_array_equal(_bits(got).numpy(), exp.view(np.int32))

    if apply_mode != "mixed":
        return
    f32 = got.cpu()
    for layout in ("NTCHW", "NCTHW", "NTHWC"):
        for dt in (torch.float32, torch.bfloat16, torch.float16):
            o = torch.ops.bgdebias.bgmix_resize_blend(src, geom, T, H, W, d_pool, *draws, layout, dt).cpu()
            ref = {"NTCHW": f32, "NCTHW": f32.permute(0, 2, 1, 3, 4), "NTHWC": f32.permute(0, 1, 3, 4, 2)}[layout].to(dt)
            assert o.dtype == dt and torch.equal(_bits(o), _bits(ref)), (layout, dt)
    u8pool = torch.from_numpy(pool.round().astype(np.uint8)).to(dev)
    exp_u8 = bo.mix_batch(fg, pool.round().astype(np.uint8).astype(np.float32), idx, top, left, app, crop=(H, W), alpha=0.5)
    o = torch.ops.bgdebias.bgmix_resize_blend(src, geom, T, H, W, u8pool, *draws, "NTCHW")
    np.testing.assert_array_equal(_bits(o).numpy(), exp_u8.view(np.int32))


def test_small_and_odd_windows(env):
    """Up- and down-scaling in both stages, 1-pixel windows at the far corner, other output sizes, odd row strides."""
    ops, _, _ = env
    rng = np.random.default_rng(7)
    clips = [rng.integers(0, 256, (3, h, w, 3), dtype=np.uint8) for h, w in ((17, 29), (64, 33), (5, 7), (1, 1))]
    buf, g5 = ops.pack_clips(clips)
    H, W = 6, 9
    rows, exp = [], []
    for b, clip in enumerate(clips):
        for Hr, Wr in ((H, W), (40, 23), (11, 100), (1, 3)):
            for ch, cw in ((1, 1), (Hr, Wr), (max(1, Hr // 2), max(1, Wr - 1))):
                for y0, x0 in ((0, 0), (Hr - ch, Wr - cw)):
                    rows.append(g5[b].tolist() + [Hr, Wr, y0, x0, ch, cw])
                    exp.append(_two_stage_cv2(clip, Hr, Wr, y0, x0, ch, cw, H, W))
    got = torch.ops.bgdebias.resize_bilinear(buf.cuda(), torch.tensor(rows), 3, H, W).cpu().numpy()
    np.testing.assert_array_equal(got, np.stack(exp))


def test_opcheck(env):
    ops, _, _ = env
    rng = np.random.default_rng(1)
    buf, g5 = ops.pack_clips([rng.integers(0, 256, (2, h, w, 3), dtype=np.uint8) for h, w in ((12, 15), (15, 12))])
    geom = torch.cat([g5, torch.tensor([[16, 20, 1, 2, 12, 14], [20, 16, 0, 0, 20, 16]])], 1)
    dev = torch.device("cuda")
    src = buf.to(dev)
    torch.library.opcheck(torch.ops.bgdebias.resize_bilinear.default, (src, geom, 2, 8, 8))
    i32 = lambda v: torch.tensor(v, dtype=torch.int32, device=dev)         # noqa: E731
    pool = torch.rand(3, 3, 10, 10, device=dev) * 255
    for layout, dt in (("NTCHW", None), ("NTHWC", torch.bfloat16)):
        torch.library.opcheck(torch.ops.bgdebias.bgmix_resize_blend.default,
                              (src, geom, 2, 8, 8, pool, i32([2, 0]), i32([1, 0]), i32([0, 2]),
                               torch.tensor([1, 0], dtype=torch.uint8, device=dev), ops.make_fg_lut(MEAN, STD, dev),
                               torch.tensor(MEAN), torch.tensor(STD), 0.5, layout, dt))


def test_rejected_geometry_launches_nothing(env):
    ops, cabi, _ = env
    dev = torch.device("cuda")
    buf, g5 = ops.pack_clips([np.zeros((2, 20, 30, 3), np.uint8)])
    src = buf.to(dev)
    base = g5[0].tolist()
    pool = torch.zeros(1, 3, 8, 8, device=dev)
    z32 = lambda n: torch.zeros(n, dtype=torch.int32, device=dev)          # noqa: E731
    lut = ops.make_fg_lut(MEAN, STD, dev)
    calls = {
        "resize_bilinear": lambda rows, s=src: torch.ops.bgdebias.resize_bilinear(s, torch.tensor(rows, dtype=torch.int64), 2, 8, 8),
        "bgmix_resize_blend": lambda rows, s=src: torch.ops.bgdebias.bgmix_resize_blend(
            s, torch.tensor(rows, dtype=torch.int64), 2, 8, 8, pool, z32(len(rows)), z32(len(rows)), z32(len(rows)),
            torch.ones(len(rows), dtype=torch.uint8, device=dev), lut, torch.tensor(MEAN), torch.tensor(STD), 0.5, "NTCHW"),
    }
    bad = {
        "window below": [base + [16, 24, 9, 0, 8, 8]],
        "window right": [base + [16, 24, 0, 17, 8, 8]],
        "window taller than Hr": [base + [16, 24, 0, 0, 17, 8]],
        "negative y0": [base + [16, 24, -1, 0, 8, 8]],
        "negative x0": [base + [16, 24, 0, -1, 8, 8]],
        "zero Hr": [base + [0, 24, 0, 0, 1, 1]],
        "zero Wr": [base + [16, 0, 0, 0, 1, 1]],
        "zero ch": [base + [16, 24, 0, 0, 0, 8]],
        "zero cw": [base + [16, 24, 0, 0, 8, 0]],
        "second entry bad": [base + [16, 24, 0, 0, 16, 24], base + [8, 8, 0, 1, 8, 8]],
    }
    for name, call in calls.items():
        call([base + [16, 24, 8, 16, 8, 8]])                               # the last window that fits
        torch.cuda.synchronize()
        n0 = cabi.kernel_launch_count()
        for what, rows in bad.items():
            with pytest.raises(ValueError, match="libbgdebias_b200: resize"):
                call(rows)
        with pytest.raises(ValueError, match="ends at byte"):
            call([base + [16, 24, 0, 0, 8, 8]], s=src[:src.numel() - 8])
        with pytest.raises(ValueError, match=r"geom must be int64 \[B, 5 or 11\]"):
            call([base + [16, 24, 0, 0]])
        torch.cuda.synchronize()
        assert cabi.kernel_launch_count() == n0, name


# ---- the dataset route against the crops route ----------------------------------------------------------------------------
class _Frames:
    """Picklable training pipeline stopped after RawFrameDecode: a list of uint8 [h, w, 3] RGB frames per video."""
    def __init__(self, clips):
        self.clips = clips

    def __call__(self, info):
        return dict(imgs=list(self.clips[info["sample"]]), label=torch.tensor([info["label"]]))


class _CropsOnHost(_Frames):
    """The crops route's worker: Resize(scale=(-1, 256)) and MultiScaleCrop on the host, with the same rules and draws."""
    def __init__(self, clips, tp):
        super().__init__(clips)
        self.tp = tp

    def __call__(self, info):
        out = super().__call__(info)
        h, w = out["imgs"][0].shape[:2]
        Hr, Wr, y0, x0, ch, cw = self.tp.draw(h, w)
        out["imgs"] = [cv2.resize(f, (Wr, Hr), interpolation=cv2.INTER_LINEAR)[y0:y0 + ch, x0:x0 + cw] for f in out["imgs"]]
        return out


class _Reader:
    def __init__(self, imgs):
        self.imgs = imgs

    def __call__(self, path):
        return self.imgs[int(os.path.basename(path).split(".")[0][2:]) % len(self.imgs)]


def _datasets(cl, tmp_path, clips, bg_imgs, steps, **kw):
    for i in range(len(bg_imgs)):
        (tmp_path / f"bg{i}.jpg").write_bytes(b"stub")
    infos = [dict(frame_dir=str(tmp_path / f"bg{i}"), total_frames=len(bg_imgs), label=i, sample=i) for i in range(len(clips))]
    common = dict(bg_dir=str(tmp_path), device_mix=True, prob=0.5, bg_reader=_Reader(bg_imgs), device="cuda",
                  extract_bg_if_not_found=False, map_bg_to_video=False, filename_tmpl="bg{}.jpg", start_index=0, **kw)
    new = cl.BackgroundMixDataset(infos, _Frames(clips), device_train_pipeline=steps, **common)
    old = cl.BackgroundMixDataset(infos, _CropsOnHost(clips, cl.TrainPipeline(steps)), **common)
    return new, old


FORMS = [(torch.float32, torch.contiguous_format, "NTCHW"), (torch.float32, torch.contiguous_format, "NCTHW"),
         (torch.bfloat16, torch.channels_last, "NTCHW"), (torch.float16, torch.contiguous_format, "NTCHW")]


def _compare(cabi, new, old, B, n_batches, launches):
    for it in range(n_batches):
        batches = {}
        for name, ds in (("new", new), ("old", old)):
            random.seed(40 + it)
            torch.manual_seed(40 + it)
            batches[name] = ds.host_collate([ds[(it * B + i) % len(ds)] for i in range(B)])
        nb, ob = batches["new"], batches["old"]
        assert nb["fg_geom"].shape[1] == 11 and ob["fg_geom"].shape[1] == 5
        for k in ("bg_idx", "bg_top", "bg_left", "bg_apply"):
            assert torch.equal(nb[k], ob[k]), k
        for dt, mf, layout in FORMS:
            n0 = cabi.kernel_launch_count()
            a = new.device_finish(nb, layout=layout, dtype=dt, memory_format=mf)["imgs"]
            if launches is not None:
                assert cabi.kernel_launch_count() - n0 == launches
            b = old.device_finish(ob, layout=layout, dtype=dt, memory_format=mf)["imgs"]
            assert a.shape == b.shape and a.stride() == b.stride() and a.dtype == b.dtype == dt
            assert torch.equal(a, b), (it, dt, mf, layout)


@pytest.mark.parametrize("pool_kind", ["dense", "ragged", "random_frame"])
def test_device_finish_equals_the_crops_route(env, tmp_path, pool_kind):
    ops, cabi, cl = env
    rng = np.random.default_rng(5)
    T, B = 8, 6
    clips = [rng.integers(0, 256, (T, h, w, 3), dtype=np.uint8) for h, w in SIZES * 2]
    bg_sizes = {"dense": [(256, 341)], "ragged": [(240, 320), (240, 427), (256, 300), (300, 400)],
                "random_frame": [(240, 320), (256, 340)]}[pool_kind]
    bg_imgs = [torch.from_numpy(rng.integers(0, 256, (3, h, w), dtype=np.uint8)) for h, w in bg_sizes * 2]
    kw = dict(back_ground_from_bg_dir=pool_kind != "random_frame")
    new, old = _datasets(cl, tmp_path, clips, bg_imgs, _steps(), **kw)
    if pool_kind != "random_frame":
        assert (new.device_pool().tensor is not None) == (pool_kind == "dense")
    _compare(cabi, new, old, B, 3, {"dense": 1, "ragged": 2, "random_frame": None}[pool_kind])


def test_device_finish_equals_the_crops_route_through_peers(env, tmp_path):
    ops, cabi, cl = env
    from bgdebias_b200 import pool
    rng = np.random.default_rng(9)
    T, B = 8, 6
    clips = [rng.integers(0, 256, (T, h, w, 3), dtype=np.uint8) for h, w in SIZES * 2]
    bg_imgs = [torch.from_numpy(rng.integers(0, 256, (3, h, w), dtype=np.uint8))
               for h, w in [(240, 320), (240, 427), (256, 300), (300, 400), (256, 256)]]
    new, old = _datasets(cl, tmp_path, clips, bg_imgs, _steps(num_fixed_crops=5, random_crop=True))
    names = [os.path.realpath(tmp_path / f"bg{i}.jpg") for i in range(len(bg_imgs))]
    counts = [2, 0, 3]
    owner = np.concatenate([np.full(c, r, np.int64) for r, c in enumerate(counts)])
    slot = np.concatenate([np.arange(c, dtype=np.int64) for c in counts])
    h, w = [int(t.shape[1]) for t in bg_imgs], [int(t.shape[2]) for t in bg_imgs]
    shards, at = [], 0
    for r, c in enumerate(counts):                                        # the W shards of an emulated node, all held here
        local = pool.RaggedPool(256, "cuda")
        local.append(bg_imgs[at:at + c])
        at += c
        shards.append(pool.ShardedPool(local, names, owner, slot, h, w, r, len(counts)))
    bases = [sp.local.data.data_ptr() if sp.local.used else 0 for sp in shards]
    sizes = [sp.local.used for sp in shards]
    src_offset = [int(shards[o].local.slots["offset"][s]) for o, s in zip(owner, slot)]
    rep = pool.RaggedPool(256, "cuda")
    rep.append(bg_imgs)
    new.attach_peer_pool(names, pool.PeerPool(shards[0], bases, sizes, src_offset))
    old.attach_pool(names, rep)
    new.bg_files = old.bg_files = list(names)
    _compare(cabi, new, old, B, 3, None)


def test_dataloader_workers_then_device_finish(env, tmp_path):
    """A training dataset behind a DataLoader with 2 worker processes: workers ship native uint8 frames and the two-stage
    geometry; device_finish mixes each batch in one launch, bit-equal to cv2 on the host plus the oracle."""
    ops, cabi, cl = env
    rng = np.random.default_rng(3)
    T = 8
    clips = [rng.integers(0, 256, (T, h, w, 3), dtype=np.uint8) for h, w in SIZES * 2]
    bg_imgs = [torch.from_numpy(rng.integers(0, 256, (3, 256, 341), dtype=np.uint8)) for _ in range(3)]
    new, _ = _datasets(cl, tmp_path, clips, bg_imgs, _steps())
    pool_t = new.device_pool().tensor
    assert pool_t is not None
    loader = torch.utils.data.DataLoader(new, batch_size=4, shuffle=False, num_workers=2, collate_fn=new.host_collate,
                                         pin_memory=True)
    seen = 0
    for batch in loader:
        assert batch["imgs"].dtype == torch.uint8 and not batch["imgs"].is_cuda and batch["fg_geom"].shape[1] == 11
        B = batch["fg_geom"].shape[0]
        n0 = cabi.kernel_launch_count()
        out = new.device_finish(batch)
        assert cabi.kernel_launch_count() - n0 == 1
        assert tuple(out["imgs"].shape) == (B, T, 3, 224, 224) and out["imgs"].dtype == torch.float32
        fg = np.stack([_two_stage_cv2(clips[seen + b], *batch["fg_geom"][b, 5:].tolist()) for b in range(B)])
        rows = new.device_pool().rows(batch["bg_idx"].clamp(min=0).to(torch.int32).cuda()).cpu()
        exp = bo.mix_batch(fg, pool_t.cpu().numpy(), rows.tolist(), batch["bg_top"].tolist(),
                           batch["bg_left"].tolist(), batch["bg_apply"].tolist(), crop=(224, 224), alpha=0.5)
        np.testing.assert_array_equal(_bits(out["imgs"]).numpy(), exp.view(np.int32))
        seen += B
    assert seen == len(clips)
