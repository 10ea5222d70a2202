"""GPU parity of the ragged-pool BG-mix path (csrc/raggedmix.cu): backgrounds of mixed sizes, the random-frame mode and
the on-device Resize(bg_resize), against the reference's own outputs (tests/golden/bgmix_ragged_reference.npz, written
by oracle/gen_golden_ragged.py from the unmodified BackgroundMixDataset), the oracle and torchvision.  Tolerance from
BASELINE.json: 1e-6 relative (fp32); the kernels round every operation like the reference, so bit equality is asserted too."""
import hashlib
import pathlib
import random
import tempfile

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from conftest import GOLDEN                                   # noqa: E402
from oracle import aa_resize_oracle as ao, bgmix_oracle as bo  # noqa: E402
from test_oracle_aa_resize import SIZES, fullsize_inputs       # noqa: E402

_NPZ = np.load(GOLDEN / "bgmix_ragged_reference.npz")
POOL_CASES = ["mixed_widths", "portrait_mix", "down_and_up", "skipped_axes"]
FRAME_CASES = ["type_a", "type_a_p"]
RTOL = ATOL = 1e-6


@pytest.fixture(scope="module")
def env():
    import bgdebias_b200.ops as ops
    from bgdebias_b200 import _cabi, comix_loader, pool
    assert torch.cuda.is_available()
    _cabi.lib()
    return ops, _cabi, comix_loader, pool


def _assert_same(got, exp):
    np.testing.assert_allclose(got, exp, rtol=RTOL, atol=ATOL)
    np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32))


@pytest.mark.parametrize("h,w,size", SIZES)
def test_device_resize_equals_torchvision_bit_for_bit(env, h, w, size):
    """bgd_aa_resize_u8_f32 against Resize(size)(img.float()) -- the call of comix_loader.py:72,140."""
    from torchvision.transforms import Resize
    ops, cabi, cl, pool_mod = env
    rng = np.random.default_rng(h * 1000 + w)
    imgs = [rng.integers(0, 256, (3, h, w), dtype=np.uint8), rng.integers(0, 256, (3, h + 3, w + 5), dtype=np.uint8)]
    rp = pool_mod.RaggedPool(size, "cuda")
    rp.append(imgs)
    for i, img in enumerate(imgs):
        ref = Resize(size)(torch.from_numpy(img).float()).numpy()
        got = rp.resized(i).cpu().numpy()
        assert got.shape == ref.shape and rp.hw(i) == ref.shape[1:]
        np.testing.assert_array_equal(got.view(np.uint32), ref.view(np.uint32))


def _dataset(cl, name, fg, ra, reader, bg_dir, **kw):
    th, tw, size, alpha, with_ra, prob, seed = _NPZ[name + "/params"]
    return cl.BackgroundMixDataset(kw.pop("infos"), lambda info: dict(imgs=torch.from_numpy(fg[info["sample"]]), label=torch.tensor([info["label"]]),
                                                                      randAug=bool(ra[info["sample"]])),
                                   bg_dir=str(bg_dir), bg_resize=int(size), bg_crop_size=(int(th), int(tw)), alpha=float(alpha), prob=float(prob),
                                   with_randAug=bool(with_ra), device_mix=True, bg_reader=reader, **kw), int(seed)


@pytest.mark.parametrize("name", POOL_CASES)
def test_mixed_size_pool_through_the_dataset_matches_the_reference(env, name):
    """device_mix=True on a pool of mixed sizes: same kwargs and seeds as the reference run, uint8 clips, one launch per
    batch; the crop offsets are drawn from the DRAWN image's size (comix_loader.py:126-141)."""
    ops, cabi, cl, pool_mod = env
    fg, ra, order = _NPZ[name + "/fg"], _NPZ[name + "/randAug"], _NPZ[name + "/bg_files_order"]
    n_bg = int(_NPZ[name + "/n_bg"])
    pool = [_NPZ[f"{name}/pool_{i:03d}"] for i in range(n_bg)]
    with tempfile.TemporaryDirectory() as tmp:
        bg_dir = pathlib.Path(tmp) / "bg"
        bg_dir.mkdir()
        names = [f"v{i:03d}" for i in range(n_bg)]
        for n in names:
            (bg_dir / (n + ".jpg")).write_bytes(b"stub")
        infos = [dict(frame_dir=f"/nowhere/{names[i % n_bg]}", total_frames=fg.shape[1], label=i, sample=i) for i in range(len(fg))]
        path_to_idx = {str((bg_dir / (n + ".jpg")).resolve()): i for i, n in enumerate(names)}
        ds, seed = _dataset(cl, name, fg, ra, lambda p: pool[path_to_idx[str(pathlib.Path(p).resolve())]], bg_dir, infos=infos)
        assert [path_to_idx[str(pathlib.Path(p).resolve())] for p in ds.bg_files] == list(order)
        for dense_budget in (None, 0):                                # the store's choice, then the ragged path forced
            ds._store = None if dense_budget is None else pool_mod.BackgroundStore(ds.bg_resize, ds.device, dense_budget_bytes=0)
            ds._pool = None
            random.seed(seed)
            torch.manual_seed(seed)
            samples = [ds.prepare_train_frames(i) for i in range(len(fg))]
            batch = ds.gpu_collate(samples)
            assert [int(s["bg_idx"]) for s in samples] == _NPZ[name + "/bg_idx"].tolist()
            _assert_same(batch["imgs"].cpu().numpy(), _NPZ[name + "/expected"])
        assert ds.device_pool().tensor is None                        # mixed sizes (or no budget): no dense cache


@pytest.mark.parametrize("name", FRAME_CASES)
def test_random_frame_mode_through_the_dataset_matches_the_reference(env, name, tmp_path):
    """back_ground_from_bg_dir=False ("type A", comix_loader.py:133-136) under device_mix=True: the decoded frames travel
    with the batch and are its pool; bg_idx = -2."""
    ops, cabi, cl, pool_mod = env
    fg, ra = _NPZ[name + "/fg"], _NPZ[name + "/randAug"]
    paths = [str(p) for p in _NPZ[name + "/frame_paths"]]
    frames = {p: _NPZ[f"{name}/frame_{i:03d}"] for i, p in enumerate(paths)}
    n_frames, vid_of = _NPZ[name + "/video_frames"], _NPZ[name + "/video_of_sample"]
    infos = [dict(frame_dir=f"/nowhere/{name}/vid{int(v):02d}", total_frames=int(n_frames[v]), label=i, sample=i) for i, v in enumerate(vid_of)]
    drawn = []
    ds, seed = _dataset(cl, name, fg, ra, lambda p: (drawn.append(paths.index(p)), frames[p])[1], tmp_path / "bg", infos=infos,
                        back_ground_from_bg_dir=False)
    assert ds.bg_files == []
    random.seed(seed)
    torch.manual_seed(seed)
    samples = [ds.prepare_train_frames(i) for i in range(len(fg))]
    assert [int(s["bg_idx"]) for s in samples] == _NPZ[name + "/bg_idx"].tolist() and drawn == _NPZ[name + "/drawn"].tolist()
    batch = ds.host_collate(samples)
    assert len(batch["bg_imgs"]) == sum(1 for s in samples if s["bg_idx"] == -2) and not batch["imgs"].is_cuda
    out = ds.device_finish(batch)
    assert set(out) == {"imgs", "bg_idx", "label", "randAug"}
    _assert_same(out["imgs"].cpu().numpy(), _NPZ[name + "/expected"])
    # a batch in which nothing was mixed is the plain normalisation
    none = ds.host_collate([dict(s, bg_apply=0, bg_idx=-1) for s in samples if "bg_img" not in s] or
                           [dict({k: v for k, v in samples[0].items() if k != "bg_img"}, bg_apply=0, bg_idx=-1)])
    got = ds.device_finish(none)["imgs"].cpu().numpy()
    exp = np.stack([bo.fg_normalize(f.numpy(), bo.fg_lut()) for f in none["imgs"]])
    _assert_same(got, exp)


def test_fullsize_mixed_width_pool_digest(env, tmp_path):
    """240x320 / 240x427 / 240x352 / 256x256 backgrounds (the widths HMDB51 and Sth-Sth-v2 mix) -> Resize(256) ->
    RandomCrop(224), 8 x 224 x 224 clips: the reference's bytes, by digest."""
    ops, cabi, cl, pool_mod = env
    fg, pool = fullsize_inputs(_NPZ)
    order = _NPZ["fullsize/bg_files_order"]
    names = [f"v{i:03d}" for i in range(len(pool))]
    for n in names:
        (tmp_path / (n + ".jpg")).write_bytes(b"stub")
    infos = [dict(frame_dir=f"/nowhere/{names[i % len(pool)]}", total_frames=8, label=i, sample=i) for i in range(4)]
    path_to_idx = {str((tmp_path / (n + ".jpg")).resolve()): i for i, n in enumerate(names)}
    ds = cl.BackgroundMixDataset(infos, lambda info: dict(imgs=torch.from_numpy(fg[info["sample"]]), label=torch.tensor([0]), randAug=False),
                                 bg_dir=str(tmp_path), with_randAug=True, device_mix=True,
                                 bg_reader=lambda p: pool[path_to_idx[str(pathlib.Path(p).resolve())]])
    assert [path_to_idx[str(pathlib.Path(p).resolve())] for p in ds.bg_files] == list(order)
    torch.manual_seed(int(_NPZ["fullsize/seed_torch"]))
    samples = [ds.prepare_train_frames(i) for i in range(4)]
    out = ds.gpu_collate(samples)["imgs"].cpu().numpy()
    assert [int(s["bg_idx"]) for s in samples] == _NPZ["fullsize/bg_idx"].tolist()
    np.testing.assert_array_equal(out[:, ::3, :, ::37, ::41].view(np.uint32), _NPZ["fullsize/sample_values"].view(np.uint32))
    assert hashlib.sha256(out.tobytes()).digest() == _NPZ["fullsize/sha256"].tobytes()


@pytest.mark.parametrize("W,layout", [(32, "NTCHW"), (30, "NTCHW"), (32, "NCTHW")])
def test_ragged_blend_op_against_the_oracle(env, W, layout):
    """The ragged blend op directly: random pool of mixed sizes, unmixed samples, scalar path (W % 4 != 0), both layouts."""
    ops, cabi, cl, pool_mod = env
    rng = np.random.default_rng(W)
    B, T, H, size = 7, 3, 28, 36
    sizes = [(36, 48), (40, 36), (80, 120), (36, 36), (31, 77)]
    imgs = [rng.integers(0, 256, (3,) + s, dtype=np.uint8) for s in sizes]
    rp = pool_mod.RaggedPool(size, "cuda")
    rp.append(imgs[:2]); rp.append(imgs[2:])                      # growth keeps the first images
    fg = rng.integers(0, 256, (B, T, H, W, 3), dtype=np.uint8)
    idx = rng.integers(0, len(imgs), B)
    app = np.array([1, 1, 0, 1, 1, 0, 1], np.uint8)
    hw = [rp.hw(int(i)) for i in idx]
    top = np.array([rng.integers(0, h - H + 1) for h, w in hw]); left = np.array([rng.integers(0, w - W + 1) for h, w in hw])
    resized = [ao.aa_resize(im, size) for im in imgs]
    exp = np.stack([bo.mix_clip(fg[b], resized[idx[b]], int(top[b]), int(left[b]), (H, W), 0.4, bool(app[b])) for b in range(B)])
    if layout == "NCTHW":
        exp = np.ascontiguousarray(exp.transpose(0, 2, 1, 3, 4))
    dev = torch.device("cuda")
    t32 = lambda a: torch.tensor(np.asarray(a), dtype=torch.int32, device=dev)
    args = (rp.data, rp.slots_tensor, rp.tables.tensor, t32(idx), t32(top), t32(left), torch.from_numpy(app).to(dev))
    mean, std = torch.tensor(bo.DEFAULT_MEAN), torch.tensor(bo.DEFAULT_STD)
    got = torch.ops.bgdebias.bgmix_blend_ragged(torch.from_numpy(fg).to(dev), *args, ops.make_fg_lut(bo.DEFAULT_MEAN, bo.DEFAULT_STD, dev),
                                                mean, std, 0.4, layout).cpu().numpy()
    _assert_same(got, exp)


def test_store_accepts_any_mix_of_sizes_and_dense_equals_ragged(env):
    """BackgroundStore: a second image size no longer raises; for a store of one size the dense fp32 cache (built on the
    device) and the ragged path give the same bits, and both equal torchvision's Resize."""
    from torchvision.transforms import Resize
    ops, cabi, cl, pool_mod = env
    rng = np.random.default_rng(5)
    imgs = {f"a{i}": rng.integers(0, 256, (3, 36, 48), dtype=np.uint8) for i in range(5)}
    store = pool_mod.BackgroundStore(40, "cuda")
    store.ensure(list(imgs), lambda n: imgs[n])
    dense = store.tensor
    assert dense is not None and tuple(dense.shape) == (5, 3, 40, 53) and store.hw == (40, 53)
    for i, n in enumerate(imgs):
        np.testing.assert_array_equal(dense[i].cpu().numpy().view(np.uint32),
                                      Resize(40)(torch.from_numpy(imgs[n]).float()).numpy().view(np.uint32))
    B, T, H, W = 6, 2, 32, 32
    fg = torch.from_numpy(rng.integers(0, 256, (B, T, H, W, 3), dtype=np.uint8)).cuda()
    dev = fg.device
    idx = torch.tensor([0, 4, 2, 2, 1, 3], dtype=torch.int32, device=dev)
    top = torch.tensor([0, 8, 3, 5, 1, 2], dtype=torch.int32, device=dev); left = torch.tensor([21, 0, 7, 9, 4, 11], dtype=torch.int32, device=dev)
    app = torch.ones(B, dtype=torch.uint8, device=dev)
    lut = ops.make_fg_lut(bo.DEFAULT_MEAN, bo.DEFAULT_STD, dev)
    mean, std = torch.tensor(bo.DEFAULT_MEAN), torch.tensor(bo.DEFAULT_STD)
    a = torch.ops.bgdebias.bgmix_blend(fg, dense, idx, top, left, app, lut, mean, std, 0.5, "NTCHW")
    r = store.ragged
    b = torch.ops.bgdebias.bgmix_blend_ragged(fg, r.data, r.slots_tensor, r.tables.tensor, idx, top, left, app, lut, mean, std, 0.5, "NTCHW")
    assert torch.equal(a, b)
    store.ensure(["other"], lambda n: rng.integers(0, 256, (3, 36, 64), dtype=np.uint8))     # a second size: accepted
    assert store.tensor is None and len(store) == 6 and store.hw_of(5) == (40, 71)
    with pytest.raises(ValueError):
        store.hw
    v = store.view(["other", "a0"])
    assert v.tensor is None and v.hw_of(0) == (40, 71) and v.hw_of(1) == (40, 53)


def test_sthv2_sized_uint8_pool_arithmetic_and_blend(env):
    """A Sth-Sth-v2-shaped pool (240 x 427 backgrounds, BASELINE configs[3]): 220,847 backgrounds are 67.9 GB as uint8 --
    resident on one 180 GB B200 -- against 308 GB as resized fp32.  Blend a batch from a 2,048-image slice of it."""
    ops, cabi, cl, pool_mod = env
    n_total, h, w = 220_847, 240, 427
    Hb, Wb = pool_mod.resized_hw(h, w, 256)
    assert (Hb, Wb) == (256, 455)
    assert n_total * 3 * h * w < 70e9 < 180e9 < n_total * 3 * Hb * Wb * 4
    n = 2048
    dev = torch.device("cuda")
    rp = pool_mod.RaggedPool(256, dev)
    g = torch.Generator().manual_seed(3)
    chunk = [torch.randint(0, 256, (3, h, w), dtype=torch.uint8, generator=g) for _ in range(64)]
    for _ in range(n // 64):
        rp.append(chunk)
    assert len(rp) == n and rp.used >= n * 3 * h * w
    rng = np.random.default_rng(1)
    B, T = 16, 8
    fg = rng.integers(0, 256, (B, T, 224, 224, 3), dtype=np.uint8)
    idx = rng.integers(0, n, B); top = rng.integers(0, Hb - 223, B); left = rng.integers(0, Wb - 223, B)
    t32 = lambda a: torch.tensor(np.asarray(a), dtype=torch.int32, device=dev)
    got = torch.ops.bgdebias.bgmix_blend_ragged(torch.from_numpy(fg).to(dev), rp.data, rp.slots_tensor, rp.tables.tensor, t32(idx), t32(top),
                                                t32(left), torch.ones(B, dtype=torch.uint8, device=dev),
                                                ops.make_fg_lut(bo.DEFAULT_MEAN, bo.DEFAULT_STD, dev), torch.tensor(bo.DEFAULT_MEAN),
                                                torch.tensor(bo.DEFAULT_STD), 0.5, "NTCHW").cpu().numpy()
    resized = {int(i) % 64: None for i in idx}
    for k in resized:
        resized[k] = ao.aa_resize(chunk[k].numpy(), 256)
    exp = np.stack([bo.mix_clip(fg[b], resized[int(idx[b]) % 64], int(top[b]), int(left[b]), (224, 224), 0.5, True) for b in range(B)])
    _assert_same(got, exp)


class _U8Clips:
    """Picklable stand-in for the mmaction pipeline up to (not including) Normalize."""
    def __init__(self, fg, ra):
        self.fg, self.ra = fg, ra

    def __call__(self, info):
        return dict(imgs=torch.from_numpy(self.fg[info["sample"]]), label=torch.tensor([info["label"]]), randAug=bool(self.ra[info["sample"]]))


def test_real_jpeg_pool_of_two_sizes_behind_dataloader_workers(env, tmp_path):
    """The whole M1-M3 chain on real files with the default reader: JPEGs of two sizes on disk (what the extraction CLI
    writes for a dataset of mixed widths), DataLoader worker processes draw bg_idx and the crop from each image's own
    resized size (header probe, no CUDA in the workers), the training process decodes every file once (read_image) and
    blends per batch.  Expected = the oracle on torchvision's decode of the same files."""
    import cv2
    from torchvision.io import ImageReadMode, read_image
    ops, cabi, cl, pool_mod = env
    rng = np.random.default_rng(23)
    T, H, W, n = 2, 32, 32, 12
    names = [f"v{i:02d}" for i in range(6)]
    for i, nm in enumerate(names):
        h, w = (36, 48) if i % 2 == 0 else (40, 72)
        base = cv2.resize(rng.integers(0, 256, (6, 8, 3), dtype=np.uint8), (w, h), interpolation=cv2.INTER_CUBIC)   # smooth: survives JPEG
        cv2.imwrite(str(tmp_path / f"{nm}.jpg"), base)
    fg = rng.integers(0, 256, (n, T, H, W, 3), dtype=np.uint8)
    ra = rng.integers(0, 2, n).astype(bool)
    infos = [dict(frame_dir=f"/x/{names[i % 6]}", total_frames=T, label=i, sample=i) for i in range(n)]
    ds = cl.BackgroundMixDataset(infos, _U8Clips(fg, ra), bg_dir=str(tmp_path), bg_resize=40, bg_crop_size=(H, W), with_randAug=True,
                                 device_mix=True)
    assert len(ds.bg_files) == n
    loader = torch.utils.data.DataLoader(ds, batch_size=4, shuffle=False, num_workers=2, collate_fn=ds.host_collate, pin_memory=True)
    decoded = {p: read_image(p, mode=ImageReadMode.RGB).numpy() for p in set(ds.bg_files)}
    seen = 0
    for batch in loader:
        out = ds.device_finish(batch)["imgs"].cpu().numpy()
        B = batch["imgs"].shape[0]
        for b in range(B):
            i = int(batch["bg_idx"][b])
            assert (i == -1) == bool(ra[seen + b])
            if i < 0:
                exp = bo.fg_normalize(fg[seen + b], bo.fg_lut())
            else:
                img = decoded[ds.bg_files[i]]
                Hb, Wb = ao.resized_hw(img.shape[1], img.shape[2], 40)
                assert 0 <= int(batch["bg_top"][b]) <= Hb - H and 0 <= int(batch["bg_left"][b]) <= Wb - W
                exp = bo.mix_clip(fg[seen + b], ao.aa_resize(img, 40), int(batch["bg_top"][b]), int(batch["bg_left"][b]), (H, W), 0.5, True)
            _assert_same(out[b], exp)
        seen += B
    assert seen == n and ds.device_pool().tensor is None and len(ds._store) == 6


def test_pool_without_resize_and_uniform_dense_choice(env):
    """bg_resize=None (a pool already at crop scale): no table, no pass -- the ragged blend reads the bytes as they are; a
    uniform store within budget serves the dense path, the same store with no budget the ragged path, same bits."""
    ops, cabi, cl, pool_mod = env
    rng = np.random.default_rng(4)
    imgs = [rng.integers(0, 256, (3, 40, 56), dtype=np.uint8) for _ in range(4)]
    B, T, H, W = 5, 2, 32, 32
    fg = rng.integers(0, 256, (B, T, H, W, 3), dtype=np.uint8)
    idx, top, left = [3, 0, 1, 2, 3], [0, 8, 3, 5, 1], [24, 0, 7, 9, 4]
    exp = np.stack([bo.mix_clip(fg[b], imgs[idx[b]].astype(np.float32), top[b], left[b], (H, W), 0.5, True) for b in range(B)])
    dev = torch.device("cuda")
    t32 = lambda a: torch.tensor(a, dtype=torch.int32, device=dev)
    lut, mean, std = ops.make_fg_lut(bo.DEFAULT_MEAN, bo.DEFAULT_STD, dev), torch.tensor(bo.DEFAULT_MEAN), torch.tensor(bo.DEFAULT_STD)
    for budget in (None, 0):
        store = pool_mod.BackgroundStore(None, dev, dense_budget_bytes=budget)
        store.ensure([f"i{k}" for k in range(4)], lambda n: imgs[int(n[1:])])
        dense = store.tensor
        assert (dense is None) == (budget == 0)
        app = torch.ones(B, dtype=torch.uint8, device=dev)
        if dense is not None:
            got = torch.ops.bgdebias.bgmix_blend(torch.from_numpy(fg).to(dev), dense, t32(idx), t32(top), t32(left), app, lut, mean, std, 0.5, "NTCHW")
        else:
            r = store.ragged
            assert int(r.slots["xtab"][0]) == -1 and int(r.slots["ytab"][0]) == -1
            got = torch.ops.bgdebias.bgmix_blend_ragged(torch.from_numpy(fg).to(dev), r.data, r.slots_tensor, r.tables.tensor, t32(idx), t32(top),
                                                        t32(left), app, lut, mean, std, 0.5, "NTCHW")
        _assert_same(got.cpu().numpy(), exp)
