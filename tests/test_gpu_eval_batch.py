"""The evaluation route on the GPU: torch.ops.bgdebias.resize_crop_normalize against a numpy restatement of the mmaction2
0.x test pipeline tail (cv2.resize of the whole frame to the rescaled size, the crop slice, the Normalize table, the
NCHW transpose), bit for bit, and the dataset's host_collate -> device_finish route behind a DataLoader against the same
pipeline run per sample on the CPU."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")

from oracle import bgmix_oracle as bo                     # noqa: E402

MEAN, STD = bo.DEFAULT_MEAN, bo.DEFAULT_STD
SIZES = [(240, 320), (240, 427), (241, 321), (239, 319), (480, 640), (320, 240), (256, 341)]


@pytest.fixture(scope="module")
def env():
    import bgdebias_b200.ops as ops
    from bgdebias_b200 import _cabi, comix_loader
    assert torch.cuda.is_available()
    _cabi.lib()
    return ops, _cabi, comix_loader


def _steps(crop, size):
    return [dict(type="Resize", scale=(-1, 256)), dict(type=crop, crop_size=size),
            dict(type="Normalize", mean=MEAN, std=STD, to_bgr=False), dict(type="FormatShape", input_format="NCHW")]


def _oracle(clip, ev, lut):
    """uint8 [T, h, w, 3] -> fp32 [K*T, 3, ch, cw]: cv2.resize to (Hr, Wr), the crop windows crop-major, table, transpose."""
    Hr, Wr, wins = ev.windows(clip.shape[1], clip.shape[2])
    ch, cw = ev.crop_hw
    resized = [cv2.resize(f, (Wr, Hr), interpolation=cv2.INTER_LINEAR) for f in clip]
    crops = np.stack([r[top:top + ch, left:left + cw] for top, left in wins for r in resized])
    return bo.fg_normalize(crops, lut)


def _mmcv_normalize(imgs_u8):
    """mmcv.imnormalize_ as mmaction's Normalize calls it, on a list of uint8 HWC images -> fp32 [N, 3, H, W]."""
    out = []
    for img in imgs_u8:
        x = img.astype(np.float32)
        cv2.subtract(x, np.float64(np.asarray(MEAN, np.float64).reshape(1, -1)), x)
        cv2.multiply(x, 1 / np.float64(np.asarray(STD, np.float64).reshape(1, -1)), x)
        out.append(x.transpose(2, 0, 1))
    return np.stack(out)


@pytest.mark.parametrize("crop, size", [("CenterCrop", 224), ("ThreeCrop", 256)])
@pytest.mark.parametrize("T", [1, 8, 16])
def test_bit_exact_against_cv2(env, crop, size, T):
    ops, cabi, cl = env
    ev = cl.EvalPipeline(_steps(crop, size))
    rng = np.random.default_rng(T)
    clips = [rng.integers(0, 256, (T, h, w, 3), dtype=np.uint8) for h, w in SIZES]
    buf, g5 = ops.pack_clips(clips)
    geom = ev.geometry(g5)
    dev = torch.device("cuda")
    lut = ops.make_fg_lut(MEAN, STD, dev)
    src = buf.to(dev)
    K, (ch, cw) = ev.n_crops, ev.crop_hw
    n0 = cabi.kernel_launch_count()
    got = torch.ops.bgdebias.resize_crop_normalize(src, geom, T, ch, cw, lut, "NTCHW")
    assert cabi.kernel_launch_count() - n0 == 1
    assert got.dtype == torch.float32 and tuple(got.shape) == (len(clips) * K, T, 3, ch, cw)
    got = got.view(len(clips), K * T, 3, ch, cw).cpu().numpy()
    h_lut = bo.fg_lut(MEAN, STD)
    for b, clip in enumerate(clips):
        np.testing.assert_array_equal(got[b].view(np.uint32), _oracle(clip, ev, h_lut).view(np.uint32), err_msg=str(clip.shape))

    f32 = torch.from_numpy(got).view(len(clips) * K, T, 3, ch, cw)
    for dt in (torch.bfloat16, torch.float16):
        low = torch.ops.bgdebias.resize_crop_normalize(src, geom, T, ch, cw, lut, "NTCHW", dt).cpu()
        assert low.dtype == dt and torch.equal(low.view(torch.int16), f32.to(dt).view(torch.int16))
    for dt in (torch.float32, torch.bfloat16):
        il = torch.ops.bgdebias.resize_crop_normalize(src, geom, T, ch, cw, lut, "NTHWC", dt).cpu()
        assert tuple(il.shape) == (len(clips) * K, T, ch, cw, 3)
        assert torch.equal(il.permute(0, 1, 4, 2, 3), f32.to(dt))


def test_windows_anywhere_in_the_resized_image(env):
    """Arbitrary windows (not only the crop rules' offsets), up- and down-scaling, 1-pixel windows at the far corner."""
    ops, _, _ = env
    rng = np.random.default_rng(7)
    dev = torch.device("cuda")
    clips = [rng.integers(0, 256, (3, h, w, 3), dtype=np.uint8) for h, w in ((17, 29), (64, 33), (5, 7))]
    buf, g5 = ops.pack_clips(clips)
    H, W = 6, 9
    rows, exp = [], []
    h_lut = bo.fg_lut(MEAN, STD)
    for b, clip in enumerate(clips):
        for Hr, Wr in ((H, W), (40, 23), (11, 100)):
            for top, left in ((0, 0), (Hr - H, Wr - W), (int(rng.integers(0, Hr - H + 1)), int(rng.integers(0, Wr - W + 1)))):
                rows.append(g5[b].tolist() + [Hr, Wr, top, left])
                r = np.stack([cv2.resize(f, (Wr, Hr), interpolation=cv2.INTER_LINEAR)[top:top + H, left:left + W] for f in clip])
                exp.append(bo.fg_normalize(r, h_lut))
    got = torch.ops.bgdebias.resize_crop_normalize(buf.to(dev), torch.tensor(rows), 3, H, W, ops.make_fg_lut(MEAN, STD, dev),
                                                   "NTCHW").cpu().numpy()
    np.testing.assert_array_equal(got.view(np.uint32), np.stack(exp).view(np.uint32))


def test_opcheck(env):
    ops, _, cl = env
    rng = np.random.default_rng(1)
    buf, g5 = ops.pack_clips([rng.integers(0, 256, (2, h, w, 3), dtype=np.uint8) for h, w in ((12, 15), (15, 12))])
    dev = torch.device("cuda")
    ev = cl.EvalPipeline([dict(type="Resize", scale=(-1, 16))] + _steps("ThreeCrop", 16)[1:])
    geom = ev.geometry(g5)
    lut = ops.make_fg_lut(MEAN, STD, dev)
    for layout, dt in (("NTCHW", None), ("NTHWC", torch.bfloat16)):
        torch.library.opcheck(torch.ops.bgdebias.resize_crop_normalize.default, (buf.to(dev), geom, 2, 16, 16, lut, layout, dt))


def test_rejected_geometry(env):
    ops, cabi, _ = env
    dev = torch.device("cuda")
    buf, g5 = ops.pack_clips([np.zeros((2, 20, 30, 3), np.uint8)])
    src, lut = buf.to(dev), ops.make_fg_lut(MEAN, STD, dev)
    base = g5[0].tolist()
    call = lambda rows, s=src, layout="NTCHW": torch.ops.bgdebias.resize_crop_normalize(  # noqa: E731
        s, torch.tensor(rows, dtype=torch.int64), 2, 8, 8, lut, layout)
    call([base + [16, 24, 8, 16]])                                          # the last window that fits
    n0 = cabi.kernel_launch_count()
    bad = {
        "window below": [base + [16, 24, 9, 0]],
        "window right": [base + [16, 24, 0, 17]],
        "negative top": [base + [16, 24, -1, 0]],
        "zero Hr": [base + [0, 24, 0, 0]],
        "zero Wr": [base + [16, 0, 0, 0]],
        "zero source height": [[base[0], 0] + base[2:] + [16, 24, 0, 0]],
        "second entry bad": [base + [16, 24, 0, 0], base + [8, 8, 0, 1]],
    }
    for name, rows in bad.items():
        with pytest.raises(ValueError, match="libbgdebias_b200: resize"):
            call(rows)
    with pytest.raises(ValueError, match="ends at byte"):
        call([base + [16, 24, 0, 0]], s=src[:src.numel() - 8])           # short buffer
    with pytest.raises(ValueError, match="layout"):
        call([base + [16, 24, 0, 0]], layout="NCTHW")
    with pytest.raises(ValueError, match=r"geom must be int64 \[B, 9\]"):
        torch.ops.bgdebias.resize_crop_normalize(src, g5, 2, 8, 8, lut, "NTCHW")
    torch.cuda.synchronize()
    assert cabi.kernel_launch_count() == n0


class _Frames:
    """Picklable test pipeline stopped after RawFrameDecode: a list of uint8 [h, w, 3] RGB frames per video."""
    def __init__(self, clips):
        self.clips = clips

    def __call__(self, info):
        return dict(imgs=list(self.clips[info["sample"]]), label=torch.tensor([info["label"]]))


class _NoReader:
    def __call__(self, path):
        raise AssertionError(f"the evaluation route read a background: {path}")


@pytest.mark.parametrize("crop, size", [("CenterCrop", 224), ("ThreeCrop", 256)])
def test_dataloader_workers_then_device_finish(env, tmp_path, crop, size):
    """A test-mode dataset behind a DataLoader with 2 worker processes: the workers ship native uint8 frames, device_finish
    runs the tail in one launch; bit-equal to Resize -> crop -> Normalize -> FormatShape per sample on the CPU."""
    ops, cabi, cl = env
    rng = np.random.default_rng(3)
    T, sizes = 8, SIZES + [(240, 320), (320, 240), (240, 427)]
    clips = [rng.integers(0, 256, (T, h, w, 3), dtype=np.uint8) for h, w in sizes]
    names = [f"v{i:02d}" for i in range(len(clips))]
    for nm in names:
        (tmp_path / (nm + ".jpg")).write_bytes(b"stub")
    infos = [dict(frame_dir=f"/x/{nm}", total_frames=T, label=i, sample=i) for i, nm in enumerate(names)]
    steps = _steps(crop, size)
    ds = cl.BackgroundMixDataset(infos, _Frames(clips), bg_dir=str(tmp_path), test_mode=True, prob=1.0, device_mix=True,
                                 device_test_pipeline=steps, bg_reader=_NoReader())
    ev = ds._eval
    K, (ch, cw) = ev.n_crops, ev.crop_hw
    loader = torch.utils.data.DataLoader(ds, batch_size=4, shuffle=False, num_workers=2, collate_fn=ds.host_collate,
                                         pin_memory=True)
    seen = 0
    for batch in loader:
        assert batch["imgs"].dtype == torch.uint8 and not batch["imgs"].is_cuda
        B = batch["fg_geom"].shape[0]
        n0 = cabi.kernel_launch_count()
        out = ds.device_finish(batch)
        assert cabi.kernel_launch_count() - n0 == 1
        assert set(out) == {"imgs", "label"} and out["imgs"].is_cuda
        assert tuple(out["imgs"].shape) == (B, K * T, 3, ch, cw) and out["imgs"].dtype == torch.float32
        got = out["imgs"].cpu().numpy()
        for b in range(B):
            clip = clips[seen + b]
            Hr, Wr, wins = ev.windows(clip.shape[1], clip.shape[2])
            resized = [cv2.resize(f, (Wr, Hr), interpolation=cv2.INTER_LINEAR) for f in clip]
            cropped = []
            for top, left in wins:                                   # mmaction's crop-major cropped.extend(crop)
                cropped.extend([r[top:top + ch, left:left + cw] for r in resized])
            np.testing.assert_array_equal(got[b].view(np.uint32), _mmcv_normalize(cropped).view(np.uint32))
        assert out["label"].tolist() == [[seen + b] for b in range(B)]
        cl_bf16 = ds.device_finish(batch, dtype=torch.bfloat16, memory_format=torch.channels_last)["imgs"]
        assert cl_bf16.dtype == torch.bfloat16 and tuple(cl_bf16.shape) == (B, K * T, 3, ch, cw)
        assert cl_bf16.flatten(0, 1).is_contiguous(memory_format=torch.channels_last)
        assert torch.equal(cl_bf16.cpu(), torch.from_numpy(got).to(torch.bfloat16))
        seen += B
    assert seen == len(clips)
    assert ds._store is None and ds._pool is None                       # the background pool was never built
