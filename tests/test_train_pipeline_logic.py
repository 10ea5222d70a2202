"""Host side of the training route (no GPU): the mmaction2 0.x Resize / MultiScaleCrop rules of comix_loader.TrainPipeline
against a line-by-line restatement of MultiScaleCrop.__call__, the validation of ``device_train_pipeline``, the training
form of ``host_collate``, and the order of the Python / torch draws against a worker that runs the CPU steps."""
import random

import numpy as np
import pytest
import torch

from bgdebias_b200 import comix_loader as cl

MEAN, STD = [123.675, 116.28, 103.53], [58.395, 57.12, 57.375]
SCALES = (1, 0.875, 0.75, 0.66)
SIZES = [(240, 320), (240, 427), (256, 340), (320, 240), (233, 301)]


def _steps(scales=SCALES, random_crop=False, num_fixed_crops=13, gap=1, out=(224, 224), **msc):
    return [dict(type="Resize", scale=(-1, 256)),
            dict(type="MultiScaleCrop", input_size=224, scales=scales, random_crop=random_crop, max_wh_scale_gap=gap,
                 num_fixed_crops=num_fixed_crops, **msc),
            dict(type="Resize", scale=out, keep_ratio=False),
            dict(type="Normalize", mean=MEAN, std=STD, to_bgr=False), dict(type="FormatShape", input_format="NCHW")]


def _mm_multiscale_crop(img_h, img_w, input_size, scales, max_wh_scale_gap, random_crop, num_fixed_crops):
    """mmaction2 0.x MultiScaleCrop.__call__ (the crop box), written out as mmaction writes it."""
    input_size = (input_size, input_size) if isinstance(input_size, int) else input_size
    base_size = min(img_h, img_w)
    crop_sizes = [int(base_size * s) for s in scales]
    candidate_sizes = []
    for i, h in enumerate(crop_sizes):
        for j, w in enumerate(crop_sizes):
            if abs(i - j) <= max_wh_scale_gap:
                candidate_sizes.append([w, h])
    crop_size = random.choice(candidate_sizes)
    for i in range(2):
        if abs(crop_size[i] - input_size[i]) < 3:
            crop_size[i] = input_size[i]
    crop_w, crop_h = crop_size
    if random_crop:
        x_offset = random.randint(0, img_w - crop_w)
        y_offset = random.randint(0, img_h - crop_h)
    else:
        w_step = (img_w - crop_w) // 4
        h_step = (img_h - crop_h) // 4
        candidate_offsets = [(0, 0), (4 * w_step, 0), (0, 4 * h_step), (4 * w_step, 4 * h_step), (2 * w_step, 2 * h_step)]
        if num_fixed_crops == 13:
            candidate_offsets.extend([(0, 2 * h_step), (4 * w_step, 2 * h_step), (2 * w_step, 4 * h_step),
                                      (2 * w_step, 0 * h_step), (1 * w_step, 1 * h_step), (3 * w_step, 1 * h_step),
                                      (1 * w_step, 3 * h_step), (3 * w_step, 3 * h_step)])
        x_offset, y_offset = random.choice(candidate_offsets)
    return y_offset, x_offset, crop_h, crop_w


@pytest.mark.parametrize("hw", SIZES)
@pytest.mark.parametrize("kw", [dict(num_fixed_crops=5), dict(num_fixed_crops=13), dict(random_crop=True),
                                dict(gap=0), dict(gap=3, scales=(1, 0.8))])
def test_draws_follow_multiscale_crop(hw, kw):
    tp = cl.TrainPipeline(_steps(**kw))
    Hr, Wr = cl.rescale_short_side(*hw, 256)
    seen = set()
    for seed in range(300):
        random.seed(seed)
        got = tp.draw(*hw)
        random.seed(seed)
        exp = _mm_multiscale_crop(Hr, Wr, 224, tp.scales, tp.max_wh_scale_gap, tp.random_crop, tp.num_fixed_crops)
        assert got == (Hr, Wr) + exp
        seen.add(got[4:])
    base = min(Hr, Wr)
    sizes = [int(base * s) for s in tp.scales]
    snap = lambda v: 224 if abs(v - 224) < 3 else v                          # noqa: E731
    pairs = {(snap(h), snap(w)) for i, h in enumerate(sizes) for j, w in enumerate(sizes) if abs(i - j) <= tp.max_wh_scale_gap}
    assert seen == pairs                                                     # every scale pair is drawn, nothing else


def test_draw_consumes_what_mmaction_consumes():
    tp = cl.TrainPipeline(_steps())
    random.seed(3)
    tp.draw(240, 320)
    after = random.random()
    random.seed(3)
    _mm_multiscale_crop(256, 341, 224, SCALES, 1, False, 13)
    assert random.random() == after


def test_known_boxes():
    """240x320 -> 256x341; crop sizes 256, 224, 192, 168 (0.66 * 256 = 168.96); fixed offsets on the 4-step grid."""
    tp = cl.TrainPipeline(_steps(num_fixed_crops=5))
    assert cl.rescale_short_side(240, 320, 256) == (256, 341)
    boxes = set()
    for seed in range(400):
        random.seed(seed)
        boxes.add(tp.draw(240, 320))
    assert (256, 341, 0, 0, 256, 256) in boxes
    assert (256, 341, 0, 116, 224, 224) in boxes                              # x = 4 * ((341 - 224) // 4)
    assert (256, 341, 16, 58, 224, 224) in boxes                              # centre: 2 * 8, 2 * 29
    assert all(h in (256, 224, 192, 168) and w in (256, 224, 192, 168) for _, _, _, _, h, w in boxes)
    for Hr, Wr, y0, x0, ch, cw in boxes:
        assert 0 <= y0 <= Hr - ch and 0 <= x0 <= Wr - cw


@pytest.mark.parametrize("steps, match", [
    (_steps()[:4], "FormatShape step is missing"),
    (_steps()[:1] + _steps()[2:], "step 1, 'Resize'"),
    ([dict(type="RandAugment", n=2, m=10)] + _steps(), "step 0, 'RandAugment'"),
    (_steps() + [dict(type="Collect", keys=["imgs"])], "step 5, 'Collect'"),
    ([dict(type="Resize", scale=(-1, 256), lazy=True)] + _steps()[1:], "Resize: lazy=True"),
    ([dict(type="Resize", scale=(340, 256), keep_ratio=False)] + _steps()[1:], "Resize: keep_ratio=False"),
    (_steps(lazy=True), "MultiScaleCrop: lazy=True"),
    (_steps(num_fixed_crops=7), "MultiScaleCrop: num_fixed_crops"),
    (_steps(scales=()), "MultiScaleCrop: scales"),
    (_steps(gap=-1), "MultiScaleCrop: max_wh_scale_gap"),
    (_steps(random_crop=1), "MultiScaleCrop: random_crop"),
    (_steps()[:2] + [dict(type="Resize", scale=(224, 224))] + _steps()[3:], "Resize: keep_ratio"),
    (_steps()[:2] + [dict(type="Resize", scale=(224, 224), keep_ratio=False, interpolation="bicubic")] + _steps()[3:],
     "Resize: interpolation='bicubic'"),
    (_steps()[:3] + [dict(type="Normalize", mean=MEAN, std=STD, to_bgr=True)] + _steps()[4:], "Normalize: to_bgr=True"),
    (_steps()[:4] + [dict(type="FormatShape", input_format="NCTHW")], "FormatShape: only input_format='NCHW'"),
    (_steps()[:2] + [dict(type="Flip", flip_ratio=0.5)] + _steps()[2:], "step 2, 'Flip'"),
])
def test_validation_names_the_step(steps, match):
    with pytest.raises(ValueError, match=match):
        cl.TrainPipeline(steps)


class _Frames:
    """Picklable stand-in for a training pipeline that stops after RawFrameDecode: a list of uint8 [h, w, 3] frames."""
    def __init__(self, clips):
        self.clips = clips

    def __call__(self, info):
        return dict(imgs=list(self.clips[info["sample"]]), label=torch.tensor([info["label"]]))


class _CpuSteps:
    """The same pipeline with the CPU Resize(scale=(-1, 256)) and MultiScaleCrop after it; records each crop box."""
    def __init__(self, clips, steps):
        self.frames, self.tp = _Frames(clips), cl.TrainPipeline(steps)
        self.boxes = []

    def __call__(self, info):
        import cv2
        out = self.frames(info)
        h, w = out["imgs"][0].shape[:2]
        Hr, Wr = cl.rescale_short_side(h, w, 256)
        tp = self.tp
        y0, x0, ch, cw = _mm_multiscale_crop(Hr, Wr, 224, tp.scales, tp.max_wh_scale_gap, tp.random_crop, tp.num_fixed_crops)
        out["imgs"] = [cv2.resize(f, (Wr, Hr), interpolation=cv2.INTER_LINEAR)[y0:y0 + ch, x0:x0 + cw] for f in out["imgs"]]
        self.boxes.append((Hr, Wr, y0, x0, ch, cw))
        return out


class _BgReader:
    def __init__(self, sizes):
        self.sizes = sizes

    def __call__(self, path):
        h, w = self.sizes[int(path.rsplit("bg", 1)[1].split(".")[0]) % len(self.sizes)]
        return torch.zeros((3, h, w), dtype=torch.uint8)


def _dataset(tmp_path, clips, pipeline=None, **kw):
    for i in range(len(clips)):
        (tmp_path / f"bg{i}.jpg").write_bytes(b"stub")
    infos = [dict(frame_dir=f"/x/bg{i}", total_frames=len(c), label=i, sample=i) for i, c in enumerate(clips)]
    return cl.BackgroundMixDataset(infos, pipeline or _Frames(clips), bg_dir=str(tmp_path),
                                   bg_reader=_BgReader([(240, 320), (256, 455), (300, 260)]), device="cpu", **kw)


def _clips(T=2):
    rng = np.random.default_rng(0)
    return [rng.integers(0, 256, (T, h, w, 3), dtype=np.uint8) for h, w in SIZES * 2]


def test_dataset_refusals(tmp_path):
    clips = _clips()
    with pytest.raises(ValueError, match="with_randAug"):
        _dataset(tmp_path, clips, device_mix=True, with_randAug=True, device_train_pipeline=_steps())
    with pytest.raises(ValueError, match="test_mode=False"):
        _dataset(tmp_path, clips, device_mix=True, test_mode=True, device_train_pipeline=_steps())
    with pytest.raises(ValueError, match="device_mix=True"):
        _dataset(tmp_path, clips, device_train_pipeline=_steps())
    eval_steps = [dict(type="Resize", scale=(-1, 256)), dict(type="CenterCrop", crop_size=224),
                  dict(type="Normalize", mean=MEAN, std=STD, to_bgr=False), dict(type="FormatShape", input_format="NCHW")]
    with pytest.raises(ValueError, match="exclusive"):
        _dataset(tmp_path, clips, device_mix=True, device_train_pipeline=_steps(), device_test_pipeline=eval_steps)
    with pytest.raises(ValueError, match="bg_crop_size"):
        _dataset(tmp_path, clips, device_mix=True, device_train_pipeline=_steps(out=(224, 200)))
    with pytest.raises(ValueError, match="bg_crop_size"):                   # mmaction's (w, h) against (h, w)
        _dataset(tmp_path, clips, device_mix=True, bg_crop_size=(224, 200), device_train_pipeline=_steps(out=(224, 200)))
    _dataset(tmp_path, clips, device_mix=True, bg_crop_size=(200, 224), device_train_pipeline=_steps(out=(224, 200)))


def test_host_collate_two_stage_geometry(tmp_path):
    from bgdebias_b200 import ops
    clips = _clips(T=3)
    ds = _dataset(tmp_path, clips, device_mix=True, prob=0.5, device_train_pipeline=_steps())
    random.seed(1)
    torch.manual_seed(1)
    samples = [ds[i] for i in range(len(clips))]
    batch = ds.host_collate(samples)
    buf, g5 = ops.pack_clips(clips)
    assert torch.equal(batch["imgs"], buf) and batch["fg_frames"] == 3
    assert batch["fg_geom"].dtype == torch.int64 and tuple(batch["fg_geom"].shape) == (len(clips), len(ops.TWO_STAGE_COLS))
    assert torch.equal(batch["fg_geom"][:, :5], g5)
    assert batch["fg_geom"][:, 5:].tolist() == [list(s["fg_window"]) for s in samples]
    for s, clip in zip(samples, clips):
        Hr, Wr, y0, x0, ch, cw = s["fg_window"]
        assert (Hr, Wr) == cl.rescale_short_side(clip.shape[1], clip.shape[2], 256)
        assert 0 <= y0 <= Hr - ch and 0 <= x0 <= Wr - cw
    assert set(batch) >= {"imgs", "fg_geom", "fg_frames", "bg_idx", "bg_top", "bg_left", "bg_apply", "label"}


@pytest.mark.parametrize("kw", [dict(), dict(random_crop=True), dict(num_fixed_crops=5)])
@pytest.mark.parametrize("bg_dir_mode", [True, False])
def test_rng_order_matches_the_cpu_steps(tmp_path, kw, bg_dir_mode):
    """Seeded alike, the device route and a worker that runs Resize + MultiScaleCrop on the host draw the same crop boxes
    and the same bg_idx / bg_top / bg_left / bg_apply, sample after sample (also in random-frame mode)."""
    pytest.importorskip("cv2")
    clips = _clips()
    steps = _steps(**kw)
    common = dict(device_mix=True, prob=0.5, back_ground_from_bg_dir=bg_dir_mode, filename_tmpl="bg{}.jpg", start_index=0)
    dev = _dataset(tmp_path, clips, device_train_pipeline=steps, **common)
    cpu_steps = _CpuSteps(clips, steps)
    ref = _dataset(tmp_path, clips, pipeline=cpu_steps, **common)
    out = {}
    for name, ds in (("dev", dev), ("ref", ref)):
        random.seed(11)
        torch.manual_seed(11)
        out[name] = [ds[i % len(clips)] for i in range(3 * len(clips))]
    assert [s["fg_window"] for s in out["dev"]] == cpu_steps.boxes
    for key in ("bg_idx", "bg_top", "bg_left", "bg_apply"):
        assert [s[key] for s in out["dev"]] == [s[key] for s in out["ref"]], key
    assert 0 < sum(s["bg_apply"] for s in out["dev"]) < len(out["dev"])
