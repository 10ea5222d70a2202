"""Host side of the evaluation route (no GPU): test-mode items run the pipeline alone, the mmaction2 0.x Resize /
CenterCrop / ThreeCrop rules of comix_loader.EvalPipeline, the validation of ``device_test_pipeline`` and the evaluation
form of ``host_collate``."""
import random

import numpy as np
import pytest
import torch

from bgdebias_b200 import comix_loader as cl

MEAN, STD = [123.675, 116.28, 103.53], [58.395, 57.12, 57.375]


def _steps(crop="CenterCrop", size=224, scale=(-1, 256)):
    return [dict(type="Resize", scale=scale), dict(type=crop, crop_size=size),
            dict(type="Normalize", mean=MEAN, std=STD, to_bgr=False), dict(type="FormatShape", input_format="NCHW")]


class _Frames:
    """Picklable stand-in for a test pipeline that stops after RawFrameDecode: a list of uint8 [h, w, 3] frames."""
    def __init__(self, clips, randaug=None):
        self.clips, self.randaug = clips, randaug

    def __call__(self, info):
        out = dict(imgs=list(self.clips[info["sample"]]), label=torch.tensor([info["label"]]))
        if self.randaug is not None:
            out["randAug"] = self.randaug
        return out


def _raise(path):
    raise AssertionError(f"the evaluation route read a background: {path}")


def _dataset(tmp_path, clips, **kw):
    names = [f"v{i}" for i in range(len(clips))]
    for nm in names:
        (tmp_path / (nm + ".jpg")).write_bytes(b"stub")
    infos = [dict(frame_dir=f"/x/{nm}", total_frames=len(clips[i]), label=i, sample=i) for i, nm in enumerate(names)]
    return cl.BackgroundMixDataset(infos, _Frames(clips, kw.pop("randaug", None)), bg_dir=str(tmp_path), bg_reader=_raise,
                                   device="cpu", **kw)


@pytest.mark.parametrize("kw", [dict(prob=1.0), dict(prob=1.0, with_randAug=True, randaug=False),
                                dict(prob=1.0, with_randAug=True),
                                dict(prob=1.0, device_mix=True, device_test_pipeline=_steps()),
                                dict(with_randAug=True, device_mix=True, device_test_pipeline=_steps())])
def test_test_mode_item_is_the_pipeline_alone(tmp_path, kw):
    """A test-mode item never mixes: no bg_* keys, no draw from Python's or torch's generator, no background read."""
    clips = [np.zeros((2, 6, 8, 3), np.uint8) + i for i in range(3)]
    ds = _dataset(tmp_path, clips, test_mode=True, **kw)
    random.seed(5)
    torch.manual_seed(5)
    py_state, torch_state = random.getstate(), torch.get_rng_state()
    for i in range(len(ds)):
        item = ds[i]
        assert not [k for k in item if k.startswith("bg_")]
        assert np.array_equal(np.stack(item["imgs"]), clips[i])
    assert random.getstate() == py_state
    assert torch.equal(torch.get_rng_state(), torch_state)


@pytest.mark.parametrize("hw, resized", [((240, 320), (256, 341)), ((240, 427), (256, 455)), ((320, 240), (341, 256)),
                                         ((256, 340), (256, 340)), ((256, 256), (256, 256)), ((480, 640), (256, 341)),
                                         ((241, 321), (256, 341)), ((239, 319), (256, 342)), ((101, 153), (256, 388)),
                                         ((720, 405), (455, 256))])
def test_rescale_short_side(hw, resized):
    """mmcv.rescale_size((w, h), (inf, 256)): f = 256 / min(h, w), new = int(x * f + 0.5)."""
    for scale in ((-1, 256), (256, -1)):
        ev = cl.EvalPipeline(_steps(scale=scale))
        Hr, Wr, _ = ev.windows(*hw)
        assert (Hr, Wr) == resized
        f = 256 / min(hw)
        assert (Wr, Hr) == (int(hw[1] * f + 0.5), int(hw[0] * f + 0.5))


def test_center_crop_offsets():
    ev = cl.EvalPipeline(_steps())
    assert ev.windows(240, 320) == (256, 341, [(16, 58)])
    assert ev.windows(320, 240) == (341, 256, [(58, 16)])
    assert ev.windows(240, 427) == (256, 455, [(16, 115)])
    assert ev.windows(256, 300) == (256, 300, [(16, 38)])
    rect = cl.EvalPipeline(_steps(size=(200, 100)))                      # (w, h), mmaction's _pair order
    assert rect.crop_hw == (100, 200)
    assert rect.windows(240, 320) == (256, 341, [(78, 70)])
    with pytest.raises(ValueError, match="larger than the resized frame"):
        cl.EvalPipeline(_steps(size=300)).windows(240, 320)


def test_three_crop_offsets():
    ev = cl.EvalPipeline(_steps("ThreeCrop", 256))
    assert ev.n_crops == 3
    # 341 - 256 = 85 pixels of slack: step 42, the right crop starts at 2 * 42 = 84, not 85
    assert ev.windows(240, 320) == (256, 341, [(0, 0), (0, 84), (0, 42)])
    assert ev.windows(240, 427) == (256, 455, [(0, 0), (0, 198), (0, 99)])
    assert ev.windows(320, 240) == (341, 256, [(0, 0), (84, 0), (42, 0)])            # portrait: vertical
    assert ev.windows(256, 256) == (256, 256, [(0, 0), (0, 0), (0, 0)])
    with pytest.raises(ValueError, match="ThreeCrop"):
        cl.EvalPipeline(_steps("ThreeCrop", 224)).windows(240, 320)                # spans neither side
    with pytest.raises(ValueError, match="ThreeCrop"):
        cl.EvalPipeline(_steps("ThreeCrop", (400, 256))).windows(240, 320)         # spans the height, wider than the frame


def test_geometry_is_clip_major_then_crop():
    from bgdebias_b200 import ops
    ev = cl.EvalPipeline(_steps("ThreeCrop", 256))
    _, g5 = ops.pack_clips([torch.zeros((2, 240, 320, 3), dtype=torch.uint8), torch.zeros((2, 320, 241, 3), dtype=torch.uint8)])
    g = ev.geometry(g5)
    assert g.dtype == torch.int64 and tuple(g.shape) == (6, 9)
    assert torch.equal(g[:3, :5], g5[0].expand(3, 5)) and torch.equal(g[3:, :5], g5[1].expand(3, 5))
    assert g[:3, 5:].tolist() == [[256, 341, 0, 0], [256, 341, 0, 84], [256, 341, 0, 42]]
    assert g[3:, 5:].tolist() == [[340, 256, 0, 0], [340, 256, 84, 0], [340, 256, 42, 0]]


@pytest.mark.parametrize("steps, match", [
    (_steps()[:3], "FormatShape step is missing"),
    (_steps() + [dict(type="Collect", keys=["imgs"])], "'Collect'"),
    ([_steps()[0], dict(type="TenCrop", crop_size=224)] + _steps()[2:], "'TenCrop'"),
    ([_steps()[0], dict(type="FiveCrop", crop_size=224)] + _steps()[2:], "'FiveCrop'"),
    ([_steps()[0], dict(type="RandomCrop", size=224)] + _steps()[2:], "'RandomCrop'"),
    (_steps()[1:2] + _steps()[:1] + _steps()[2:], "'CenterCrop'"),
    ([dict(type="Resize", scale=(-1, 256), keep_ratio=False)] + _steps()[1:], "Resize: keep_ratio"),
    ([dict(type="Resize", scale=(-1, 256), interpolation="bicubic")] + _steps()[1:], "Resize: interpolation"),
    ([dict(type="Resize", scale=(340, 256))] + _steps()[1:], "Resize: only scale"),
    ([dict(type="Resize", scale=(224, 224), keep_ratio=False)] + _steps()[1:], "Resize: keep_ratio"),
    (_steps()[:2] + [dict(type="Normalize", mean=MEAN, std=STD, to_bgr=True)] + _steps()[3:], "Normalize: to_bgr"),
    (_steps()[:2] + [dict(type="Normalize", mean=MEAN[:2], std=STD)] + _steps()[3:], "Normalize: mean and std"),
    (_steps()[:3] + [dict(type="FormatShape", input_format="NCTHW")], "FormatShape: only"),
    ([_steps()[0], dict(type="CenterCrop", crop_size=0)] + _steps()[2:], "CenterCrop: crop_size"),
])
def test_device_test_pipeline_refusals(steps, match):
    with pytest.raises(ValueError, match=match):
        cl.EvalPipeline(steps)


def test_device_test_pipeline_needs_test_mode_and_device_mix(tmp_path):
    clips = [np.zeros((2, 6, 8, 3), np.uint8)]
    with pytest.raises(ValueError, match="needs device_test_pipeline"):
        _dataset(tmp_path, clips, test_mode=True, device_mix=True)
    with pytest.raises(ValueError, match="evaluation tail"):
        _dataset(tmp_path, clips, device_mix=True, device_test_pipeline=_steps())
    with pytest.raises(ValueError, match="'Collect'"):
        _dataset(tmp_path, clips, test_mode=True, device_mix=True, device_test_pipeline=_steps() + [dict(type="Collect")])


def test_host_collate_eval_batch(tmp_path):
    """Samples without draws: native-size uint8 clips packed with ops.pack_clips (ragged sizes), label carried."""
    rng = np.random.default_rng(0)
    clips = [rng.integers(0, 256, (3, h, w, 3), dtype=np.uint8) for h, w in ((24, 32), (24, 43), (31, 17))]
    ds = _dataset(tmp_path, clips, test_mode=True, device_mix=True, device_test_pipeline=_steps("ThreeCrop", 24))
    batch = ds.host_collate([ds[i] for i in range(len(ds))])
    assert set(batch) == {"imgs", "fg_geom", "fg_frames", "label"}
    assert batch["imgs"].dtype == torch.uint8 and batch["imgs"].dim() == 1 and not batch["imgs"].is_cuda
    assert batch["fg_frames"] == 3 and batch["label"].tolist() == [[0], [1], [2]]
    for c, (off, h, w, rs, fs) in zip(clips, batch["fg_geom"].tolist()):
        assert (h, w, rs, fs) == (c.shape[1], c.shape[2], 3 * c.shape[2], 3 * c.shape[1] * c.shape[2])
        assert np.array_equal(batch["imgs"][off:off + c.size].numpy().reshape(c.shape), c)
    # one size for the whole batch is packed as well: the device route always reads the packed form
    same = [clips[0], clips[0] + 1]
    b2 = cl.BackgroundMixDataset.host_collate([dict(imgs=torch.from_numpy(c), label=torch.tensor([0])) for c in same])
    assert b2["imgs"].dim() == 1 and tuple(b2["fg_geom"].shape) == (2, 5)


def test_device_finish_refuses_eval_batch_without_tail(tmp_path):
    clips = [np.zeros((2, 6, 8, 3), np.uint8)]
    ds = _dataset(tmp_path, clips, test_mode=True, prob=1.0)
    batch = ds.host_collate([ds[0]])
    with pytest.raises(ValueError, match="device_test_pipeline"):
        ds.device_finish(batch)
