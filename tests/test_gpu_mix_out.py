"""16-bit and channels-last outputs of the batch blends (bgmix_blend, bgmix_blend_ragged, bgmix_resize_blend with out_dtype /
layout="NTHWC", and BackgroundMixDataset.device_finish(dtype=..., memory_format=...)).

The output is defined as the fp32 blend rounded once to nearest even, so every 16-bit result must equal torch's .to(dtype)
of the fp32 result bit for bit -- of the oracle's fp32 batch (oracle/bgmix_oracle.py with aa_resize_oracle.py /
resize_oracle.py, built as tests/test_gpu_bgmix.py, test_gpu_ragged.py and test_gpu_resize.py build it) and of the same op's
fp32 output.  NTHWC is the same values stored [B, T, H, W, 3]."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import aa_resize_oracle as ao  # noqa: E402
from oracle import bgmix_oracle as bo      # noqa: E402
from oracle import resize_oracle as ro     # noqa: E402

DTYPES = [torch.float32, torch.bfloat16, torch.float16]
LAYOUTS = ["NTCHW", "NCTHW", "NTHWC"]
_BITS = {torch.float32: torch.int32, torch.bfloat16: torch.int16, torch.float16: torch.int16}


def _load_env():
    import bgdebias_b200.ops as ops
    from bgdebias_b200 import _cabi, comix_loader, pool
    assert torch.cuda.is_available()
    _cabi.lib()
    return ops, _cabi, comix_loader, pool


@pytest.fixture(scope="module")
def env():
    return _load_env()


def _arrange(x_ntchw: torch.Tensor, layout: str) -> torch.Tensor:
    """[B, T, 3, H, W] -> the op's layout, contiguous."""
    if layout == "NCTHW":
        return x_ntchw.permute(0, 2, 1, 3, 4).contiguous()
    if layout == "NTHWC":
        return x_ntchw.permute(0, 1, 3, 4, 2).contiguous()
    return x_ntchw.contiguous()


def _assert_bits(got: torch.Tensor, exp: torch.Tensor):
    assert got.dtype == exp.dtype and tuple(got.shape) == tuple(exp.shape) and got.is_contiguous()
    g, e = got.cpu(), exp.cpu()
    assert torch.equal(g.view(_BITS[g.dtype]), e.view(_BITS[e.dtype]))


def _check_all_forms(run, exp_ntchw: np.ndarray, cabi):
    """run(layout, out_dtype) -> device tensor.  Each (dtype, layout) equals the oracle's fp32 batch converted by torch and
    the op's own fp32 output converted; one launch per call."""
    exp32 = torch.from_numpy(exp_ntchw)
    ref32 = run("NTCHW", None)
    _assert_bits(ref32, exp32)
    for layout in LAYOUTS:
        for dt in DTYPES:
            n0 = cabi.kernel_launch_count()
            got = run(layout, dt)
            assert cabi.kernel_launch_count() - n0 == 1
            _assert_bits(got, _arrange(exp32.to(dt), layout))
            _assert_bits(got, _arrange(ref32.to(dt), layout))


def _i32(a, dev):
    return torch.as_tensor(np.asarray(a), dtype=torch.int32, device=dev)


# --------------------------------------------------------------------------- #
# ops
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("T", [1, 8])
@pytest.mark.parametrize("pool_dtype", ["f32", "u8"])
@pytest.mark.parametrize("hw", [(32, 32), (30, 27)])          # 4-pixel vectors; W % 4 != 0: one pixel per thread
def test_dense_pool(env, hw, pool_dtype, T):
    ops, cabi, cl, pool_mod = env
    rng = np.random.default_rng(T * 100 + hw[1])
    B, (H, W) = 5, hw
    Hb, Wb = H + 9, W + 21
    fg = rng.integers(0, 256, (B, T, H, W, 3), dtype=np.uint8)
    pool = (rng.uniform(0, 255, (4, 3, Hb, Wb)).astype(np.float32) if pool_dtype == "f32"
            else rng.integers(0, 256, (4, 3, Hb, Wb), dtype=np.uint8))
    idx = rng.integers(0, 4, B); top = rng.integers(0, Hb - H + 1, B); left = rng.integers(0, Wb - W + 1, B)
    app = np.array([1, 0, 1, 1, 0], np.uint8)
    exp = bo.mix_batch(fg, pool.astype(np.float32), idx, top, left, app, crop=(H, W), alpha=0.3)
    dev = torch.device("cuda")
    args = (torch.from_numpy(fg).to(dev), torch.from_numpy(pool).to(dev), _i32(idx, dev), _i32(top, dev), _i32(left, dev),
            torch.from_numpy(app).to(dev), ops.make_fg_lut(bo.DEFAULT_MEAN, bo.DEFAULT_STD, dev),
            torch.tensor(bo.DEFAULT_MEAN), torch.tensor(bo.DEFAULT_STD), 0.3)
    _check_all_forms(lambda layout, dt: torch.ops.bgdebias.bgmix_blend(*args, layout, dt), exp, cabi)


def _ragged_case(env, W, size=36, seed=0):
    ops, cabi, cl, pool_mod = env
    rng = np.random.default_rng(seed + W)
    B, T, H = 7, 3, 28
    # (160, 200) -> 36 rows: a 32-row tile spans more than the tile kernel's 48 source rows (per-value fallback)
    sizes = [(36, 48), (40, 36), (80, 120), (36, 36), (31, 77), (160, 200)]
    imgs = [rng.integers(0, 256, (3,) + s, dtype=np.uint8) for s in sizes]
    rp = pool_mod.RaggedPool(size, "cuda")
    rp.append(imgs)
    fg = rng.integers(0, 256, (B, T, H, W, 3), dtype=np.uint8)
    idx = np.array([5, 2, 0, 1, 5, 3, 4])
    app = np.array([1, 1, 0, 1, 1, 0, 1], np.uint8)
    hw = [rp.hw(int(i)) for i in idx]
    top = np.array([rng.integers(0, h - H + 1) for h, w in hw]); left = np.array([rng.integers(0, w - W + 1) for h, w in hw])
    resized = [ao.aa_resize(im, size) for im in imgs]
    exp = np.stack([bo.mix_clip(fg[b], resized[idx[b]], int(top[b]), int(left[b]), (H, W), 0.4, bool(app[b])) for b in range(B)])
    dev = torch.device("cuda")
    args = (torch.from_numpy(fg).to(dev), rp.data, rp.slots_tensor, rp.tables.tensor, _i32(idx, dev), _i32(top, dev),
            _i32(left, dev), torch.from_numpy(app).to(dev), ops.make_fg_lut(bo.DEFAULT_MEAN, bo.DEFAULT_STD, dev),
            torch.tensor(bo.DEFAULT_MEAN), torch.tensor(bo.DEFAULT_STD), 0.4)
    return args, exp


@pytest.mark.parametrize("W", [32, 30])                        # tile kernel; per-value kernel, one pixel per thread
def test_ragged_pool(env, W):
    args, exp = _ragged_case(env, W)
    _check_all_forms(lambda layout, dt: torch.ops.bgdebias.bgmix_blend_ragged(*args, layout, dt), exp, env[1])


_PER_VALUE_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
import test_gpu_mix_out as t
env = t._load_env()
args, exp = t._ragged_case(env, 32, seed=1)
t._check_all_forms(lambda layout, dt: torch.ops.bgdebias.bgmix_blend_ragged(*args, layout, dt), exp, env[1])
print("per-value ok")
"""


def test_ragged_pool_per_value_vector_form(env):
    """The per-value kernel with 4-pixel vectors (selected by BGD_RAGGED_PER_VALUE, read once per process)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _PER_VALUE_SCRIPT, root], env=dict(os.environ, BGD_RAGGED_PER_VALUE="1"),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "per-value ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("pool_dtype", [torch.float32, torch.uint8])
def test_fused_resize_blend_of_packed_crops(env, pool_dtype):
    ops, cabi, cl, pool_mod = env
    rng = np.random.default_rng(7)
    T, H, W, P = 4, 56, 56, 6
    shapes = [(64, 64), (56, 56), (48, 56), (42, 48), (56, 64), (64, 56), (48, 48), (42, 42), (50, 62)]
    clips = [rng.integers(0, 256, (T, h, w, 3), dtype=np.uint8) for h, w in shapes]
    B = len(clips)
    pool = rng.integers(0, 256, (P, 3, 64, 85)).astype(np.float32)
    idx = rng.integers(0, P, B); top = rng.integers(0, 64 - H + 1, B); left = rng.integers(0, 85 - W + 1, B)
    app = (rng.random(B) < 0.6).astype(np.uint8); app[0], app[1] = 1, 0
    buf, geom = ops.pack_clips(clips)
    dev = torch.device("cuda")
    args = (buf.to(dev), geom, T, H, W, torch.from_numpy(pool).to(dev, pool_dtype), _i32(idx, dev), _i32(top, dev),
            _i32(left, dev), torch.as_tensor(app, device=dev), ops.make_fg_lut(bo.DEFAULT_MEAN, bo.DEFAULT_STD, dev),
            torch.tensor(bo.DEFAULT_MEAN), torch.tensor(bo.DEFAULT_STD), 0.5)
    exp = bo.mix_batch(np.stack([ro.resize_clip(c, H, W) for c in clips]), pool, idx, top, left, app, crop=(H, W))
    _check_all_forms(lambda layout, dt: torch.ops.bgdebias.bgmix_resize_blend(*args, layout, dt), exp, cabi)


def test_full_size_batch(env):
    """The 64 x 8 x 224 x 224 batch of bench.py's mix leg against a 240 x 320 fp32 pool, Bernoulli(0.25) mixing."""
    ops, cabi, cl, pool_mod = env
    rng = np.random.default_rng(64)
    B, T, H, W, P = 64, 8, 224, 224, 16
    fg = rng.integers(0, 256, (B, T, H, W, 3), dtype=np.uint8)
    pool = rng.uniform(0, 255, (P, 3, 240, 320)).astype(np.float32)
    idx = rng.integers(0, P, B); top = rng.integers(0, 240 - H + 1, B); left = rng.integers(0, 320 - W + 1, B)
    app = (rng.random(B) < 0.25).astype(np.uint8); app[0] = 1
    exp = bo.mix_batch(fg, pool, idx, top, left, app, crop=(H, W))
    dev = torch.device("cuda")
    args = (torch.from_numpy(fg).to(dev), torch.from_numpy(pool).to(dev), _i32(idx, dev), _i32(top, dev), _i32(left, dev),
            torch.from_numpy(app).to(dev), ops.make_fg_lut(bo.DEFAULT_MEAN, bo.DEFAULT_STD, dev),
            torch.tensor(bo.DEFAULT_MEAN), torch.tensor(bo.DEFAULT_STD), 0.5)
    ref32 = torch.ops.bgdebias.bgmix_blend(*args, "NTCHW")
    _assert_bits(ref32, torch.from_numpy(exp))
    for layout, dt in (("NTHWC", torch.bfloat16), ("NTCHW", torch.float16), ("NTHWC", torch.float32)):
        _assert_bits(torch.ops.bgdebias.bgmix_blend(*args, layout, dt), _arrange(ref32.to(dt), layout))


def test_opcheck(env):
    ops, cabi, cl, pool_mod = env
    dev = torch.device("cuda")
    rng = np.random.default_rng(3)
    B, T, H, W = 3, 2, 16, 16
    fg = torch.from_numpy(rng.integers(0, 256, (B, T, H, W, 3), dtype=np.uint8)).to(dev)
    lut = ops.make_fg_lut(bo.DEFAULT_MEAN, bo.DEFAULT_STD, dev)
    mean, std = torch.tensor(bo.DEFAULT_MEAN), torch.tensor(bo.DEFAULT_STD)
    draws = (_i32([0, 1, 0], dev), _i32([1, 0, 2], dev), _i32([3, 0, 1], dev), torch.tensor([1, 0, 1], dtype=torch.uint8, device=dev))
    pool = torch.from_numpy(rng.uniform(0, 255, (2, 3, 20, 24)).astype(np.float32)).to(dev)
    torch.library.opcheck(torch.ops.bgdebias.bgmix_blend.default,
                          (fg, pool, *draws, lut, mean, std, 0.5, "NTHWC"), {"out_dtype": torch.bfloat16})
    rp = pool_mod.RaggedPool(20, dev)
    rp.append([rng.integers(0, 256, (3, 20, 26), dtype=np.uint8), rng.integers(0, 256, (3, 30, 24), dtype=np.uint8)])
    torch.library.opcheck(torch.ops.bgdebias.bgmix_blend_ragged.default,
                          (fg, rp.data, rp.slots_tensor, rp.tables.tensor, *draws, lut, mean, std, 0.5, "NTHWC"),
                          {"out_dtype": torch.bfloat16})
    buf, geom = ops.pack_clips([rng.integers(0, 256, (T, h, w, 3), dtype=np.uint8) for h, w in ((18, 20), (16, 16), (14, 12))])
    torch.library.opcheck(torch.ops.bgdebias.bgmix_resize_blend.default,
                          (buf.to(dev), geom, T, H, W, pool, *draws, lut, mean, std, 0.5, "NTHWC"), {"out_dtype": torch.bfloat16})


def test_rejected_arguments(env):
    ops, cabi, cl, pool_mod = env
    dev = torch.device("cuda")
    fg = torch.zeros((1, 1, 8, 8, 3), dtype=torch.uint8, device=dev)
    pool = torch.zeros((1, 3, 8, 8), dtype=torch.float32, device=dev)
    z, one = torch.zeros(1, dtype=torch.int32, device=dev), torch.ones(1, dtype=torch.uint8, device=dev)
    lut = ops.make_fg_lut(bo.DEFAULT_MEAN, bo.DEFAULT_STD, dev)
    mean, std = torch.tensor(bo.DEFAULT_MEAN), torch.tensor(bo.DEFAULT_STD)
    rp = pool_mod.RaggedPool(None, dev)
    rp.append([np.zeros((3, 8, 8), np.uint8)])
    buf, geom = ops.pack_clips([torch.zeros((1, 8, 8, 3), dtype=torch.uint8)])
    calls = [lambda dt, lay="NTCHW": torch.ops.bgdebias.bgmix_blend(fg, pool, z, z, z, one, lut, mean, std, 0.5, lay, dt),
             lambda dt, lay="NTCHW": torch.ops.bgdebias.bgmix_blend_ragged(fg, rp.data, rp.slots_tensor, rp.tables.tensor, z, z,
                                                                          z, one, lut, mean, std, 0.5, lay, dt),
             lambda dt, lay="NTCHW": torch.ops.bgdebias.bgmix_resize_blend(buf.to(dev), geom, 1, 8, 8, pool, z, z, z, one, lut,
                                                                          mean, std, 0.5, lay, dt)]
    for call in calls:
        for dt in (torch.float64, torch.uint8):
            with pytest.raises(ValueError):
                call(dt)
        with pytest.raises(ValueError):
            call(torch.bfloat16, "NHWC")
        assert call(torch.float16, "NTHWC").shape == (1, 1, 8, 8, 3)
    # the fp32 entry points keep their contract: NTHWC is not one of their layouts
    L = cabi.lib()
    out = torch.empty((1, 1, 8, 8, 3), dtype=torch.float32, device=dev)
    rc = L.bgd_bgmix_blend_f32(fg.data_ptr(), 1, 1, 8, 8, pool.data_ptr(), 1, 8, 8, z.data_ptr(), z.data_ptr(), z.data_ptr(),
                               one.data_ptr(), lut.data_ptr(), cabi.f32x3(bo.DEFAULT_MEAN), cabi.f32x3(bo.DEFAULT_STD), 0.5,
                               cabi.LAYOUT_NTHWC, out.data_ptr(), None)
    assert rc == cabi.BGD_ERR_INVALID


# --------------------------------------------------------------------------- #
# dataset
# --------------------------------------------------------------------------- #
class _Reader:
    """bg_reader: a fixed random uint8 [3, h, w] image per path (sizes cycle through `sizes`)."""
    def __init__(self, sizes, seed):
        self.sizes, self.rng, self.cache = sizes, np.random.default_rng(seed), {}

    def __call__(self, path):
        if path not in self.cache:
            self.cache[path] = self.rng.integers(0, 256, (3,) + self.sizes[len(self.cache) % len(self.sizes)], dtype=np.uint8)
        return self.cache[path]


def _dataset_batch(env, tmp_path, bg_sizes, crops, from_bg_dir=True):
    """A host_collate batch of 7 samples (mixed and unmixed) from a device_mix dataset; crops=True: the clips are
    MultiScaleCrop-like crops of mixed sizes (packed, resized on the device)."""
    ops, cabi, cl, pool_mod = env
    rng = np.random.default_rng(len(bg_sizes) + 10 * crops + 100 * from_bg_dir)
    n, T, H, W = 7, 2, 32, 32
    shapes = [(36, 36), (32, 32), (28, 32), (24, 28), (32, 36), (36, 32), (28, 28)] if crops else [(H, W)] * n
    clips = [rng.integers(0, 256, (T, h, w, 3), dtype=np.uint8) for h, w in shapes]
    ra = np.array([0, 1, 0, 0, 1, 0, 0], bool)
    names = [f"v{i:02d}" for i in range(4)]
    for nm in names:
        (tmp_path / (nm + ".jpg")).write_bytes(b"stub")
    infos = [dict(frame_dir=f"/x/{names[i % 4]}", total_frames=5, label=i, sample=i) for i in range(n)]
    pipeline = lambda info: dict(imgs=torch.from_numpy(clips[info["sample"]]), label=torch.tensor([info["label"]]),  # noqa: E731
                                 randAug=bool(ra[info["sample"]]))
    ds = cl.BackgroundMixDataset(infos, pipeline, bg_dir=str(tmp_path), bg_resize=40, bg_crop_size=(H, W), with_randAug=True,
                                 device_mix=True, bg_reader=_Reader(bg_sizes, 5), back_ground_from_bg_dir=from_bg_dir)
    torch.manual_seed(11)
    return ds, ds.host_collate([ds.prepare_train_frames(i) for i in range(n)])


@pytest.mark.parametrize("case", ["dense", "ragged", "random_frame", "crops_dense", "crops_ragged"])
def test_device_finish_dtype_and_channels_last(env, tmp_path, case):
    ops, cabi, cl, pool_mod = env
    bg_sizes = [(36, 48)] if case in ("dense", "crops_dense") else [(36, 48), (36, 64), (50, 40)]
    ds, batch = _dataset_batch(env, tmp_path, bg_sizes, crops=case.startswith("crops"), from_bg_dir=case != "random_frame")
    if case == "random_frame":
        assert "bg_imgs" in batch
    else:
        assert (ds.device_pool().tensor is not None) == (case in ("dense", "crops_dense"))
    launches = 2 if case == "crops_ragged" else 1             # resize_bilinear, then the ragged blend
    for layout in ("NTCHW", "NCTHW"):
        ref = ds.device_finish(batch, layout=layout)["imgs"]
        assert ref.dtype == torch.float32 and ref.is_contiguous()
        for dt in DTYPES:
            for mf in (torch.contiguous_format, torch.channels_last):
                n0 = cabi.kernel_launch_count()
                got = ds.device_finish(batch, layout=layout, dtype=dt, memory_format=mf)["imgs"]
                assert cabi.kernel_launch_count() - n0 == launches
                assert got.dtype == dt and got.shape == ref.shape
                assert torch.equal(got.cpu().view(_BITS[dt]), ref.to(dt).cpu().view(_BITS[dt]))
                if mf == torch.contiguous_format:
                    assert got.is_contiguous()
                elif layout == "NTCHW":
                    assert got.flatten(0, 1).is_contiguous(memory_format=torch.channels_last)
                else:
                    assert got.is_contiguous(memory_format=torch.channels_last_3d)
    if case == "dense":
        samples = [ds.prepare_train_frames(i) for i in range(3)]
        got = ds.gpu_collate(samples, dtype=torch.bfloat16, memory_format=torch.channels_last)["imgs"]
        ref = ds.device_finish(ds.host_collate(samples))["imgs"]
        assert torch.equal(got.cpu().view(torch.int16), ref.to(torch.bfloat16).cpu().view(torch.int16))
        for mf in (torch.preserve_format, torch.channels_last_3d):
            with pytest.raises(ValueError):
                ds.device_finish(batch, memory_format=mf)
        with pytest.raises(ValueError):
            ds.device_finish(batch, dtype=torch.float64)
