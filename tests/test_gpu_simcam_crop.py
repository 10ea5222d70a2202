"""GPU parity of the batched RandomResizedCrop (torch.ops.bgdebias.resized_crop_aa, C ABI bgd_resized_crop_aa_u8_f32)
and of the staged sim_cam extraction (bg_extract_multiple with sim_cam_motion_bg_extract: decoder threads, pinned
slabs, one crop launch and one NaN-reduce launch per slab).

Bit-exact throughout: crops are compared with torchvision's RandomResizedCrop(100) / resized_crop as float32 bit
patterns, backgrounds as JPEG bytes against the per-folder drop-in and the reference's own outputs
(tests/golden/simcam_reference.npz)."""
import pathlib
import sys

import cv2
import numpy as np
import pytest
import torch

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from conftest import GOLDEN, median_case_names            # noqa: E402
from oracle import simcam_oracle as so                    # noqa: E402

pytestmark = pytest.mark.gpu
_NPZ = np.load(GOLDEN / "simcam_reference.npz")
CASES = median_case_names(_NPZ)
SIZES = [(60, 80), (101, 99), (100, 100), (240, 320), (240, 427), (256, 340), (480, 640), (720, 1280)]


@pytest.fixture(scope="module")
def eb():
    assert torch.cuda.is_available()
    import bgdebias_b200.ops  # noqa: F401
    from bgdebias_b200 import extract_background
    return extract_background


def _pack(frames, gaps):
    """uint8 [3, H, W] frames back to back with `gaps` bytes before each (unaligned offsets) -> (buffer, [(off, H, W)])."""
    layout, parts, off = [], [], 0
    for f, g in zip(frames, gaps):
        parts.append(np.full(g, 77, np.uint8))
        off += g
        layout.append((off, f.shape[1], f.shape[2]))
        parts.append(f.reshape(-1))
        off += f.size
    parts.append(np.full(3, 77, np.uint8))
    return torch.from_numpy(np.concatenate(parts)), layout


def _crop(eb, buf, layout, draws, out=(100, 100)):
    from bgdebias_b200.pool import AATables
    tables = AATables("cuda")
    rows = []
    for (off, H, W), (i, j, h, w) in zip(layout, draws):
        xtab, kx = tables.lookup(w, out[1])
        ytab, ky = tables.lookup(h, out[0])
        rows.append((off, H, W, i, j, h, w, xtab, ytab, kx, ky))
    desc = torch.tensor(rows, dtype=torch.int64)
    return torch.ops.bgdebias.resized_crop_aa(buf.cuda(), desc, tables.tensor, out[0], out[1]).cpu().numpy()


def _frames(rng, sizes):
    out = []
    for H, W in sizes:
        f = rng.integers(0, 256, (3, H, W), dtype=np.uint8)
        f[:, rng.random((H, W)) < 0.03] = 0
        out.append(f)
    return out


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def test_kernel_equals_random_resized_crop_mixed_sizes_one_launch(eb):
    from torchvision.transforms import RandomResizedCrop
    rng = np.random.default_rng(11)
    sizes = [SIZES[k % len(SIZES)] for k in range(3 * len(SIZES))] + [(720, 1280)] * 4
    frames = _frames(rng, sizes)
    buf, layout = _pack(frames, rng.integers(0, 4, len(frames)))       # frames at unaligned byte offsets
    torch.manual_seed(5)
    draws = eb.crop_draws(sizes)
    torch.manual_seed(5)
    rrc = RandomResizedCrop(100)
    exp = np.stack([rrc(torch.from_numpy(f).float()).permute(1, 2, 0).numpy() for f in frames])
    got = _crop(eb, buf, layout, draws)
    assert got.shape == (len(frames), 100, 100, 3)
    for k in range(len(frames)):
        np.testing.assert_array_equal(_bits(got[k]), _bits(exp[k]), err_msg=f"frame {k} {sizes[k]} crop {draws[k]}")


@pytest.mark.parametrize("out", [(100, 100), (37, 50), (64, 129)])
def test_kernel_equals_resized_crop_on_chosen_windows(eb, out):
    """Crop axes equal to the output (pass skipped), up-scaled crops, whole frames, strong down-scaling of 720p
    frames (the per-value form), and output widths that are not a multiple of 4."""
    from torchvision.transforms import InterpolationMode
    from torchvision.transforms import functional as F
    rng = np.random.default_rng(out[0] * 1000 + out[1])
    OH, OW = out
    cases = [((240, 320), (7, 11, OH, 200)), ((240, 320), (3, 5, 150, OW)), ((240, 320), (0, 0, OH, OW)),
             ((101, 99), (1, 0, 100, 99)), ((60, 80), (10, 20, 23, 31)), ((60, 80), (0, 0, 60, 80)),
             ((720, 1280), (0, 0, 720, 1280)), ((720, 1280), (13, 400, 700, 850)), ((720, 1280), (100, 50, 40, 1200)),
             ((480, 640), (5, 9, 470, 17))]
    frames = _frames(rng, [s for s, _ in cases])
    buf, layout = _pack(frames, [1, 2, 3, 0, 5, 1, 7, 2, 1, 3])
    draws = [d for _, d in cases]
    got = _crop(eb, buf, layout, draws, out)
    for k, (f, (i, j, h, w)) in enumerate(zip(frames, draws)):
        exp = F.resized_crop(torch.from_numpy(f).float(), i, j, h, w, [OH, OW], InterpolationMode.BILINEAR,
                             antialias=True).permute(1, 2, 0).numpy()
        np.testing.assert_array_equal(_bits(got[k]), _bits(exp), err_msg=f"case {k} {cases[k]}")


@pytest.mark.parametrize("name", CASES)
def test_kernel_equals_reference_transformed_frames(eb, name):
    interval, max_frames, avg, seed = (int(v) for v in _NPZ[name + "/params"])
    fr = _NPZ[name + "/frames"]
    idx = so.select_file_indices(len(fr), interval, max_frames)
    frames = [np.ascontiguousarray(fr[k].transpose(2, 0, 1)) for k in idx]
    buf, layout = _pack(frames, [0] * len(frames))
    torch.manual_seed(seed)
    draws = eb.crop_draws([f.shape[1:] for f in frames])
    got = _crop(eb, buf, layout, draws)
    exp = np.nan_to_num(_NPZ[name + "/transformed"], nan=0.0)
    np.testing.assert_array_equal(_bits(got), _bits(exp))


def test_op_validation(eb):
    from bgdebias_b200.pool import AATables
    tables = AATables("cuda")
    xtab, kx = tables.lookup(200, 100)
    ytab, ky = tables.lookup(150, 100)
    t = tables.tensor
    buf = torch.zeros(3 * 240 * 320 + 5, dtype=torch.uint8, device="cuda")
    good = [5, 240, 320, 10, 20, 150, 200, xtab, ytab, kx, ky]
    op = torch.ops.bgdebias.resized_crop_aa
    assert op(buf, torch.tensor([good]), t, 100, 100).shape == (1, 100, 100, 3)

    def bad(**kw):
        row = dict(zip(("offset", "H", "W", "top", "left", "h", "w", "xtab", "ytab", "kx", "ky"), good))
        row.update(kw)
        return torch.tensor([list(row.values())])

    for desc in (bad(top=91), bad(left=121), bad(top=-1), bad(h=0), bad(offset=6), bad(offset=-1), bad(H=0),
                 bad(kx=kx + 1), bad(xtab=int(t.numel())), bad(xtab=-1), bad(ytab=-2), bad(ky=ky - 1)):
        with pytest.raises(ValueError):
            op(buf, desc, t, 100, 100)
    with pytest.raises(ValueError):
        op(buf.float(), torch.tensor([good]), t, 100, 100)                 # not uint8
    with pytest.raises(ValueError):
        op(buf, torch.tensor([good[:10]]), t, 100, 100)                    # 10 columns
    with pytest.raises(ValueError):
        op(buf, torch.tensor([good]), t.to(torch.int64), 100, 100)         # tables not int32
    with pytest.raises(ValueError):
        op(buf, torch.tensor([good]), t, 0, 100)                           # empty output
    with pytest.raises(ValueError):
        op(buf, torch.tensor([good]), t, 100, 99)                          # tables built for another output width
    with pytest.raises(ValueError):
        op(buf, bad(h=1 << 33), t, 100, 100)                               # beyond int32


# ---- staged extraction -------------------------------------------------------------------------------------------
def _write_folder(d: pathlib.Path, rng, sizes, gray=False):
    d.mkdir(parents=True)
    for k, (H, W) in enumerate(sizes):
        img = rng.integers(0, 256, (H, W) if gray else (H, W, 3), dtype=np.uint8)
        img[rng.random((H, W)) < 0.02] = 0
        assert cv2.imwrite(str(d / f"img_{k + 1:05d}.{'png' if k % 2 else 'jpg'}"), img)


def _tree(root: pathlib.Path, seed: int):
    rng = np.random.default_rng(seed)
    good = []
    for v in range(14):
        n = int(rng.integers(2, 14))
        if v % 4 == 0:
            sizes = [[(120, 160), (240, 320), (101, 99)][int(k)] for k in rng.integers(0, 3, n)]     # mixed sizes
        else:
            sizes = [[(120, 160), (240, 320), (96, 128)][v % 3]] * n
        _write_folder(root / f"v{v:02d}", rng, sizes)
        good.append(root / f"v{v:02d}")
    (root / "v_empty").mkdir()
    _write_folder(root / "v_gray", rng, [(60, 80)] * 4, gray=True)
    return good, [root / "v_empty", root / "v_gray"]


def _staged(eb, paths, out, interval, max_frames, avg, threads, slab_mb, seed):
    out.mkdir(parents=True)
    torch.manual_seed(seed)
    failures = eb.bg_extract_multiple(paths, out, False, interval, max_frames, 0, eb.sim_cam_motion_bg_extract, avg, 0,
                                      threads, slab_mb)
    return failures


@pytest.mark.parametrize("interval,max_frames,avg", [(1, 500, 0), (3, 500, 1), (1, 4, 0)])
def test_staged_path_writes_the_dropin_jpegs(eb, tmp_path, interval, max_frames, avg):
    good, bad = _tree(tmp_path / "in", 40 + interval + max_frames)
    paths = sorted(good + bad)
    # the per-folder drop-in, in the same order and from the same seed
    (tmp_path / "ref").mkdir()
    torch.manual_seed(7)
    for p in paths:
        if p in bad:
            with pytest.raises(ValueError):
                eb.sim_cam_motion_bg_extract(p, tmp_path / "ref" / (p.name + ".jpg"), False, interval, max_frames, avg)
        else:
            eb.sim_cam_motion_bg_extract(p, tmp_path / "ref" / (p.name + ".jpg"), False, interval, max_frames, avg)
    for tag, threads, slab_mb in (("one", 1, 512), ("many", 8, 1)):
        out = tmp_path / tag
        failures = _staged(eb, paths, out, interval, max_frames, avg, threads, slab_mb, 7)
        assert sorted(pathlib.Path(f).name for f, _ in failures) == ["v_empty", "v_gray"], failures
        written = sorted(f.name for f in out.iterdir())
        assert written == sorted(p.name + ".jpg" for p in good)
        for p in good:
            assert (out / (p.name + ".jpg")).read_bytes() == (tmp_path / "ref" / (p.name + ".jpg")).read_bytes(), (tag, p.name)


@pytest.mark.parametrize("name", CASES)
def test_staged_path_writes_the_reference_jpeg(eb, tmp_path, name):
    interval, max_frames, avg, seed = (int(v) for v in _NPZ[name + "/params"])
    d = tmp_path / "in" / "video"
    d.mkdir(parents=True)
    for i, f in enumerate(_NPZ[name + "/frames"]):
        assert cv2.imwrite(str(d / f"img_{i + 1:05d}.png"), cv2.cvtColor(f, cv2.COLOR_RGB2BGR))
    failures = _staged(eb, [d], tmp_path / "out", interval, max_frames, avg, 2, 512, seed)
    assert failures == []
    assert (tmp_path / "out" / "video.jpg").read_bytes() == _NPZ[name + "/jpeg"].tobytes()
