"""The sim_cam ("type C") oracle against the reference's own outputs (tests/golden/simcam_reference.npz,
written by oracle/gen_golden_simcam.py from cil_tools/extract_background.py:78-99) and against numpy's
nanmedian / nanmean, which the reference calls (:94-98)."""
import pathlib
import sys
import warnings

import numpy as np
import pytest

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from conftest import GOLDEN, median_case_names            # noqa: E402
from oracle import simcam_oracle as so                    # noqa: E402

_NPZ = np.load(GOLDEN / "simcam_reference.npz")
CASES = median_case_names(_NPZ)


@pytest.mark.parametrize("name", CASES)
def test_reduction_matches_reference_output(name):
    interval, max_frames, avg, seed = (int(v) for v in _NPZ[name + "/params"])
    tf = _NPZ[name + "/transformed"]
    assert tf.shape[0] == len(so.select_file_indices(len(_NPZ[name + "/frames"]), interval, max_frames))
    np.testing.assert_array_equal(so.cast_u8(so.nan_temporal_reduce(tf, avg)), _NPZ[name + "/expected"])


@pytest.mark.parametrize("name", CASES)
def test_transform_is_reproducible_here(name):
    """Same torch / torchvision as the fixture generator: the RNG draws and the antialiased resize of
    RandomResizedCrop(100) reproduce the captured frames bit for bit."""
    import torch
    interval, max_frames, avg, seed = (int(v) for v in _NPZ[name + "/params"])
    frames = _NPZ[name + "/frames"]
    torch.manual_seed(seed)
    tf = so.transform_frames(frames[so.select_file_indices(len(frames), interval, max_frames)])
    np.testing.assert_array_equal(tf.view(np.uint32), _NPZ[name + "/transformed"].view(np.uint32))
    torch.manual_seed(seed)
    np.testing.assert_array_equal(so.sim_cam_background(frames, interval, max_frames, avg), _NPZ[name + "/expected"])


def test_file_selection():
    # image_files[:-1:interval], cut at max_frames (extract_background.py:86-88)
    assert so.select_file_indices(10, 1, 500) == list(range(9))
    assert so.select_file_indices(10, 3, 500) == [0, 3, 6]
    assert so.select_file_indices(10, 2, 3) == [0, 2, 4]
    assert so.select_file_indices(1, 1, 5) == [] and so.select_file_indices(0, 1, 5) == []


@pytest.mark.parametrize("T", [1, 2, 3, 8, 33, 120])
@pytest.mark.parametrize("avg", [0, 1])
def test_against_numpy(T, avg):
    rng = np.random.default_rng(100 * T + avg)
    x = (rng.random((T, 37, 3), dtype=np.float32) * 255).astype(np.float32)
    x[rng.random(x.shape) < 0.3] = np.nan
    x[:, 0] = np.nan                                   # all missing
    x[1:, 1] = np.nan                                  # one valid
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        exp = (np.nanmedian if avg == 0 else np.nanmean)(list(x), axis=0)
    got = so.nan_temporal_reduce(x, avg)
    assert exp.dtype == np.float32 and np.array_equal(np.isnan(got), np.isnan(exp))
    np.testing.assert_array_equal(np.nan_to_num(got).view(np.uint32), np.nan_to_num(exp).view(np.uint32))   # bit-exact
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        np.testing.assert_array_equal(so.cast_u8(got), exp.astype(np.uint8))


@pytest.mark.parametrize("name", CASES)
def test_stored_reference_file_agrees(name, tmp_path):
    """The comparison of test_reference_function_end_to_end on the folders whose reference outputs are stored: the
    restatement under the stored torch seed, written as sim_cam_motion_bg_extract writes it (:99, one channel swap), is
    the reference's file byte for byte."""
    import cv2
    import torch
    interval, max_frames, avg, seed = (int(v) for v in _NPZ[name + "/params"])
    torch.manual_seed(seed)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        img = so.sim_cam_background(_NPZ[name + "/frames"], interval, max_frames, avg)
    assert cv2.imwrite(str(tmp_path / "o.jpg"), cv2.cvtColor(img, cv2.COLOR_BGR2RGB))
    assert (tmp_path / "o.jpg").read_bytes() == _NPZ[name + "/jpeg"].tobytes()


@pytest.mark.reference
def test_reference_function_end_to_end(tmp_path):
    import cv2
    import torch
    from oracle import _ref_import
    ref = _ref_import.load_extract_background()
    rng = np.random.default_rng(3)
    frames = rng.integers(0, 256, (6, 50, 70, 3), dtype=np.uint8)
    d = tmp_path / "v"
    d.mkdir()
    for i, f in enumerate(frames):
        cv2.imwrite(str(d / f"img_{i + 1:05d}.png"), cv2.cvtColor(f, cv2.COLOR_RGB2BGR))
    for avg in (0, 1):
        torch.manual_seed(5)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref.sim_cam_motion_bg_extract(d, tmp_path / "o.png", False, 1, 500, avg)
        written = cv2.imread(str(tmp_path / "o.png"))                 # BGR order of what was written
        torch.manual_seed(5)
        exp = so.sim_cam_background(frames, 1, 500, avg)
        np.testing.assert_array_equal(cv2.cvtColor(written, cv2.COLOR_BGR2RGB), exp)   # :99 swaps the channels once
