"""The median oracle (NumPy + C restatements) against the reference's own outputs.

tests/golden/median_reference.npz was produced by running the reference's
``bg_extraction_tmf`` (cil_tools/extract_background.py:42-75 on FFV1 videos, and
libs/loader/comix_loader.py:148-164 on PNG folders) -- see oracle/gen_golden.py.
"""
import numpy as np
import pytest

from oracle import c_oracle, median_oracle as mo

from conftest import GOLDEN, median_case_names

_NPZ = np.load(GOLDEN / "median_reference.npz")
CASES = median_case_names(_NPZ)


def _used_frames(name):
    frames = _NPZ[name + "/frames"]
    interval, max_frames = (int(v) for v in _NPZ[name + "/params"])
    idx = mo.select_frame_indices(len(frames), interval, max_frames)
    return frames[idx], interval, max_frames


@pytest.mark.parametrize("name", CASES)
def test_numpy_restatement_matches_reference(name):
    frames = _NPZ[name + "/frames"]
    interval, max_frames = (int(v) for v in _NPZ[name + "/params"])
    got = mo.bg_extraction_tmf_frames(frames, interval, max_frames)
    assert got.dtype == np.uint8
    np.testing.assert_array_equal(got, _NPZ[name + "/expected"])


@pytest.mark.parametrize("name", CASES)
def test_integer_form_matches_reference(name):
    used, _, _ = _used_frames(name)
    np.testing.assert_array_equal(mo.temporal_median_int(used), _NPZ[name + "/expected"])


@pytest.mark.parametrize("name", CASES)
def test_c_oracle_matches_reference(name):
    used, _, _ = _used_frames(name)
    np.testing.assert_array_equal(c_oracle.temporal_median(used), _NPZ[name + "/expected"])


@pytest.mark.parametrize("name", [n for n in CASES if n + "/expected_rawframes" in _NPZ.files])
def test_rawframes_variant_uses_all_frames(name):
    # comix_loader.py:157-161: no interval, no cap
    frames = _NPZ[name + "/frames"]
    np.testing.assert_array_equal(mo.temporal_median_np(frames), _NPZ[name + "/expected_rawframes"])


def test_frame_selection_off_by_one_and_interval():
    # extract_background.py:52 `len(frames) <= max_frames` keeps max_frames + 1 frames
    assert mo.select_frame_indices(20, 1, 4) == [0, 1, 2, 3, 4]
    assert mo.select_frame_indices(40, 2, 5) == [0, 2, 4, 6, 8, 10]
    assert mo.select_frame_indices(50, 3, 500) == list(range(0, 50, 3))
    assert mo.select_frame_indices(520, 1, 500) == list(range(501))
    assert mo.select_frame_indices(0, 1, 500) == []
    assert mo.select_frame_indices(3, 1, 0) == [0]
    with pytest.raises(ZeroDivisionError):
        mo.select_frame_indices(3, 0, 5)


def test_pure_python_form_small():
    rng = np.random.default_rng(5)
    for T in (1, 2, 3, 4, 5, 8, 9):
        fr = rng.integers(0, 256, (T, 7), dtype=np.uint8)
        assert mo.temporal_median_py(fr.T.tolist()) == mo.temporal_median_np(fr).tolist()


def test_order_invariance_and_varlen():
    rng = np.random.default_rng(6)
    fr = rng.integers(0, 256, (37, 5, 4, 3), dtype=np.uint8)
    perm = rng.permutation(37)
    np.testing.assert_array_equal(mo.temporal_median_int(fr), mo.temporal_median_int(fr[perm]))
    offs = [0, 1, 3, 10, 37]
    v = mo.temporal_median_varlen(fr, offs)
    vc = c_oracle.temporal_median_varlen(fr, offs)
    np.testing.assert_array_equal(v, vc)
    for i in range(4):
        np.testing.assert_array_equal(v[i], mo.temporal_median_np(fr[offs[i]:offs[i + 1]]))


def test_empty_input_fails_like_reference():
    # reference: np.median([]) is nan and cv2.imwrite raises (extract_background.py:73-74)
    with pytest.raises(ValueError):
        mo.temporal_median_int(np.zeros((0, 4), np.uint8))
    with pytest.raises(ValueError):
        c_oracle.temporal_median(np.zeros((0, 4), np.uint8))


def test_reference_splits():
    # extract_background.py:128-133
    s = mo.reference_contiguous_splits(10, 4)
    assert [list(r) for r in s] == [[0, 1, 2], [3, 4, 5], [6, 7, 8], [9]]
    s = mo.reference_contiguous_splits(3, 4)
    assert [len(r) for r in s] == [1, 1, 1, 0]


@pytest.mark.parametrize("name", CASES)
def test_stored_reference_video_agrees(name, tmp_path):
    """The comparison of test_live_reference_agrees on the videos whose reference outputs are stored: the frames are
    written as an FFV1 video, read back with cv2.VideoCapture as bg_extraction_tmf reads them (extract_background.py:
    42-75), and the restatement of the decoded frames must give the reference's output."""
    import cv2
    from oracle import gen_golden
    interval, max_frames = (int(v) for v in _NPZ[name + "/params"])
    vid = str(tmp_path / "v.avi")
    gen_golden.write_ffv1(vid, _NPZ[name + "/frames"])
    cap = cv2.VideoCapture(vid)
    decoded = []
    ok, f = cap.read()
    while ok:
        decoded.append(f)
        ok, f = cap.read()
    cap.release()
    np.testing.assert_array_equal(mo.bg_extraction_tmf_frames(np.array(decoded), interval, max_frames),
                                  _NPZ[name + "/expected"])


@pytest.mark.reference
def test_live_reference_agrees(tmp_path):
    """Build container only: run the reference itself on a fresh random video."""
    import pathlib
    from oracle import _ref_import, gen_golden
    ref = _ref_import.load_extract_background()
    fr = np.random.default_rng(99).integers(0, 256, (21, 16, 24, 3), dtype=np.uint8)
    vid = str(tmp_path / "v.avi")
    gen_golden.write_ffv1(vid, fr)
    out = ref.bg_extraction_tmf(pathlib.Path(vid), tmp_path / "o.jpg", True, 2, 7, 0)
    np.testing.assert_array_equal(out, mo.bg_extraction_tmf_frames(fr, 2, 7))
