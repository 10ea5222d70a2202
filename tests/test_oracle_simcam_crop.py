"""CPU checks of the host side of the batched sim_cam crop (extract_background.crop_draws and the in-order staging loop):
replaying RandomResizedCrop's draws from the frame sizes alone, then the antialiased resize of the crop window
(oracle/aa_resize_oracle.py, the arithmetic the CUDA kernel restates), is bit-equal to torchvision's
``RandomResizedCrop(100)(frame.float())`` (cil_tools/extract_background.py:81,89-90) and leaves the torch RNG where
the real transform leaves it; the draw order does not depend on the number of decoder threads."""
import pathlib
import random
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from oracle import aa_resize_oracle as ao                 # noqa: E402

SIZES = [(60, 80), (101, 99), (100, 100), (240, 320), (240, 427), (256, 340), (480, 640), (720, 1280)]


@pytest.fixture(scope="module")
def eb():
    from bgdebias_b200 import extract_background
    return extract_background


def _frame(rng, H, W):
    img = rng.integers(0, 256, (3, H, W), dtype=np.uint8)
    img[:, rng.random((H, W)) < 0.05] = 0                 # zeros: the reference marks them missing afterwards
    return img


@pytest.mark.parametrize("size", SIZES, ids=[f"{h}x{w}" for h, w in SIZES])
def test_replayed_draws_and_window_resize_equal_random_resized_crop(eb, size):
    from torchvision.transforms import RandomResizedCrop
    H, W = size
    rng = np.random.default_rng(H * 7919 + W)
    n_seeds = 3 if H * W > 400_000 else 8
    for seed in range(n_seeds):
        img = _frame(rng, H, W)
        torch.manual_seed(seed)
        exp = RandomResizedCrop(100)(torch.from_numpy(img).float()).numpy()
        torch.manual_seed(seed)
        (i, j, h, w), = eb.crop_draws([(H, W)])
        got = ao.aa_resize(img[:, i:i + h, j:j + w], (100, 100))
        assert got.dtype == np.float32 and got.shape == (3, 100, 100)
        np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32), err_msg=f"{size} seed {seed} crop {(i, j, h, w)}")


def test_draws_cover_upscaled_and_unresized_axes(eb):
    torch.manual_seed(0)
    draws = eb.crop_draws([(101, 99)] * 400 + [(60, 80)] * 100)
    assert any(h < 100 or w < 100 for _, _, h, w in draws)                   # up-scaled crops
    assert any(h == 100 or w == 100 for _, _, h, w in draws[:400])            # an axis whose pass is skipped


def test_rng_state_after_replay_equals_state_after_real_transforms(eb):
    from torchvision.transforms import RandomResizedCrop
    sizes = [SIZES[k % len(SIZES)] for k in range(37)]
    torch.manual_seed(1234)
    rrc = RandomResizedCrop(100)
    for H, W in sizes:
        rrc(torch.zeros((3, H, W)))
    real = torch.get_rng_state()
    torch.manual_seed(1234)
    eb.crop_draws(sizes)
    assert torch.equal(torch.get_rng_state(), real)


def test_draw_sequence_does_not_depend_on_decoder_threads(eb):
    """The staged loop's structure: folders decoded by a pool that finishes out of order, draws made on the consuming
    thread as folders come back in submission order."""
    rng = np.random.default_rng(3)
    folders = [[SIZES[int(k)] for k in rng.integers(0, len(SIZES), int(n))] for n in rng.integers(1, 9, 40)]

    def decode(sizes):
        time.sleep(random.random() * 0.004)                # decoders finish in any order
        return sizes

    def run(threads, window):
        torch.manual_seed(99)
        with ThreadPoolExecutor(threads) as pool:
            return [eb.crop_draws(sizes) for sizes in eb.in_submission_order(pool, decode, folders, window)]

    one = run(1, 4)
    torch.manual_seed(99)
    serial = [eb.crop_draws(sizes) for sizes in folders]                     # the reference worker's order
    assert one == serial
    assert run(8, 32) == serial
    assert run(3, 5) == serial
