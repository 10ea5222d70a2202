import pathlib
import sys

import pytest

ROOT = pathlib.Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

GOLDEN = ROOT / "tests" / "golden"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: runs the original project's code (its source tree at BGD_REFERENCE_ROOT)")


def pytest_collection_modifyitems(config, items):
    from oracle import _ref_import
    have_ref = _ref_import.available()
    skip_ref = pytest.mark.skip(reason="the original project's source tree is not present (BGD_REFERENCE_ROOT)")
    for item in items:
        if "reference" in item.keywords and not have_ref:
            item.add_marker(skip_ref)


@pytest.fixture(scope="session")
def golden_median():
    import numpy as np
    return np.load(GOLDEN / "median_reference.npz")


@pytest.fixture(scope="session")
def golden_bgmix():
    import numpy as np
    return np.load(GOLDEN / "bgmix_reference.npz")


def median_case_names(npz):
    return sorted({k.split("/")[0] for k in npz.files})
