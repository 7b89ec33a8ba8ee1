import os
import sys

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def lib():
    """libxrseg.so: the product library (include/xrseg.h only)."""
    from xr_image_segmentation_b200 import _lib
    if not os.path.exists(_lib.library_path()) or not os.path.exists(_lib.library_path(True)):
        _lib.build_library()
    return _lib.load_library()


@pytest.fixture(scope="session")
def dlib(lib):
    """libxrseg_debug.so: the same sources + the parity hooks of include/xrseg_debug.h."""
    from xr_image_segmentation_b200 import _lib
    return _lib.load_library(True)


@pytest.fixture(scope="session")
def golden(lib):
    from xr_image_segmentation_b200 import inference as I
    model = I.ModelLoader.Load(os.path.join(GOLDEN, "yolo11n_seg.xrsw"))
    inputs = dict(np.load(os.path.join(GOLDEN, "inputs.npz")))
    expected = dict(np.load(os.path.join(GOLDEN, "expected.npz")))
    labels = open(os.path.join(GOLDEN, "labels.txt")).read()
    return dict(model=model, inputs=inputs, expected=expected, labels=labels)


@pytest.fixture(scope="session")
def golden_sentis(golden):
    """The golden XRSW pack (the reference asset's uint8 tensors with their scale / zero point) put back into a .sentis
    container with the asset's NMS thresholds (SURVEY.md fact 3): what the asset's loaders read, without the asset."""
    from oracle.sentis import write_sentis
    from xr_image_segmentation_b200 import weights as W
    pack = golden["model"].pack
    _, _, n, _, payload, _ = W.HEADER.unpack_from(pack, 0)
    convs = []
    for i in range(n):
        (_, cout, cin_g, k, _, _, _, tr, dtype, ws, wz, bs, bz, w_off, b_off) = \
            W.RECORD.unpack_from(pack, W.HEADER.size + i * W.RECORD.size)
        assert dtype == 3
        shape = (cin_g, cout, k, k) if tr else (cout, cin_g, k, k)
        wq = np.frombuffer(pack, np.uint8, int(np.prod(shape)), payload + w_off).reshape(shape)
        convs.append((wq, ws, wz, np.frombuffer(pack, np.uint8, cout, payload + b_off), bs, bz, bool(tr)))
    return write_sentis(convs, 0.43, 0.301)


@pytest.fixture(scope="session")
def golden_weights(golden):
    from xr_image_segmentation_b200 import weights as W
    scale, layers = W.read_pack(golden["model"].pack)
    assert scale == "n"
    return [(w, b) for _, w, b in layers]
