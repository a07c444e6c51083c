"""CPU: finding the YOLOv5 Detect head convs in a .mars blob, and the class-count-generic decode of the heads reference flow."""
import numpy as np
import pytest

from heads_ref import decode_anchor_grid_nc
from util import MICRO


@pytest.mark.parametrize("nc", [80, 3])
@pytest.mark.parametrize("nhwc", [False, True])
@pytest.mark.parametrize("size", [320, 640])
@pytest.mark.parametrize("width", [0.25, 0.5])
def test_find_yolo_heads_in_stride_order(pkg, width, size, nhwc, nc):
    m = pkg.marsfile.build_yolov5(width=width, size=size, nhwc=nhwc, nc=nc)
    ids = pkg.capi.find_yolo_heads(m.to_bytes())
    assert len(ids) == 3
    for level, tid in enumerate(ids):
        t = m.tensors[tid]
        assert t.name == "/model.24/m.%d/Conv_output_0" % level
        g = size // (8 << level)
        assert t.shape == ([1, g, g, 3 * (5 + nc)] if nhwc else [1, 3 * (5 + nc), g, g])


def test_find_yolo_heads_without_a_detect_block(pkg):
    mf = pkg.marsfile
    blobs = [mf.build_tiny(160).to_bytes(), mf.build_nanodet_like().to_bytes()]
    blobs += [mf.build_single_layer(kind, **kw).to_bytes() for kind, kw in MICRO]
    for b in blobs:
        assert pkg.capi.find_yolo_heads(b) == []
    assert pkg.capi.find_yolo_heads(b"not a model") == []


def test_decode_nc80_matches_the_oracle(ob):
    rng = np.random.default_rng(4)
    for trial in range(8):
        gh, gw = int(rng.integers(1, 24)), int(rng.integers(1, 24))
        head = rng.integers(-128, 128, size=(3, gh, gw, 85), dtype=np.int8)
        if trial % 2:
            head = (head // 40 * 40).astype(np.int8)  # ties in the class argmax
        scale = float(rng.choice([0.01, 0.05, 0.2]))
        level, conf = trial % 3, float(rng.choice([0.1, 0.25, 0.5]))
        maxd = int(rng.choice([1000, 37]))
        want = np.zeros(maxd, dtype=ob.BOX_DTYPE)
        n = ob.lib().mo_decode_anchor_grid(head.ctypes.data, gh, gw, scale, level, conf, want.ctypes.data, 0, maxd)
        got = decode_anchor_grid_nc(head, scale, level, conf, 80, 0, maxd)
        assert got.size == n and got.tobytes() == want[:n].tobytes(), trial
