"""GPU: the host-pointer YOLO helpers (corner NMS, letterbox inverse, anchor-grid decode) against the oracle, over the sizes,
ties, special values and count / cap cases their device kernels handle separately."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NMS_SIZES = [1, 2, 31, 32, 33, 255, 256, 257, 1000, 1023, 1024]


def random_boxes(pkg, rng, n):
    b = np.zeros(n, dtype=pkg.capi.BOX_DTYPE)
    xy = rng.integers(0, 200, size=(n, 2)).astype(np.float32)
    wh = rng.integers(1, 60, size=(n, 2)).astype(np.float32)
    b["x0"], b["y0"], b["x1"], b["y1"] = xy[:, 0], xy[:, 1], xy[:, 0] + wh[:, 0], xy[:, 1] + wh[:, 1]
    b["confidence"] = (rng.integers(0, 10, size=n) / 10).astype(np.float32)  # heavy ties: input order decides
    b["class_id"] = rng.choice(np.array([-1, 0, 1, 2, 126, 127, 5000, 2**31 - 1], dtype=np.int32), size=n)
    return b


@pytest.mark.parametrize("n", NMS_SIZES)
def test_nms_boxes_sizes_ties_and_class_ids(pkg, ob, n):
    rng = np.random.default_rng(1000 + n)
    b = random_boxes(pkg, rng, n)
    for th in (0.45, 0.0):
        assert pkg.capi.nms_boxes(b, th).tobytes() == ob.nms_corner(b, th).tobytes(), th


@pytest.mark.parametrize("n", NMS_SIZES)
def test_nms_boxes_nan_inf_and_signed_zero_confidences(pkg, ob, n):
    """presorted the way both sorts agree on: descending, NaN last, ties and -0 / +0 in input order (the oracle's insertion
    sort leaves a sorted array in place; on unsorted input a NaN stops its inner loop)"""
    rng = np.random.default_rng(2000 + n)
    b = random_boxes(pkg, rng, n)
    special = np.array([np.nan, np.inf, -np.inf, 0.0, -0.0], dtype=np.float32)
    k = rng.integers(0, n, size=max(1, n // 4))
    b["confidence"][k] = rng.choice(special, size=k.size)
    b = b[np.argsort(-b["confidence"], kind="stable")]
    for th in (0.45, 0.0):
        assert pkg.capi.nms_boxes(b, th).tobytes() == ob.nms_corner(b, th).tobytes(), th


def test_nms_boxes_rejects_more_than_1024(pkg):
    b = random_boxes(pkg, np.random.default_rng(5), 1025)
    assert pkg.lib().mars_yolo_nms_boxes(b.ctypes.data, len(b), 0.45) == -1


@pytest.mark.parametrize("net", [(640, 640), (320, 640)])
def test_scale_detections_frames(pkg, ob, net):
    net_w, net_h = net
    rng = np.random.default_rng(net_w)
    L, O = pkg.lib(), ob.lib()
    frames = [(1920, 1080), (1080, 1920), (net_w, net_h), (2 * net_w, 2 * net_h), (333, 777), (777, 333), (1, 1)]
    for fw, fh in frames:
        b = np.zeros(300, dtype=pkg.capi.BOX_DTYPE)
        for f in ("x0", "y0", "x1", "y1"):  # inside the input and beyond both edges, so both clamps act
            b[f] = rng.uniform(-50, max(net_w, net_h) + 50, size=len(b)).astype(np.float32)
        b["confidence"] = rng.uniform(0, 1, size=len(b)).astype(np.float32)
        b["class_id"] = rng.integers(0, 80, size=len(b))
        g, o = b.copy(), b.copy()
        L.mars_yolo_scale_detections(g.ctypes.data, len(g), fw, fh, net_w, net_h)
        O.mo_scale_detections(o.ctypes.data, len(o), fw, fh, net_w, net_h)
        assert g.tobytes() == o.tobytes(), (fw, fh)


def decode_both(pkg, ob, head, gh, gw, scale, level, conf, prefill, cnt, maxd):
    d1, d2 = prefill.copy(), prefill.copy()
    n1 = pkg.lib().mars_yolo_decode_anchor_grid(head.ctypes.data, gh, gw, scale, level, conf, d1.ctypes.data, cnt, maxd)
    n2 = ob.lib().mo_decode_anchor_grid(head.ctypes.data, gh, gw, scale, level, conf, d2.ctypes.data, cnt, maxd)
    return n1, n2, d1, d2


@pytest.mark.parametrize("level,gh,gw", [(0, 12, 20), (1, 7, 3), (2, 1, 9), (2, 5, 5)])
def test_decode_anchor_grid_counts_and_caps(pkg, ob, level, gh, gw):
    rng = np.random.default_rng(10 * level + gh)
    head = rng.integers(-128, 128, size=(3, gh, gw, 85), dtype=np.int8)
    cells = 3 * gh * gw
    cap = 2 * cells
    prefill = np.zeros(cap, dtype=pkg.capi.BOX_DTYPE)
    prefill.view(np.uint8)[:] = rng.integers(0, 256, size=prefill.nbytes, dtype=np.uint8)
    full = None
    for scale, conf in ((0.05, 0.25), (0.02, 0.1)):
        for cnt, maxd in ((0, cap), (5, cap), (0, 1), (cells // 3, cells // 3 + 3), (1, 2)):
            n1, n2, d1, d2 = decode_both(pkg, ob, head, gh, gw, scale, level, conf, prefill, cnt, maxd)
            assert n1 == n2 and cnt <= n1 <= maxd, (scale, conf, cnt, maxd, n1, n2)
            assert d1.tobytes() == d2.tobytes(), (scale, conf, cnt, maxd)
            assert d1[:cnt].tobytes() == prefill[:cnt].tobytes() and d1[n1:].tobytes() == prefill[n1:].tobytes()
            if (scale, cnt, maxd) == (0.05, 0, cap):
                full = n1
            if maxd - cnt < 4:
                assert n1 == maxd, "the cap case needs more candidates than room"
        for cnt in (cap, cap + 3):  # no room: the count comes back and dets is not touched
            n1, n2, d1, d2 = decode_both(pkg, ob, head, gh, gw, scale, level, conf, prefill, cnt, cap)
            assert n1 == n2 == cnt and d1.tobytes() == prefill.tobytes() and d2.tobytes() == prefill.tobytes()
    assert full and full > 0
