"""CPU: finding the NanoDet GFL head convs in a .mars blob, and the GFL decode: its C statement against the numpy
restatement, known answers, and an independent float64 evaluation of NanoDet's Integral + distance2bbox."""
import hashlib

import numpy as np
import pytest

from gfl_ref import CENTRE, c_decode_gfl, decode_gfl
from heads_ref import BOX_DTYPE, sigmoid_table
from util import MICRO


@pytest.mark.parametrize("nc", [80, 3])
@pytest.mark.parametrize("nhwc", [False, True])
@pytest.mark.parametrize("size", [320, 416])
def test_find_gfl_heads_in_stride_order(pkg, size, nhwc, nc):
    m = pkg.marsfile.build_nanodet_like(size=size, nhwc=nhwc, nc=nc)
    ids = pkg.capi.find_gfl_heads(m.to_bytes(), nc=nc)
    assert len(ids) == 3
    for level, tid in enumerate(ids):
        t = m.tensors[tid]
        assert t.name == "/head%d.out/Conv_output_0" % level
        g, c = size // (8 << level), nc + 32
        assert t.shape == ([1, g, g, c] if nhwc else [1, c, g, g])
    assert pkg.capi.find_gfl_heads(m.to_bytes(), nc=nc + 1) == []
    assert pkg.capi.find_gfl_heads(m.to_bytes(), nc=nc, reg_max=6) == []


@pytest.mark.parametrize("nhwc", [False, True])
def test_find_gfl_heads_four_levels(pkg, nhwc):
    m = pkg.marsfile.build_nanodet_like(size=320, nhwc=nhwc, levels=4)
    ids = pkg.capi.find_gfl_heads(m.to_bytes())
    assert [m.tensors[t].name for t in ids] == ["/head%d.out/Conv_output_0" % k for k in range(4)]
    assert m.tensors[ids[3]].shape == ([1, 5, 5, 112] if nhwc else [1, 112, 5, 5])


def test_find_gfl_heads_without_gfl_heads(pkg):
    mf = pkg.marsfile
    blobs = [mf.build_yolov5(width=0.25, size=320).to_bytes(), mf.build_yolov5(width=0.5, size=640, nhwc=True).to_bytes(),
             mf.build_tiny(160).to_bytes()]
    blobs += [mf.build_single_layer(kind, **kw).to_bytes() for kind, kw in MICRO]
    for b in blobs:
        assert pkg.capi.find_gfl_heads(b) == []
    assert pkg.capi.find_gfl_heads(b"not a model") == []
    for kw in (dict(), dict(nhwc=True), dict(nc=3), dict(size=416), dict(levels=4), dict(nhwc=True, nc=3, levels=4)):
        assert pkg.capi.find_yolo_heads(mf.build_nanodet_like(**kw).to_bytes()) == [], kw


def test_find_heads_in_a_blob_cut_short(pkg):
    """the finders parse a blob as mars_load_memory does: weights that run past its end make it no model"""
    mf = pkg.marsfile
    for blob, find in ((mf.build_nanodet_like().to_bytes(), pkg.capi.find_gfl_heads),
                       (mf.build_yolov5(width=0.25, size=320).to_bytes(), pkg.capi.find_yolo_heads)):
        assert len(find(blob)) == 3
        assert find(blob[:-1]) == []


def test_default_nanodet_blobs_unchanged(pkg):
    for size, want in ((320, "35fba38eaf8c246645f270ffdabeb2ff1501326f4332c2fbe6e44bfb39476676"),
                       (416, "79d2667b2ac239e664d9d6fd13dac7b5321ea8c1891d902e41d69864db09b54f")):
        b = pkg.marsfile.build_nanodet_like(size=size, seed=7).to_bytes()
        assert len(b) == 1165032 and hashlib.sha256(b).hexdigest() == want, size


def random_heads():
    """(head, nc, reg_max, scale, stride, centre, net_w, net_h, conf, cnt, maxd) cases: tied and saturated class scores, both
    centres, strides 8 to 64, caps 1000 and 37, appends after cnt > 0"""
    rng = np.random.default_rng(11)
    cases = []
    for trial in range(16):
        nc, reg_max = [(80, 7), (3, 7), (1, 1), (20, 16)][trial % 4]
        stride = 8 << (trial % 4)
        gh, gw = int(rng.integers(1, 40)), int(rng.integers(1, 40))
        head = rng.integers(-128, 128, size=(gh, gw, nc + 4 * (reg_max + 1)), dtype=np.int8)
        if trial % 3 == 1:
            head[..., :nc] = head[..., :nc] // 64 * 64  # byte ties in the classes
        scale = float(rng.choice([0.01, 0.05, 0.2, 0.5]))  # 0.2 and 0.5 saturate the sigmoid table: different bytes, equal scores
        conf = float(rng.choice([0.05, 0.3, 0.6, 0.9]))
        maxd = int(rng.choice([1000, 37]))
        cnt = int(rng.integers(0, 10)) if trial % 2 else 0
        cases.append((head, nc, reg_max, scale, stride, CENTRE["half" if trial % 2 else "corner"], gw * stride, gh * stride, conf, cnt,
                      maxd))
    return cases


def test_c_statement_equals_numpy_restatement():
    capped = saturated = 0
    for i, (head, nc, reg_max, scale, stride, centre, net_w, net_h, conf, cnt, maxd) in enumerate(random_heads()):
        prior = np.zeros(cnt, dtype=BOX_DTYPE)
        prior["confidence"] = np.arange(cnt)
        want = c_decode_gfl(head, nc, reg_max, scale, stride, centre, net_w, net_h, conf, prior, cnt, maxd)
        got = decode_gfl(head, nc, reg_max, scale, stride, centre, net_w, net_h, conf, cnt, maxd)
        assert want[:cnt].tobytes() == prior.tobytes()
        assert len(got) == len(want) - cnt and got.tobytes() == want[cnt:].tobytes(), i
        capped += len(got) == maxd - cnt
        s = sigmoid_table(scale)[head[..., :nc].astype(np.int32) + 128]
        b = head[..., :nc]
        top = s == s.max(axis=-1, keepdims=True)  # saturated scores: the maximum score on several classes with different bytes
        saturated += bool(((top.sum(axis=-1) > 1) & (np.where(top, b, 127).min(axis=-1) != np.where(top, b, -128).max(axis=-1))).any())
    assert capped > 0 and capped < len(random_heads()) and saturated > 0


def test_known_answers():
    nc, reg_max, stride = 2, 7, 16
    nb = reg_max + 1
    C = nc + 4 * nb
    # all bins equal: every e_j = E[0] = 1, den = R + 1, dist = sum_j j * fl(1 / (R + 1)) in float32
    head = np.zeros((2, 3, C), dtype=np.int8)
    head[..., 0] = 100
    head[..., nc:] = 5
    dist = np.float32(0)
    for j in range(nb):
        dist = dist + np.float32(j) * (np.float32(1) / np.float32(nb))
    d = dist * np.float32(stride)
    for centre, off in ((CENTRE["half"], 0.5), (CENTRE["corner"], 0.0)):
        got = c_decode_gfl(head, nc, reg_max, 0.05, stride, centre, 1000, 1000, 0.25)
        assert len(got) == 6
        assert np.array_equal(decode_gfl(head, nc, reg_max, 0.05, stride, centre, 1000, 1000, 0.25), got)
        cx = (np.arange(3, dtype=np.float32) + np.float32(off)) * np.float32(stride)
        assert np.array_equal(got["x1"][:3], cx + d) and np.array_equal(got["y1"][3:], np.full(3, (np.float32(1) + np.float32(off)) * stride + d))
    # one-hot bins at scale 1.0: E[255] = expf(-255) is 0 in float32, so the distance is exactly j * stride
    head = np.full((1, 8, C), -128, dtype=np.int8)
    head[0, :, 1] = 90
    for x in range(8):
        for s, j in enumerate(((x % nb), (x + 3) % nb, 7 - x % nb, 2)):
            head[0, x, nc + s * nb + j] = 100
    got = c_decode_gfl(head, nc, reg_max, 1.0, stride, CENTRE["corner"], 4096, 4096, 0.5)
    assert np.array_equal(decode_gfl(head, nc, reg_max, 1.0, stride, CENTRE["corner"], 4096, 4096, 0.5), got)
    for x in range(8):
        l, t, r, b = (x % nb), (x + 3) % nb, 7 - x % nb, 2
        cx = x * stride
        assert got[x]["x0"] == max(cx - l * stride, 0) and got[x]["y0"] == 0
        assert got[x]["x1"] == cx + r * stride and got[x]["y1"] == b * stride
        assert got[x]["class_id"] == 1
    # a score exactly equal to conf_thresh is not a candidate; just above it is
    sig = sigmoid_table(0.05)
    head = np.zeros((1, 2, C), dtype=np.int8)
    head[0, :, 0] = 40
    thr = float(sig[40 + 128])
    assert len(c_decode_gfl(head, nc, reg_max, 0.05, stride, 0, 64, 64, thr)) == 0
    assert len(decode_gfl(head, nc, reg_max, 0.05, stride, 0, 64, 64, thr)) == 0
    assert len(c_decode_gfl(head, nc, reg_max, 0.05, stride, 0, 64, 64, float(np.nextafter(np.float32(thr), np.float32(0))))) == 2


def test_edges_match_float64_integral_and_distance2bbox():
    """NanoDet's Integral (softmax over the bins, expectation against 0..reg_max) and distance2bbox (clipped to the input) in
    float64 on the dequantised head: every box edge of every cell within 1e-3 px"""
    rng = np.random.default_rng(5)
    for trial, (nc, reg_max) in enumerate([(80, 7), (3, 7), (5, 16), (1, 3)]):
        for level in range(4):
            stride = 8 << level
            gh = gw = 640 // stride
            head = rng.integers(-128, 128, size=(gh, gw, nc + 4 * (reg_max + 1)), dtype=np.int8)
            scale = [0.02, 0.05, 0.1, 0.08][trial]
            centre = level % 2
            got = c_decode_gfl(head, nc, reg_max, scale, stride, centre, 640, 640, -1.0, maxd=gh * gw)
            assert len(got) == gh * gw  # every cell is a candidate at conf -1
            nb = reg_max + 1
            logits = head[..., nc:].astype(np.float64).reshape(gh, gw, 4, nb) * float(np.float32(scale))
            p = np.exp(logits - logits.max(axis=-1, keepdims=True))
            p /= p.sum(axis=-1, keepdims=True)
            dist = (p * np.arange(nb)).sum(axis=-1) * stride
            off = 0.5 if centre == 0 else 0.0
            yy, xx = np.meshgrid(np.arange(gh), np.arange(gw), indexing="ij")
            cx, cy = ((xx + off) * stride).ravel(), ((yy + off) * stride).ravel()
            d = dist.reshape(-1, 4)
            want = np.stack([np.clip(cx - d[:, 0], 0, 640), np.clip(cy - d[:, 1], 0, 640),
                             np.clip(cx + d[:, 2], 0, 640), np.clip(cy + d[:, 3], 0, 640)], axis=1)
            have = np.stack([got["x0"], got["y0"], got["x1"], got["y1"]], axis=1).astype(np.float64)
            assert np.abs(have - want).max() < 1e-3, (nc, reg_max, level, np.abs(have - want).max())
            scores = 1.0 / (1.0 + np.exp(-head[..., :nc].astype(np.float64).reshape(-1, nc) * float(np.float32(scale))))
            assert np.allclose(got["confidence"], scores.max(axis=1), rtol=1e-6, atol=1e-7)
