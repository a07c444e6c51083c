"""Reference flow of the YOLOv5 heads decode (mars_b200_set_yolo_heads), for the tests.

The oracle runs the model layer by layer and the bytes of each head conv are copied right after that conv (later layers may
overwrite them through the planner's round-robin buffers).  Each head is permuted to [3, gh, gw, 5 + nc] and decoded with the
arithmetic of the oracle's mo_decode_anchor_grid (oracle/mars_oracle.c), restated here in numpy float32 with the class count as a
parameter; the 1000-candidate cap is chained across the three levels.  Then the oracle's mo_nms_corner and, for a frame size,
mo_scale_detections.
"""
import collections
import ctypes as C
import ctypes.util

import numpy as np

BOX_DTYPE = np.dtype([("x0", "<f4"), ("y0", "<f4"), ("x1", "<f4"), ("y1", "<f4"), ("confidence", "<f4"), ("class_id", "<i4")])
ANCHORS = np.array([[10, 13, 16, 30, 33, 23], [30, 61, 62, 45, 59, 119], [116, 90, 156, 198, 373, 326]], dtype=np.float32)
STRIDES = (8, 16, 32)
MAX_CAND = 1000
FMT_NHWC = 7
LAYER_CONV2D = 0

Desc = collections.namedtuple("Desc", "format shape scale")
_expf = None


def sigmoid_table(scale):
    """1 / (1 + expf(-(v * scale))) for v = -128..127 with the host libm's expf, one float32 rounding per operation"""
    global _expf
    if _expf is None:
        _expf = C.CDLL(ctypes.util.find_library("m")).expf
        _expf.restype, _expf.argtypes = C.c_float, [C.c_float]
    s = np.float32(scale)
    out = np.zeros(256, dtype=np.float32)
    for v in range(-128, 128):
        x = np.float32(v) * s
        e = np.float32(_expf(float(-x)))
        out[v + 128] = np.float32(1.0) / (np.float32(1.0) + e)
    return out


def decode_anchor_grid_nc(head, scale, level, conf_thresh, nc, cnt=0, maxd=MAX_CAND):
    """head: int8 [3, gh, gw, 5 + nc] -> corner boxes in (anchor, y, x) order, at most maxd - cnt of them"""
    _, gh, gw, no = head.shape
    assert no == 5 + nc
    sig = sigmoid_table(scale)
    conf_t = np.float32(conf_thresh)
    p = head.reshape(-1, no).astype(np.int32)
    obj = sig[p[:, 4] + 128]
    cls = p[:, 5:]
    best = cls.argmax(axis=1)  # first maximum
    bv = cls.max(axis=1)
    conf = obj * sig[bv + 128]
    keep = np.nonzero(~(obj < conf_t) & ~(conf < conf_t))[0][: max(maxd - cnt, 0)]
    a, rem = keep // (gh * gw), keep % (gh * gw)
    y, x = (rem // gw).astype(np.float32), (rem % gw).astype(np.float32)
    q = p[keep]
    two, half, stride = np.float32(2.0), np.float32(0.5), np.float32(STRIDES[level])
    cx = ((sig[q[:, 0] + 128] * two - half) + x) * stride
    cy = ((sig[q[:, 1] + 128] * two - half) + y) * stride
    tw, th = sig[q[:, 2] + 128] * two, sig[q[:, 3] + 128] * two
    w = (tw * tw) * ANCHORS[level][2 * a]
    h = (th * th) * ANCHORS[level][2 * a + 1]
    hw, hh = w / two, h / two
    d = np.zeros(keep.size, dtype=BOX_DTYPE)
    d["x0"], d["y0"], d["x1"], d["y1"] = cx - hw, cy - hh, cx + hw, cy + hh
    d["confidence"], d["class_id"] = conf[keep], best[keep]
    return d


def head_to_grid(raw, desc):
    """bytes of a head conv output -> int8 [3, gh, gw, 5 + nc]"""
    v = np.asarray(raw).view(np.int8)
    if desc.format == FMT_NHWC:
        _, gh, gw, c = desc.shape[:4]
        return np.ascontiguousarray(v.reshape(gh, gw, 3, c // 3).transpose(2, 0, 1, 3))
    _, c, gh, gw = desc.shape[:4]
    return np.ascontiguousarray(v.reshape(3, c // 3, gh, gw).transpose(0, 2, 3, 1))


def heads_flow(ob, blob, x, head_ids, arena_bytes=8 << 20, conf=0.25, nms_thresh=0.45, frame=None):
    """kept corner boxes of one image (frame = (w, h): in frame coordinates)"""
    om = ob.OracleModel(blob, arena_bytes=arena_bytes)
    index = {om.tensor_desc(i).id: i for i in range(om.num_tensors)}
    om.set_input(x)
    heads = {}
    for li in range(om.num_layers):
        assert om.run_layer(li) == 0
        L = om.layer_desc(li)
        out = L.output_tensor_ids[0]
        if L.type == LAYER_CONV2D and out in head_ids:
            t = index[out]
            d = om.tensor_desc(t)
            desc = Desc(int(d.format), [int(v) for v in d.shape[: d.ndims]], float(d.scale))  # the oracle's table dies with it
            off, n = om.tensor_offset(t), int(np.prod([max(v, 0) for v in desc.shape]))
            heads[out] = (om.arena()[off: off + n].copy(), desc)
    net = om.tensor_desc(om.input_index())
    net_w, net_h = (int(net.shape[2]), int(net.shape[1])) if net.format == FMT_NHWC else (int(net.shape[3]), int(net.shape[2]))
    om.close()
    cand = np.zeros(0, dtype=BOX_DTYPE)
    for level, hid in enumerate(head_ids):
        raw, d = heads[hid]
        g = head_to_grid(raw, d)
        cand = np.concatenate([cand, decode_anchor_grid_nc(g, d.scale, level, conf, g.shape[3] - 5, cand.size)])
    kept = ob.nms_corner(cand, nms_thresh)
    if frame is not None and kept.size:
        kept = np.ascontiguousarray(kept)
        ob.lib().mo_scale_detections(kept.ctypes.data, kept.size, frame[0], frame[1], net_w, net_h)
    return kept
