"""Reference flow of the NanoDet GFL heads decode (mars_b200_set_gfl_heads), for the tests.

c_decode_gfl runs the C statement of the decode (tests/gfl_oracle.c, compiled with -ffp-contract=off into a temporary directory
on first use); decode_gfl restates it in numpy float32, one rounding per operation, on a head laid out [gh, gw, nc + 4 (reg_max + 1)].  gfl_flow follows heads_ref.heads_flow: the oracle runs the model layer by layer, the
bytes of each head conv are copied right after that conv, each head is decoded with the 1000-candidate cap chained over the levels,
then the oracle's mo_nms_corner and, for a frame size, mo_scale_detections.
"""
import ctypes as C
import ctypes.util
import os
import subprocess
import tempfile

import numpy as np

from heads_ref import BOX_DTYPE, FMT_NHWC, LAYER_CONV2D, MAX_CAND, Desc, sigmoid_table

CENTRE = {"half": 0, "corner": 1}
_expf = None
_clib = None


def c_decode_gfl(head, nc, reg_max, scale, stride, centre, net_w, net_h, conf_thresh, dets=None, cnt=0, maxd=MAX_CAND):
    """the C statement (tests/gfl_oracle.c) on one [gh, gw, C] head: boxes appended after dets[:cnt], returns [:count]"""
    global _clib
    if _clib is None:
        src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "gfl_oracle.c")
        so = os.path.join(tempfile.mkdtemp(prefix="gfl_oracle_"), "libgfl_oracle.so")
        subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-o", so, src, "-lm"], check=True)
        _clib = C.CDLL(so)
        _clib.gfl_decode.restype = C.c_int
        _clib.gfl_decode.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_float, C.c_void_p, C.c_int, C.c_int]
    gh, gw, _ = head.shape
    out = np.zeros(maxd, dtype=BOX_DTYPE)
    if cnt:
        out[:cnt] = dets[:cnt]
    h = np.ascontiguousarray(head, dtype=np.int8)
    n = _clib.gfl_decode(h.ctypes.data, gh, gw, nc, reg_max, scale, stride, centre, net_w, net_h, conf_thresh, out.ctypes.data, cnt, maxd)
    return out[:n].copy()


def exp_table(scale):
    """E[d] = expf(-(d * scale)) for d = 0..255 with the host libm's expf"""
    global _expf
    if _expf is None:
        _expf = C.CDLL(ctypes.util.find_library("m")).expf
        _expf.restype, _expf.argtypes = C.c_float, [C.c_float]
    s = np.float32(scale)
    return np.array([_expf(float(-(np.float32(d) * s))) for d in range(256)], dtype=np.float32)


def decode_gfl(head, nc, reg_max, scale, stride, centre, net_w, net_h, conf_thresh, cnt=0, maxd=MAX_CAND):
    """head: int8 [gh, gw, nc + 4 (reg_max + 1)] -> corner boxes in (y, x) order, at most maxd - cnt of them"""
    gh, gw, ch = head.shape
    nb = reg_max + 1
    assert ch == nc + 4 * nb
    sig, E = sigmoid_table(scale), exp_table(scale)
    p = head.reshape(-1, ch).astype(np.int32)
    scores = sig[p[:, :nc] + 128]
    score = scores.max(axis=1)
    label = scores.argmax(axis=1)  # the first class with the maximum score (floats compared)
    keep = np.nonzero(score > np.float32(conf_thresh))[0][: max(maxd - cnt, 0)]
    q = p[keep]
    fs = np.float32(stride)
    dist = []
    for s in range(4):
        v = q[:, nc + s * nb: nc + (s + 1) * nb]
        e = E[v.max(axis=1, keepdims=True) - v]
        den = e[:, 0].copy()
        for j in range(1, nb):
            den = den + e[:, j]
        acc = np.zeros(keep.size, dtype=np.float32)
        for j in range(nb):
            acc = acc + np.float32(j) * (e[:, j] / den)
        dist.append(acc * fs)
    off = np.float32(0.5 if centre == CENTRE["half"] else 0.0)
    cx = ((keep % gw).astype(np.float32) + off) * fs
    cy = ((keep // gw).astype(np.float32) + off) * fs
    d = np.zeros(keep.size, dtype=BOX_DTYPE)
    d["x0"] = np.maximum(cx - dist[0], np.float32(0))
    d["y0"] = np.maximum(cy - dist[1], np.float32(0))
    d["x1"] = np.minimum(cx + dist[2], np.float32(net_w))
    d["y1"] = np.minimum(cy + dist[3], np.float32(net_h))
    d["confidence"], d["class_id"] = score[keep], label[keep]
    return d


def head_to_hwc(raw, desc):
    """bytes of a head conv output -> int8 [gh, gw, C]"""
    v = np.asarray(raw).view(np.int8)
    if desc.format == FMT_NHWC:
        _, gh, gw, c = desc.shape[:4]
        return v.reshape(gh, gw, c)
    _, c, gh, gw = desc.shape[:4]
    return np.ascontiguousarray(v.reshape(c, gh, gw).transpose(1, 2, 0))


def gfl_heads(ob, blob, x, head_ids, arena_bytes=8 << 20, depthwise=False):
    """the oracle's bytes of each head conv right after it ran, its descriptor, and the network input size (w, h)"""
    om = ob.OracleModel(blob, arena_bytes=arena_bytes, depthwise=depthwise)
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
            desc = Desc(int(d.format), [int(v) for v in d.shape[: d.ndims]], float(d.scale))
            off, n = om.tensor_offset(t), int(np.prod([max(v, 0) for v in desc.shape]))
            heads[out] = (head_to_hwc(om.arena()[off: off + n].copy(), desc), desc)
    net = om.tensor_desc(om.input_index())
    net_wh = (int(net.shape[2]), int(net.shape[1])) if net.format == FMT_NHWC else (int(net.shape[3]), int(net.shape[2]))
    om.close()
    return [heads[h] for h in head_ids], net_wh


def gfl_candidates(heads, net_wh, nc=80, reg_max=7, centre="half", conf=0.25):
    cand = np.zeros(0, dtype=BOX_DTYPE)
    for level, (g, d) in enumerate(heads):
        cand = np.concatenate([cand, decode_gfl(g, nc, reg_max, d.scale, 8 << level, CENTRE[centre], net_wh[0], net_wh[1], conf,
                                                cand.size)])
    return cand


def gfl_flow(ob, blob, x, head_ids, nc=80, reg_max=7, centre="half", arena_bytes=8 << 20, conf=0.25, nms_thresh=0.45, frame=None,
             depthwise=False):
    """kept corner boxes of one image (frame = (w, h): in frame coordinates)"""
    heads, net_wh = gfl_heads(ob, blob, x, head_ids, arena_bytes, depthwise)
    kept = ob.nms_corner(gfl_candidates(heads, net_wh, nc, reg_max, centre, conf), nms_thresh)
    if frame is not None and kept.size:
        kept = np.ascontiguousarray(kept)
        ob.lib().mo_scale_detections(kept.ctypes.data, kept.size, frame[0], frame[1], net_wh[0], net_wh[1])
    return kept


def cell_scores(heads, nc):
    """the score (maximum class sigmoid) of every cell of every level, in candidate order"""
    return np.concatenate([sigmoid_table(d.scale)[g[..., :nc].astype(np.int32) + 128].max(axis=-1).ravel() for g, d in heads])


def thresholds(scores, cap=MAX_CAND):
    """confidence thresholds from the candidate counts of a set of images (scores: each image's cell_scores) under which some
    images hit the cap and some end below it: one threshold that splits the images when there is one with a candidate on
    both sides, else one at which every image hits the cap and one at which none does"""
    vals = np.unique(np.concatenate(scores))
    srt = [np.sort(s) for s in scores]
    counts = np.stack([s.size - np.searchsorted(s, vals, side="right") for s in srt], axis=1)  # [value, image]: #(score > value)
    split = np.nonzero((counts.max(axis=1) >= cap) & (counts.min(axis=1) < cap) & (counts.min(axis=1) > 0))[0]
    if split.size:
        return [float(vals[split[0]])]
    return [float(vals[np.nonzero(counts.min(axis=1) >= cap)[0][-1]]), float(vals[np.nonzero(counts.max(axis=1) < cap)[0][0]])]
