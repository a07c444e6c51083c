"""Reference composition of tiled detection (mars_b200_preprocess_rois + heads step + mars_b200_merge_rois_resident), for the
tests: the oracle heads flow of each region's crop in region coordinates (heads_ref.heads_flow with frame = the region's size),
each box shifted into its frame by one float32 add of the region's origin per coordinate, the boxes of a frame's regions
concatenated in region order, a stable descending sort by confidence, the first 1000, then the oracle's mo_nms_corner."""
import numpy as np

from heads_ref import BOX_DTYPE, heads_flow

MERGE_CAP = 1000


def region_boxes(ob, blob, letterbox, frame, roi, head_ids, size, conf, nms_thresh):
    """kept boxes of one region (region coordinates), as the region's slot holds them"""
    _, x, y, w, h = (int(v) for v in roi)
    crop = np.ascontiguousarray(frame[y: y + h, x: x + w])
    return heads_flow(ob, blob, letterbox(crop, size, size), head_ids, conf=conf, nms_thresh=nms_thresh, frame=(w, h))


def merge(ob, per_region, rois, n_frames, merge_thresh):
    """per_region[r]: kept boxes of region r -> the merged boxes of each frame"""
    out = []
    for f in range(n_frames):
        parts = []
        for r, roi in enumerate(rois):
            if int(roi[0]) != f:
                continue
            b = np.array(per_region[r], dtype=BOX_DTYPE, copy=True)
            ox, oy = np.float32(int(roi[1])), np.float32(int(roi[2]))
            b["x0"] += ox
            b["x1"] += ox
            b["y0"] += oy
            b["y1"] += oy
            parts.append(b)
        u = np.concatenate(parts) if parts else np.zeros(0, dtype=BOX_DTYPE)
        u = u[np.argsort(-u["confidence"], kind="stable")][:MERGE_CAP]
        out.append(ob.nms_corner(np.ascontiguousarray(u), merge_thresh) if u.size else u)
    return out


def union_size(per_region, rois, f):
    return sum(len(per_region[r]) for r, roi in enumerate(rois) if int(roi[0]) == f)
