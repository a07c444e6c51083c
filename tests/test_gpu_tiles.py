"""GPU: tiled detection -- regions of frames letterboxed into slots (mars_b200_preprocess_rois, the NV12 device form) and their
boxes merged per frame (mars_b200_merge_rois_resident, mars_b200_submit_rois[_nv12]_heads_batch).  Every check is byte for
byte: a region's slot against mars_b200_letterbox of the cropped frame, the merge against the oracle composition of
tiles_ref."""
import ctypes as C

import numpy as np
import pytest

from nv12_ref import nv12_frame, nv12_to_rgb
from test_gpu_frames import blob, check, pitched, slot_inputs
from test_preproc import frame
from tiles_ref import merge, region_boxes, union_size

pytestmark = pytest.mark.gpu


def model(pkg, batch, size=640, nhwc=False):
    return pkg.MarsModel(blob(size, nhwc), arena_bytes=32 << 20, device=0, batch=batch)


def regions_of(W, H, f, rng, k=3):
    """whole frame, 1 x 1 regions in two corners, regions touching each edge, and k random ones at odd origins"""
    out = [(f, 0, 0, W, H), (f, W - 1, H - 1, 1, 1), (f, 0, 0, min(W, 641), min(H, 639))]
    if W > 2 and H > 2:
        out += [(f, 1, 1, 1, 1), (f, W - (W - 1) // 2, H - (H - 1) // 2, (W - 1) // 2, (H - 1) // 2), (f, 1, H // 3, W - 1, H - H // 3)]
    for _ in range(k):
        x, y = int(rng.integers(0, W)) | 1, int(rng.integers(0, H)) | 1
        if x < W and y < H:
            out.append((f, x, y, int(rng.integers(1, W - x + 1)), int(rng.integers(1, H - y + 1))))
    return out


def fits(pkg, roi, tw=640):
    """regions whose letterbox is at least one pixel wide and tall (the others are rejected, test_rejections)"""
    w, h = roi[3], roi[4]
    s = min(tw / w, tw / h)
    return int(np.float32(w) * np.float32(s)) > 0 and int(np.float32(h) * np.float32(s)) > 0


def check_regions(pkg, got, frames_rgb, rois, nhwc, tw=640):
    for r, (f, x, y, w, h) in enumerate(rois):
        want = pkg.capi.letterbox(frames_rgb[f][y: y + h, x: x + w], tw, tw, nhwc)
        assert got[r].view(np.int8).tobytes() == want.tobytes(), (r, (f, x, y, w, h))


@pytest.mark.parametrize("nhwc", [False, True])
def test_rgb_region_slots(pkg, nhwc):
    rng = np.random.default_rng(4)
    sizes = [(3840, 2160, 34), (1920, 1080, 11), (333, 999, 33), (7, 5, 32), (641, 639, 36)]
    frames = [frame(w, h, s) for (w, h, s) in sizes]
    frames[1] = pitched(frames[1], 77, rng)  # a padded row pitch
    assert frames[1].strides[0] != 1920 * 3
    rois = []
    for f, (w, h, _) in enumerate(sizes):
        if f == 2:
            continue  # a frame without regions between two with regions
        rois += [r for r in regions_of(w, h, f, rng) if fits(pkg, r)]
    gm = model(pkg, len(rois) + len(sizes) + 1, nhwc=nhwc)
    gm.preprocess_rois(1, frames, rois)  # deliberately not slot 0
    check_regions(pkg, slot_inputs(gm, 1, len(rois)), frames, rois, nhwc)
    # a whole-frame region's slot is the slot preprocess_frames writes for the frame
    base = len(rois) + 1
    gm.preprocess_frames(base, frames)
    whole = slot_inputs(gm, base, len(frames))
    got = slot_inputs(gm, 1, len(rois))
    with_whole = set()
    for r, (f, x, y, w, h) in enumerate(rois):
        if (x, y, w, h) == (0, 0, sizes[f][0], sizes[f][1]):
            assert got[r].tobytes() == whole[f].tobytes(), r
            with_whole.add(f)
    assert with_whole == {0, 1, 3, 4}
    gm.close()


def test_nv12_device_regions(pkg):
    import torch
    rng = np.random.default_rng(5)
    sizes = [(1920, 1080), (333, 999), (641, 639), (7, 5)]
    frames = [nv12_frame(w, h, 50 + i) + (i % 4,) for i, (w, h) in enumerate(sizes)]
    rgb = [nv12_to_rgb(y, uv, c) for (y, uv, c) in frames]
    rois = [r for f, (w, h) in enumerate(sizes) for r in regions_of(w, h, f, rng) if fits(pkg, r)]
    assert any(r[1] % 2 and r[2] % 2 for r in rois)
    keep, table = [], []
    for i, (y, uv, c) in enumerate(frames):
        h, w = y.shape
        ey = 0 if i % 2 == 0 else 13  # every other frame with padded planes
        dy = torch.from_numpy(np.pad(y, ((0, 0), (0, ey)), constant_values=5)).cuda()
        duv = torch.from_numpy(np.pad(uv.reshape(uv.shape[0], -1), ((0, 0), (0, ey)), constant_values=9)).cuda()
        keep += [dy, duv]
        table.append((dy.data_ptr(), duv.data_ptr(), w, h, w + ey, uv.shape[1] * 2 + ey, c))
    torch.cuda.synchronize()
    assert {c for (_, _, c) in frames} == {0, 1, 2, 3}
    gm = model(pkg, len(rois))
    gm.preprocess_rois_nv12_device(0, table, rois)
    check_regions(pkg, slot_inputs(gm, 0, len(rois)), rgb, rois, False)
    gm.close()


def test_rejections_write_no_slot(pkg):
    import torch
    L, capi = pkg.lib(), pkg.capi
    gm = model(pkg, 4)
    good = [frame(64, 48, 1), frame(20, 5000, 5)]
    ok = [(0, 0, 0, 64, 48), (0, 3, 5, 7, 9), (1, 0, 0, 20, 5000)]
    gm.preprocess_rois(0, good, ok + [(1, 1, 1, 3, 3)])
    before = slot_inputs(gm, 0, 4)
    nv = [nv12_frame(64, 48, 1), nv12_frame(20, 5000, 5)]
    dev = [(torch.from_numpy(y).cuda(), torch.from_numpy(np.ascontiguousarray(uv)).cuda()) for (y, uv) in nv]
    torch.cuda.synchronize()
    dtable = capi.device_nv12_frames([(dy.data_ptr(), duv.data_ptr(), dy.shape[1], dy.shape[0], 0, 0, 0) for (dy, duv) in dev])
    htable, _keep = capi.host_frames(good)
    cases = [
        (2, 0, 0, 1, 1),        # frame outside [0, n_frames)
        (-1, 0, 0, 1, 1),
        (0, 0, 0, 4, 4),        # frame index decreasing after region 2 (frame 1)
        (1, -1, 0, 4, 4),       # x < 0
        (1, 0, -1, 4, 4),       # y < 0
        (1, 0, 0, 0, 4),        # w <= 0
        (1, 0, 0, 4, -2),       # h <= 0
        (1, 17, 0, 4, 4),       # past the right edge
        (1, 0, 4997, 4, 4),     # past the bottom edge
        (1, 0, 0, 1, 5000),     # the letterbox of a 1 x 5000 region is 0 pixels wide
    ]
    for bad in cases:
        r = capi.roi_table(ok + [bad])
        for fn, t in ((L.mars_b200_preprocess_rois, htable), (L.mars_b200_preprocess_rois_nv12_device, dtable)):
            assert fn(gm.m, 0, 2, t, 4, r.ctypes.data) != 0, bad
            assert "region 3" in L.mars_b200_last_error().decode(), (bad, L.mars_b200_last_error())
    # more regions than slots in range: the first one past the capacity is named
    r = capi.roi_table(ok + [(1, 0, 0, 4, 4)] * 2)
    assert L.mars_b200_preprocess_rois(gm.m, 0, 2, htable, 5, r.ctypes.data) != 0
    assert "region 4" in L.mars_b200_last_error().decode()
    assert L.mars_b200_preprocess_rois(gm.m, 1, 2, htable, 4, r.ctypes.data) != 0
    assert "region 3" in L.mars_b200_last_error().decode()
    # a frame check fails: the frame is named
    bad_frames, _k = capi.host_frames(good)
    bad_frames[1] = capi.FRAME(None, 20, 5000, 0)
    assert L.mars_b200_preprocess_rois(gm.m, 0, 2, bad_frames, 3, capi.roi_table(ok).ctypes.data) != 0
    assert "frame 1" in L.mars_b200_last_error().decode()
    assert L.mars_b200_preprocess_rois(gm.m, 0, 2, htable, 3, None) != 0  # NULL region table
    after = slot_inputs(gm, 0, 4)
    for i in range(4):
        assert before[i].tobytes() == after[i].tobytes(), i
    # the merge checks its regions the same way (no frame sizes there)
    for bad in cases[:7]:
        r = capi.roi_table(ok + [bad])
        assert L.mars_b200_merge_rois_resident(gm.m, 0, 2, 4, r.ctypes.data, 0.45) != 0, bad
        assert "region 3" in L.mars_b200_last_error().decode()
    gm.close()
    # the submit validates the same way, and needs heads
    hm = pkg.MarsModel(blob(320, width=0.25), device=0, batch=8)
    boxes, counts = np.zeros((2, 1000), dtype=capi.BOX_DTYPE), np.zeros(2, dtype=np.int32)
    with pytest.raises(capi.MarsError) as e:
        hm.submit_rois_heads_batch(0, good, ok, boxes, counts)
    assert "heads" in str(e.value)
    hm.set_yolo_heads()
    for bad in cases:
        r = capi.roi_table(ok + [bad])
        assert L.mars_b200_submit_rois_heads_batch(hm.m, 0, 2, htable, 4, r.ctypes.data, boxes.ctypes.data, counts.ctypes.data, 1000,
                                                   0.45, 0.45) != 0, bad
        assert "region 3" in L.mars_b200_last_error().decode()
        hm.wait_batch(0)  # nothing was queued
    r = capi.roi_table(ok * 2)  # 6 regions: more than half of 8 slots
    assert L.mars_b200_submit_rois_heads_batch(hm.m, 0, 2, htable, 6, r.ctypes.data, boxes.ctypes.data, counts.ctypes.data, 1000, 0.45,
                                               0.45) != 0
    hm.close()


SIZE, CONF = 320, 0.05


def tiled(pkg, shapes, with_full=True):
    """320 x 320 tiles overlapping by 64 (and the whole frame) of each frame, frames in order"""
    return np.concatenate([pkg.capi.tile_rois(w, h, SIZE, SIZE, 64, 64, with_full=with_full, frame=f) for f, (w, h) in enumerate(shapes)])


def oracle(pkg, ob, bl, ids, frames_rgb, rois, nms_thresh, merge_thresh):
    per_region = [region_boxes(ob, bl, pkg.capi.letterbox, frames_rgb[int(r[0])], r, ids, SIZE, CONF, nms_thresh) for r in rois]
    return per_region, merge(ob, per_region, rois, len(frames_rgb), merge_thresh)


@pytest.mark.parametrize("nms_thresh,merge_thresh", [(0.45, 0.45), (1.5, 0.6)])
def test_merge_resident(pkg, ob, nms_thresh, merge_thresh):
    """nms_thresh 1.5 keeps every candidate of a region, so the union of a frame passes the cap of 1000 and the synthetic
    weights' tied confidences exercise the tie order of the cut"""
    bl = blob(SIZE, width=0.25)
    ids = pkg.capi.find_yolo_heads(bl)
    shapes = [(700, 500), (1000, 400)]
    frames = [frame(w, h, 60 + i) for i, (w, h) in enumerate(shapes)]
    rois = tiled(pkg, shapes)
    per_region, want = oracle(pkg, ob, bl, ids, frames, rois, nms_thresh, merge_thresh)
    assert sum(len(w) for w in want) > 0
    if nms_thresh > 1:
        assert union_size(per_region, rois, 1) > 1000, union_size(per_region, rois, 1)
    gm = pkg.MarsModel(bl, device=0, batch=len(rois) + 1)
    gm.set_yolo_heads(None, CONF)
    gm.preprocess_rois(1, frames, rois)
    gm.step_heads_resident(1, len(rois), nms_thresh)
    gm.merge_rois_resident(1, len(frames), rois, merge_thresh)
    check(gm.download_frame_boxes(1, len(frames)), want)
    check(gm.download_boxes(1, len(rois)), per_region)  # the slots keep their boxes in region coordinates
    gm.close()


def test_submit_rgb_and_nv12(pkg, ob):
    """both submits from pinned frames, alternating the two pools over two rounds (the step is captured as a graph in the first
    and replayed in the second), against the oracle composition and the resident path"""
    bl = blob(SIZE, width=0.25)
    ids = pkg.capi.find_yolo_heads(bl)
    L = pkg.lib()
    mixes = [[(600, 400), (400, 300)], [(333, 500), (640, 360)], [(321, 321), (900, 200)]]
    nv_bytes = [w * h + 2 * ((w + 1) // 2) * ((h + 1) // 2) for mix in mixes for (w, h) in mix]
    rgb_bytes = [w * h * 3 for mix in mixes for (w, h) in mix]
    ptr = L.nna_malloc(sum(nv_bytes) + sum(rgb_bytes))
    assert ptr
    pinned = np.ctypeslib.as_array((C.c_uint8 * (sum(nv_bytes) + sum(rgb_bytes))).from_address(ptr))
    nv, rgb, at, k = [], [], 0, 0
    for mix in mixes:
        fn, fr = [], []
        for (w, h) in mix:
            y0, uv0 = nv12_frame(w, h, 200 + k)
            y = pinned[at: at + w * h].reshape(h, w)
            uv = pinned[at + w * h: at + nv_bytes[k]].reshape(uv0.shape)
            y[...], uv[...] = y0, uv0
            at += nv_bytes[k]
            v = pinned[at: at + w * h * 3].reshape(h, w, 3)
            v[...] = nv12_to_rgb(y0, uv0, k % 4)
            at += w * h * 3
            fn.append((y, uv, k % 4))
            fr.append(v)
            k += 1
        nv.append(fn)
        rgb.append(fr)
    rois = [tiled(pkg, mix) for mix in mixes]
    want = [oracle(pkg, ob, bl, ids, rgb[b], rois[b], 0.45, 0.5)[1] for b in range(len(mixes))]
    assert sum(len(w) for ws in want for w in ws) > 0
    half = max(len(r) for r in rois)
    gm = pkg.MarsModel(bl, device=0, batch=2 * half)
    gm.set_yolo_heads(None, CONF)
    out = [(np.zeros((2, 1000), dtype=pkg.capi.BOX_DTYPE), np.zeros(2, dtype=np.int32)) for _ in range(2)]
    for submit, frames in ((gm.submit_rois_heads_batch, rgb), (gm.submit_rois_nv12_heads_batch, nv)):
        for rnd in range(2):
            for b in range(len(mixes)):
                pool = b % 2
                if b >= 2:
                    gm.wait_batch(pool)
                    check(out[pool], want[b - 2])
                out[pool][1][:] = -1
                submit(pool, frames[b], rois[b], out[pool][0], out[pool][1], thresh=0.45, merge_thresh=0.5)
            for b in (len(mixes) - 2, len(mixes) - 1):
                gm.wait_batch(b % 2)
                check(out[b % 2], want[b])
    # the resident path gives the same
    for b in range(len(mixes)):
        gm.preprocess_rois(0, rgb[b], rois[b])
        gm.step_heads_resident(0, len(rois[b]), 0.45)
        gm.merge_rois_resident(0, 2, rois[b], 0.5)
        check(gm.download_frame_boxes(0, 2), want[b])
    gm.close()
    L.nna_free(ptr)
