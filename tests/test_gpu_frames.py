"""GPU: letterboxing batches of frames of mixed sizes and row pitches (mars_b200_preprocess_frames, the device-frame form and
mars_b200_submit_frames_heads_batch).  Every check is byte for byte: against the reference's golden hashes
(tests/golden/preproc.json), the numpy restatement of test_preproc.py, the single-frame mars_b200_letterbox, and for the
submit the oracle flow of the heads decode (heads_ref) in frame coordinates."""
import ctypes as C
import functools

import numpy as np
import pytest

from heads_ref import heads_flow
from test_preproc import PRE, frame, letterbox_numpy, sha

pytestmark = pytest.mark.gpu

# (w, h, seed): the golden 1920x1080 and 500x375 cases, then one pixel, tiny, tall, 4K, identity and one-pixel-off sizes
MIXED = [(1920, 1080, 11), (500, 375, 13), (1, 1, 31), (7, 5, 32), (333, 999, 33), (3840, 2160, 34), (640, 640, 35), (641, 639, 36)]
NHWC_EXTRA = [(1280, 720, 12)]  # the golden NHWC case


@functools.lru_cache(maxsize=None)
def blob(size, nhwc=False, width=0.125):
    from __graft_entry__ import load_package
    return load_package().marsfile.build_yolov5(width=width, size=size, seed=9, nhwc=nhwc).to_bytes()


def model(pkg, batch, size=640, nhwc=False):
    return pkg.MarsModel(blob(size, nhwc), arena_bytes=32 << 20, device=0, batch=batch)


def slot_inputs(gm, first, n):
    off = gm.tensor_offset(gm.m.contents.header.input_tensor_ids[0])
    nb = gm.input_bytes
    return [gm.arena_download(first + i)[off:off + nb].copy() for i in range(n)]


def golden(w, h, nhwc, seed, tw=640):
    for v in PRE.values():
        if v["case"] == [w, h, tw, tw, int(nhwc), seed]:
            return v["sha256"]
    return None


def check_against_references(pkg, got, cases, nhwc, tw=640):
    for i, (w, h, seed) in enumerate(cases):
        f = frame(w, h, seed)
        want = pkg.capi.letterbox(f, tw, tw, nhwc)
        assert got[i].view(np.int8).tobytes() == want.tobytes(), (w, h)
        g = golden(w, h, nhwc, seed, tw)
        if g is not None:
            assert sha(got[i]) == g, (w, h)
        elif w * h <= 1 << 20:  # the numpy restatement is slow on 4K frames; the single-frame kernel covers those
            assert got[i].view(np.int8).tobytes() == letterbox_numpy(pkg.capi, f, tw, tw, nhwc).tobytes(), (w, h)


def pitched(f, extra, rng):
    """the frame inside a buffer whose rows are w * 3 + extra bytes apart, random bytes in the padding"""
    h, w, _ = f.shape
    pitch = w * 3 + extra
    raw = rng.integers(0, 256, h * pitch, dtype=np.uint8)
    v = np.lib.stride_tricks.as_strided(raw, (h, w, 3), (pitch, 3, 1))
    v[...] = f
    return v


@pytest.mark.parametrize("nhwc", [False, True])
def test_mixed_batch_host(pkg, nhwc):
    cases = MIXED + (NHWC_EXTRA if nhwc else [])
    gm = model(pkg, len(cases) + 1, nhwc=nhwc)
    gm.preprocess_frames(1, [frame(w, h, s) for (w, h, s) in cases])  # deliberately not slot 0
    check_against_references(pkg, slot_inputs(gm, 1, len(cases)), cases, nhwc)
    gm.close()


def test_row_pitch(pkg):
    rng = np.random.default_rng(1)
    gm = model(pkg, 2 * len(MIXED))
    frames = [frame(w, h, s) for (w, h, s) in MIXED]
    gm.preprocess_frames(0, frames)
    views = [pitched(f, int(e), rng) for f, e in zip(frames, rng.integers(1, 200, len(frames)))]
    assert all(v.strides[0] != v.shape[1] * 3 for v in views)
    gm.preprocess_frames(len(MIXED), views)
    a, b = slot_inputs(gm, 0, len(MIXED)), slot_inputs(gm, len(MIXED), len(MIXED))
    for i in range(len(MIXED)):
        assert a[i].tobytes() == b[i].tobytes(), MIXED[i]
    gm.close()


def test_uniform_batch_equals_preprocess_batch(pkg):
    frames = np.stack([frame(1280, 720, 40 + i) for i in range(4)])
    gm = model(pkg, 8)
    gm.preprocess(0, frames)
    gm.preprocess_frames(4, list(frames))
    a, b = slot_inputs(gm, 0, 4), slot_inputs(gm, 4, 4)
    for i in range(4):
        assert a[i].tobytes() == b[i].tobytes(), i
    gm.close()


def test_device_frames_equal_host_frames(pkg):
    import torch
    rng = np.random.default_rng(2)
    frames = [frame(w, h, s) for (w, h, s) in MIXED]
    gm = model(pkg, 2 * len(MIXED))
    gm.preprocess_frames(0, frames)
    keep, table = [], []
    for i, f in enumerate(frames):
        h, w, _ = f.shape
        extra = 0 if i % 2 == 0 else int(rng.integers(1, 100))  # every other frame in a wider device buffer
        buf = torch.from_numpy(rng.integers(0, 256, (h, w * 3 + extra), dtype=np.uint8)).cuda()
        buf[:, : w * 3] = torch.from_numpy(f.reshape(h, w * 3)).cuda()
        keep.append(buf)
        table.append((buf.data_ptr(), w, h, 0 if extra == 0 else w * 3 + extra))
    torch.cuda.synchronize()
    gm.preprocess_frames_device(len(MIXED), table)
    a, b = slot_inputs(gm, 0, len(MIXED)), slot_inputs(gm, len(MIXED), len(MIXED))  # arena_download orders after the launches
    for i in range(len(MIXED)):
        assert a[i].tobytes() == b[i].tobytes(), MIXED[i]
    # a host address is not a device frame
    with pytest.raises(pkg.capi.MarsError) as e:
        gm.preprocess_frames_device(0, [(frames[0].ctypes.data, 1920, 1080, 0)])
    assert "frame 0" in str(e.value)
    gm.close()


def test_rejections_write_no_slot(pkg):
    import torch
    L, capi = pkg.lib(), pkg.capi
    gm = model(pkg, 4)
    good = [frame(64, 48, 1), frame(100, 37, 5)]
    gm.preprocess_frames(0, good + [frame(20, 14, 3)])
    before = slot_inputs(gm, 0, 4)
    tall = np.zeros((5000, 1, 3), np.uint8)  # 1 x 5000: the letterbox is 0 pixels wide
    on_device = [torch.from_numpy(f).cuda() for f in good + [tall]]
    torch.cuda.synchronize()

    def table(bad, device):
        if device:
            t = capi.device_frames([(d.data_ptr(), d.shape[1], d.shape[0], 0) for d in on_device])
        else:
            t, _ = capi.host_frames(good + [tall])
        if bad is not None:
            t[2] = bad
        return t

    f0 = good[0]
    cases = [
        capi.FRAME(None, 64, 48, 0),                       # NULL rgb
        capi.FRAME(f0.ctypes.data, 0, 48, 0),              # w <= 0
        capi.FRAME(f0.ctypes.data, 64, -1, 0),             # h <= 0
        capi.FRAME(f0.ctypes.data, 64, 48, 64 * 3 - 1),    # row_stride < w * 3
        None,                                              # the 1 x 5000 frame itself
    ]
    for bad in cases:
        for device, fn in ((False, L.mars_b200_preprocess_frames), (True, L.mars_b200_preprocess_frames_device)):
            assert fn(gm.m, 0, 3, table(bad, device)) != 0, (bad, device)
            assert "frame 2" in L.mars_b200_last_error().decode(), (bad, device)
    assert L.mars_b200_preprocess_frames(gm.m, 0, 3, None) != 0  # NULL table
    assert L.mars_b200_preprocess_frames_device(gm.m, 0, 3, None) != 0
    t, _keep = capi.host_frames(good)
    assert L.mars_b200_preprocess_frames(gm.m, 3, 2, t) != 0  # slots 3..4 of 4
    assert L.mars_b200_preprocess_frames(gm.m, -1, 2, t) != 0
    after = slot_inputs(gm, 0, 4)
    for i in range(4):
        assert before[i].tobytes() == after[i].tobytes(), i
    gm.close()
    # an input tensor that is not a 4-d int8 tensor
    fm = pkg.MarsModel(pkg.marsfile.build_tiny(32, f32=True).to_bytes(), device=0)
    with pytest.raises(capi.MarsError):
        fm.preprocess_frames(0, [good[0]])
    fm.close()
    # the frames submit validates the same way, and needs heads like submit_heads_batch
    hm = pkg.MarsModel(blob(320, width=0.25), device=0, batch=4)
    boxes, counts = np.zeros((2, 1000), dtype=capi.BOX_DTYPE), np.zeros(2, dtype=np.int32)
    with pytest.raises(capi.MarsError) as e:
        hm.submit_frames_heads_batch(0, good, boxes, counts)
    assert "heads" in str(e.value)
    hm.set_yolo_heads()
    with pytest.raises(capi.MarsError) as e:
        hm.submit_frames_heads_batch(0, [good[0], tall], boxes, counts)
    assert "frame 1" in str(e.value)
    hm.wait_batch(0)  # nothing was queued
    hm.close()


# size mixes of the pipelined submit, two frames per pool
MIXES = [[(1920, 1080), (640, 360)], [(1280, 720), (333, 999)], [(7, 5), (3840, 2160)],
         [(641, 639), (500, 375)], [(1920, 1080), (1920, 1080)], [(1, 1), (800, 600)]]


def test_pipelined_submit(pkg, ob):
    size, conf = 320, 0.1
    bl = blob(size, width=0.25)
    ids = pkg.capi.find_yolo_heads(bl)
    L = pkg.lib()
    rng = np.random.default_rng(7)
    # the frames in pinned host memory (nna_malloc), as a server would hold them for the upload to overlap the kernels
    total = sum(w * h * 3 for mix in MIXES for (w, h) in mix)
    ptr = L.nna_malloc(total)
    assert ptr
    pinned = np.ctypeslib.as_array((C.c_uint8 * total).from_address(ptr))
    frames, at = [], 0
    for mix in MIXES:
        fs = []
        for (w, h) in mix:
            v = pinned[at: at + w * h * 3].reshape(h, w, 3)
            v[...] = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
            fs.append(v)
            at += w * h * 3
        frames.append(fs)
    want = [[heads_flow(ob, bl, pkg.capi.letterbox(f, size, size), ids, conf=conf, frame=(f.shape[1], f.shape[0])) for f in fs]
            for fs in frames]
    assert sum(len(w) for ws in want for w in ws) > 0
    gm = pkg.MarsModel(bl, device=0, batch=4)
    gm.set_yolo_heads(None, conf)
    out = [(np.zeros((2, 1000), dtype=pkg.capi.BOX_DTYPE), np.zeros(2, dtype=np.int32)) for _ in range(2)]
    for rnd in range(2):  # the step is captured as a graph in the first round and replayed in the second
        for k, fs in enumerate(frames):
            pool = k % 2
            if k >= 2:
                gm.wait_batch(pool)
                check(out[pool], want[k - 2])
            gm.submit_frames_heads_batch(pool, fs, out[pool][0], out[pool][1], thresh=0.45)
        for k in (len(frames) - 2, len(frames) - 1):
            gm.wait_batch(k % 2)
            check(out[k % 2], want[k])
    # the same as preprocess_frames + step_heads_resident + download_boxes
    for k, fs in enumerate(frames):
        gm.preprocess_frames(0, fs)
        gm.step_heads_resident(0, 2, 0.45)
        check(gm.download_boxes(0, 2), want[k])
    gm.close()
    L.nna_free(ptr)


def check(got, want):
    boxes, counts = got
    for i, w in enumerate(want):
        assert counts[i] == len(w), "frame %d: %d boxes, the oracle flow keeps %d" % (i, counts[i], len(w))
        assert boxes[i, : len(w)].tobytes() == w.tobytes(), "frame %d" % i


def test_batch_over_the_scratch_chunk(pkg):
    """32 frames of 3840 x 2160 need 32 x 2160 x 640 x 12 bytes = 531 MB of float rows: two launches of at most 256 MiB"""
    rng = np.random.default_rng(3)
    base = rng.integers(0, 256, (2160, 3840, 3), dtype=np.uint8)
    frames = [np.roll(base, 7 * f, axis=0) for f in range(32)]
    gm = model(pkg, 32)
    gm.preprocess_frames(0, frames)
    got = slot_inputs(gm, 0, 32)
    for f in range(32):
        assert got[f].view(np.int8).tobytes() == pkg.capi.letterbox(frames[f], 640, 640).tobytes(), f
    gm.close()
