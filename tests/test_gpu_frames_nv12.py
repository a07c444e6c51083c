"""GPU: letterboxing NV12 frames (mars_b200_preprocess_frames_nv12, the device-frame form and
mars_b200_submit_frames_nv12_heads_batch).  The contract: an NV12 frame letterboxes to a slot tensor byte-identical to that
of the RGB8 frame the conversion of nv12_ref gives, letterboxed by mars_b200_letterbox -- the RGB chain is the oracle."""
import ctypes as C

import numpy as np
import pytest

from heads_ref import heads_flow
from nv12_ref import nv12_frame, nv12_to_rgb
from test_gpu_frames import MIXED, blob, check, pitched, slot_inputs
from test_preproc import letterbox_numpy

pytestmark = pytest.mark.gpu


def model(pkg, batch, size=640, nhwc=False):
    return pkg.MarsModel(blob(size, nhwc), arena_bytes=32 << 20, device=0, batch=batch)


def frames_of(cases):
    """(y, uv, colour) per case; the colour variants interleave"""
    return [nv12_frame(w, h, s) + (i % 4,) for i, (w, h, s) in enumerate(cases)]


def check_against_rgb(pkg, got, frames, nhwc, tw=640):
    for i, (y, uv, colour) in enumerate(frames):
        rgb = nv12_to_rgb(y, uv, colour)
        want = pkg.capi.letterbox(rgb, tw, tw, nhwc)
        assert got[i].view(np.int8).tobytes() == want.tobytes(), (y.shape, colour)
        if y.size <= 1 << 20:
            assert got[i].view(np.int8).tobytes() == letterbox_numpy(pkg.capi, rgb, tw, tw, nhwc).tobytes(), (y.shape, colour)


def padded(plane, extra, rng):
    """a [h, w] or [h, w, 2] plane inside a buffer whose rows are `extra` bytes wider, random bytes in the padding"""
    plane = np.ascontiguousarray(plane)
    h, row = plane.shape[0], plane[0].size
    raw = rng.integers(0, 256, (h, row + extra), dtype=np.uint8)
    raw[:, :row] = plane.reshape(h, row)
    # explicit strides: a reshape would give a one-row plane its tight row stride back
    return np.lib.stride_tricks.as_strided(raw, plane.shape, (row + extra,) + plane.strides[1:])


def nvdec_surface(y, uv, pitch=2048):
    """one allocation as a hardware decoder lays it out: luma rows `pitch` apart, the chroma plane at pitch * align(h, 16)"""
    h, w = y.shape
    at = pitch * ((h + 15) // 16 * 16)
    buf = np.full(at + pitch * uv.shape[0], 77, np.uint8)
    buf[:at].reshape(-1, pitch)[:h, :w] = y
    buf[at:].reshape(-1, pitch)[:, :uv.shape[1] * 2] = uv.reshape(uv.shape[0], -1)
    return buf, at


@pytest.mark.parametrize("nhwc", [False, True])
def test_mixed_batch_host(pkg, nhwc):
    frames = frames_of(MIXED)
    assert {c for _, _, c in frames} == {0, 1, 2, 3}
    gm = model(pkg, len(frames) + 1, nhwc=nhwc)
    gm.preprocess_frames_nv12(1, frames)  # deliberately not slot 0
    check_against_rgb(pkg, slot_inputs(gm, 1, len(frames)), frames, nhwc)
    gm.close()


def test_every_variant_on_every_size(pkg):
    gm = model(pkg, 4 * len(MIXED))
    frames = [nv12_frame(w, h, s) + (c,) for c in range(4) for (w, h, s) in MIXED]
    gm.preprocess_frames_nv12(0, frames)
    check_against_rgb(pkg, slot_inputs(gm, 0, len(frames)), frames, False)
    gm.close()


def test_pitches_and_plane_placement(pkg):
    """padded plane rows and an NVDEC-like single allocation give the slots of the tight frames, which equal the converted
    RGB8 frames letterboxed by mars_b200_preprocess_frames from row-padded buffers"""
    rng = np.random.default_rng(1)
    frames = frames_of(MIXED)
    n = len(MIXED)
    gm = model(pkg, 4 * n)
    gm.preprocess_frames_nv12(0, frames)
    views = [(padded(y, int(rng.integers(1, 200)), rng), padded(uv, int(rng.integers(1, 200)), rng), c) for (y, uv, c) in frames]
    for (y, uv, _) in views:
        assert y.strides[0] != y.shape[1] and uv.strides[0] != uv.shape[1] * 2
    gm.preprocess_frames_nv12(n, views)
    # one host allocation per frame as a decoder lays it out (pitch 2048; the 4K frame gets pitch 4096)
    surfaces, table = [], (pkg.capi.NV12_FRAME * n)()
    for i, (y, uv, c) in enumerate(frames):
        pitch = 2048 if y.shape[1] <= 2048 else 4096
        buf, at = nvdec_surface(y, uv, pitch)
        surfaces.append(buf)
        table[i] = pkg.capi.NV12_FRAME(buf.ctypes.data, buf.ctypes.data + at, y.shape[1], y.shape[0], pitch, pitch, c)
    gm._check(pkg.lib().mars_b200_preprocess_frames_nv12(gm.m, 2 * n, n, table), "preprocess_frames_nv12")
    gm.preprocess_frames(3 * n, [pitched(nv12_to_rgb(y, uv, c), int(rng.integers(1, 200)), rng) for (y, uv, c) in frames])
    tight, padd, surf, rgb = (slot_inputs(gm, k * n, n) for k in range(4))
    for i in range(n):
        assert tight[i].tobytes() == padd[i].tobytes() == surf[i].tobytes() == rgb[i].tobytes(), MIXED[i]
    gm.close()


def test_device_frames_equal_host_frames(pkg):
    import torch
    rng = np.random.default_rng(2)
    frames = frames_of(MIXED)
    n = len(MIXED)
    gm = model(pkg, 2 * n + 1)
    gm.preprocess_frames_nv12(0, frames)
    keep, table = [], []
    for i, (y, uv, c) in enumerate(frames):
        h, w = y.shape
        ey, euv = (0, 0) if i % 2 == 0 else (int(rng.integers(1, 100)), int(rng.integers(1, 100)))  # every other frame padded
        dy = torch.from_numpy(np.pad(y, ((0, 0), (0, ey)), constant_values=5)).cuda()
        duv = torch.from_numpy(np.pad(uv.reshape(uv.shape[0], -1), ((0, 0), (0, euv)), constant_values=9)).cuda()
        keep += [dy, duv]
        table.append((dy.data_ptr(), duv.data_ptr(), w, h, w + ey if ey else 0, uv.shape[1] * 2 + euv if euv else 0, c))
    # the NVDEC-like surface of the first frame: one device allocation, chroma at pitch * align(h, 16)
    y, uv, c = frames[0]
    buf, at = nvdec_surface(y, uv)
    dbuf = torch.from_numpy(buf).cuda()
    table.append((dbuf.data_ptr(), dbuf.data_ptr() + at, y.shape[1], y.shape[0], 2048, 2048, c))
    torch.cuda.synchronize()
    gm.preprocess_frames_nv12_device(n, table)
    a, b = slot_inputs(gm, 0, n), slot_inputs(gm, n, n + 1)  # arena_download orders after the launches
    for i in range(n):
        assert a[i].tobytes() == b[i].tobytes(), MIXED[i]
    assert a[0].tobytes() == b[n].tobytes()
    # a host address is not a device frame, in either plane
    for bad in ((y.ctypes.data, dbuf.data_ptr() + at), (dbuf.data_ptr(), uv.ctypes.data)):
        with pytest.raises(pkg.capi.MarsError) as e:
            gm.preprocess_frames_nv12_device(0, [table[1], (bad[0], bad[1], y.shape[1], y.shape[0], 2048, 2048, c)])
        assert "frame 1" in str(e.value)
    gm.close()


def test_rejections_write_no_slot(pkg):
    import torch
    L, capi = pkg.lib(), pkg.capi
    gm = model(pkg, 4)
    good = [nv12_frame(64, 48, 1) + (0,), nv12_frame(101, 37, 5) + (3,)]
    gm.preprocess_frames_nv12(0, good + [nv12_frame(20, 14, 3) + (1,)])
    before = slot_inputs(gm, 0, 4)
    tall = nv12_frame(1, 5000, 4) + (0,)  # 1 x 5000: the letterbox is 0 pixels wide
    dev = [(torch.from_numpy(y).cuda(), torch.from_numpy(np.ascontiguousarray(uv)).cuda()) for (y, uv, _) in good + [tall]]
    torch.cuda.synchronize()

    def table(bad, device):
        if device:
            t = capi.device_nv12_frames([(dy.data_ptr(), duv.data_ptr(), dy.shape[1], dy.shape[0], 0, 0, f[2])
                                         for (dy, duv), f in zip(dev, good + [tall])])
        else:
            t, _ = capi.host_nv12_frames(good + [tall])
        if bad is not None:
            t[2] = bad(t[0])
        return t

    def with_(**kw):
        def f(base):
            v = {k: getattr(base, k) for k, _ in capi.NV12_FRAME._fields_}
            v.update(kw)
            return capi.NV12_FRAME(**v)
        return f

    cases = [
        with_(y=None),                       # NULL y
        with_(uv=None),                      # NULL uv
        with_(w=0),                          # w <= 0
        with_(h=-1),                         # h <= 0
        with_(y_stride=63),                  # y_stride < w
        with_(uv_stride=63),                 # uv_stride < 2 * ceil(w / 2)
        with_(colour=4),                     # not a variant
        with_(colour=-1),
        None,                                # the 1 x 5000 frame itself
    ]
    for bad in cases:
        for device, fn in ((False, L.mars_b200_preprocess_frames_nv12), (True, L.mars_b200_preprocess_frames_nv12_device)):
            assert fn(gm.m, 0, 3, table(bad, device)) != 0, device
            assert "frame 2" in L.mars_b200_last_error().decode(), (device, L.mars_b200_last_error())
    assert L.mars_b200_preprocess_frames_nv12(gm.m, 0, 3, None) != 0  # NULL table
    assert L.mars_b200_preprocess_frames_nv12_device(gm.m, 0, 3, None) != 0
    t, _keep = capi.host_nv12_frames(good)
    assert L.mars_b200_preprocess_frames_nv12(gm.m, 3, 2, t) != 0  # slots 3..4 of 4
    after = slot_inputs(gm, 0, 4)
    for i in range(4):
        assert before[i].tobytes() == after[i].tobytes(), i
    gm.close()
    # the submit validates the same way, and needs heads like submit_frames_heads_batch
    hm = pkg.MarsModel(blob(320, width=0.25), device=0, batch=6)
    boxes, counts = np.zeros((3, 1000), dtype=capi.BOX_DTYPE), np.zeros(3, dtype=np.int32)
    with pytest.raises(capi.MarsError) as e:
        hm.submit_frames_nv12_heads_batch(0, good, boxes, counts)
    assert "heads" in str(e.value)
    hm.set_yolo_heads()
    for bad in cases:
        t, _k = capi.host_nv12_frames(good + [tall])
        if bad is not None:
            t[2] = bad(t[0])
        assert L.mars_b200_submit_frames_nv12_heads_batch(hm.m, 0, 3, t, boxes.ctypes.data, counts.ctypes.data, 1000, 0.45) != 0
        assert "frame 2" in L.mars_b200_last_error().decode()
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
    # the frames in pinned host memory (nna_malloc): each frame's luma plane, then its chroma plane
    nbytes = [w * h + 2 * ((w + 1) // 2) * ((h + 1) // 2) for mix in MIXES for (w, h) in mix]
    ptr = L.nna_malloc(sum(nbytes))
    assert ptr
    pinned = np.ctypeslib.as_array((C.c_uint8 * sum(nbytes)).from_address(ptr))
    frames, at, k = [], 0, 0
    for mix in MIXES:
        fs = []
        for (w, h) in mix:
            y0, uv0 = nv12_frame(w, h, 100 + k)
            y = pinned[at: at + w * h].reshape(h, w)
            uv = pinned[at + w * h: at + nbytes[k]].reshape(uv0.shape)
            y[...], uv[...] = y0, uv0
            fs.append((y, uv, k % 4))
            at += nbytes[k]
            k += 1
        frames.append(fs)
    want = [[heads_flow(ob, bl, pkg.capi.letterbox(nv12_to_rgb(y, uv, c), size, size), ids, conf=conf, frame=(y.shape[1], y.shape[0]))
             for (y, uv, c) in fs] for fs in frames]
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
            gm.submit_frames_nv12_heads_batch(pool, fs, out[pool][0], out[pool][1], thresh=0.45)
        for k in (len(frames) - 2, len(frames) - 1):
            gm.wait_batch(k % 2)
            check(out[k % 2], want[k])
    # the same as preprocess_frames_nv12 + step_heads_resident + download_boxes
    for k, fs in enumerate(frames):
        gm.preprocess_frames_nv12(0, fs)
        gm.step_heads_resident(0, 2, 0.45)
        check(gm.download_boxes(0, 2), want[k])
    gm.close()
    L.nna_free(ptr)


def test_batch_over_the_scratch_chunk(pkg):
    """32 NV12 frames of 3840 x 2160: 531 MB of float rows, two launches of at most 256 MiB, staged launch by launch"""
    y0, uv0 = nv12_frame(3840, 2160, 3)
    frames = [(np.roll(y0, 7 * f, axis=0), np.roll(uv0, 3 * f, axis=0), f % 4) for f in range(32)]
    gm = model(pkg, 32)
    gm.preprocess_frames_nv12(0, frames)
    got = slot_inputs(gm, 0, 32)
    for f, (y, uv, c) in enumerate(frames):
        assert got[f].view(np.int8).tobytes() == pkg.capi.letterbox(nv12_to_rgb(y, uv, c), 640, 640).tobytes(), f
    gm.close()
