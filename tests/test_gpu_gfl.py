"""GPU: decoding NanoDet GFL head convs inside the program (mars_b200_set_gfl_heads) through every heads entry point, byte for
byte against the oracle flow (gfl_ref)."""
import ctypes as C
import functools
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from gfl_ref import MAX_CAND, c_decode_gfl, cell_scores, decode_gfl, gfl_candidates, gfl_flow, gfl_heads, thresholds
from nv12_ref import nv12_frame, nv12_to_rgb
from test_gfl_host import random_heads
from tiles_ref import merge

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZE, ARENA = 320, 16 << 20


@functools.lru_cache(maxsize=None)
def model(nhwc=False, nc=80, levels=3):
    from __graft_entry__ import load_package
    return load_package().marsfile.build_nanodet_like(size=SIZE, seed=7, nhwc=nhwc, nc=nc, levels=levels).to_bytes()


def inputs(n, seed=0):
    return np.random.default_rng(seed).integers(-128, 128, size=(n, 3 * SIZE * SIZE), dtype=np.int8)


def gfl_model(pkg, blob, batch, nc=80, centre="half", conf=0.25, arena=ARENA, opt=3, depthwise=0):
    gm = pkg.MarsModel(blob, arena_bytes=arena, device=0, batch=batch)
    gm.set_opt_level(opt)
    gm.set_depthwise_mode(depthwise)
    gm.set_gfl_heads(None, nc, 7, centre, conf)
    return gm


def step(gm, xs, steps=1):
    runs = []
    for _ in range(steps):
        gm.upload_inputs(0, len(xs), xs, xs.shape[1])  # the input lives in a work buffer later layers overwrite
        gm.step_heads_resident(0, len(xs), 0.45)
        runs.append(gm.download_boxes(0, len(xs)))
    return runs


def check(got, want):
    boxes, counts = got
    for i, w in enumerate(want):
        assert counts[i] == len(w), "image %d: %d boxes, the oracle flow keeps %d" % (i, counts[i], len(w))
        assert boxes[i, : len(w)].tobytes() == w.tobytes(), "image %d" % i


def two_buffer_arena(pkg, blob):
    """an arena in which the planner falls back to two work buffers"""
    gm = pkg.MarsModel(blob, arena_bytes=64 << 20, device=0)
    a = gm.weights_size + 2 * gm.buffer_size + gm.buffer_size // 2
    gm.close()
    return a


@pytest.mark.parametrize("nhwc,nc,levels,centre,depthwise,arena", [
    (False, 80, 3, "half", 0, ARENA),
    (True, 80, 3, "corner", 1, ARENA),
    (False, 3, 4, "corner", 1, ARENA),
    (True, 3, 4, "half", 0, ARENA),
    (False, 3, 3, "half", 1, ARENA),
    (False, 80, 3, "half", 1, "two"),
    (True, 3, 4, "corner", 1, "two"),
])
def test_bit_exact_against_the_oracle_flow(pkg, ob, nhwc, nc, levels, centre, depthwise, arena):
    blob = model(nhwc, nc, levels)
    ids = pkg.capi.find_gfl_heads(blob, nc=nc)
    assert len(ids) == levels
    if arena == "two":
        arena = two_buffer_arena(pkg, blob)
    xs = inputs(4, seed=1)
    heads = [gfl_heads(ob, blob, x, ids, arena, bool(depthwise)) for x in xs]
    capped = below = 0
    for conf in thresholds([cell_scores(h, nc) for h, _ in heads]):
        cand = [gfl_candidates(h, wh, nc, 7, centre, conf) for h, wh in heads]
        capped += sum(len(c) == MAX_CAND for c in cand)
        below += sum(len(c) < MAX_CAND for c in cand)
        want = [ob.nms_corner(c, 0.45) for c in cand]
        gm = gfl_model(pkg, blob, len(xs), nc, centre, conf, arena, depthwise=depthwise)
        if gm.num_buffers == 2:
            # two work buffers: heads share one, so each head is overwritten before the next one exists (decoded in order)
            idx = {gm.m.contents.tensors[i].desc.id: i for i in range(gm.header.num_tensors)}
            assert len({gm.tensor_offset(idx[t]) for t in ids}) < levels
        check(step(gm, xs)[0], want)
        gm.close()
    assert capped and below  # both regimes: images that hit the 1000-candidate cap and images that end below it


def test_same_results_at_every_opt_level_graph_and_submit(pkg, ob):
    blob = model()
    ids = pkg.capi.find_gfl_heads(blob)
    xs = inputs(4, seed=2)
    want = [gfl_flow(ob, blob, x, ids, arena_bytes=ARENA) for x in xs]
    assert sum(len(w) for w in want)
    for opt in (0, 1, 2, 3):
        gm = gfl_model(pkg, blob, 4, opt=opt)
        for got in step(gm, xs, steps=3):  # plain, captured, replayed
            check(got, want)
        gm.upload_inputs(0, 4, xs, xs.shape[1])
        gm.enqueue_step_heads_resident(0, 4, 0.45)
        check(gm.download_boxes(0, 4), want)
        gm.close()
    gm = gfl_model(pkg, blob, 4)
    out = [(np.zeros((2, 1000), dtype=pkg.capi.BOX_DTYPE), np.zeros(2, dtype=np.int32)) for _ in range(2)]
    for rnd in range(2):
        for pool in (0, 1):
            gm.submit_heads_batch(pool, 2, xs[2 * pool:], xs.shape[1], out[pool][0], out[pool][1])
        for pool in (0, 1):
            gm.wait_batch(pool)
            check(out[pool], want[2 * pool: 2 * pool + 2])
    gm.close()
    # without CUDA graphs (MARS_GRAPH is read once per process)
    code = ("import sys, numpy as np; sys.path.insert(0, %r); from __graft_entry__ import load_package; pkg = load_package(); "
            "xs = np.load(sys.argv[1]); gm = pkg.MarsModel(open(sys.argv[2], 'rb').read(), arena_bytes=%d, device=0, batch=4); "
            "gm.set_gfl_heads(); [(gm.upload_inputs(0, 4, xs, xs.shape[1]), gm.step_heads_resident(0, 4, 0.45)) for _ in range(3)]; "
            "b, c = gm.download_boxes(0, 4); np.save(sys.argv[3], b); np.save(sys.argv[4], c)" % (ROOT, ARENA))
    with tempfile.TemporaryDirectory() as d:
        paths = [os.path.join(d, f) for f in ("x.npy", "m.mars", "b.npy", "c.npy")]
        np.save(paths[0], xs)
        open(paths[1], "wb").write(blob)
        subprocess.run([sys.executable, "-c", code] + paths, check=True, env=dict(os.environ, MARS_GRAPH="0"))
        check((np.load(paths[2]), np.load(paths[3])), want)


def test_large_batch_equals_small_batch(pkg):
    blob = model(nc=3)
    xs = inputs(3, seed=3)
    gm = gfl_model(pkg, blob, 3, nc=3, conf=0.7)
    [(b3, c3)] = step(gm, xs)
    gm.close()
    assert c3.sum() > 0
    gm = gfl_model(pkg, blob, 600, nc=3, conf=0.7)
    [(b600, c600)] = step(gm, xs[np.arange(600) % 3])
    for i in range(600):
        assert c600[i] == c3[i % 3] and b600[i, : c600[i]].tobytes() == b3[i % 3, : c3[i % 3]].tobytes(), i
    gm.close()


FRAMES = [(1920, 1080), (1280, 720), (1280, 720), (1920, 1080)]


def frames_rgb(seed):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for (w, h) in FRAMES]


def test_frame_coordinates(pkg, ob):
    blob = model(nc=3)
    ids = pkg.capi.find_gfl_heads(blob, nc=3)
    frames = frames_rgb(5)
    gm = gfl_model(pkg, blob, len(frames), nc=3, conf=0.6)
    gm.preprocess_frames(0, frames)
    gm.step_heads_resident(0, len(frames), 0.45)
    want = [gfl_flow(ob, blob, pkg.capi.letterbox(f, SIZE, SIZE), ids, nc=3, arena_bytes=ARENA, conf=0.6, frame=(f.shape[1], f.shape[0]))
            for f in frames]
    assert all(len(w) for w in want)
    check(gm.download_boxes(0, len(frames)), want)
    gm.preprocess_frames(0, frames)  # the inputs again (the run overwrote them), then back to network coordinates
    gm.set_frame_size(0, len(frames), 0, 0)
    gm.step_heads_resident(0, len(frames), 0.45)
    want = [gfl_flow(ob, blob, pkg.capi.letterbox(f, SIZE, SIZE), ids, nc=3, arena_bytes=ARENA, conf=0.6) for f in frames]
    check(gm.download_boxes(0, len(frames)), want)
    gm.close()


def pinned_frames(L, mixes, seed):
    """NV12 frames and the RGB8 frames their conversion produces, both in pinned host memory"""
    nv_bytes = [w * h + 2 * ((w + 1) // 2) * ((h + 1) // 2) for mix in mixes for (w, h) in mix]
    total = sum(nv_bytes) + sum(w * h * 3 for mix in mixes for (w, h) in mix)
    ptr = L.nna_malloc(total)
    assert ptr
    pinned = np.ctypeslib.as_array((C.c_uint8 * total).from_address(ptr))
    nv, rgb, at, k = [], [], 0, 0
    for mix in mixes:
        fn, fr = [], []
        for (w, h) in mix:
            y0, uv0 = nv12_frame(w, h, seed + k)
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
    return ptr, nv, rgb


def test_submit_frames_rgb_and_nv12(pkg, ob):
    """both frame submits alternating two pools over two rounds (captured in the first, replayed in the second)"""
    blob = model(nc=3)
    ids = pkg.capi.find_gfl_heads(blob, nc=3)
    L = pkg.lib()
    mixes = [[(1920, 1080), (1280, 720)], [(1280, 720), (640, 360)], [(1920, 1080), (333, 500)]]
    ptr, nv, rgb = pinned_frames(L, mixes, 300)
    want = [[gfl_flow(ob, blob, pkg.capi.letterbox(f, SIZE, SIZE), ids, nc=3, arena_bytes=ARENA, conf=0.6, frame=(f.shape[1], f.shape[0]))
             for f in fs] for fs in rgb]
    assert sum(len(w) for ws in want for w in ws)
    gm = gfl_model(pkg, blob, 4, nc=3, conf=0.6)
    out = [(np.zeros((2, 1000), dtype=pkg.capi.BOX_DTYPE), np.zeros(2, dtype=np.int32)) for _ in range(2)]
    for submit, frames in ((gm.submit_frames_heads_batch, rgb), (gm.submit_frames_nv12_heads_batch, nv)):
        for rnd in range(2):
            for k, fs in enumerate(frames):
                pool = k % 2
                if k >= 2:
                    gm.wait_batch(pool)
                    check(out[pool], want[k - 2])
                out[pool][1][:] = -1
                submit(pool, fs, out[pool][0], out[pool][1], thresh=0.45)
            for k in (len(frames) - 2, len(frames) - 1):
                gm.wait_batch(k % 2)
                check(out[k % 2], want[k])
    gm.close()
    L.nna_free(ptr)


def test_submit_rois_nv12_merge(pkg, ob):
    """tiled NV12 detection: 320 x 320 tiles overlapping by 64 plus the whole frame, merged per frame, against tiles_ref.merge of
    the per-region oracle flow"""
    blob = model(nc=3)
    ids = pkg.capi.find_gfl_heads(blob, nc=3)
    L = pkg.lib()
    mixes = [[(700, 500), (640, 360)], [(333, 500), (900, 200)]]
    ptr, nv, rgb = pinned_frames(L, mixes, 400)
    rois = [np.concatenate([pkg.capi.tile_rois(w, h, SIZE, SIZE, 64, 64, with_full=True, frame=f) for f, (w, h) in enumerate(mix)])
            for mix in mixes]
    want = []
    for fs, rs in zip(rgb, rois):
        per_region = []
        for (f, x, y, w, h) in (tuple(int(v) for v in r) for r in rs):
            crop = np.ascontiguousarray(fs[f][y: y + h, x: x + w])
            per_region.append(gfl_flow(ob, blob, pkg.capi.letterbox(crop, SIZE, SIZE), ids, nc=3, arena_bytes=ARENA, conf=0.6, frame=(w, h)))
        want.append(merge(ob, per_region, rs, 2, 0.5))
    assert sum(len(w) for ws in want for w in ws)
    half = max(len(r) for r in rois)
    gm = gfl_model(pkg, blob, 2 * half, nc=3, conf=0.6)
    out = [(np.zeros((2, 1000), dtype=pkg.capi.BOX_DTYPE), np.zeros(2, dtype=np.int32)) for _ in range(2)]
    for rnd in range(2):
        for b in range(len(mixes)):
            out[b][1][:] = -1
            gm.submit_rois_nv12_heads_batch(b, nv[b], rois[b], out[b][0], out[b][1], thresh=0.45, merge_thresh=0.5)
        for b in range(len(mixes)):
            gm.wait_batch(b)
            check(out[b], want[b])
    gm.close()
    L.nna_free(ptr)


def test_decode_gfl_matches_the_c_statement(pkg):
    for i, (head, nc, reg_max, scale, stride, centre, net_w, net_h, conf, cnt, maxd) in enumerate(random_heads()):
        prior = np.zeros(cnt, dtype=pkg.capi.BOX_DTYPE)
        prior["confidence"] = np.arange(cnt)
        want = c_decode_gfl(head, nc, reg_max, scale, stride, centre, net_w, net_h, conf, prior, cnt, maxd)
        got = pkg.capi.decode_gfl(head, nc, reg_max, scale, stride, net_w, net_h, conf, centre, prior, cnt, maxd)
        assert got.tobytes() == want.tobytes(), i
        assert got[cnt:].tobytes() == decode_gfl(head, nc, reg_max, scale, stride, centre, net_w, net_h, conf, cnt, maxd).tobytes()


def test_no_side_effects_when_configured(pkg, ob):
    """output tensors and (opt <= 2) the whole arena equal the oracle with GFL heads configured; step_resident's output0
    detections are unchanged (on the YOLOv5 graph, whose three heads are also GFL heads with nc = 223)"""
    blob, n = model(), 2
    xs = inputs(n, seed=4)
    for opt in (0, 1, 2, 3):
        plain = pkg.MarsModel(blob, arena_bytes=ARENA, device=0, batch=n)
        heads = pkg.MarsModel(blob, arena_bytes=ARENA, device=0, batch=n)
        heads.set_gfl_heads()
        for gm in (plain, heads):
            gm.set_opt_level(opt)
            gm.upload_inputs(0, n, xs, xs.shape[1])
            gm.step_resident(0, n, 0.45, False)  # output0 of the NanoDet graph is not a [1, N, 85] head: no detect
        outs, pouts = heads.download_outputs(0, n), plain.download_outputs(0, n)
        for i in range(n):
            om = ob.OracleModel(blob, arena_bytes=ARENA)
            om.set_input(xs[i])
            om.run()
            assert np.array_equal(outs[i], om.output_bytes()) and np.array_equal(pouts[i], outs[i]), (opt, i)
            if opt <= 2:
                got = heads.arena_download(i)
                assert np.array_equal(got, om.arena()[: got.size]), (opt, i)
            om.close()
        plain.close()
        heads.close()
    yb = pkg.marsfile.build_yolov5(width=0.25, size=320, seed=9).to_bytes()
    yids = pkg.capi.find_yolo_heads(yb)
    ys = np.random.default_rng(7).integers(-128, 128, size=(n, 3 * 320 * 320), dtype=np.int8)
    plain = pkg.MarsModel(yb, device=0, batch=n)
    heads = pkg.MarsModel(yb, device=0, batch=n)
    heads.set_gfl_heads(yids, nc=223, reg_max=7)
    for gm in (plain, heads):
        gm.upload_inputs(0, n, ys, ys.shape[1])
        gm.step_resident(0, n, 0.45, True)
    d0, c0 = plain.download_detections(0, n)
    d1, c1 = heads.download_detections(0, n)
    assert np.array_equal(c0, c1) and d0.tobytes() == d1.tobytes()
    plain.close()
    heads.close()


def test_describe_and_switching_kinds(pkg, ob):
    blob = model()
    gm = pkg.MarsModel(blob, arena_bytes=ARENA, device=0)
    before = gm.describe()
    gm.set_gfl_heads(enable=False)
    assert gm.describe() == before
    gm.set_gfl_heads(centre="corner", conf_thresh=0.5)
    text = gm.describe()
    lines = [l for l in text.splitlines() if "gfl_head" in l]
    assert len(lines) == 3 and "yolo_head" not in text
    assert "level 2 stride 32 nc 80 reg_max 7 nchw centre corner conf 0.5" in lines[2]
    gm.set_gfl_heads(enable=False)
    assert gm.describe() == before
    gm.close()
    # a YOLOv5 graph's three 255-channel heads are also GFL heads with nc = 223, reg_max = 7: YOLO -> GFL -> off on one model
    yb = pkg.marsfile.build_yolov5(width=0.25, size=320, seed=9).to_bytes()
    yids = pkg.capi.find_yolo_heads(yb)
    xs = np.random.default_rng(6).integers(-128, 128, size=(2, 3 * 320 * 320), dtype=np.int8)
    gm = pkg.MarsModel(yb, device=0, batch=2)
    before = gm.describe()
    gm.set_yolo_heads()
    assert gm.describe().count("yolo_head") == 3
    yolo = step(gm, xs)[0]
    gm.set_gfl_heads(yids, nc=223, reg_max=7, conf_thresh=0.3)
    text = gm.describe()
    assert text.count("gfl_head") == 3 and "yolo_head" not in text
    want = [gfl_flow(ob, yb, x, yids, nc=223, conf=0.3) for x in xs]
    assert sum(len(w) for w in want)
    check(step(gm, xs)[0], want)
    gm.set_gfl_heads(yids, nc=223, reg_max=7, conf_thresh=0.3)  # unchanged: nothing recompiles
    check(step(gm, xs)[0], want)
    gm.set_yolo_heads()
    r = step(gm, xs)[0]
    assert np.array_equal(r[1], yolo[1]) and r[0].tobytes() == yolo[0].tobytes()
    gm.set_gfl_heads(enable=False)  # n = 0 on either setter switches decoding off
    assert gm.describe() == before
    with pytest.raises(pkg.capi.MarsError) as e:
        gm.step_heads_resident(0, 1)
    assert e.value.code == -7 and "no detection heads configured" in str(e.value)
    gm.close()


def test_set_gfl_heads_rejections(pkg):
    mf = pkg.marsfile
    m = mf.build_nanodet_like(size=SIZE, seed=7, levels=4)
    blob = m.to_bytes()
    ids = pkg.capi.find_gfl_heads(blob)
    gm = pkg.MarsModel(blob, arena_bytes=ARENA, device=0)
    conv_out = next(L.outputs[0] for L in m.layers if L.type == 0 and L.outputs[0] not in ids)
    cases = [([m.inputs[0], ids[1], ids[2]], {}, "not the output of a CONV2D layer"),
             ([conv_out, ids[1], ids[2]], {}, "channels"),
             (ids[:3], dict(nc=79), "channels"),
             ([ids[1], ids[0], ids[2]], {}, "level order"),
             ([ids[0], ids[1], ids[3]], {}, "level 2 needs stride 32"),
             (ids[:2], {}, "heads given"),
             (ids + ids[:1], {}, "heads given"),
             (ids[:3], dict(nc=0), "nc = 0"),
             (ids[:3], dict(reg_max=0), "reg_max = 0"),
             (ids[:3], dict(reg_max=17), "reg_max = 17"),
             (ids[:3], dict(centre=2), "centre = 2"),
             (ids[:3], dict(conf_thresh=float("nan")), "not finite"),
             (None, dict(nc=3), "no GFL head convolutions"),
             (None, dict(reg_max=0), "reg_max = 0")]
    for bad, kw, text in cases:
        with pytest.raises(pkg.capi.MarsError) as e:
            gm.set_gfl_heads(bad, **kw)
        assert e.value.code == -7 and text in str(e.value), (bad, kw, str(e.value))
    assert "yolo_head" not in gm.describe() and "gfl_head" not in gm.describe()  # a rejected call changes nothing
    with pytest.raises(pkg.capi.MarsError) as e:
        gm.step_heads_resident(0, 1)
    assert e.value.code == -7
    gm.close()
    for t, field, value, text in ((ids[1], "scale", 0.0, "scale"), (ids[1], "scale", float("inf"), "scale"),
                                  (ids[2], "dtype", 0, "int8"), (ids[0], "shape", [112, 40, 40], "int8")):
        mm = mf.build_nanodet_like(size=SIZE, seed=7, levels=4)
        setattr(mm.tensors[t], field, value)
        gm = pkg.MarsModel(mm.to_bytes(), arena_bytes=ARENA, device=0)
        with pytest.raises(pkg.capi.MarsError) as e:
            gm.set_gfl_heads(ids)
        assert e.value.code == -7 and text in str(e.value) and "head" in str(e.value), (field, str(e.value))
        gm.close()
