"""GPU: decoding the three YOLOv5 head convs inside the program (mars_b200_set_yolo_heads) against the oracle flow (heads_ref)."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from heads_ref import heads_flow

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@functools.lru_cache(maxsize=None)
def model(width, size, nhwc=False, nc=80):
    from __graft_entry__ import load_package
    return load_package().marsfile.build_yolov5(width=width, size=size, seed=9, nhwc=nhwc, nc=nc).to_bytes()


def inputs(size, n, seed=0):
    return np.random.default_rng(seed).integers(-128, 128, size=(n, 3 * size * size), dtype=np.int8)


def gpu_boxes(pkg, blob, xs, arena, conf=0.25, opt=3, steps=1):
    gm = pkg.MarsModel(blob, arena_bytes=arena, device=0, batch=len(xs))
    gm.set_opt_level(opt)
    gm.set_yolo_heads(None, conf)
    runs = []
    for _ in range(steps):
        # the input tensor lives in a work buffer that later layers overwrite: like the reference's caller, write it before every run
        gm.upload_inputs(0, len(xs), xs, xs.shape[1])
        gm.step_heads_resident(0, len(xs), 0.45)
        runs.append(gm.download_boxes(0, len(xs)))
    return gm, runs


def check(boxes, counts, want):
    for i, w in enumerate(want):
        assert counts[i] == len(w), "image %d: %d boxes, the oracle flow keeps %d" % (i, counts[i], len(w))
        assert boxes[i, : len(w)].tobytes() == w.tobytes(), "image %d" % i


def two_buffer_arena(pkg, blob):
    """an arena in which the planner falls back to two work buffers, as the reference's 8 MiB does for the shipped yolov5n"""
    gm = pkg.MarsModel(blob, arena_bytes=64 << 20, device=0)
    a = gm.weights_size + 2 * gm.buffer_size + gm.buffer_size // 2
    gm.close()
    return a


@pytest.mark.parametrize("width,size,arena,nhwc,nc,conf", [
    (0.25, 640, 8 << 20, False, 80, 0.25),
    (0.25, 640, "two", False, 80, 0.25),
    (0.25, 640, "two", False, 80, 0.6),
    (0.25, 640, 64 << 20, False, 80, 0.25),
    (0.5, 320, 32 << 20, False, 80, 0.25),
    (0.25, 320, 8 << 20, True, 80, 0.25),
    (0.25, 320, 8 << 20, False, 3, 0.25),
])
def test_bit_exact_against_the_oracle_flow(pkg, ob, width, size, arena, nhwc, nc, conf):
    blob = model(width, size, nhwc, nc)
    ids = pkg.capi.find_yolo_heads(blob)
    xs = inputs(size, 4, seed=1)
    two = arena == "two"
    if two:
        arena = two_buffer_arena(pkg, blob)
    gm, [(boxes, counts)] = gpu_boxes(pkg, blob, xs, arena, conf)
    if two:
        # two work buffers: the heads share one, so each head is overwritten before the next one exists (decoded in order)
        idx = {gm.m.contents.tensors[i].desc.id: i for i in range(gm.header.num_tensors)}
        assert gm.num_buffers == 2
        assert len({gm.tensor_offset(idx[t]) for t in ids}) < 3
    check(boxes, counts, [heads_flow(ob, blob, x, ids, arena, conf) for x in xs])
    gm.close()


def test_frame_coordinates(pkg, ob):
    blob, size = model(0.25, 320), 320
    ids = pkg.capi.find_yolo_heads(blob)
    frames = np.random.default_rng(5).integers(0, 256, size=(2, 1080, 1920, 3), dtype=np.uint8)
    gm = pkg.MarsModel(blob, device=0, batch=3)
    gm.set_yolo_heads(None, 0.1)
    gm.preprocess(0, frames)
    gm.step_heads_resident(0, 2, 0.45)
    boxes, counts = gm.download_boxes(0, 2)
    for i in range(2):
        x = pkg.capi.letterbox(frames[i], size, size)
        want = heads_flow(ob, blob, x, ids, conf=0.1, frame=(1920, 1080))
        assert len(want) and counts[i] == len(want)
        assert boxes[i, : len(want)].tobytes() == want.tobytes()
    gm.preprocess(0, frames)  # the inputs again (the run overwrote them), then back to network coordinates
    gm.set_frame_size(0, 2, 0, 0)
    gm.step_heads_resident(0, 2, 0.45)
    boxes, counts = gm.download_boxes(0, 2)
    want = heads_flow(ob, blob, pkg.capi.letterbox(frames[0], size, size), ids, conf=0.1)
    assert counts[0] == len(want) and boxes[0, : len(want)].tobytes() == want.tobytes()
    gm.close()


def test_same_results_at_every_opt_level_graph_and_submit(pkg, ob):
    blob, size = model(0.25, 320), 320
    ids = pkg.capi.find_yolo_heads(blob)
    xs = inputs(size, 4, seed=2)
    want = [heads_flow(ob, blob, x, ids) for x in xs]
    for opt in (0, 1, 2, 3):
        gm, runs = gpu_boxes(pkg, blob, xs, 8 << 20, opt=opt, steps=3)  # plain, captured, replayed
        for boxes, counts in runs:
            check(boxes, counts, want)
        # the enqueue-only form and the asynchronous batch path
        gm.upload_inputs(0, 4, xs, xs.shape[1])
        gm.enqueue_step_heads_resident(0, 4, 0.45)
        boxes, counts = gm.download_boxes(0, 4)
        check(boxes, counts, want)
        gm.close()
    gm = pkg.MarsModel(blob, device=0, batch=4)
    gm.set_yolo_heads()
    out = [(np.zeros((2, 1000), dtype=pkg.capi.BOX_DTYPE), np.zeros(2, dtype=np.int32)) for _ in range(2)]
    for rnd in range(2):
        for pool in (0, 1):
            gm.submit_heads_batch(pool, 2, xs[2 * pool:], xs.shape[1], out[pool][0], out[pool][1])
        for pool in (0, 1):
            gm.wait_batch(pool)
            check(out[pool][0], out[pool][1], want[2 * pool: 2 * pool + 2])
    gm.close()
    # without CUDA graphs (MARS_GRAPH is read once per process)
    code = ("import sys, numpy as np; sys.path.insert(0, %r); from __graft_entry__ import load_package; pkg = load_package(); "
            "xs = np.load(sys.argv[1]); gm = pkg.MarsModel(open(sys.argv[2], 'rb').read(), device=0, batch=4); gm.set_yolo_heads(); "
            "[(gm.upload_inputs(0, 4, xs, xs.shape[1]), gm.step_heads_resident(0, 4, 0.45)) for _ in range(3)]; "
            "b, c = gm.download_boxes(0, 4); np.save(sys.argv[3], b); np.save(sys.argv[4], c)" % ROOT)
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        paths = [os.path.join(d, f) for f in ("x.npy", "m.mars", "b.npy", "c.npy")]
        np.save(paths[0], xs)
        open(paths[1], "wb").write(blob)
        subprocess.run([sys.executable, "-c", code] + paths, check=True, env=dict(os.environ, MARS_GRAPH="0"))
        check(np.load(paths[2]), np.load(paths[3]), want)


def test_large_batch_equals_small_batch(pkg):
    blob, size = model(0.25, 320), 320
    xs = inputs(size, 3, seed=3)
    _, [(b3, c3)] = gpu_boxes(pkg, blob, xs, 8 << 20)
    big = xs[np.arange(600) % 3]
    gm, [(b600, c600)] = gpu_boxes(pkg, blob, big, 8 << 20)
    for i in range(600):
        assert c600[i] == c3[i % 3] and b600[i, : c600[i]].tobytes() == b3[i % 3, : c3[i % 3]].tobytes(), i
    gm.close()


def test_no_side_effects_when_configured(pkg, ob):
    blob, size, n = model(0.25, 320), 320, 2
    xs = inputs(size, n, seed=4)
    for opt in (0, 1, 2, 3):
        plain = pkg.MarsModel(blob, device=0, batch=n)
        heads = pkg.MarsModel(blob, device=0, batch=n)
        heads.set_yolo_heads()
        for gm in (plain, heads):
            gm.set_opt_level(opt)
            gm.upload_inputs(0, n, xs, xs.shape[1])
            gm.step_resident(0, n, 0.45, True)
        d0, c0 = plain.download_detections(0, n)
        d1, c1 = heads.download_detections(0, n)
        assert np.array_equal(c0, c1) and d0.tobytes() == d1.tobytes()
        outs = heads.download_outputs(0, n)
        for i in range(n):
            om = ob.OracleModel(blob)
            om.set_input(xs[i])
            om.run()
            assert np.array_equal(outs[i], om.output_bytes()), (opt, i)
            if opt <= 2:
                got = heads.arena_download(i)
                assert np.array_equal(got, om.arena()[: got.size]), (opt, i)
            om.close()
        plain.close()
        heads.close()


def test_describe_unchanged_when_not_configured(pkg):
    blob = model(0.25, 320)
    gm = pkg.MarsModel(blob, device=0)
    before = gm.describe()
    gm.set_yolo_heads(enable=False)
    assert gm.describe() == before
    gm.set_yolo_heads()
    text = gm.describe()
    assert text.count("yolo_head") == 3 and "level 2 stride 32 nc 80 nchw" in text
    gm.set_yolo_heads(enable=False)
    assert gm.describe() == before
    gm.close()


def test_set_yolo_heads_rejections(pkg):
    mf = pkg.marsfile
    m = mf.build_yolov5(width=0.25, size=320, seed=9)
    blob = m.to_bytes()
    ids = pkg.capi.find_yolo_heads(blob)
    gm = pkg.MarsModel(blob, device=0)
    conv_out = next(L.outputs[0] for L in m.layers if L.type == 0 and L.outputs[0] not in ids)
    cases = [([m.inputs[0], ids[1], ids[2]], "not the output of a CONV2D layer"),
             ([conv_out, ids[1], ids[2]], "channels"),
             ([ids[2], ids[1], ids[0]], "level order"),
             (ids[:2], "heads given")]
    for bad, text in cases:
        with pytest.raises(pkg.capi.MarsError) as e:
            gm.set_yolo_heads(bad)
        assert e.value.code == -7 and text in str(e.value), (bad, str(e.value))
    with pytest.raises(pkg.capi.MarsError) as e:
        gm.step_heads_resident(0, 1)
    assert e.value.code == -7
    gm.close()
    m.tensors[ids[1]].scale = 0.0
    gm = pkg.MarsModel(m.to_bytes(), device=0)
    with pytest.raises(pkg.capi.MarsError) as e:
        gm.set_yolo_heads()
    assert e.value.code == -7 and "scale" in str(e.value)
    gm.close()
    gm = pkg.MarsModel(mf.build_tiny(160).to_bytes(), device=0)
    with pytest.raises(pkg.capi.MarsError) as e:
        gm.set_yolo_heads()
    assert e.value.code == -7 and "no YOLOv5 Detect head" in str(e.value)
    gm.close()
