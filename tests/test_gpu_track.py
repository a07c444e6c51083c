"""GPU: the multi-object tracker (k_track, mars_b200_set_tracking) through every entry point, byte for byte against the C statement
(track_ref.OracleTracker)."""
import functools

import numpy as np
import pytest

from nv12_ref import nv12_frame, nv12_to_rgb
from track_ref import BOX_DTYPE, OracleTracker, params

pytestmark = pytest.mark.gpu

YOLO_SIZE, GFL_SIZE = 320, 320


@functools.lru_cache(maxsize=None)
def yolo_blob():
    from __graft_entry__ import load_package
    return load_package().marsfile.build_yolov5(width=0.25, size=YOLO_SIZE, seed=9).to_bytes()


@functools.lru_cache(maxsize=None)
def gfl_blob():
    from __graft_entry__ import load_package
    return load_package().marsfile.build_nanodet_like(size=GFL_SIZE, seed=7).to_bytes()


def heads_model(pkg, kind, batch):
    if kind == "yolo":
        gm = pkg.MarsModel(yolo_blob(), arena_bytes=8 << 20, device=0, batch=batch)
        gm.set_yolo_heads(None, 0.25)
    else:
        gm = pkg.MarsModel(gfl_blob(), arena_bytes=16 << 20, device=0, batch=batch)
        gm.set_gfl_heads(None, 80, 7, "half", 0.25)
    return gm


def host_model(pkg, n_streams, p=None):
    """the tracker alone needs no heads: any model serves mars_b200_track_boxes"""
    gm = pkg.MarsModel(yolo_blob(), arena_bytes=8 << 20, device=0)
    gm.set_tracking(n_streams, **({} if p is None else {f: getattr(p, f) for f, _ in p._fields_}))
    return gm


def check(got, counts, want, what):
    for i, w in enumerate(want):
        assert counts[i] == len(w), "%s entry %d: %d tracks, the oracle has %d" % (what, i, counts[i], len(w))
        assert got[i, : len(w)].tobytes() == w.tobytes(), "%s entry %d" % (what, i)


# ---- detection sequences -------------------------------------------------------------------------------------------------------
def random_frames(seed, frames, n_obj, ties=False, size=640.0):
    """per frame a BOX_DTYPE array: n_obj objects on random walks (overlapping freely), each detected with probability 0.85 at a
    random confidence in (0.05, 1), plus clutter, a few degenerate or non-finite boxes, classes 0..2, shuffled.  ties: coordinates on
    an 8 px grid, confidences from {0.3, 0.7, 0.9} and duplicated boxes, so that equal similarities are everywhere."""
    rng = np.random.default_rng(seed)
    pos = rng.uniform(0, size, (n_obj, 2))
    wh = rng.uniform(20, 120, (n_obj, 2))
    vel = rng.normal(0, 4, (n_obj, 2))
    cls = rng.integers(0, 3, n_obj)
    out = []
    for _ in range(frames):
        vel += rng.normal(0, 0.5, vel.shape)
        pos += vel
        rows = []
        for k in range(n_obj):
            if rng.random() < 0.85:
                x, y = pos[k] + rng.normal(0, 2, 2)
                c = float(rng.choice([0.3, 0.7, 0.9])) if ties else float(rng.uniform(0.05, 1.0))
                b = (x, y, x + wh[k, 0], y + wh[k, 1], c, int(cls[k]))
                if ties:
                    b = tuple(np.round(np.array(b[:4]) / 8) * 8) + b[4:]
                rows.append(b)
                if ties and rng.random() < 0.3:
                    rows.append(b)
        for _ in range(int(rng.integers(0, 4))):
            x, y = rng.uniform(0, size, 2)
            rows.append((x, y, x + rng.uniform(10, 60), y + rng.uniform(10, 60), float(rng.uniform(0.05, 1.0)), int(rng.integers(0, 3))))
        if rng.random() < 0.2:
            rows.append((5.0, 5.0, 5.0, 40.0, 0.9, 0))
            rows.append((float("nan"), 5.0, 30.0, 40.0, 0.9, 0))
        order = rng.permutation(len(rows))
        out.append(np.array([rows[i] for i in order], dtype=BOX_DTYPE))
    return out


def run_host(gm, oracle, seqs, calls):
    """calls: per call the list of streams it names; each names the next frame of its streams"""
    nxt = {}
    for c, streams in enumerate(calls):
        boxes = []
        for s in streams:
            boxes.append(seqs[s][nxt.get(s, 0)])
            nxt[s] = nxt.get(s, 0) + 1
        got, counts = gm.track_boxes(streams, boxes)
        want = [oracle.step(s, b) for s, b in zip(streams, boxes)]
        check(got, counts, want, "call %d" % c)


@pytest.mark.parametrize("ties,class_aware", [(False, 0), (True, 0), (False, 1), (True, 1)])
def test_track_boxes_equal_the_oracle(pkg, ties, class_aware):
    S, frames = 256, 60
    p = params(class_aware=class_aware)
    seqs = [random_frames(1000 * ties + s, frames + 20, int(np.random.default_rng(s).integers(1, 40)), ties) for s in range(S)]
    gm, oracle = host_model(pkg, S, p), OracleTracker(S, p)
    calls = [list(range(S))] * frames
    rng = np.random.default_rng(5)
    for _ in range(20):  # calls naming different subsets of the streams, in shuffled order
        calls.append([int(v) for v in rng.permutation(S)[: int(rng.integers(1, S))]])
    run_host(gm, oracle, seqs, calls)
    gm.close()


def crowded(seed, frames):
    """1000 detections per frame: a 40 x 25 grid of boxes (every one of them a birth candidate on frame 1, so 256 tracks live from
    then on), jittered from frame to frame, with half of them duplicated on later frames"""
    rng = np.random.default_rng(seed)
    gx, gy = np.meshgrid(np.arange(40) * 24.0, np.arange(25) * 24.0)
    base = np.stack([gx.ravel(), gy.ravel()], axis=1)
    out = []
    for f in range(frames):
        xy = base + rng.normal(0, 2, base.shape)
        b = np.zeros(1000, dtype=BOX_DTYPE)
        b["x0"], b["y0"], b["x1"], b["y1"] = xy[:, 0], xy[:, 1], xy[:, 0] + 30, xy[:, 1] + 30
        b["confidence"] = rng.choice([0.3, 0.7, 0.9], 1000)
        if f > 0:
            b[500:] = b[rng.permutation(500)]
        out.append(b)
    return out


def test_crowded_frames(pkg):
    S, frames = 3, 5
    seqs = [crowded(s, frames) for s in range(S)]
    gm, oracle = host_model(pkg, S), OracleTracker(S)
    run_host(gm, oracle, seqs, [list(range(S))] * frames)
    gm.close()


def test_reset_resize_and_rejections(pkg):
    S = 8
    seqs = [random_frames(s, 40, 6) for s in range(S)]
    gm, oracle = host_model(pkg, S), OracleTracker(S)
    run_host(gm, oracle, seqs, [list(range(S))] * 5)
    pos = {s: 5 for s in range(S)}

    def step(streams):
        boxes = [seqs[s][pos[s]] for s in streams]
        for s in streams:
            pos[s] += 1
        got, counts = gm.track_boxes(streams, boxes)
        check(got, counts, [oracle.step(s, b) for s, b in zip(streams, boxes)], "after rejections")

    b = [seqs[0][0]]
    L = pkg.lib()
    for streams, boxes in (([S], b), ([-1], b), ([1, 1], b * 2), ([0], [np.zeros(1001, dtype=BOX_DTYPE)])):
        with pytest.raises(pkg.capi.MarsError, match="track_boxes"):
            gm.track_boxes(streams, boxes)
    for bad in (dict(low_thresh=0.6), dict(low_thresh=-0.1), dict(sim_high=1.0), dict(sim_low=-0.5), dict(max_lost=-1),
                dict(high_thresh=float("nan")), dict(new_thresh=float("inf")), dict(class_aware=2)):
        with pytest.raises(pkg.capi.MarsError, match="set_tracking"):
            gm.set_tracking(S, **bad)
    with pytest.raises(pkg.capi.MarsError, match="reset_tracks"):
        gm.reset_tracks(S - 1, 2)
    with pytest.raises(pkg.capi.MarsError, match="track_resident"):  # no heads configured
        gm.track_resident(0, [0])
    assert b"track_resident" in L.mars_b200_last_error()
    step(list(range(S)))  # the rejected calls changed nothing
    gm.reset_tracks(2, 3)
    oracle.reset(2, 3)
    step([7, 3, 2, 0])
    gm.set_tracking(S + 4)  # resize: everything starts over
    oracle = OracleTracker(S + 4)
    step(list(range(S)))
    gm.set_tracking(0)
    with pytest.raises(pkg.capi.MarsError, match="tracking is not set"):
        gm.track_boxes([0], b)
    gm.close()


# ---- on the heads path -----------------------------------------------------------------------------------------------------------
def perturbed_inputs(size, n, frames, seed):
    """n slowly changing inputs: each frame rewrites 2 % of the bytes of the previous one"""
    rng = np.random.default_rng(seed)
    x = rng.integers(-128, 128, size=(n, 3 * size * size), dtype=np.int8)
    out = []
    for _ in range(frames):
        m = rng.random(x.shape) < 0.02
        x = np.where(m, rng.integers(-128, 128, size=x.shape, dtype=np.int8), x)
        out.append(x.copy())
    return out


@pytest.mark.parametrize("kind,frame_size", [("yolo", False), ("yolo", True), ("gfl", False), ("gfl", True)])
def test_resident_equals_the_oracle_on_the_kept_boxes(pkg, kind, frame_size):
    B, S, frames = 6, 10, 8
    gm = heads_model(pkg, kind, B)
    gm.set_tracking(S)
    oracle = OracleTracker(S)
    if frame_size:
        gm.set_frame_size(0, B, 1280, 720)
    rng = np.random.default_rng(3)
    total = 0
    for f, xs in enumerate(perturbed_inputs(YOLO_SIZE if kind == "yolo" else GFL_SIZE, B, frames, 11)):
        streams = [int(v) for v in rng.permutation(S)[:B]] if f % 2 else list(range(B))
        gm.upload_inputs(0, B, xs, xs.shape[1])
        gm.step_heads_resident(0, B, 0.45)
        gm.track_resident(0, streams)
        boxes, counts = gm.download_boxes(0, B)
        got, tc = gm.download_tracks(0, B)
        want = [oracle.step(s, boxes[i, : counts[i]]) for i, s in enumerate(streams)]
        check(got, tc, want, "frame %d" % f)
        total += int(tc.sum())
    assert total > 0
    gm.close()


def test_tracking_leaves_the_boxes_unchanged(pkg):
    B = 4
    xs = perturbed_inputs(YOLO_SIZE, B, 1, 2)[0]
    gm = heads_model(pkg, "yolo", B)
    gm.upload_inputs(0, B, xs, xs.shape[1])
    gm.step_heads_resident(0, B, 0.45)
    before = gm.download_boxes(0, B)
    gm.set_tracking(B)
    gm.upload_inputs(0, B, xs, xs.shape[1])
    gm.step_heads_resident(0, B, 0.45)
    gm.track_resident(0, list(range(B)))
    after = gm.download_boxes(0, B)
    assert before[0].tobytes() == after[0].tobytes() and np.array_equal(before[1], after[1]) and before[1].sum() > 0
    gm.close()


@pytest.mark.parametrize("nv12", [False, True])
def test_submit_equals_the_resident_composition(pkg, nv12):
    """pooled submits alternating between the pools, the same streams in consecutive submits, against preprocess + step +
    track_resident on a second model"""
    B, S, K = 3, 5, 8
    sizes = [(640, 360), (500, 500), (320, 240)]
    rng = np.random.default_rng(9)
    base = [nv12_frame(w, h, 40 + i) for i, (w, h) in enumerate(sizes)]
    batches = []
    for k in range(K):
        fs = []
        for i, (y, uv) in enumerate(base):
            y = y.copy()
            y[rng.random(y.shape) < 0.02] = rng.integers(0, 256)
            fs.append((y, uv, i % 4))
        batches.append(fs)
    streams = [[(k + i) % S for i in range(B)] if k % 3 else [0, 1, 2] for k in range(K)]
    sub = heads_model(pkg, "yolo", 2 * B)
    ref = heads_model(pkg, "yolo", B)
    sub.set_tracking(S)
    ref.set_tracking(S)
    out = [(np.zeros((B, 256), dtype=pkg.capi.TRACK_DTYPE), np.zeros(B, dtype=np.int32)) for _ in range(2)]
    want, total = [], 0
    for k, fs in enumerate(batches):
        if nv12:
            ref.preprocess_frames_nv12(0, fs)
        else:
            ref.preprocess_frames(0, [nv12_to_rgb(y, uv, c) for (y, uv, c) in fs])
        ref.step_heads_resident(0, B, 0.45)
        ref.track_resident(0, streams[k])
        want.append(ref.download_tracks(0, B))
        total += int(want[-1][1].sum())
    assert total > 0
    for k, fs in enumerate(batches):
        pool = k % 2
        if k >= 2:
            sub.wait_batch(pool)
            check(*out[pool], [w[: n] for w, n in zip(*want[k - 2])], "batch %d" % (k - 2))
        if nv12:
            sub.submit_frames_nv12_track_batch(pool, fs, streams[k], out[pool][0], out[pool][1])
        else:
            sub.submit_frames_track_batch(pool, [nv12_to_rgb(y, uv, c) for (y, uv, c) in fs], streams[k], out[pool][0], out[pool][1])
    for k in (K - 2, K - 1):
        sub.wait_batch(k % 2)
        check(*out[k % 2], [w[: n] for w, n in zip(*want[k])], "batch %d" % k)
    bad = np.zeros((B, 256), dtype=pkg.capi.TRACK_DTYPE), np.zeros(B, dtype=np.int32)
    with pytest.raises(pkg.capi.MarsError, match="named twice"):
        sub.submit_frames_track_batch(0, [nv12_to_rgb(y, uv, c) for (y, uv, c) in batches[0]], [1, 1, 2], bad[0], bad[1])
    sub.close()
    ref.close()
