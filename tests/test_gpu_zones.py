"""GPU: zones and counting lines on tracked streams (k_zones, mars_b200_set_zones) through every entry point, byte for byte against
the C statement behind the tracker's (zones_ref.ChainedOracle)."""
import numpy as np
import pytest

from nv12_ref import nv12_frame, nv12_to_rgb
from test_gpu_track import crowded, heads_model, perturbed_inputs, random_frames
from track_ref import BOX_DTYPE
from zones_ref import MAX_LINES, MAX_ZONES, ChainedOracle, line, random_geometry, records_equal, zone

pytestmark = pytest.mark.gpu


def set_both(pkg, gm, oracle, s, zones, lines):
    gm.set_zones(s, [pkg.capi.ZONE.from_buffer_copy(bytes(z)) for z in zones], [pkg.capi.LINE.from_buffer_copy(bytes(ln)) for ln in lines])
    oracle.zn.set(s, zones, lines)


def check(tracks, counts, zrec, want, what):
    for i, (wt, wz) in enumerate(want):
        assert counts[i] == len(wt) and tracks[i, : len(wt)].tobytes() == wt.tobytes(), "%s entry %d: tracks" % (what, i)
        d = records_equal(zrec[i], wz)
        assert d is None, "%s entry %d: %s" % (what, i, d)


def grid_geometry(rng, side=320):
    """zones and lines with every vertex and end on the 16 px grid of the tie scenes"""
    g = lambda v: float(np.clip(np.round(v / 16) * 16, 0, side))  # noqa: E731
    zones = []
    for _ in range(int(rng.integers(1, MAX_ZONES + 1))):
        c, n = rng.uniform(48, side - 48, 2), int(rng.integers(3, 17))
        ang, rad = np.sort(rng.uniform(0, 2 * np.pi, n)), rng.uniform(32, 160, n)
        zones.append(zone([(g(c[0] + r * np.cos(a)), g(c[1] + r * np.sin(a))) for a, r in zip(ang, rad)], int(rng.choice([-1, 0, 1])),
                          int(rng.integers(0, 2)), int(rng.choice([0, 1, 3]))))
    lines = []
    for _ in range(int(rng.integers(1, MAX_LINES + 1))):
        a = [g(v) for v in rng.uniform(0, side, 2)]
        b = a
        while b == a:
            b = [g(v) for v in rng.uniform(0, side, 2)]
        lines.append(line(a[0], a[1], b[0], b[1], int(rng.choice([-1, 0, 1])), int(rng.integers(0, 2))))
    return zones, lines


def grid_frames(seed, frames, n_obj, side=320):
    """32 x 32 boxes on the 16 px grid that mostly stand still (the tracked box of a still object stays exact, so its anchors sit
    on grid points: on vertices, edges and lines), sometimes step by 16 px and sometimes jump (a new track, exact from birth)"""
    rng = np.random.default_rng(seed)
    pos = rng.integers(0, side // 16, (n_obj, 2)) * 16.0
    cls = rng.integers(0, 3, n_obj)
    out = []
    for _ in range(frames):
        u = rng.random(n_obj)
        pos[u > 0.9] = rng.integers(0, side // 16, (int(np.sum(u > 0.9)), 2)) * 16.0
        step = (u > 0.75) & (u <= 0.9)
        pos[step] += rng.choice([-16.0, 16.0], (int(step.sum()), 2))
        rows = [(p[0], p[1], p[0] + 32, p[1] + 32, 0.9, int(c)) for p, c in zip(pos, cls) if rng.random() < 0.95]
        out.append(np.array(rows, dtype=BOX_DTYPE))
    return out


def on_a_line(tracks, lines):
    """shown tracks in exact float32 ties with a line (side 0), counted with the definition's operations"""
    n = 0
    f = np.float32
    for ln in lines:
        for t in tracks:
            px = (t["x0"] + t["x1"]) * f(0.5)
            py = (t["y0"] + t["y1"]) * f(0.5) if ln.anchor == 1 else t["y1"]
            v = (f(ln.x1) - f(ln.x0)) * (py - f(ln.y0)) - (f(ln.y1) - f(ln.y0)) * (px - f(ln.x0))
            n += int(v == 0)
    return n


@pytest.mark.parametrize("ties", [False, True])
def test_track_boxes_zones_equal_the_oracle(pkg, ties):
    S, frames = 256, 60
    rng = np.random.default_rng(17 + ties)
    if ties:
        seqs = [grid_frames(s, frames + 20, int(rng.integers(1, 24))) for s in range(S)]
    else:
        seqs = [random_frames(s, frames + 20, int(np.random.default_rng(s).integers(1, 40))) for s in range(S)]
    gm = pkg.MarsModel(heads_blob(pkg), arena_bytes=8 << 20, device=0)
    gm.set_tracking(S)
    oracle = ChainedOracle(S)
    for s in range(S):
        if s % 5 != 4:  # every fifth stream has no geometry
            zones, lines = grid_geometry(rng) if ties else random_geometry(rng, 640.0, 640.0, int(rng.integers(0, 9)), int(rng.integers(3, 17)),
                                                                           int(rng.integers(1, 9)))
            set_both(pkg, gm, oracle, s, zones, lines)
    calls = [list(range(S))] * frames
    for _ in range(20):  # shuffled subsets
        calls.append([int(v) for v in rng.permutation(S)[: int(rng.integers(1, S))]])
    nxt, events, ties_seen = {}, 0, 0
    for c, streams in enumerate(calls):
        boxes = [seqs[s][nxt.get(s, 0)] for s in streams]
        for s in streams:
            nxt[s] = nxt.get(s, 0) + 1
        got, counts, zr = gm.track_boxes_zones(streams, boxes)
        want = [oracle.step(s, b) for s, b in zip(streams, boxes)]
        check(got, counts, zr, want, "call %d" % c)
        events += int(zr["n_events"].sum())
        if ties:
            ties_seen += sum(on_a_line(w[0], oracle.zn.geom[s].line[: oracle.zn.geom[s].n_lines]) for s, w in zip(streams, want))
    assert events > 1000
    assert not ties or ties_seen > 0
    gm.close()


def heads_blob(pkg):
    from test_gpu_track import yolo_blob
    return yolo_blob()


def test_plain_track_calls_keep_the_analytics_advancing(pkg):
    """track_boxes without zone output between zone calls: the analytics still see every frame; the tracked boxes are the same"""
    S, frames = 16, 30
    rng = np.random.default_rng(4)
    seqs = [random_frames(100 + s, frames, 20) for s in range(S)]
    gm = pkg.MarsModel(heads_blob(pkg), arena_bytes=8 << 20, device=0)
    gm.set_tracking(S)
    oracle = ChainedOracle(S)
    for s in range(S):
        set_both(pkg, gm, oracle, s, *random_geometry(rng, 640.0, 640.0, 4, 8, 4))
    streams = list(range(S))
    for f in range(frames):
        boxes = [seqs[s][f] for s in streams]
        want = [oracle.step(s, b) for s, b in zip(streams, boxes)]
        if f % 3 == 1:
            got, counts = gm.track_boxes(streams, boxes)
            for i, (wt, _) in enumerate(want):
                assert counts[i] == len(wt) and got[i, : len(wt)].tobytes() == wt.tobytes()
        else:
            check(*gm.track_boxes_zones(streams, boxes), want, "frame %d" % f)
    gm.close()


def test_crowded_frames_over_the_event_cap(pkg):
    S, frames = 3, 5
    seqs = [crowded(s, frames) for s in range(S)]
    gm = pkg.MarsModel(heads_blob(pkg), arena_bytes=8 << 20, device=0)
    gm.set_tracking(S)
    oracle = ChainedOracle(S)
    for s in range(S):  # 8 overlapping 16-gons over the tracked rows of the grid, 8 lines through them
        a = np.arange(16) * 2 * np.pi / 16
        zones = [zone([(float(np.float32(60 + 120 * k + 110 * np.cos(t))), float(np.float32(130 + 10 * s + 140 * np.sin(t)))) for t in a], -1,
                      k % 2, 1 + k % 3) for k in range(MAX_ZONES)]
        lines = [line(0.0, 12.0 + 24 * k + 3 * s, 960.0, 20.0 + 24 * k, -1, k % 2) for k in range(MAX_LINES)]
        set_both(pkg, gm, oracle, s, zones, lines)
    over = 0
    for f in range(frames):
        got, counts, zr = gm.track_boxes_zones(list(range(S)), [seqs[s][f] for s in range(S)])
        want = [oracle.step(s, seqs[s][f]) for s in range(S)]
        check(got, counts, zr, want, "frame %d" % f)
        assert f > 0 or np.all(counts == 256)
        over += int(np.sum(zr["n_events"] > 128))
    assert over > 0
    gm.close()


def test_set_zones_reset_set_tracking_and_rejections(pkg):
    S = 8
    seqs = [random_frames(s, 60, 8) for s in range(S)]
    rng = np.random.default_rng(2)
    gm = pkg.MarsModel(heads_blob(pkg), arena_bytes=8 << 20, device=0)
    C = pkg.capi
    with pytest.raises(C.MarsError, match="tracking is not set"):
        gm.set_zones(0, [C.ZONE([(0, 0), (1, 0), (0, 1)])])
    gm.set_tracking(S)
    oracle = ChainedOracle(S)
    pos = {s: 0 for s in range(S)}

    def step(streams, zones_out=True):
        boxes = [seqs[s][pos[s]] for s in streams]
        for s in streams:
            pos[s] += 1
        want = [oracle.step(s, b) for s, b in zip(streams, boxes)]
        before = gm.launch_count
        if zones_out:
            check(*gm.track_boxes_zones(streams, boxes), want, "step")
        else:
            gm.track_boxes(streams, boxes)
        return gm.launch_count - before

    assert step(list(range(S)), False) == 1  # no geometry anywhere: k_track alone, as before zones existed
    assert step(list(range(S))) == 2  # the zone form always runs k_zones
    geo = {s: random_geometry(rng, 640.0, 640.0, 3, 6, 3) for s in range(S)}
    for s in range(S):
        set_both(pkg, gm, oracle, s, *geo[s])
    assert step(list(range(S)), False) == 2  # geometry somewhere: every tracker call runs the analytics
    step(list(range(S)))
    sq = [(0.0, 0.0), (10.0, 0.0), (10.0, 10.0)]
    bad = [(dict(stream=S), "stream"), (dict(stream=-1), "stream"), (dict(zones=[C.ZONE(sq)] * 9), "zones"),
           (dict(zones=[C.ZONE(sq[:2])]), "zone 0: n_verts"), (dict(zones=[C.ZONE(sq), C.ZONE(sq * 6)]), "zone 1: n_verts"),
           (dict(zones=[C.ZONE(sq[:2] + [(float("nan"), 1.0)])]), "zone 0: vertex 2"), (dict(zones=[C.ZONE(sq, class_id=-2)]), "zone 0: class_id"),
           (dict(zones=[C.ZONE(sq, anchor=2)]), "zone 0: anchor"), (dict(zones=[C.ZONE(sq, min_dwell=-1)]), "zone 0: min_dwell"),
           (dict(lines=[C.LINE(1, 2, 1, 2)]), "line 0: ends coincide"), (dict(lines=[C.LINE(0, 0, 1, 1), C.LINE(0, 0, float("inf"), 1)]),
                                                                         "line 1: ends"),
           (dict(lines=[C.LINE(0, 0, 1, 1, class_id=-3)]), "line 0: class_id"), (dict(lines=[C.LINE(0, 0, 1, 1, anchor=7)]), "line 0: anchor"),
           (dict(lines=[C.LINE(0, 0, 1, 1)] * 9), "lines")]
    for kw, msg in bad:
        args = dict(stream=1, zones=[C.ZONE(sq)], lines=[C.LINE(0, 0, 5, 5)])
        args.update(kw)
        with pytest.raises(C.MarsError, match="set_zones") as e:
            gm.set_zones(args["stream"], args["zones"], args["lines"])
        assert msg in str(e.value), (msg, str(e.value))
    step(list(range(S)))  # the rejected calls changed nothing
    set_both(pkg, gm, oracle, 3, *random_geometry(rng, 640.0, 640.0, 2, 5, 2))  # new geometry: that stream's analytics start over
    step([3, 1, 0])
    set_both(pkg, gm, oracle, 5, (), ())  # switched off: frame number and zeros
    step([5, 6])
    gm.reset_tracks(2, 3)  # tracks and analytics of 2, 3, 4 start over; their geometry stays
    oracle.reset(2, 3)
    step([4, 3, 2, 7])
    step(list(range(S)))
    gm.set_tracking(S + 4)  # drops every geometry
    oracle = ChainedOracle(S + 4)
    assert step(list(range(S)), False) == 1
    step(list(range(S)))
    gm.close()


# ---- on the heads path -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,frame_size", [("yolo", False), ("yolo", True), ("gfl", False), ("gfl", True)])
def test_resident_equals_the_oracle_on_the_downloaded_tracks(pkg, kind, frame_size):
    B, S, frames = 6, 10, 8
    gm = heads_model(pkg, kind, B)
    gm.set_tracking(S)
    oracle = ChainedOracle(S)
    W, H = (1280.0, 720.0) if frame_size else (320.0, 320.0)
    if frame_size:
        gm.set_frame_size(0, B, int(W), int(H))
    rng = np.random.default_rng(5)
    for s in range(S - 1):  # the last stream has no geometry
        set_both(pkg, gm, oracle, s, *random_geometry(rng, W, H, 4, 12, 4))
    events = 0
    for f, xs in enumerate(perturbed_inputs(320, B, frames, 13)):
        streams = [int(v) for v in rng.permutation(S)[:B]] if f % 2 else list(range(S - B, S))
        gm.upload_inputs(0, B, xs, xs.shape[1])
        gm.step_heads_resident(0, B, 0.45)
        gm.track_resident(0, streams)
        boxes, counts = gm.download_boxes(0, B)
        got, tc = gm.download_tracks(0, B)
        zr = gm.download_zones(0, B)
        want = [oracle.step(s, boxes[i, : counts[i]]) for i, s in enumerate(streams)]
        check(got, tc, zr, want, "frame %d" % f)
        events += int(zr["n_events"].sum())
    assert events > 0
    gm.close()


@pytest.mark.parametrize("nv12", [False, True])
def test_zone_submits_equal_the_resident_flow(pkg, nv12):
    """pooled zone submits alternating between the pools (one plain track submit among them), against preprocess + step +
    track_resident + download_zones on a second model"""
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
    sub, ref = heads_model(pkg, "yolo", 2 * B), heads_model(pkg, "yolo", B)
    for gm in (sub, ref):
        gm.set_tracking(S)
        grng = np.random.default_rng(21)
        for s in range(S):
            zones, lines = random_geometry(grng, 640.0, 500.0, 4, 10, 4)
            gm.set_zones(s, [pkg.capi.ZONE.from_buffer_copy(bytes(z)) for z in zones], [pkg.capi.LINE.from_buffer_copy(bytes(ln)) for ln in lines])
    want, events = [], 0
    for k, fs in enumerate(batches):
        if nv12:
            ref.preprocess_frames_nv12(0, fs)
        else:
            ref.preprocess_frames(0, [nv12_to_rgb(y, uv, c) for (y, uv, c) in fs])
        ref.step_heads_resident(0, B, 0.45)
        ref.track_resident(0, streams[k])
        want.append(ref.download_tracks(0, B) + (ref.download_zones(0, B),))
        events += int(want[-1][2]["n_events"].sum())
    assert events > 0
    T = pkg.capi.TRACK_DTYPE
    out = [(np.zeros((B, 256), dtype=T), np.zeros(B, dtype=np.int32), np.zeros(B, dtype=pkg.capi.ZONE_FRAME_DTYPE)) for _ in range(2)]
    plain = 4  # a plain track submit: its zone records are not read back, the analytics advance all the same

    def compare(k):
        t, c, z = out[k % 2]
        wt, wc, wz = want[k]
        for i in range(B):
            assert c[i] == wc[i] and t[i, : wc[i]].tobytes() == wt[i, : wc[i]].tobytes(), "batch %d entry %d" % (k, i)
            if k != plain:
                d = records_equal(z[i], wz[i])
                assert d is None, "batch %d entry %d: %s" % (k, i, d)

    for k, fs in enumerate(batches):
        pool = k % 2
        if k >= 2:
            sub.wait_batch(pool)
            compare(k - 2)
        frames = fs if nv12 else [nv12_to_rgb(y, uv, c) for (y, uv, c) in fs]
        t, c, z = out[pool]
        if k == plain:
            (sub.submit_frames_nv12_track_batch if nv12 else sub.submit_frames_track_batch)(pool, frames, streams[k], t, c)
        else:
            (sub.submit_frames_nv12_zones_batch if nv12 else sub.submit_frames_zones_batch)(pool, frames, streams[k], t, c, z)
    for k in (K - 2, K - 1):
        sub.wait_batch(k % 2)
        compare(k)
    with pytest.raises(pkg.capi.MarsError, match="named twice"):
        sub.submit_frames_zones_batch(0, [nv12_to_rgb(y, uv, c) for (y, uv, c) in batches[0]], [1, 1, 2], *out[0])
    with pytest.raises(pkg.capi.MarsError, match="no zone record table"):
        sub.submit_frames_zones_batch(0, [nv12_to_rgb(y, uv, c) for (y, uv, c) in batches[0]], [0, 1, 2], out[0][0], out[0][1], None)
    sub.close()
    ref.close()


def test_set_zones_is_ordered_before_the_next_tracker_call(pkg):
    """geometry set again on every stream between consecutive tracker calls: each call sees the new geometry and a cleared state"""
    S, frames = 64, 12
    rng = np.random.default_rng(31)
    seqs = [random_frames(300 + s, frames, 30) for s in range(S)]
    gm = pkg.MarsModel(heads_blob(pkg), arena_bytes=8 << 20, device=0)
    gm.set_tracking(S)
    oracle = ChainedOracle(S)
    for f in range(frames):
        for s in range(S):
            set_both(pkg, gm, oracle, s, *random_geometry(rng, 640.0, 640.0, int(rng.integers(1, 9)), 16, int(rng.integers(1, 9))))
        boxes = [seqs[s][f] for s in range(S)]
        check(*gm.track_boxes_zones(list(range(S)), boxes), [oracle.step(s, b) for s, b in zip(range(S), boxes)], "frame %d" % f)
    gm.close()
