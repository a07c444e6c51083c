"""CPU: the C statement of the multi-object tracker (tests/track_oracle.c) against an independent float64 restatement, and known
answers of the definition (include/mars_b200.h, mars_b200_set_tracking)."""
import numpy as np
import pytest

from track_ref import BOX_DTYPE, MAX_TRACKS, Float64Tracker, OracleTracker, lanes_sequence, params


def dets(*rows):
    """(x0, y0, x1, y1, conf[, class]) rows -> BOX_DTYPE array"""
    return np.array([tuple(r) + (0,) * (6 - len(r)) for r in rows], dtype=BOX_DTYPE)


def ids(out):
    return [int(v) for v in out["track_id"]]


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_oracle_equals_the_float64_reference(seed):
    """Lanes keep the objects apart, so every similarity is far from its gate: the float32 statement and the float64 filter take
    the same decisions, and IDs and detection indices must be identical.  The boxes differ by rounding only: the filter's gains
    are below 1, so the float32 error does not grow with the sequence.  Coordinates stay below 2048, where a float32 ulp is at most
    2^-12 px; the observed difference is about 2 ulps (2e-4 px), and the bound is 8 ulps (2^-9 px)."""
    seq = lanes_sequence(seed, frames=400)
    o, r = OracleTracker(1), Float64Tracker()
    worst, births, lost_found, seen = 0.0, set(), 0, {}
    for f, d in enumerate(seq):
        got, want = o.step(0, d), r.step(d)
        assert ids(got) == [w[0] for w in want], "frame %d" % f
        assert [int(v) for v in got["det_index"]] == [w[1] for w in want], "frame %d" % f
        for g, w in zip(got, want):
            worst = max(worst, float(np.max(np.abs(np.array([g["x0"], g["y0"], g["x1"], g["y1"]], dtype=np.float64) - w[2]))))
            assert float(g["confidence"]) == np.float32(w[3]) and int(g["class_id"]) == w[4]
            births.add(int(g["track_id"]))
            if int(g["track_id"]) in seen and seen[int(g["track_id"])] < f - 1:
                lost_found += 1
            seen[int(g["track_id"])] = f
    assert worst < 2.0 ** -9, worst
    assert min(r.margins) > 1e-3  # no decision was close to its gate
    assert len(births) > 20 and lost_found > 0  # births, and tracks found again after a gap


def run(o, frames, stream=0):
    return [o.step(stream, d) for d in frames]


def box(x, y=100.0, w=50.0, h=80.0, conf=0.9, cls=0):
    return (x, y, x + w, y + h, conf, cls)


def test_first_frame_activates_later_births_wait_for_a_match():
    o = OracleTracker(1)
    a = o.step(0, dets(box(100)))
    assert ids(a) == [1]  # frame 1: born activated
    b = o.step(0, dets(box(102), box(400)))
    assert ids(b) == [1]  # the new track 2 is unconfirmed: not shown
    c = o.step(0, dets(box(104), box(401)))
    assert ids(c) == [1, 2] and list(c["det_index"]) == [0, 1]  # confirmed by its second match


def test_unconfirmed_track_removed_after_one_miss():
    o = OracleTracker(1)
    o.step(0, dets(box(100)))
    o.step(0, dets(box(100), box(400)))  # track 2 born unconfirmed
    o.step(0, dets(box(100)))  # missed once: removed
    out = o.step(0, dets(box(100), box(400)))
    assert ids(out) == [1]  # box(400) starts track 3, unconfirmed
    out = o.step(0, dets(box(100), box(400)))
    assert ids(out) == [1, 3]


@pytest.mark.parametrize("max_lost", [0, 3, 30])
def test_lost_track_removed_exactly_after_max_lost_frames(max_lost):
    p = params(max_lost=max_lost)
    for gap in (max_lost, max_lost + 1):
        o = OracleTracker(1, p)
        o.step(0, dets(box(100)))  # frame 1, last = 1
        for _ in range(gap):
            o.step(0, dets())  # frames 2 .. gap + 1: lost
        # frame gap + 2: frame - last = gap + 1; the track survives frame - last = max_lost + 1 only as long as gap + 1 <= max_lost + 1
        out = o.step(0, dets(box(100)))
        if gap <= max_lost:
            assert ids(out) == [1], (max_lost, gap)  # found again: the ID is kept
        else:
            assert ids(out) == [], (max_lost, gap)  # removed at frame - last = max_lost + 1 (frame gap + 1); a new track 2 waits


def test_reactivation_keeps_the_id():
    o = OracleTracker(1)
    run(o, [dets(box(100 + 4 * k)) for k in range(5)])
    run(o, [dets() for _ in range(5)])  # lost; the prediction keeps moving at 4 px per frame
    out = o.step(0, dets(box(100 + 4 * 10)))
    assert ids(out) == [1]


def test_occlusion_bridged_only_by_a_low_score_detection():
    for low in (True, False):
        o = OracleTracker(1)
        run(o, [dets(box(100 + 2 * k)) for k in range(3)])
        out = o.step(0, dets(box(106, conf=0.3)) if low else dets())
        assert ids(out) == ([1] if low else [])
        out = o.step(0, dets(box(108, conf=0.3)) if low else dets())
        assert ids(out) == ([1] if low else [])


def test_class_aware_gating():
    for aware in (0, 1):
        o = OracleTracker(1, params(class_aware=aware))
        o.step(0, dets(box(100, cls=1)))
        out = o.step(0, dets(box(101, cls=2)))
        assert ids(out) == ([] if aware else [1]), aware  # class-aware: track 1 is lost, the box starts an unconfirmed track


def test_track_cap_consumes_no_id():
    o = OracleTracker(1)
    grid = [box(10 + 60 * (i % 30), 10 + 100 * (i // 30), w=40, h=60) for i in range(260)]
    out = o.step(0, dets(*grid))
    assert ids(out) == list(range(1, MAX_TRACKS + 1))  # 256 born on frame 1; detections 256..259 start nothing
    out = o.step(0, dets(*grid, box(5000, 5000)))
    assert len(out) == MAX_TRACKS and ids(out) == list(range(1, MAX_TRACKS + 1))
    o2 = OracleTracker(1)
    o2.step(0, dets(*grid[:255]))
    o2.step(0, dets(*grid[:255]))
    out = o2.step(0, dets(*grid[:254], box(5000, 5000), box(6000, 6000)))  # 255 live: one birth, ID 256; the second consumes nothing
    o2.step(0, dets(*grid[:254], box(5000, 5000)))  # track 255 was lost, track 256 confirmed
    out = o2.step(0, dets(*grid[:254], box(5000, 5000)))
    assert int(out["track_id"].max()) == 256


def test_degenerate_and_non_finite_boxes_are_ignored():
    nan, inf = float("nan"), float("inf")
    o = OracleTracker(1)
    bad = dets((10, 10, 10, 50, 0.9), (10, 10, 50, 5, 0.9), (nan, 10, 50, 50, 0.9), (10, 10, 50, inf, 0.9), (10, 10, 50, 50, nan),
               (10, 10, 50, 50, inf), box(200))
    out = o.step(0, bad)
    assert ids(out) == [1] and list(out["det_index"]) == [6]


def test_conf_equal_to_high_is_neither_high_nor_low():
    o = OracleTracker(1)
    o.step(0, dets(box(100)))
    out = o.step(0, dets(box(101, conf=0.5)))
    assert ids(out) == []  # not high (no stage 1), not low (no stage 2): track 1 is lost
    out = o.step(0, dets(box(102, conf=0.5000001)))
    assert ids(out) == [1]


def test_ties_resolved_by_track_id_then_detection_index():
    o = OracleTracker(1)
    o.step(0, dets(box(100), box(100), box(100)))  # three identical tracks 1, 2, 3
    out = o.step(0, dets(box(100), box(100)))  # equal similarities everywhere: track 1 <- det 0, track 2 <- det 1, track 3 lost
    assert ids(out) == [1, 2] and list(out["det_index"]) == [0, 1]
    o = OracleTracker(1)
    o.step(0, dets(box(100), box(300)))
    out = o.step(0, dets(box(300), box(100), box(100)))  # track 1 has two equal candidates: the smaller index wins
    assert ids(out) == [1, 2] and list(out["det_index"]) == [1, 0]


def test_streams_are_independent_and_reset_starts_over():
    o = OracleTracker(3)
    o.step(0, dets(box(100)))
    o.step(2, dets(box(100), box(300)))
    assert ids(o.step(1, dets(box(100)))) == [1]
    assert ids(o.step(2, dets(box(100), box(300)))) == [1, 2]
    o.reset(2, 1)
    assert ids(o.step(2, dets(box(500)))) == [1]
