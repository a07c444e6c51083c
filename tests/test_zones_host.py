"""CPU: the C statement of the zone and line analytics (tests/zones_oracle.c) against an independent float64 restatement, and known
answers of the definition (include/mars_b200.h, mars_b200_set_zones)."""
import numpy as np
import pytest

from track_ref import BOX_DTYPE, TRACK_DTYPE, params
from zones_ref import (BOTTOM, CENTRE, CROSS_NEG, CROSS_POS, DWELL, ENTER, EXIT, GONE, MAX_EVENTS, ChainedOracle, Float64Zones,
                       OracleZones, as64, line, random_geometry, walk_scene, zone)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_oracle_equals_the_float64_restatement(seed):
    """Random walks at the limits (8 zones of 16 vertices, 8 lines) whose anchors keep 1e-2 px from every edge, vertex row, line and
    line-end extension: float32 and float64 take the same decisions, so events, occupancy and totals must be identical."""
    rng = np.random.default_rng(100 + seed)
    zones, lines = random_geometry(rng)
    o = OracleZones(1)
    o.set(0, zones, lines)
    r = Float64Zones(*as64(zones, lines))
    kinds = np.zeros(6, dtype=np.int64)
    for f, (live, shown) in enumerate(walk_scene(seed, zones, lines, frames=300, n_obj=30), start=1):
        got = o.step(0, f, live, shown)
        events, occ, pos, neg = r.step(f, live, shown)
        n = int(got["n_events"])
        assert n == len(events), "frame %d" % f
        want = [tuple(int(v) for v in e) for e in got["events"][: min(n, MAX_EVENTS)]]
        assert want == [tuple(e) for e in events[:MAX_EVENTS]], "frame %d" % f
        assert list(got["occupancy"]) == occ and list(got["crossed_pos"]) == pos and list(got["crossed_neg"]) == neg, "frame %d" % f
        for e in events:
            kinds[e[2]] += 1
    assert np.all(kinds > 0), kinds  # every kind of event happened


# ---- known answers -------------------------------------------------------------------------------------------------------------
def at(tid, px, py, cls=0):
    """a shown track whose bottom anchor is (px, py) and whose centre anchor is (px, py - 10)"""
    return (px - 10.0, py - 20.0, px + 10.0, py, 0.9, cls, tid, 0)


class Stream:
    """one stream of the C statement, frame by frame: shown = [at(...), ...], live = extra IDs that are live but not shown"""

    def __init__(self, zones=(), lines=()):
        self.o, self.f = OracleZones(1), 0
        self.o.set(0, zones, lines)

    def step(self, *shown, lost=()):
        self.f += 1
        sh = np.array(sorted(shown, key=lambda r: r[6]), dtype=TRACK_DTYPE)
        live = sorted(set(int(v) for v in sh["track_id"]) | set(lost))
        return self.o.step(0, self.f, live, sh)


def evs(rec):
    return [tuple(int(v) for v in e) for e in rec["events"][: min(int(rec["n_events"]), MAX_EVENTS)]]


SQUARE = [(0.0, 0.0), (100.0, 0.0), (100.0, 100.0), (0.0, 100.0)]


@pytest.mark.parametrize("point,inside", [((50, 0), True), ((50, 100), False), ((0, 50), True), ((100, 50), False), ((0, 0), True),
                                          ((100, 0), False), ((0, 100), False), ((100, 100), False), ((50, 50), True), ((-1, 50), False)])
def test_half_open_rule_on_edges_and_vertices(point, inside):
    """the crossing number counts the top and left edges of the square in, the bottom and right edges out"""
    s = Stream([zone(SQUARE)])
    rec = s.step(at(1, *point))
    assert int(rec["occupancy"][0]) == inside
    assert evs(rec) == ([(1, 0, ENTER, 0, 1)] if inside else [])


H = line(0.0, 50.0, 100.0, 50.0)  # side +1 below (larger y), -1 above


def crossings(recs):
    return [(int(e[2]), int(e[4])) for r in recs for e in r["events"][: int(r["n_events"])] if e[2] in (CROSS_POS, CROSS_NEG)]


def test_stopping_on_the_line_then_going_on_counts_once():
    s = Stream(lines=[H])
    recs = [s.step(at(1, 50, y)) for y in (40, 50, 50, 60, 60, 70)]
    assert crossings(recs) == [(CROSS_POS, 1)]
    assert list(recs[-1]["crossed_pos"][:1]) == [1] and list(recs[-1]["crossed_neg"][:1]) == [0]
    assert [int(e[0]) for e in recs[3]["events"][:1]] == [1]


def test_walking_around_a_lines_end_never_counts():
    s = Stream(lines=[H])
    recs = [s.step(at(1, x, y)) for x, y in ((50, 40), (150, 40), (150, 60), (50, 60), (50, 70))]
    assert crossings(recs) == []
    back = s.step(at(1, 50, 40))  # and the way back over the segment counts
    assert crossings([back]) == [(CROSS_NEG, 1)]


def test_a_crossing_during_a_lost_gap_counts_on_reappearance():
    s = Stream(lines=[H])
    recs = [s.step(at(1, 50, 40))] + [s.step(lost=[1]) for _ in range(3)] + [s.step(at(1, 50, 60))]
    assert crossings(recs[:4]) == [] and crossings(recs[4:]) == [(CROSS_POS, 1)]


def test_class_filters_and_a_class_switch():
    s = Stream([zone(SQUARE, class_id=1)], [line(0.0, 150.0, 100.0, 150.0, class_id=1)])
    assert evs(s.step(at(1, 50, 50, cls=0))) == []  # class 0 is not counted in the class-1 zone
    assert evs(s.step(at(1, 50, 50, cls=1))) == [(1, 1, ENTER, 0, 0)]
    assert evs(s.step(at(1, 50, 50, cls=0))) == [(1, 0, EXIT, 0, 1)]
    assert evs(s.step(at(1, 50, 50, cls=1))) == [(1, 1, ENTER, 0, 0)]
    # the line: class 0 crosses uncounted, but sigma follows it, so class 1 crossing back counts
    assert crossings([s.step(at(1, 50, 140, cls=1)), s.step(at(1, 50, 160, cls=0))]) == []
    assert crossings([s.step(at(1, 50, 140, cls=1))]) == [(CROSS_NEG, 1)]


@pytest.mark.parametrize("min_dwell", [0, 1, 3])
def test_dwell(min_dwell):
    s = Stream([zone(SQUARE, min_dwell=min_dwell)])
    recs = [s.step(at(1, 50, 50)) for _ in range(6)]
    dwell = [(f, int(e[4])) for f, r in enumerate(recs, 1) for e in r["events"][: int(r["n_events"])] if e[2] == DWELL]
    assert dwell == ([] if min_dwell == 0 else [(min_dwell, min_dwell)])
    assert evs(recs[0])[0] == (1, 0, ENTER, 0, 1)
    if min_dwell == 1:
        assert evs(recs[0]) == [(1, 0, ENTER, 0, 1), (1, 0, DWELL, 0, 1)]
    out = s.step(at(1, 50, 150))
    assert evs(out) == [(1, 0, EXIT, 0, 6)]
    again = [s.step(at(1, 50, 50)) for _ in range(4)]  # a new stay dwells again
    assert [int(e[2]) for r in again for e in r["events"][: int(r["n_events"])]] == [ENTER] + ([DWELL] if min_dwell else [])


def test_enter_on_first_sight_and_later():
    s = Stream([zone(SQUARE)])
    assert evs(s.step(at(1, 50, 50), at(2, 150, 50))) == [(1, 0, ENTER, 0, 1)]
    assert evs(s.step(at(1, 50, 50), at(2, 50, 60))) == [(2, 0, ENTER, 0, 0)]


def test_gone_when_max_lost_expires_inside_a_zone():
    o = ChainedOracle(1, params(max_lost=2))
    o.zn.set(0, [zone([(0.0, 0.0), (400.0, 0.0), (400.0, 400.0), (0.0, 400.0)])])
    det = np.array([(100.0, 100.0, 150.0, 180.0, 0.9, 3)], dtype=BOX_DTYPE)
    none = np.zeros(0, dtype=BOX_DTYPE)
    tracks, rec = o.step(0, det)
    assert len(tracks) == 1 and evs(rec) == [(1, 3, ENTER, 0, 1)] and int(rec["occupancy"][0]) == 1
    for f in (2, 3):
        tracks, rec = o.step(0, none)  # lost: state kept, no occupancy
        assert len(tracks) == 0 and evs(rec) == [] and int(rec["occupancy"][0]) == 0 and int(rec["frame"]) == f
    tracks, rec = o.step(0, none)  # frame 4: 4 - 1 > max_lost, the tracker removes it
    assert evs(rec) == [(1, 3, GONE, 0, 3)]
    assert evs(o.step(0, none)[1]) == []


def test_event_order_and_truncation():
    zones = [zone(SQUARE, min_dwell=1), zone([(0.0, 0.0), (300.0, 0.0), (300.0, 300.0), (0.0, 300.0)], anchor=CENTRE)]
    s = Stream(zones, [H])
    s.step(at(5, 50, 40), at(9, 200, 200))
    # track 5 crosses H and leaves the square; track 7 is new inside both; track 9 is removed while inside zone 1
    rec = s.step(at(5, 50, 120), at(7, 50, 50))
    assert evs(rec) == [(5, 0, CROSS_POS, 0, 1), (5, 0, EXIT, 0, 1), (7, 0, ENTER, 0, 1), (7, 0, DWELL, 0, 1), (7, 0, ENTER, 1, 1),
                        (9, 0, GONE, 1, 1)]
    # 100 tracks entering both zones: 300 events, the first 128 written in order
    big = Stream(zones)
    rec = big.step(*[at(t, 50, 50) for t in range(1, 101)])
    assert int(rec["n_events"]) == 300 and int(rec["occupancy"][0]) == 100 and int(rec["occupancy"][1]) == 100
    want = [(t, 0, k, z, 1) for t in range(1, 101) for k, z in ((ENTER, 0), (DWELL, 0), (ENTER, 1))][:MAX_EVENTS]
    assert evs(rec) == want


def test_a_stream_without_geometry_gets_its_frame_and_zeros():
    s = Stream()
    rec = s.step(at(1, 50, 50))
    assert int(rec["frame"]) == 1 and rec.tobytes()[4:] == bytes(len(rec.tobytes()) - 4)


def test_capi_layouts_match_the_oracle(pkg):
    import ctypes
    from zones_ref import EVENT_DTYPE, FRAME_DTYPE, Line, Zone
    c = pkg.capi
    assert c.ZONE_FRAME_DTYPE == FRAME_DTYPE and c.ZONE_EVENT_DTYPE == EVENT_DTYPE
    assert ctypes.sizeof(c.ZONE) == ctypes.sizeof(Zone) and ctypes.sizeof(c.LINE) == ctypes.sizeof(Line)
    z = c.ZONE([(1.0, 2.0), (3.0, 4.0), (5.0, 7.0)], class_id=2, anchor=c.ANCHOR_CENTRE, min_dwell=4)
    assert bytes(z) == bytes(zone([(1.0, 2.0), (3.0, 4.0), (5.0, 7.0)], 2, CENTRE, 4))
    assert bytes(c.LINE(1, 2, 3, 4)) == bytes(line(1.0, 2.0, 3.0, 4.0, -1, BOTTOM))
