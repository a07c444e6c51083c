"""Reference flows of the zone and line analytics (mars_b200_set_zones), for the tests.

OracleZones runs the C statement (tests/zones_oracle.c, compiled with -ffp-contract=off into a temporary directory on first use), one
state per stream.  ChainedOracle puts it behind the tracker's C statement (track_ref.OracleTracker), taking the live track IDs from
the oracle tracker's stream table, as k_zones follows k_track.  Float64Zones is an independent restatement in float64 that sorts
each frame's events instead of walking the tracks in order.  walk_scene generates shown / lost / removed tracks on random walks
whose anchors keep at least `margin` px from every zone edge and vertex row, every line, and whose steps keep every line end at
least `margin` px off their own line, so that float32 and float64 take the same decisions.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from track_ref import MAX_TRACKS, TRACK_DTYPE, OracleTracker

MAX_ZONES, MAX_VERTS, MAX_LINES, MAX_EVENTS = 8, 16, 8, 128
BOTTOM, CENTRE = 0, 1
ENTER, DWELL, EXIT, GONE, CROSS_POS, CROSS_NEG = 0, 1, 2, 3, 4, 5
EVENT_DTYPE = np.dtype([("track_id", "<i4"), ("class_id", "<i4"), ("kind", "<i2"), ("index", "<i2"), ("value", "<i4")])
FRAME_DTYPE = np.dtype([("frame", "<i4"), ("n_events", "<i4"), ("occupancy", "<i4", MAX_ZONES), ("crossed_pos", "<i4", MAX_LINES),
                        ("crossed_neg", "<i4", MAX_LINES), ("events", EVENT_DTYPE, MAX_EVENTS)])
_clib = None


class Zone(C.Structure):
    """mars_b200_zone_t"""
    _fields_ = [("x", C.c_float * MAX_VERTS), ("y", C.c_float * MAX_VERTS), ("n_verts", C.c_int32), ("class_id", C.c_int32),
                ("anchor", C.c_int32), ("min_dwell", C.c_int32)]


class Line(C.Structure):
    """mars_b200_line_t"""
    _fields_ = [("x0", C.c_float), ("y0", C.c_float), ("x1", C.c_float), ("y1", C.c_float), ("class_id", C.c_int32), ("anchor", C.c_int32)]


class Geom(C.Structure):
    _fields_ = [("n_zones", C.c_int32), ("n_lines", C.c_int32), ("zone", Zone * MAX_ZONES), ("line", Line * MAX_LINES)]


def zone(points, class_id=-1, anchor=BOTTOM, min_dwell=0):
    z = Zone(n_verts=len(points), class_id=class_id, anchor=anchor, min_dwell=min_dwell)
    for i, (x, y) in enumerate(points):
        z.x[i], z.y[i] = x, y
    return z


def line(x0, y0, x1, y1, class_id=-1, anchor=BOTTOM):
    return Line(x0, y0, x1, y1, class_id, anchor)


def _lib():
    global _clib
    if _clib is None:
        src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "zones_oracle.c")
        so = os.path.join(tempfile.mkdtemp(prefix="zones_oracle_"), "libzones_oracle.so")
        subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-o", so, src, "-lm"], check=True)
        _clib = C.CDLL(so)
        for f in ("zn_stream_bytes", "zn_geom_bytes", "zn_frame_bytes"):
            getattr(_clib, f).restype = C.c_int
        _clib.zn_step.restype = None
        _clib.zn_step.argtypes = [C.c_void_p, C.POINTER(Geom), C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
        assert _clib.zn_geom_bytes() == C.sizeof(Geom) and _clib.zn_frame_bytes() == FRAME_DTYPE.itemsize
    return _clib


class OracleZones:
    """the C statement, one geometry and one state per stream"""

    def __init__(self, n_streams):
        self.geom = [Geom() for _ in range(n_streams)]
        self.state = np.zeros((n_streams, _lib().zn_stream_bytes()), dtype=np.uint8)

    def set(self, stream, zones=(), lines=()):
        g = Geom(n_zones=len(zones), n_lines=len(lines))
        for i, z in enumerate(zones):
            g.zone[i] = z
        for i, ln in enumerate(lines):
            g.line[i] = ln
        self.geom[stream] = g
        self.state[stream] = 0

    def reset(self, first, n):
        self.state[first: first + n] = 0

    def step(self, stream, frame, live_ids, shown):
        """live_ids: the tracker's track IDs after this frame; shown: its TRACK_DTYPE output -> one FRAME_DTYPE record"""
        live = np.ascontiguousarray(live_ids, dtype=np.int32)
        sh = np.ascontiguousarray(shown, dtype=TRACK_DTYPE)
        out = np.zeros(1, dtype=FRAME_DTYPE)
        _lib().zn_step(self.state[stream].ctypes.data, C.byref(self.geom[stream]), frame, live.ctypes.data, live.size, sh.ctypes.data,
                       sh.size, out.ctypes.data)
        return out[0]


# the tracker oracle's stream_t: frame, issued, live, then MAX_TRACKS track_t of 27 words (track_id is word 22)
_TRACK_WORDS, _TRACK_ID_WORD = 27, 22


class ChainedOracle:
    """OracleTracker followed by OracleZones, as k_zones follows k_track"""

    def __init__(self, n_streams, p=None):
        self.trk = OracleTracker(n_streams, p)
        self.zn = OracleZones(n_streams)
        assert self.trk.state.shape[1] == 4 * (3 + MAX_TRACKS * _TRACK_WORDS)

    def reset(self, first, n):
        self.trk.reset(first, n)
        self.zn.reset(first, n)

    def step(self, stream, boxes):
        """boxes: the frame's kept boxes -> (TRACK_DTYPE tracked boxes, FRAME_DTYPE zone record)"""
        tracks = self.trk.step(stream, boxes)
        words = self.trk.state[stream].view(np.int32)
        frame, live = int(words[0]), int(words[2])
        ids = words[3: 3 + live * _TRACK_WORDS].reshape(live, _TRACK_WORDS)[:, _TRACK_ID_WORD]
        return tracks, self.zn.step(stream, frame, ids, tracks)


def records_equal(got, want):
    """byte equality of zone records, with a readable difference"""
    if got.tobytes() == want.tobytes():
        return None
    for f in ("frame", "n_events", "occupancy", "crossed_pos", "crossed_neg"):
        if not np.array_equal(got[f], want[f]):
            return "%s: %s != %s" % (f, got[f], want[f])
    n = min(int(want["n_events"]), MAX_EVENTS)
    for k in range(MAX_EVENTS):
        if got["events"][k].tobytes() != want["events"][k].tobytes():
            return "event %d of %d: %s != %s" % (k, n, got["events"][k], want["events"][k])
    return "bytes differ"


# ---- the float64 restatement ----------------------------------------------------------------------------------------------------
def anchors64(box, kind):
    """box: (x0, y0, x1, y1) float32 values -> the anchor in float64"""
    x0, y0, x1, y1 = (float(v) for v in box)
    return ((x0 + x1) / 2, (y0 + y1) / 2 if kind == CENTRE else y1)


def inside64(poly, p):
    """even-odd rule: the number of polygon edges a ray from p towards +x crosses"""
    xs, ys = np.asarray(poly[0], dtype=np.float64), np.asarray(poly[1], dtype=np.float64)
    xj, yj = np.roll(xs, 1), np.roll(ys, 1)
    span = (ys > p[1]) != (yj > p[1])
    with np.errstate(divide="ignore", invalid="ignore"):
        xcut = xs + (xj - xs) * (p[1] - ys) / (yj - ys)
    return bool(np.count_nonzero(span & (p[0] < xcut)) % 2)


def side64(seg, p):
    (ax, ay), (bx, by) = seg
    v = (bx - ax) * (p[1] - ay) - (by - ay) * (p[0] - ax)
    return int(np.sign(v))


def meets64(seg, p, q):
    (ax, ay), (bx, by) = seg
    dx, dy = q[0] - p[0], q[1] - p[1]
    oa, ob = dx * (ay - p[1]) - dy * (ax - p[0]), dx * (by - p[1]) - dy * (bx - p[0])
    return not (oa * ob > 0)


class Float64Zones:
    """one stream: zones as ((xs, ys), class, anchor, min_dwell), lines as (((x0, y0), (x1, y1)), class, anchor)"""

    def __init__(self, zones, lines):
        self.zones, self.lines = zones, lines
        self.tracks = {}  # track_id -> dict(box, cls, sigma, inside, dwelt, entry)
        self.pos, self.neg = [0] * len(lines), [0] * len(lines)

    def step(self, frame, live_ids, shown):
        live = set(int(v) for v in live_ids)
        events, occ = [], [0] * len(self.zones)  # events: (track_id, group, index, order, kind, class, value)
        for tid in sorted(self.tracks):
            if tid not in live:
                t = self.tracks.pop(tid)
                for z in range(len(self.zones)):
                    if t["inside"][z]:
                        events.append((tid, 1, z, 0, GONE, t["cls"], frame - t["entry"][z]))
        for r in shown:
            tid, cls, box = int(r["track_id"]), int(r["class_id"]), (r["x0"], r["y0"], r["x1"], r["y1"])
            first = tid not in self.tracks
            t = self.tracks.setdefault(tid, dict(box=box, cls=cls, sigma=[0] * len(self.lines), inside=[False] * len(self.zones),
                                                 dwelt=[False] * len(self.zones), entry=[0] * len(self.zones)))
            for l, (seg, lcls, anc) in enumerate(self.lines):
                p, q = anchors64(t["box"], anc), anchors64(box, anc)
                sq = side64(seg, q)
                if not first and sq and t["sigma"][l] == -sq and lcls in (-1, cls) and meets64(seg, p, q):
                    events.append((tid, 0, l, 0, CROSS_POS if sq > 0 else CROSS_NEG, cls, None))
                if sq:
                    t["sigma"][l] = sq
            for z, (poly, zcls, anc, min_dwell) in enumerate(self.zones):
                now = zcls in (-1, cls) and inside64(poly, anchors64(box, anc))
                if now and not t["inside"][z]:
                    events.append((tid, 1, z, 0, ENTER, cls, 1 if first else 0))
                    t["inside"][z], t["dwelt"][z], t["entry"][z] = True, False, frame
                if now and min_dwell > 0 and not t["dwelt"][z] and frame - t["entry"][z] + 1 >= min_dwell:
                    events.append((tid, 1, z, 1, DWELL, cls, frame - t["entry"][z] + 1))
                    t["dwelt"][z] = True
                if not now and t["inside"][z]:
                    events.append((tid, 1, z, 0, EXIT, cls, frame - t["entry"][z]))
                    t["inside"][z] = t["dwelt"][z] = False
                occ[z] += now
            t["box"], t["cls"] = box, cls
        out = []
        for tid, _, index, _, kind, cls, value in sorted(events, key=lambda e: e[:4]):
            if kind == CROSS_POS:
                self.pos[index] += 1
                value = self.pos[index]
            elif kind == CROSS_NEG:
                self.neg[index] += 1
                value = self.neg[index]
            out.append((tid, cls, kind, index, value))
        return out, occ, list(self.pos), list(self.neg)


# ---- scenes -------------------------------------------------------------------------------------------------------------------
def random_geometry(rng, width=1920.0, height=1080.0, n_zones=MAX_ZONES, n_verts=MAX_VERTS, n_lines=MAX_LINES):
    """star-shaped zones of n_verts vertices and lines anywhere, with classes from {-1, 0, 1}, both anchors and dwell thresholds"""
    zones, lines = [], []
    for _ in range(n_zones):
        c = rng.uniform([0.1 * width, 0.1 * height], [0.9 * width, 0.9 * height])
        ang = np.sort(rng.uniform(0, 2 * np.pi, n_verts))
        rad = rng.uniform(0.05, 0.3, n_verts) * min(width, height)
        pts = [(float(np.float32(c[0] + r * np.cos(a))), float(np.float32(c[1] + r * np.sin(a)))) for a, r in zip(ang, rad)]
        zones.append(zone(pts, int(rng.choice([-1, 0, 1])), int(rng.integers(0, 2)), int(rng.choice([0, 1, 2, 5, 20]))))
    for _ in range(n_lines):
        a = rng.uniform([0, 0], [width, height])
        b = a + rng.normal(0, 500, 2)
        lines.append(line(*(float(np.float32(v)) for v in (a[0], a[1], b[0], b[1])), int(rng.choice([-1, 0, 1])), int(rng.integers(0, 2))))
    return zones, lines


def as64(zones, lines):
    """the ctypes geometry in the form Float64Zones takes"""
    z64 = [((list(z.x)[: z.n_verts], list(z.y)[: z.n_verts]), z.class_id, z.anchor, z.min_dwell) for z in zones]
    l64 = [(((ln.x0, ln.y0), (ln.x1, ln.y1)), ln.class_id, ln.anchor) for ln in lines]
    return z64, l64


class _Clearance:
    """the geometry of one anchor kind as arrays: zone edges (i, j = i - 1) and lines"""

    def __init__(self, zones, lines):
        e = [(x, y, np.roll(x, 1), np.roll(y, 1)) for (x, y), _, _, _ in ((tuple(np.asarray(v) for v in z[0]),) + z[1:] for z in zones)]
        self.xi, self.yi, self.xj, self.yj = (np.concatenate([t[k] for t in e]) if e else np.zeros(0) for k in range(4))
        self.seg = np.array([[a[0], a[1], b[0], b[1]] for (a, b), _, _ in lines], dtype=np.float64).reshape(-1, 4)

    def ok(self, p, q, margin):
        """anchor q (and the step from p, when there is one) keeps its margins"""
        if self.yi.size:
            if np.min(np.abs(self.yi - q[1])) < margin:
                return False
            span = (self.yi > q[1]) != (self.yj > q[1])
            xcut = self.xi[span] + (self.xj[span] - self.xi[span]) * (q[1] - self.yi[span]) / (self.yj[span] - self.yi[span])
            if xcut.size and np.min(np.abs(xcut - q[0])) < margin:
                return False
        if self.seg.size:
            ax, ay, bx, by = self.seg.T
            if np.min(np.abs((bx - ax) * (q[1] - ay) - (by - ay) * (q[0] - ax)) / np.hypot(bx - ax, by - ay)) < margin:
                return False
            if p is not None:
                d = np.hypot(q[0] - p[0], q[1] - p[1])
                for ex, ey in ((ax, ay), (bx, by)):
                    if d == 0 or np.min(np.abs((q[0] - p[0]) * (ey - p[1]) - (q[1] - p[1]) * (ex - p[0]))) / d < margin:
                        return False
        return True


def walk_scene(seed, zones, lines, frames=300, n_obj=40, margin=1e-2, width=1920.0, height=1080.0):
    """per frame (live_ids, shown TRACK_DTYPE): objects on random walks with IDs in order of birth; each frame an object is shown,
    lost (not shown, still live) or removed for good, and new objects are born.  A step whose anchors would come closer than
    `margin` to the geometry is drawn again (the object is lost for the frame when ten draws fail).  Classes 0..2, switching now
    and then."""
    rng = np.random.default_rng(seed)
    z64, l64 = as64(zones, lines)
    clear = {k: _Clearance([z for z in z64 if z[2] == k], [ln for ln in l64 if ln[2] == k]) for k in (BOTTOM, CENTRE)}
    objs, issued, out = {}, 0, []
    for f in range(frames):
        while len(objs) < n_obj and rng.random() < 0.5:
            issued += 1
            w, h = rng.uniform(30, 120, 2)
            objs[issued] = dict(xy=rng.uniform([0, 0], [width - w, height - h]), v=rng.normal(0, 6, 2), wh=(w, h), cls=int(rng.integers(0, 3)),
                                last=None)
        for tid in list(objs):
            if rng.random() < 0.01:
                del objs[tid]
        shown = []
        for tid in sorted(objs):
            o = objs[tid]
            if rng.random() < 0.05:
                o["cls"] = int(rng.integers(0, 3))
            lost = rng.random() < 0.1
            for _ in range(10):
                v = o["v"] + rng.normal(0, 1.5, 2)
                xy = o["xy"] + v
                box = np.array([xy[0], xy[1], xy[0] + o["wh"][0], xy[1] + o["wh"][1]], dtype=np.float32)
                if lost or all(clear[k].ok(None if o["last"] is None else anchors64(o["last"], k), anchors64(box, k), margin)
                               for k in (BOTTOM, CENTRE)):
                    break
            else:
                lost = True
            o["v"], o["xy"] = np.clip(v, -12, 12), np.clip(xy, [-50, -50], [width, height])
            if not lost:
                o["last"] = box
                shown.append((*box, 0.9, o["cls"], tid, 0))
        out.append((np.array(sorted(objs), dtype=np.int32), np.array(shown, dtype=TRACK_DTYPE)))
    return out
