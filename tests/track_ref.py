"""Reference flows of the multi-object tracker (mars_b200_set_tracking), for the tests.

OracleTracker runs the C statement of the tracker (tests/track_oracle.c, compiled with -ffp-contract=off into a temporary directory
on first use), one state per stream.  Float64Tracker is an independent restatement in float64: ByteTrack's Kalman filter in its
literal 8x8 form (F, H, diagonal Q and R, the update through a Cholesky solve) and the same schedule with the literal greedy
matching.  lanes_sequence generates detections whose decisions cannot flip on rounding: objects in separate horizontal lanes
(boxes of different objects never overlap), births, exits, changing velocities and occlusions.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
from scipy.linalg import cho_factor, cho_solve

BOX_DTYPE = np.dtype([("x0", "<f4"), ("y0", "<f4"), ("x1", "<f4"), ("y1", "<f4"), ("confidence", "<f4"), ("class_id", "<i4")])
TRACK_DTYPE = np.dtype([("x0", "<f4"), ("y0", "<f4"), ("x1", "<f4"), ("y1", "<f4"), ("confidence", "<f4"), ("class_id", "<i4"),
                        ("track_id", "<i4"), ("det_index", "<i4")])
MAX_TRACKS, MAX_DETS = 256, 1000
DEFAULTS = dict(high_thresh=0.5, low_thresh=0.1, new_thresh=0.6, sim_high=0.2, sim_low=0.5, sim_unconfirmed=0.3, max_lost=30,
                class_aware=0)
_clib = None


class Params(C.Structure):
    """mars_b200_track_params_t"""
    _fields_ = [("high_thresh", C.c_float), ("low_thresh", C.c_float), ("new_thresh", C.c_float), ("sim_high", C.c_float),
                ("sim_low", C.c_float), ("sim_unconfirmed", C.c_float), ("max_lost", C.c_int32), ("class_aware", C.c_int32)]


def params(**kw):
    return Params(**{**DEFAULTS, **kw})


def _lib():
    global _clib
    if _clib is None:
        src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "track_oracle.c")
        so = os.path.join(tempfile.mkdtemp(prefix="track_oracle_"), "libtrack_oracle.so")
        subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-o", so, src, "-lm"], check=True)
        _clib = C.CDLL(so)
        _clib.trk_stream_bytes.restype = C.c_int
        _clib.trk_step.restype = C.c_int
        _clib.trk_step.argtypes = [C.c_void_p, C.POINTER(Params), C.c_void_p, C.c_int, C.c_void_p]
    return _clib


class OracleTracker:
    """the C statement, one state per stream"""

    def __init__(self, n_streams, p=None):
        self.p = p if p is not None else params()
        self.state = np.zeros((n_streams, _lib().trk_stream_bytes()), dtype=np.uint8)

    def reset(self, first, n):
        self.state[first: first + n] = 0

    def step(self, stream, boxes):
        """boxes: BOX_DTYPE array (the frame's kept boxes) -> TRACK_DTYPE array"""
        b = np.ascontiguousarray(boxes, dtype=BOX_DTYPE)
        out = np.zeros(MAX_TRACKS, dtype=TRACK_DTYPE)
        n = _lib().trk_step(self.state[stream].ctypes.data, C.byref(self.p), b.ctypes.data, len(b), out.ctypes.data)
        return out[:n].copy()


# ---- the float64 restatement -----------------------------------------------------------------------------------------------
WP, WV = 1.0 / 20, 1.0 / 160
F = np.eye(8)
F[:4, 4:] = np.eye(4)
H = np.eye(4, 8)


def iou64(a, b):
    x0, y0, x1, y1 = max(a[0], b[0]), max(a[1], b[1]), min(a[2], b[2]), min(a[3], b[3])
    inter = max(0.0, x1 - x0) * max(0.0, y1 - y0)
    return inter / ((a[2] - a[0]) * (a[3] - a[1]) + (b[2] - b[0]) * (b[3] - b[1]) - inter + 1e-6)


def measure64(b):
    w, h = b[2] - b[0], b[3] - b[1]
    return np.array([b[0] + w / 2, b[1] + h / 2, w / h, h])


class Track64:
    def __init__(self, z, tid, det, j, frame, activated):
        h = z[3]
        std = np.array([2 * WP * h, 2 * WP * h, 1e-2, 2 * WP * h, 10 * WV * h, 10 * WV * h, 1e-5, 10 * WV * h])
        self.mean, self.cov = np.r_[z, np.zeros(4)], np.diag(std ** 2)
        self.id, self.state, self.activated, self.last = tid, "tracked", activated, frame
        self.conf, self.cls, self.j = float(det["confidence"]), int(det["class_id"]), j

    def predict(self):
        if self.state == "lost":
            self.mean[7] = 0.0
        h = self.mean[3]
        q = np.array([WP * h, WP * h, 1e-2, WP * h, WV * h, WV * h, 1e-5, WV * h])
        self.mean = F @ self.mean
        self.cov = F @ self.cov @ F.T + np.diag(q ** 2)

    def update(self, z):
        h = self.mean[3]
        R = np.diag(np.array([WP * h, WP * h, 1e-1, WP * h]) ** 2)
        S = H @ self.cov @ H.T + R
        K = cho_solve(cho_factor(S, lower=True), (self.cov @ H.T).T).T
        self.mean = self.mean + K @ (z - H @ self.mean)
        self.cov = self.cov - K @ S @ K.T

    def box(self):
        cx, cy, a, h = self.mean[:4]
        w = a * h
        return np.array([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2])


class Float64Tracker:
    """the same schedule in float64, one stream; margins collects |sim - gate| of every pair with a positive similarity"""

    def __init__(self, **kw):
        self.p = {**DEFAULTS, **kw}
        self.tracks, self.frame, self.issued = [], 0, 0
        self.margins = []

    def _greedy(self, tracks, dets, idx, with_conf, gate, tm, dm):
        pairs = []
        for t in tracks:
            for j in idx:
                d = dets[j]
                if self.p["class_aware"] and int(d["class_id"]) != t.cls:
                    continue
                sim = iou64(t.box(), [float(d[k]) for k in ("x0", "y0", "x1", "y1")])
                if with_conf:
                    sim *= float(d["confidence"])
                if sim > 0:
                    self.margins.append(abs(sim - gate))
                if sim > gate:
                    pairs.append((-sim, t.id, j, t))
        for _, _, j, t in sorted(pairs, key=lambda q: q[:3]):
            if t.id not in tm and j not in dm:
                tm[t.id], dm[j] = j, t

    def step(self, dets):
        p = self.p
        self.frame += 1
        f = self.frame
        ok = [bool(np.all(np.isfinite([d["x0"], d["y0"], d["x1"], d["y1"], d["confidence"]]))) and float(d["x1"] - d["x0"]) > 0 and
              float(d["y1"] - d["y0"]) > 0 for d in dets]
        conf = [float(d["confidence"]) for d in dets]
        high = [j for j in range(len(dets)) if ok[j] and conf[j] > p["high_thresh"]]
        low = [j for j in range(len(dets)) if ok[j] and p["low_thresh"] < conf[j] < p["high_thresh"]]
        pool = [t for t in self.tracks if t.state == "lost" or t.activated]
        unconf = [t for t in self.tracks if t.state == "tracked" and not t.activated]
        for t in pool:
            t.predict()
        tm, dm = {}, {}
        self._greedy(pool, dets, high, True, p["sim_high"], tm, dm)
        self._greedy([t for t in pool if t.state == "tracked" and t.id not in tm], dets, low, False, p["sim_low"], tm, dm)
        self._greedy(unconf, dets, [j for j in high if j not in dm], True, p["sim_unconfirmed"], tm, dm)
        live = []
        for t in self.tracks:
            if t.id in tm:
                j = tm[t.id]
                t.update(measure64([float(dets[j][k]) for k in ("x0", "y0", "x1", "y1")]))
                t.state, t.activated, t.last = "tracked", True, f
                t.conf, t.cls, t.j = conf[j], int(dets[j]["class_id"]), j
            elif t in pool and t.state == "tracked":
                t.state = "lost"
            elif t in unconf:
                continue
            live.append(t)
        for j in high:
            if j not in dm and conf[j] >= p["new_thresh"] and len(live) < MAX_TRACKS:
                self.issued += 1
                d = dets[j]
                live.append(Track64(measure64([float(d[k]) for k in ("x0", "y0", "x1", "y1")]), self.issued, d, j, f, f == 1))
        self.tracks = [t for t in live if not (t.state == "lost" and f - t.last > p["max_lost"])]
        out = [t for t in self.tracks if t.state == "tracked" and t.activated]
        return [(t.id, t.j, t.box(), t.conf, t.cls) for t in out]


# ---- sequences --------------------------------------------------------------------------------------------------------------
def lanes_sequence(seed, frames=300, lanes=12, width=1920.0, lane_h=90.0):
    """detections (a BOX_DTYPE array per frame) of objects that each keep to one horizontal lane, so boxes of different objects
    never overlap.  Each lane hosts objects one after another: a birth at a random frame, motion with a drifting velocity and a
    small vertical oscillation, detections with ~1 px noise and confidence 0.8..0.95, stretches detected only with confidence 0.3
    (kept alive by the low-score stage), stretches without detections (lost, then found again, or expired) and an exit."""
    rng = np.random.default_rng(seed)
    per_frame = [[] for _ in range(frames)]
    for lane in range(lanes):
        t = int(rng.integers(0, 40))
        while t < frames - 5:
            life = int(rng.integers(40, 200))
            x = float(rng.uniform(0, width - 200))
            vx = float(rng.uniform(-6, 6))
            w, h = float(rng.uniform(40, 110)), float(rng.uniform(40, 70))
            cy0 = lane * lane_h + lane_h / 2
            amp, om = float(rng.uniform(0, 4)), float(rng.uniform(0.02, 0.1))
            low0 = int(rng.integers(5, 30)) if rng.random() < 0.5 else -1
            gap0 = int(rng.integers(30, 60)) if rng.random() < 0.5 else -1
            gap_len = int(rng.integers(2, 12))
            for k in range(min(life, frames - t)):
                f = t + k
                vx += float(rng.normal(0, 0.05))
                x += vx
                cy = cy0 + amp * np.sin(om * k)
                if x < -w or x > width:
                    break
                if gap0 >= 0 and gap0 <= k < gap0 + gap_len:
                    continue
                conf = 0.3 if low0 >= 0 and low0 <= k < low0 + 6 else float(rng.uniform(0.8, 0.95))
                nz = rng.normal(0, 1.0, 4)
                per_frame[f].append((x + nz[0], cy - h / 2 + nz[1], x + w + nz[2], cy + h / 2 + nz[3], conf, lane % 3))
            t += life + int(rng.integers(40, 80))  # the lane stays empty long enough for the old track to expire
    out = []
    for dets in per_frame:
        order = rng.permutation(len(dets))
        out.append(np.array([dets[i] for i in order], dtype=BOX_DTYPE))
    return out
