"""tools/zones_bench.py -- zones and counting lines on tracked streams (k_zones, mars_b200_set_zones), one GPU.

(a) k_zones device time next to k_track's (torch.profiler, CUDA activities, the kernels alone) on mars_b200_track_boxes at 64 and 512
    streams, every stream with geometry, in the two loads of tools/track_bench.py:
      typical: about 40 detections and 30 live tracks per stream, with 4 zones of 8 vertices and 4 lines per stream;
      worst:   1000 detections on a grid, 256 shown tracks, with 8 zones of 16 vertices and 8 lines per stream (the limits).
(b) the steady-state pooled stream of tools/track_bench.py (NanoDet-m-shaped 320x320 int8 graph, GFL heads, 64 pinned RGB8 640x360
    frames per micro-batch over two pools, maxd 100): submit_frames_track_batch with no geometry set against
    submit_frames_zones_batch with 4 zones and 4 lines on each of the 64 streams, alternating, two runs each.
The GPU name and power limit are read in the same run.
Usage: python tools/zones_bench.py [--frames 20] [--micro-batches 200] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from __graft_entry__ import load_package  # noqa: E402
from track_bench import ARENA, FH, FW, MAXD, MICRO, SIDE, gpu_info, pinned, typical, worst  # noqa: E402


def geometry(capi, rng, n_zones, n_verts, n_lines, w, h):
    """star-shaped zones and random lines over a w x h frame, both anchors, classes any"""
    zones, lines = [], []
    for _ in range(n_zones):
        c = rng.uniform([0.2 * w, 0.2 * h], [0.8 * w, 0.8 * h])
        ang, rad = np.sort(rng.uniform(0, 2 * np.pi, n_verts)), rng.uniform(0.05, 0.3, n_verts) * min(w, h)
        zones.append(capi.ZONE([(float(c[0] + r * np.cos(a)), float(c[1] + r * np.sin(a))) for a, r in zip(ang, rad)],
                               anchor=int(rng.integers(0, 2)), min_dwell=int(rng.choice([0, 10, 30]))))
    for _ in range(n_lines):
        a, b = rng.uniform([0, 0], [w, h]), rng.uniform([0, 0], [w, h])
        lines.append(capi.LINE(float(a[0]), float(a[1]), float(b[0]), float(b[1]), anchor=int(rng.integers(0, 2))))
    return zones, lines


def kernel_times(pkg, load, S, a):
    import torch
    from torch.profiler import ProfilerActivity, profile
    rng = np.random.default_rng(S)
    gen = typical if load == "typical" else worst
    warm = 30 if load == "typical" else 1
    seq = gen(rng, S, warm + a.frames)
    gm = pkg.MarsModel(pkg.marsfile.build_nanodet_like(size=SIDE, seed=7).to_bytes(), arena_bytes=ARENA, device=0)
    gm.set_tracking(S)
    shape, (w, h) = ((4, 8, 4), (1500.0, 1500.0)) if load == "typical" else ((8, 16, 8), (960.0, 600.0))
    for s in range(S):
        gm.set_zones(s, *geometry(pkg.capi, rng, *shape, w, h))
    streams = list(range(S))
    for f in range(warm):
        gm.track_boxes(streams, seq[f])
    torch.cuda.synchronize()
    events = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for f in range(warm, warm + a.frames):
            _, counts, zr = gm.track_boxes_zones(streams, seq[f])
            events.append(float(np.mean(zr["n_events"])))
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kz = [e.time_range.elapsed_us() / 1e3 for e in ev if "k_zones" in e.name]
    kt = [e.time_range.elapsed_us() / 1e3 for e in ev if "k_track" in e.name]
    gm.close()
    return {"load": load, "streams": S, "zones_verts_lines": shape, "calls": len(kz), "k_zones_median_ms": float(np.median(kz)),
            "k_zones_mean_ms": float(np.mean(kz)), "k_track_median_ms": float(np.median(kt)), "shown_tracks_per_stream": float(np.mean(counts)),
            "events_per_stream": float(np.mean(events))}


def stream(pkg, a):
    L = pkg.lib()
    C = pkg.capi
    gm = pkg.MarsModel(pkg.marsfile.build_nanodet_like(size=SIDE, seed=7).to_bytes(), arena_bytes=ARENA, device=0, batch=2 * MICRO)
    gm.set_gfl_heads(None, 80, 7, "half", 0.25)
    gm.set_tracking(MICRO)
    rng = np.random.default_rng(3)
    geo = [geometry(C, rng, 4, 8, 4, float(FW), float(FH)) for _ in range(MICRO)]
    n_src = 256
    src, src_p = pinned(L, n_src * FH * FW * 3)
    src[:] = np.random.default_rng(7).integers(0, 256, src.size, dtype=np.uint8)
    frames = src.reshape(n_src, FH, FW, 3)
    tracks = [pinned(L, MICRO * MAXD * 32) for _ in range(2)]
    counts = [pinned(L, MICRO * 4, np.int32) for _ in range(2)]
    zones = [pinned(L, MICRO * C.ZONE_FRAME_DTYPE.itemsize) for _ in range(2)]
    streams = np.arange(MICRO, dtype=np.int32)
    nmb = a.micro_batches

    def run(with_zones):
        for s in range(MICRO):  # outside the timed window: geometry on every stream, or none anywhere
            gm.set_zones(s, *(geo[s] if with_zones else ((), ())))
        lat, t_sub = [], [0.0, 0.0]
        t0 = time.perf_counter()
        for j in range(nmb):
            h = j & 1
            if j >= 2:
                gm.wait_batch(h)
                lat.extend([time.perf_counter() - t_sub[h]] * MICRO)
            fs = [frames[(j * MICRO + i) % n_src] for i in range(MICRO)]
            t_sub[h] = time.perf_counter()
            out = tracks[h][0].view(C.TRACK_DTYPE)
            if with_zones:
                gm.submit_frames_zones_batch(h, fs, streams, out, counts[h][0], zones[h][0].view(C.ZONE_FRAME_DTYPE), MAXD, 0.45)
            else:
                gm.submit_frames_track_batch(h, fs, streams, out, counts[h][0], MAXD, 0.45)
        for j in range(nmb - 2, nmb):
            gm.wait_batch(j & 1)
            lat.extend([time.perf_counter() - t_sub[j & 1]] * MICRO)
        wall = time.perf_counter() - t0
        lat = np.asarray(lat) * 1e3
        return {"frames_per_s": nmb * MICRO / wall, "p50_ms": float(np.percentile(lat, 50)), "p99_ms": float(np.percentile(lat, 99))}

    res = []
    for r in range(2):
        for name, z in (("submit_frames_track_batch", False), ("submit_frames_zones_batch", True)):
            run(z)  # warm-up
            res.append(dict(run=r, flavour=name, **run(z)))
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        gm.submit_frames_zones_batch(0, [frames[i] for i in range(MICRO)], streams, tracks[0][0].view(C.TRACK_DTYPE), counts[0][0],
                                     zones[0][0].view(C.ZONE_FRAME_DTYPE), MAXD, 0.45)
        gm.wait_batch(0)
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    split = {"k_zones_ms_per_micro_batch": float(sum(e.time_range.elapsed_us() for e in ev if "k_zones" in e.name) / 1e3),
             "k_track_ms_per_micro_batch": float(sum(e.time_range.elapsed_us() for e in ev if "k_track" in e.name) / 1e3),
             "shown_tracks_per_frame": float(np.mean(counts[0][0])),
             "events_per_frame": float(np.mean(zones[0][0].view(C.ZONE_FRAME_DTYPE)["n_events"]))}
    gm.close()
    for buf in [(src, src_p)] + tracks + counts + zones:
        L.nna_free(buf[1])
    return {"micro_batch": MICRO, "micro_batches": nmb, "frame": [FW, FH], "maxd": MAXD, "runs": res, "split": split}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--micro-batches", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    pkg = load_package()
    res = {"gpu": gpu_info(), "kernel": [kernel_times(pkg, load, S, a) for load in ("typical", "worst") for S in (64, 512)],
           "stream": stream(pkg, a)}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(text + "\n")


if __name__ == "__main__":
    main()
