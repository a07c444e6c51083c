"""tools/track_bench.py -- the multi-object tracker (k_track, mars_b200_set_tracking), one GPU.

(a) k_track device time (torch.profiler, CUDA activities: the kernel alone, without the uploads and read-backs of
    mars_b200_track_boxes) at 64 and 512 streams in two loads:
      typical: 30 objects on random walks, each detected with probability 0.9, plus 0..20 clutter boxes (about 40 detections and
               30 live tracks per frame), measured after 30 warm-up frames;
      worst:   1000 detections per frame on a grid, 256 live tracks from the first frame on.
(b) the steady-state pooled stream on the NanoDet-m-shaped 320x320 int8 graph of `bench.py --config streams` (build_nanodet_like
    seed 7, 16 MiB arena, GFL heads), 64 RGB8 640x360 frames per micro-batch from pinned host memory over two pools:
    submit_frames_heads_batch (maxd 100) against submit_frames_track_batch (64 streams, maxd 100), alternating, two runs each.
Usage: python tools/track_bench.py [--frames 20] [--micro-batches 200] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from __graft_entry__ import load_package  # noqa: E402

SIDE, ARENA, MICRO, MAXD, FW, FH = 320, 16 << 20, 64, 100, 640, 360


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def typical(rng, S, frames, n_obj=30):
    box = np.dtype([("x0", "<f4"), ("y0", "<f4"), ("x1", "<f4"), ("y1", "<f4"), ("confidence", "<f4"), ("class_id", "<i4")])
    pos = rng.uniform(0, 1500, (S, n_obj, 2))
    vel = rng.normal(0, 3, (S, n_obj, 2))
    wh = rng.uniform(30, 120, (S, n_obj, 2))
    out = []
    for _ in range(frames):
        vel += rng.normal(0, 0.3, vel.shape)
        pos += vel
        fr = []
        for s in range(S):
            seen = rng.random(n_obj) < 0.9
            k = int(seen.sum()) + int(rng.integers(0, 21))
            b = np.zeros(k, dtype=box)
            xy = np.concatenate([pos[s][seen] + rng.normal(0, 2, (seen.sum(), 2)), rng.uniform(0, 1500, (k - seen.sum(), 2))])
            whk = np.concatenate([wh[s][seen], rng.uniform(20, 60, (k - seen.sum(), 2))])
            b["x0"], b["y0"], b["x1"], b["y1"] = xy[:, 0], xy[:, 1], xy[:, 0] + whk[:, 0], xy[:, 1] + whk[:, 1]
            b["confidence"] = np.concatenate([rng.uniform(0.4, 0.95, seen.sum()), rng.uniform(0.05, 0.7, k - seen.sum())])
            fr.append(b)
        out.append(fr)
    return out


def worst(rng, S, frames):
    box = np.dtype([("x0", "<f4"), ("y0", "<f4"), ("x1", "<f4"), ("y1", "<f4"), ("confidence", "<f4"), ("class_id", "<i4")])
    gx, gy = np.meshgrid(np.arange(40) * 24.0, np.arange(25) * 24.0)
    base = np.stack([gx.ravel(), gy.ravel()], axis=1)
    out = []
    for _ in range(frames):
        fr = []
        for _ in range(S):
            xy = base + rng.normal(0, 2, base.shape)
            b = np.zeros(1000, dtype=box)
            b["x0"], b["y0"], b["x1"], b["y1"] = xy[:, 0], xy[:, 1], xy[:, 0] + 30, xy[:, 1] + 30
            b["confidence"] = rng.uniform(0.6, 0.95, 1000)
            fr.append(b)
        out.append(fr)
    return out


def kernel_times(pkg, load, S, a):
    """median and mean k_track time per call over a.frames profiled calls, and the live tracks / detections per stream"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    rng = np.random.default_rng(S)
    gen = typical if load == "typical" else worst
    warm = 30 if load == "typical" else 1
    seq = gen(rng, S, warm + a.frames)
    gm = pkg.MarsModel(pkg.marsfile.build_nanodet_like(size=SIDE, seed=7).to_bytes(), arena_bytes=ARENA, device=0)
    gm.set_tracking(S)
    streams = list(range(S))
    for f in range(warm):
        _, counts = gm.track_boxes(streams, seq[f])
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for f in range(warm, warm + a.frames):
            _, counts = gm.track_boxes(streams, seq[f])
    ms = [e.time_range.elapsed_us() / 1e3 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "k_track" in e.name]
    gm.close()
    return {"load": load, "streams": S, "calls": len(ms), "k_track_median_ms": float(np.median(ms)), "k_track_mean_ms": float(np.mean(ms)),
            "shown_tracks_per_stream": float(np.mean(counts)), "detections_per_stream": float(np.mean([len(b) for b in seq[-1]]))}


def pinned(L, nbytes, dtype=np.uint8):
    p = L.nna_malloc(nbytes)
    if not p:
        raise MemoryError("nna_malloc(%d)" % nbytes)
    return np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(p)).view(dtype), p


def stream(pkg, a):
    L = pkg.lib()
    gm = pkg.MarsModel(pkg.marsfile.build_nanodet_like(size=SIDE, seed=7).to_bytes(), arena_bytes=ARENA, device=0, batch=2 * MICRO)
    gm.set_gfl_heads(None, 80, 7, "half", 0.25)
    gm.set_tracking(MICRO)
    n_src = 256
    src, src_p = pinned(L, n_src * FH * FW * 3)
    src[:] = np.random.default_rng(7).integers(0, 256, src.size, dtype=np.uint8)
    frames = src.reshape(n_src, FH, FW, 3)
    boxes = [pinned(L, MICRO * MAXD * 24) for _ in range(2)]
    tracks = [pinned(L, MICRO * MAXD * 32) for _ in range(2)]
    counts = [pinned(L, MICRO * 4, np.int32) for _ in range(2)]
    streams = np.arange(MICRO, dtype=np.int32)
    nmb = a.micro_batches

    def run(track):
        lat, t_sub = [], [0.0, 0.0]
        t0 = time.perf_counter()
        for j in range(nmb):
            h = j & 1
            if j >= 2:
                gm.wait_batch(h)
                lat.extend([time.perf_counter() - t_sub[h]] * MICRO)
            fs = [frames[(j * MICRO + i) % n_src] for i in range(MICRO)]
            t_sub[h] = time.perf_counter()
            if track:
                gm.submit_frames_track_batch(h, fs, streams, tracks[h][0].view(pkg.capi.TRACK_DTYPE), counts[h][0], MAXD, 0.45)
            else:
                gm.submit_frames_heads_batch(h, fs, boxes[h][0].view(pkg.capi.BOX_DTYPE), counts[h][0], MAXD, 0.45)
        for j in range(nmb - 2, nmb):
            gm.wait_batch(j & 1)
            lat.extend([time.perf_counter() - t_sub[j & 1]] * MICRO)
        wall = time.perf_counter() - t0
        lat = np.asarray(lat) * 1e3
        return {"frames_per_s": nmb * MICRO / wall, "p50_ms": float(np.percentile(lat, 50)), "p99_ms": float(np.percentile(lat, 99))}

    res = []
    for r in range(2):
        for name, track in (("submit_frames_heads_batch", False), ("submit_frames_track_batch", True)):
            run(track)  # warm-up: the staging, the capture of the 64-frame step
            res.append(dict(run=r, flavour=name, **run(track)))
    # where the tracking time goes: k_track of one micro-batch (profiled on its own), and the load it saw
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        gm.submit_frames_track_batch(0, [frames[i] for i in range(MICRO)], streams, tracks[0][0].view(pkg.capi.TRACK_DTYPE), counts[0][0],
                                     MAXD, 0.45)
        gm.wait_batch(0)
    k_ms = [e.time_range.elapsed_us() / 1e3 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "k_track" in e.name]
    _, kept = gm.download_boxes(0, MICRO)
    split = {"k_track_ms_per_micro_batch": float(sum(k_ms)), "kept_boxes_per_frame": float(np.mean(kept)),
             "shown_tracks_per_frame": float(np.mean(counts[0][0]))}
    gm.close()
    for buf in [(src, src_p)] + boxes + tracks + counts:
        L.nna_free(buf[1])
    return {"micro_batch": MICRO, "micro_batches": nmb, "frame": [FW, FH], "maxd": MAXD, "runs": res, "track_split": split}


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
