"""tools/frames_bench.py -- letterbox pre-processing of camera frames on the device, three measurements:
  (a) uniform:  64 frames of 1920x1080 -> 640x640 through mars_b200_preprocess_batch (the path every caller had before)
  (b) mixed:    one camera batch of 64 frames -- half 1920x1080, a quarter 1280x720, a quarter 640x360 -- as one
                mars_b200_preprocess_frames call, and grouped by size through three mars_b200_preprocess_batch calls
  (c) steady:   mars_b200_submit_frames_heads_batch on the yolov5s-shaped heads model, alternating pools, pinned frames:
                frames/s and the latency from submit to boxes on the host (p50 / p99)
Frames live in pinned host memory (nna_malloc).  Device times are CUDA events around the copies + kernels; host times are
wall clock around calls that end in a device synchronisation.
usage: python tools/frames_bench.py [--part a|b|c|all] [--repeat N] [--batches N] [--pool N]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from __graft_entry__ import load_package  # noqa: E402

pkg = load_package()
L = pkg.capi.lib()
mf = pkg.marsfile


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi unavailable (%s)" % e
    return q


def pinned_frames(shapes, seed):
    """one pinned buffer holding the frames back to back; returns (views, pointer)"""
    total = sum(w * h * 3 for (w, h) in shapes)
    ptr = L.nna_malloc(total)
    assert ptr, "nna_malloc(%d)" % total
    buf = np.ctypeslib.as_array((C.c_uint8 * total).from_address(ptr))
    rng = np.random.default_rng(seed)
    out, at = [], 0
    for (w, h) in shapes:
        v = buf[at: at + w * h * 3].reshape(h, w, 3)
        v[...] = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        out.append(v)
        at += w * h * 3
    return out, ptr


def timed(fn, repeat, warmup=2):
    for _ in range(warmup):
        fn()
    dev, wall = [], []
    for _ in range(repeat):
        t0 = time.perf_counter()
        dev.append(fn())
        wall.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(dev)), float(np.median(wall)), float(np.min(wall)), float(np.max(wall))


def letterbox_model(batch):
    return pkg.MarsModel(mf.build_yolov5(width=0.5, size=640, seed=5).to_bytes(), arena_bytes=mf.ARENA_YOLOV5S_INT8, device=0, batch=batch)


def part_a(repeat):
    n = 64
    frames, ptr = pinned_frames([(1920, 1080)] * n, 0)
    gm = letterbox_model(n)
    block = np.ctypeslib.as_array((C.c_uint8 * (n * 1920 * 1080 * 3)).from_address(ptr)).reshape(n, 1080, 1920, 3)
    dev, wall, lo, hi = timed(lambda: gm.preprocess(0, block), repeat)
    gm.close()
    L.nna_free(ptr)
    return dict(part="a", frames=n, size="1920x1080", device_ms=round(dev, 3), wall_ms=round(wall, 3), wall_min_ms=round(lo, 3),
                wall_max_ms=round(hi, 3), frames_per_s=round(n / wall * 1e3, 1))


def part_b(repeat):
    groups = [((1920, 1080), 32), ((1280, 720), 16), ((640, 360), 16)]
    bufs = {size: pinned_frames([size] * k, i) for i, (size, k) in enumerate(groups)}
    # the ragged call sees the sizes interleaved, as cameras deliver them
    order = []
    for i in range(32):
        order.append(bufs[(1920, 1080)][0][i])
        if i % 2 == 0:
            order.append(bufs[(1280, 720)][0][i // 2])
        else:
            order.append(bufs[(640, 360)][0][i // 2])
    gm = letterbox_model(64)
    dev1, wall1, lo1, hi1 = timed(lambda: gm.preprocess_frames(0, order), repeat)

    def grouped():
        first, ms = 0, 0.0
        for (w, h), k in groups:
            views, ptr = bufs[(w, h)]
            block = np.ctypeslib.as_array((C.c_uint8 * (k * w * h * 3)).from_address(ptr)).reshape(k, h, w, 3)
            ms += gm.preprocess(first, block)
            first += k
        return ms

    dev2, wall2, lo2, hi2 = timed(grouped, repeat)
    gm.close()
    for _, ptr in bufs.values():
        L.nna_free(ptr)
    return dict(part="b", frames=64, mix="32x1920x1080 + 16x1280x720 + 16x640x360",
                frames_call=dict(device_ms=round(dev1, 3), wall_ms=round(wall1, 3), wall_min_ms=round(lo1, 3), wall_max_ms=round(hi1, 3),
                                 frames_per_s=round(64 / wall1 * 1e3, 1)),
                grouped_calls=dict(device_ms=round(dev2, 3), wall_ms=round(wall2, 3), wall_min_ms=round(lo2, 3), wall_max_ms=round(hi2, 3),
                                   frames_per_s=round(64 / wall2 * 1e3, 1)))


def part_c(batches, pool_n, sizes):
    gm = pkg.MarsModel(mf.build_yolov5(width=0.5, size=640, seed=5).to_bytes(), arena_bytes=mf.ARENA_YOLOV5S_INT8, device=0,
                       batch=2 * pool_n)
    gm.set_yolo_heads(None, 0.25)
    # two distinct sets of frames, one per pool
    sets = [pinned_frames([sizes[i % len(sizes)] for i in range(pool_n)], 20 + p) for p in range(2)]
    out = [(np.zeros((pool_n, 100), dtype=pkg.capi.BOX_DTYPE), np.zeros(pool_n, dtype=np.int32)) for _ in range(2)]
    sub, lat = {}, []

    def run(k):
        for i in range(k):
            pool = i % 2
            if i >= 2:
                gm.wait_batch(pool)
                lat.append((time.perf_counter() - sub[i - 2]) * 1e3)
            sub[i] = time.perf_counter()
            gm.submit_frames_heads_batch(pool, sets[pool][0], out[pool][0], out[pool][1], maxd=100)
        for i in (k - 2, k - 1):
            gm.wait_batch(i % 2)
            lat.append((time.perf_counter() - sub[i]) * 1e3)

    run(6)  # warm-up: staging, tap lists, the captured step graphs
    sub.clear()
    lat.clear()
    t0 = time.perf_counter()
    run(batches)
    dt = time.perf_counter() - t0
    gm.close()
    for _, ptr in sets:
        L.nna_free(ptr)
    nbytes = sum(w * h * 3 for (w, h) in [sizes[i % len(sizes)] for i in range(pool_n)])
    fps = batches * pool_n / dt
    return dict(part="c", model="yolov5s-shaped heads (width 0.5, 640)", pool_frames=pool_n, batches=batches,
                sizes=sorted({"%dx%d" % s for s in sizes}), frames_per_s=round(fps, 1),
                h2d_gb_per_s=round(fps * nbytes / pool_n / 1e9, 2),
                latency_ms_p50=round(float(np.percentile(lat, 50)), 3), latency_ms_p99=round(float(np.percentile(lat, 99)), 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--part", default="all", choices=["a", "b", "c", "all"])
    ap.add_argument("--repeat", type=int, default=20)
    ap.add_argument("--batches", type=int, default=60)
    ap.add_argument("--pool", type=int, default=32, help="frames per submit (half the slots)")
    a = ap.parse_args()
    print(json.dumps(dict(gpu=gpu_info())))
    if a.part in ("a", "all"):
        print(json.dumps(part_a(a.repeat)))
    if a.part in ("b", "all"):
        print(json.dumps(part_b(a.repeat)))
    if a.part in ("c", "all"):
        print(json.dumps(part_c(a.batches, a.pool, [(1920, 1080)])))
        print(json.dumps(part_c(a.batches, a.pool, [(1920, 1080), (1280, 720), (1920, 1080), (640, 360)])))


if __name__ == "__main__":
    main()
