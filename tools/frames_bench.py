"""tools/frames_bench.py -- letterbox pre-processing of camera frames on the device, three measurements:
  (a) uniform:  64 frames of 1920x1080 -> 640x640 through mars_b200_preprocess_batch (the path every caller had before)
  (b) mixed:    one camera batch of 64 frames -- half 1920x1080, a quarter 1280x720, a quarter 640x360 -- as one
                mars_b200_preprocess_frames call, and grouped by size through three mars_b200_preprocess_batch calls
  (c) steady:   mars_b200_submit_frames_heads_batch on the yolov5s-shaped heads model, alternating pools, pinned frames:
                frames/s and the latency from submit to boxes on the host (p50 / p99)
  (d) nv12:     1920x1080 NV12 frames against RGB8 frames of the same size: 64 device-resident frames letterboxed in place
                (mars_b200_preprocess_frames[_nv12]_device; ms by CUDA events, source bytes per frame, GB/s of source read), and
                the steady-state submit of (c) from pinned NV12 frames (mars_b200_submit_frames_nv12_heads_batch)
Frames live in pinned host memory (nna_malloc).  Device times are CUDA events around the copies + kernels; host times are
wall clock around calls that end in a device synchronisation.
usage: python tools/frames_bench.py [--part a|b|c|d|all] [--repeat N] [--batches N] [--pool N]"""
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


def frame_bytes(w, h, nv12=False):
    return w * h + 2 * ((w + 1) // 2) * ((h + 1) // 2) if nv12 else w * h * 3


def pinned_frames(shapes, seed, nv12=False):
    """one pinned buffer holding the frames back to back -- RGB8 [h, w, 3] arrays, or NV12 (y, uv, BT.709 limited) tuples with
    each frame's chroma plane right after its luma plane; returns (frames, pointer)"""
    total = sum(frame_bytes(w, h, nv12) for (w, h) in shapes)
    ptr = L.nna_malloc(total)
    assert ptr, "nna_malloc(%d)" % total
    buf = np.ctypeslib.as_array((C.c_uint8 * total).from_address(ptr))
    rng = np.random.default_rng(seed)
    buf[...] = rng.integers(0, 256, total, dtype=np.uint8)
    out, at = [], 0
    for (w, h) in shapes:
        if nv12:
            uv = buf[at + w * h: at + frame_bytes(w, h, True)].reshape((h + 1) // 2, (w + 1) // 2, 2)
            out.append((buf[at: at + w * h].reshape(h, w), uv, pkg.capi.YUV_BT709_LIMITED))
        else:
            out.append(buf[at: at + w * h * 3].reshape(h, w, 3))
        at += frame_bytes(w, h, nv12)
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


def part_c(batches, pool_n, sizes, nv12=False):
    gm = pkg.MarsModel(mf.build_yolov5(width=0.5, size=640, seed=5).to_bytes(), arena_bytes=mf.ARENA_YOLOV5S_INT8, device=0,
                       batch=2 * pool_n)
    gm.set_yolo_heads(None, 0.25)
    # two distinct sets of frames, one per pool
    sets = [pinned_frames([sizes[i % len(sizes)] for i in range(pool_n)], 20 + p, nv12) for p in range(2)]
    submit = gm.submit_frames_nv12_heads_batch if nv12 else gm.submit_frames_heads_batch
    out = [(np.zeros((pool_n, 100), dtype=pkg.capi.BOX_DTYPE), np.zeros(pool_n, dtype=np.int32)) for _ in range(2)]
    sub, lat = {}, []

    def run(k):
        for i in range(k):
            pool = i % 2
            if i >= 2:
                gm.wait_batch(pool)
                lat.append((time.perf_counter() - sub[i - 2]) * 1e3)
            sub[i] = time.perf_counter()
            submit(pool, sets[pool][0], out[pool][0], out[pool][1], maxd=100)
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
    nbytes = sum(frame_bytes(w, h, nv12) for (w, h) in [sizes[i % len(sizes)] for i in range(pool_n)])
    fps = batches * pool_n / dt
    return dict(part="d" if nv12 else "c", source="nv12" if nv12 else "rgb8", model="yolov5s-shaped heads (width 0.5, 640)",
                pool_frames=pool_n, batches=batches,
                sizes=sorted({"%dx%d" % s for s in sizes}), frames_per_s=round(fps, 1),
                h2d_gb_per_s=round(fps * nbytes / pool_n / 1e9, 2),
                latency_ms_p50=round(float(np.percentile(lat, 50)), 3), latency_ms_p99=round(float(np.percentile(lat, 99)), 3))


def part_d_device(repeat, calls=5):
    """64 device-resident 1920x1080 frames letterboxed in place: CUDA events on the compute stream around `calls` calls in a
    row (the host work of one call -- validation, table upload -- overlaps the launches of the previous one), per call.
    RGB8 and NV12 alternate within one model; 64 frames (199 MB NV12, 398 MB RGB8) exceed the 126 MB L2."""
    import torch
    n, w, h = 64, 1920, 1080
    gm = letterbox_model(n)
    g = torch.Generator(device="cuda").manual_seed(0)
    rgb = torch.randint(0, 256, (n, h, w * 3), dtype=torch.uint8, device="cuda", generator=g)
    luma = torch.randint(0, 256, (n, h, w), dtype=torch.uint8, device="cuda", generator=g)
    chroma = torch.randint(0, 256, (n, h // 2, w), dtype=torch.uint8, device="cuda", generator=g)
    torch.cuda.synchronize()
    stream = torch.cuda.ExternalStream(gm.compute_stream())
    t_rgb = pkg.capi.device_frames([(rgb[i].data_ptr(), w, h, 0) for i in range(n)])
    t_nv12 = pkg.capi.device_nv12_frames([(luma[i].data_ptr(), chroma[i].data_ptr(), w, h, 0, 0, pkg.capi.YUV_BT709_LIMITED)
                                          for i in range(n)])
    runs = {"rgb8": lambda: L.mars_b200_preprocess_frames_device(gm.m, 0, n, t_rgb),
            "nv12": lambda: L.mars_b200_preprocess_frames_nv12_device(gm.m, 0, n, t_nv12)}
    ms = {k: [] for k in runs}
    for it in range(repeat + 2):
        for k, fn in runs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(calls):
                assert fn() == 0, L.mars_b200_last_error()
            e1.record(stream)
            e1.synchronize()
            if it >= 2:
                ms[k].append(e0.elapsed_time(e1) / calls)
    gm.close()
    out = dict(part="d", case="device-resident letterbox", frames=n, size="%dx%d" % (w, h))
    for k, v in ms.items():
        med = float(np.median(v))
        fb = frame_bytes(w, h, k == "nv12")
        out[k] = dict(ms=round(med, 3), ms_min=round(min(v), 3), ms_max=round(max(v), 3), source_bytes_per_frame=fb,
                      source_gb_per_s=round(n * fb / med / 1e6, 1))
    out["nv12_over_rgb8"] = round(out["nv12"]["ms"] / out["rgb8"]["ms"], 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--part", default="all", choices=["a", "b", "c", "d", "all"])
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
    if a.part in ("d", "all"):
        print(json.dumps(part_d_device(a.repeat)))
        for nv12 in (False, True, False, True):  # alternated: RGB8 (part c) and NV12 on the same model and sizes
            print(json.dumps(part_c(a.batches, a.pool, [(1920, 1080)], nv12)))


if __name__ == "__main__":
    main()
