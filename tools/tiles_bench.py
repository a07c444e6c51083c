"""tools/tiles_bench.py -- tiled detection on 3840x2160 frames: 640x640 tiles overlapping by 128 plus the whole frame, 33 regions
per frame, on the yolov5s-shaped heads model of tools/frames_bench.py.  Three measurements:
  (a) region letterbox: 8 device-resident NV12 frames -> 264 slots through mars_b200_preprocess_rois_nv12_device, against the
      264 crops given as separate device frames to mars_b200_preprocess_frames_nv12_device (CUDA events on the compute stream)
  (b) merge: k_merge_rois per batch of 8 frames (mars_b200_merge_rois_resident) next to the step's per-slot corner NMS
      (mars_b200_detect_heads_resident on the 264 slots), CUDA events
  (c) steady state: mars_b200_submit_rois_nv12_heads_batch from pinned host frames, 4 frames (132 slots) per pool, frames/s and
      the latency from submit to merged boxes on the host (p50 / p99), next to untiled mars_b200_submit_frames_nv12_heads_batch on
      the same frames
The card's name, power limit and SM clock are printed in the same run.
usage: python tools/tiles_bench.py [--part a|b|c|all] [--repeat N] [--batches N]"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from frames_bench import L, gpu_info, mf, pinned_frames, pkg  # noqa: E402

W, H, TILE, OVERLAP = 3840, 2160, 640, 128


def heads_model(batch):
    gm = pkg.MarsModel(mf.build_yolov5(width=0.5, size=640, seed=5).to_bytes(), arena_bytes=mf.ARENA_YOLOV5S_INT8, device=0, batch=batch)
    gm.set_yolo_heads(None, 0.25)
    return gm


def rois_for(n_frames):
    return np.concatenate([pkg.capi.tile_rois(W, H, TILE, TILE, OVERLAP, OVERLAP, with_full=True, frame=f) for f in range(n_frames)])


def event_ms(stream, fn, calls, repeat):
    import torch
    out = []
    for it in range(repeat + 2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(calls):
            fn()
        e1.record(stream)
        e1.synchronize()
        if it >= 2:
            out.append(e0.elapsed_time(e1) / calls)
    return dict(ms=round(float(np.median(out)), 3), ms_min=round(min(out), 3), ms_max=round(max(out), 3))


def device_nv12(n):
    import torch
    g = torch.Generator(device="cuda").manual_seed(0)
    luma = torch.randint(0, 256, (n, H, W), dtype=torch.uint8, device="cuda", generator=g)
    chroma = torch.randint(0, 256, (n, H // 2, W), dtype=torch.uint8, device="cuda", generator=g)
    torch.cuda.synchronize()
    return luma, chroma


def part_a(repeat, calls=3):
    import torch
    n = 8
    rois = rois_for(n)
    gm = heads_model(len(rois))
    luma, chroma = device_nv12(n)
    frames = [(luma[i].data_ptr(), chroma[i].data_ptr(), W, H, 0, 0, pkg.capi.YUV_BT709_LIMITED) for i in range(n)]
    # the same regions as separate device frames: each crop's luma at (x, y), its chroma at (x / 2, y / 2) -- every origin is even
    assert (rois["x"] % 2 == 0).all() and (rois["y"] % 2 == 0).all()
    crops = [(luma[f].data_ptr() + y * W + x, chroma[f].data_ptr() + (y // 2) * W + x, w, h, W, W, pkg.capi.YUV_BT709_LIMITED)
             for (f, x, y, w, h) in rois.tolist()]
    t_rois = pkg.capi.roi_table(rois)
    t_frames = pkg.capi.device_nv12_frames(frames)
    t_crops = pkg.capi.device_nv12_frames(crops)
    stream = torch.cuda.ExternalStream(gm.compute_stream())
    runs = {"regions": lambda: L.mars_b200_preprocess_rois_nv12_device(gm.m, 0, n, t_frames, len(rois), t_rois.ctypes.data),
            "crops_as_frames": lambda: L.mars_b200_preprocess_frames_nv12_device(gm.m, 0, len(crops), t_crops)}
    out = dict(part="a", case="region letterbox, device-resident NV12", n_frames=n, n_regions=len(rois), size="%dx%d" % (W, H))
    for _ in range(2):  # alternated
        for k, fn in runs.items():
            assert fn() == 0, L.mars_b200_last_error()
            out.setdefault(k, []).append(event_ms(stream, lambda: fn(), calls, repeat))
    gm.close()
    return out


def part_b(repeat, calls=5):
    import torch
    n = 8
    rois = rois_for(n)
    gm = heads_model(len(rois))
    luma, chroma = device_nv12(n)
    frames = [(luma[i].data_ptr(), chroma[i].data_ptr(), W, H, 0, 0, pkg.capi.YUV_BT709_LIMITED) for i in range(n)]
    gm.preprocess_rois_nv12_device(0, frames, rois)
    gm.step_heads_resident(0, len(rois), 0.45)
    t_rois = pkg.capi.roi_table(rois)
    stream = torch.cuda.ExternalStream(gm.compute_stream())
    b, c = gm.download_boxes(0, len(rois))
    out = dict(part="b", frames=n, regions=len(rois), kept_boxes_per_region_mean=round(float(c.mean()), 1))
    out["merge_k_merge_rois"] = event_ms(stream, lambda: L.mars_b200_merge_rois_resident(gm.m, 0, n, len(rois), t_rois.ctypes.data, 0.45), calls,
                                         repeat)
    out["slot_nms_k_nms_corner_batch"] = event_ms(stream, lambda: L.mars_b200_detect_heads_resident(gm.m, 0, len(rois), 0.45), calls, repeat)
    gm.close()
    return out


def part_c(batches, pool_frames=4):
    rois = rois_for(pool_frames)
    gm = heads_model(2 * len(rois))
    sets = [pinned_frames([(W, H)] * pool_frames, 30 + p, True) for p in range(2)]
    out = [(np.zeros((pool_frames, 100), dtype=pkg.capi.BOX_DTYPE), np.zeros(pool_frames, dtype=np.int32)) for _ in range(2)]
    res = dict(part="c", model="yolov5s-shaped heads (width 0.5, 640)", pool_frames=pool_frames, regions_per_pool=len(rois),
               size="%dx%d" % (W, H), batches=batches)

    def run(submit, k, lat, sub):
        for i in range(k):
            pool = i % 2
            if i >= 2:
                gm.wait_batch(pool)
                lat.append((time.perf_counter() - sub[i - 2]) * 1e3)
            sub[i] = time.perf_counter()
            submit(pool)
        for i in (k - 2, k - 1):
            gm.wait_batch(i % 2)
            lat.append((time.perf_counter() - sub[i]) * 1e3)

    cases = {"tiled": lambda pool: gm.submit_rois_nv12_heads_batch(pool, sets[pool][0], rois, out[pool][0], out[pool][1], maxd=100),
             "untiled": lambda pool: gm.submit_frames_nv12_heads_batch(pool, sets[pool][0], out[pool][0], out[pool][1], maxd=100)}
    for _ in range(2):  # alternated
        for name, submit in cases.items():
            run(submit, 6, [], {})  # warm-up: staging, tap lists, captured step graphs
            lat, sub = [], {}
            t0 = time.perf_counter()
            run(submit, batches, lat, sub)
            dt = time.perf_counter() - t0
            res.setdefault(name, []).append(dict(frames_per_s=round(batches * pool_frames / dt, 2),
                                                 latency_ms_p50=round(float(np.percentile(lat, 50)), 3),
                                                 latency_ms_p99=round(float(np.percentile(lat, 99)), 3)))
    gm.close()
    for _, ptr in sets:
        L.nna_free(ptr)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--part", default="all", choices=["a", "b", "c", "all"])
    ap.add_argument("--repeat", type=int, default=10)
    ap.add_argument("--batches", type=int, default=30)
    a = ap.parse_args()
    print(json.dumps(dict(gpu=gpu_info())), flush=True)
    if a.part in ("a", "all"):
        print(json.dumps(part_a(a.repeat)), flush=True)
    if a.part in ("b", "all"):
        print(json.dumps(part_b(a.repeat)), flush=True)
    if a.part in ("c", "all"):
        print(json.dumps(part_c(a.batches)), flush=True)


if __name__ == "__main__":
    main()
