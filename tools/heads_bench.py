"""tools/heads_bench.py -- the YOLOv5 heads flavour (mars_b200_set_yolo_heads + step_heads_resident) against the output0
flavour (step_resident with parse_output + centre NMS) on the yolov5s-shaped 640x640 int8 graph, 1024 images on one GPU.

Three alternating runs of each flavour, `--steps` device-timed steps per run after `--warmup` steps; then one profiled pass that
splits the heads flavour's post-process into the three decode ops (per-op events, mars_b200_set_profile) and the NMS + letterbox
inverse (mars_b200_detect_heads_resident), next to the output0 flavour's decode + NMS (mars_b200_detect_resident).
Usage: python tools/heads_bench.py [--batch 1024] [--steps 20] [--warmup 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from __graft_entry__ import load_package  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def timed(gm, fn, steps):
    ms = []
    for _ in range(steps):
        ms.append(fn())
    return float(np.median(ms)), float(np.min(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    pkg = load_package()
    mf = pkg.marsfile
    blob = mf.build_yolov5(width=0.5, size=640, seed=5).to_bytes()
    B = a.batch
    gm = pkg.MarsModel(blob, arena_bytes=mf.ARENA_YOLOV5S_INT8, device=0, batch=B)
    xs = np.stack([np.random.default_rng(1000 + b).integers(-128, 128, size=3 * 640 * 640, dtype=np.int8) for b in range(B)])
    gm.upload_inputs(0, B, xs, xs.shape[1])
    plain = lambda: gm.step_resident(0, B, 0.45, True)
    heads = lambda: gm.step_heads_resident(0, B, 0.45)
    res = {"gpu": gpu_info(), "model": "yolov5s-shaped 640x640 int8 (build_yolov5 width 0.5, seed 5)", "batch": B, "steps": a.steps, "runs": []}
    for run in range(3):
        for name, fn, on in (("output0", plain, False), ("heads", heads, True)):
            gm.set_yolo_heads(None, 0.25, enable=on)  # recompiles: warm-up covers the plan, the first plain step and the capture
            timed(gm, fn, a.warmup)
            med, best = timed(gm, fn, a.steps)
            res["runs"].append({"run": run, "flavour": name, "median_ms": med, "min_ms": best, "images_per_s": B / med * 1e3})
    # profiled pass: per-op events (plain launches), then the post-process calls on their own
    gm.set_yolo_heads(None, 0.25)
    gm.set_profile(True)
    heads()
    gm.set_profile(False)
    ops = gm.op_profile()
    dec = [o["ms"] / max(o["calls"], 1) for o in ops if o["kind"] == 21]
    total_ops = sum(o["ms"] / max(o["calls"], 1) for o in ops)
    nms_heads = float(np.median([gm.detect_heads_resident(0, B, 0.45) for _ in range(10)]))
    _, counts = gm.download_boxes(0, B)
    gm.set_yolo_heads(enable=False)
    gm.step_resident(0, B, 0.45, True)
    det_plain = float(np.median([gm.detect_resident(0, B, 0.45) for _ in range(10)]))
    _, dcounts = gm.download_detections(0, B)
    res["split_ms"] = {"heads_decode_per_level": dec, "heads_decode": sum(dec), "heads_nms_scale": nms_heads,
                       "heads_postprocess": sum(dec) + nms_heads, "output0_parse_nms": det_plain, "profiled_layer_ops": total_ops}
    res["kept_per_image"] = {"heads_mean": float(np.mean(counts)), "output0_mean": float(np.mean(dcounts))}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(text + "\n")
    gm.close()


if __name__ == "__main__":
    main()
