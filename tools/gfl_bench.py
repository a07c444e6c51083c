"""tools/gfl_bench.py -- the NanoDet GFL heads decode (mars_b200_set_gfl_heads) on the NanoDet-m-shaped 320x320 int8 graph of
`bench.py --config streams` (build_nanodet_like seed 7, 16 MiB arena), one GPU.

(a) device-timed step_resident without detect (the layers alone) against step_heads_resident with GFL heads (layers, the three
    decode ops, corner NMS), at 64 and 1024 images, two alternating runs of each; then one profiled pass splitting the heads
    flavour's post-process into the decode ops (per-op events) and the NMS (mars_b200_detect_heads_resident).
(b) the steady-state pooled stream at 64 frames per micro-batch over two pools: submit_run_batch, which reads back output0
    (179 200 bytes per frame), against submit_heads_batch with maxd = 100 (2 404 bytes of box records and count per frame);
    frames/s and p50 / p99 latency from submit to the results on the host, two alternating runs of each.
Usage: python tools/gfl_bench.py [--steps 20] [--warmup 3] [--micro-batches 200] [--out FILE]
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

SIDE, ARENA, MICRO, MAXD = 320, 16 << 20, 64, 100
OP_GFL_HEAD = 22


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def pinned(L, nbytes, dtype=np.uint8):
    p = L.nna_malloc(nbytes)
    if not p:
        raise MemoryError("nna_malloc(%d)" % nbytes)
    return np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(p)).view(dtype), p


def steps(pkg, blob, xs, a):
    """(a): device-timed steps"""
    B = len(xs)
    gm = pkg.MarsModel(blob, arena_bytes=ARENA, device=0, batch=B)
    gm.upload_inputs(0, B, xs, xs.shape[1])
    plain = lambda: gm.step_resident(0, B, 0.45, False)
    heads = lambda: gm.step_heads_resident(0, B, 0.45)
    runs = []
    for run in range(2):
        for name, fn, on in (("layers", plain, False), ("gfl_heads", heads, True)):
            gm.set_gfl_heads(enable=on)  # recompiles: the warm-up covers the plan, the first plain step and the capture
            for _ in range(a.warmup):
                fn()
            ms = [fn() for _ in range(a.steps)]
            runs.append({"run": run, "flavour": name, "median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)),
                         "images_per_s": B / float(np.median(ms)) * 1e3})
    gm.set_gfl_heads()
    gm.set_profile(True)
    heads()
    gm.set_profile(False)
    ops = gm.op_profile()
    dec = [o["ms"] / max(o["calls"], 1) for o in ops if o["kind"] == OP_GFL_HEAD]
    nms = float(np.median([gm.detect_heads_resident(0, B, 0.45) for _ in range(10)]))
    _, counts = gm.download_boxes(0, B)
    gm.close()
    return {"batch": B, "runs": runs,
            "split_ms": {"gfl_decode_per_level": dec, "gfl_decode": sum(dec), "nms": nms, "postprocess": sum(dec) + nms,
                         "profiled_ops": sum(o["ms"] / max(o["calls"], 1) for o in ops)},
            "kept_per_image_mean": float(np.mean(counts))}


def stream(pkg, blob, a):
    """(b): the pooled stream, two halves of the slot pool, micro-batch k+1 submitted while k-1 is read back"""
    L = pkg.lib()
    gm = pkg.MarsModel(blob, arena_bytes=ARENA, device=0, batch=2 * MICRO)
    in_bytes, out_bytes = gm.input_bytes, gm.out_bytes
    src = np.random.default_rng(7).integers(-128, 128, size=(512, in_bytes), dtype=np.int8)
    stage = [pinned(L, MICRO * in_bytes, np.int8) for _ in range(2)]
    outs = [pinned(L, MICRO * out_bytes) for _ in range(2)]
    boxes = [pinned(L, MICRO * MAXD * 24) for _ in range(2)]
    counts = [pinned(L, MICRO * 4, np.int32) for _ in range(2)]
    nmb = a.micro_batches

    def run(heads):
        lat, t_sub = [], [0.0, 0.0]
        t0 = time.perf_counter()
        for j in range(nmb):
            h = j & 1
            if j >= 2:
                gm.wait_batch(h)
                lat.extend([time.perf_counter() - t_sub[h]] * MICRO)
            idx = np.arange(j * MICRO, (j + 1) * MICRO) % len(src)
            stage[h][0].reshape(MICRO, in_bytes)[:] = src[idx]
            t_sub[h] = time.perf_counter()
            if heads:
                gm.submit_heads_batch(h, MICRO, stage[h][0], in_bytes, boxes[h][0].view(pkg.capi.BOX_DTYPE), counts[h][0], MAXD, 0.45)
            else:
                gm.submit_run_batch(h, MICRO, stage[h][0], in_bytes, outs[h][0], out_bytes)
        for j in range(nmb - 2, nmb):
            gm.wait_batch(j & 1)
            lat.extend([time.perf_counter() - t_sub[j & 1]] * MICRO)
        wall = time.perf_counter() - t0
        lat = np.asarray(lat) * 1e3
        return {"frames_per_s": nmb * MICRO / wall, "p50_ms": float(np.percentile(lat, 50)), "p99_ms": float(np.percentile(lat, 99))}

    res = []
    for r in range(2):
        for name, heads in (("submit_run_batch", False), ("submit_heads_batch", True)):
            gm.set_gfl_heads(enable=heads)
            run(heads)  # warm-up: the compile and the capture of the 64-frame step
            res.append(dict(run=r, flavour=name, **run(heads)))
    gm.close()
    for buf in stage + outs + boxes + counts:
        L.nna_free(buf[1])
    return {"micro_batch": MICRO, "micro_batches": nmb, "maxd": MAXD, "runs": res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--micro-batches", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    pkg = load_package()
    blob = pkg.marsfile.build_nanodet_like(size=SIDE, seed=7).to_bytes()
    res = {"gpu": gpu_info(), "model": "NanoDet-m-shaped 320x320 int8 (build_nanodet_like seed 7, 16 MiB arena), GFL heads nc 80 reg_max 7",
           "bytes_per_frame": {"heads_read_by_decode": sum(112 * (SIDE // s) ** 2 for s in (8, 16, 32)), "output0": 112 * 40 * 40,
                               "boxes_maxd_100": MAXD * 24 + 4}}
    res["steps"] = [steps(pkg, blob, np.random.default_rng(1000).integers(-128, 128, size=(B, 3 * SIDE * SIDE), dtype=np.int8), a)
                    for B in (64, 1024)]
    res["stream"] = stream(pkg, blob, a)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(text + "\n")


if __name__ == "__main__":
    main()
