"""shared helpers for the parity tests"""
import hashlib
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN_DIR = os.path.join(HERE, "golden")
GOLDEN = json.load(open(os.path.join(GOLDEN_DIR, "golden.json")))
REF_MODELS = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "models")

# The reference's shipped .mars files are staged under oracle/_ref/models only where the reference has been built; they are not
# part of this repository.  Without them the GPU parity tests run on generated stand-ins of the same kind (dtype, input size and
# layer types) with synthetic weights; the yolov5n ones come from the writer whose width-0.25 graph tests/test_marsfile.py holds
# to the shipped layer table where that file is staged.  The stand-ins do not carry the shipped files' quirks (fp16 payloads
# tagged f32, biases stored as one byte per channel, ...).  The CUDA path is held bit-exact to the oracle either way; the golden
# outputs of the reference apply to the shipped files only.
STAND_INS = {
    "tiny_160_int8.mars": lambda mf: mf.build_tiny(160),
    "tiny_160_f32.mars": lambda mf: mf.build_tiny(160, f32=True),
    "test_model.mars": lambda mf: mf.build_single_layer("conv", k=3, s=1, c=3, h=64, w=64, co=16, padding=1, act=1),
    "test_simple.mars": lambda mf: mf.build_tiny(64, f32=True, chans=(16,)),
    "yolov5n_int8.mars": lambda mf: mf.build_yolov5(width=0.25, size=640, seed=5),
    "yolov5n.mars": lambda mf: mf.build_yolov5(width=0.25, size=640, seed=6, f32=True),
    "yolov5nu.mars": lambda mf: mf.build_yolov5(width=0.25, size=320, seed=7),
}


# output sha256 of each golden.json model case on its stand-in, recorded from the oracle restatement (run 2;
# tests/golden/make_standin_golden.py) -- outputs of this project, not of the reference
STANDIN_GOLDEN = json.load(open(os.path.join(GOLDEN_DIR, "standin.json")))


def model_blob(pkg, name):
    """(bytes, shipped): the reference's file when it is staged, else its generated stand-in"""
    p = os.path.join(REF_MODELS, name)
    if os.path.exists(p):
        return open(p, "rb").read(), True
    return STAND_INS[name](pkg.marsfile).to_bytes(), False


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def numel(desc):
    n = 1
    for i in range(min(desc.ndims, 6)):
        n *= max(desc.shape[i], 0)
    return n


def make_input(pattern, n):
    if pattern == "p0":  # reference src/mars/mars_test.c:82-85
        return (np.arange(n, dtype=np.int64) % 127).astype(np.int8)
    if pattern == "f32":  # reference src/mars/mars_test.c:76-80
        return ((np.arange(n, dtype=np.int64) % 256).astype(np.float32) / np.float32(255.0)).astype(np.float32)
    if pattern.startswith("rng"):
        return np.random.default_rng(int(pattern[3:])).integers(-128, 128, size=n, dtype=np.int8)
    raise ValueError(pattern)


def first_diff(a, b):
    a, b = np.asarray(a).ravel(), np.asarray(b).ravel()
    n = min(a.size, b.size)
    d = np.nonzero(a[:n] != b[:n])[0]
    return (int(d[0]), int(d.size)) if d.size else (None, 0)


# micro-models (kind, builder arguments) for kernels and shapes no shipped file exercises (SURVEY B.4).  The GPU parity tests run
# the CUDA path against the restatement on them (tests/test_gpu_parity.py); the CPU suite pins the restatement to the reference
# library on the same list (tests/test_oracle.py).
MICRO = [
    ("conv", dict(k=3, s=1)), ("conv", dict(k=3, s=2, c=5, co=7, h=17, w=13)), ("conv", dict(k=1, s=1, c=32, co=24)),
    ("conv", dict(k=6, s=2, c=3, co=16, h=32, w=32)), ("conv", dict(k=3, s=1, padding=1, act=1)),  # SAME + fused ReLU
    ("conv", dict(k=3, s=1, no_bias=True)), ("conv", dict(k=3, s=1, nhwc=True)), ("conv", dict(k=1, s=1, nhwc=True, c=16, co=16)),
    ("conv", dict(k=3, s=2, nhwc=True, padding=1)), ("conv", dict(k=3, s=1, f32=True)), ("conv", dict(k=1, s=1, f32=True, c=16)),
    ("sigmoid", {}), ("sigmoid", dict(f32=True)), ("relu", {}), ("relu6", {}), ("leaky", {}), ("leaky", dict(f32=True)),
    ("add", {}), ("mul", {}), ("add", dict(f32=True)), ("mul", dict(f32=True)), ("maxpool", dict(k=2, s=2)),
    ("maxpool", dict(k=5, s=1, h=20, w=20, c=20)), ("maxpool", dict(k=3, s=2, h=9, w=11)), ("upsample", dict(scale=2)),
    ("upsample", dict(scale=3, ratio_fallback=True)), ("concat", dict(n=4)), ("concat", dict(n=2)), ("batchnorm", {}),
    ("batchnorm", dict(f32=True)), ("depthwise", {}),
]
# int8 convs that take the tcgen05 path (tests/test_gpu_parity.py asserts impl=1 for each)
MICRO_TC = [
    # shapes that take the tcgen05 path (Ci % 32 == 0)
    ("conv", dict(k=1, s=1, c=32, co=64, h=20, w=20)), ("conv", dict(k=1, s=1, c=64, co=32, h=16, w=24)),
    ("conv", dict(k=1, s=1, c=128, co=512, h=8, w=8)), ("conv", dict(k=1, s=1, c=256, co=255, h=20, w=20)),
    ("conv", dict(k=3, s=1, c=32, co=32, h=20, w=20)), ("conv", dict(k=3, s=1, c=64, co=255, h=13, w=11)),
    ("conv", dict(k=3, s=1, c=32, co=48, h=40, w=40, padding=1)), ("conv", dict(k=3, s=2, c=64, co=128, h=40, w=40)),
    ("conv", dict(k=3, s=2, c=32, co=64, h=34, w=30, padding=1)), ("conv", dict(k=3, s=1, c=96, co=16, h=9, w=50, no_bias=True)),
    ("conv", dict(k=3, s=1, c=32, co=32, h=24, w=24, padding=0)),
    # halo loads with 2 / 1 / 4 M tiles per group, 5x5 taps, narrow N tiles (one 16-column unit), N = 48
    ("conv", dict(k=3, s=1, c=64, co=64, h=30, w=26)), ("conv", dict(k=3, s=1, c=32, co=128, h=24, w=20)),
    ("conv", dict(k=5, s=1, c=32, co=32, h=20, w=20)), ("conv", dict(k=1, s=1, c=32, co=16, h=64, w=64)),
    ("conv", dict(k=1, s=1, c=64, co=48, h=50, w=50)), ("conv", dict(k=3, s=1, c=128, co=128, h=40, w=40)),
    # the stem shape (6x6 stride 2, pads 0 or 2, <= 4 channels): space-to-depth copy read as overlapping K rows
    ("conv", dict(k=6, s=2, c=3, co=32, h=128, w=128, pad=2)), ("conv", dict(k=6, s=2, c=3, co=32, h=128, w=128, pad=2, padding=1)),
    ("conv", dict(k=6, s=2, c=3, co=16, h=130, w=136, pad=2)), ("conv", dict(k=6, s=2, c=4, co=48, h=128, w=160, pad=2, padding=1)),
    ("conv", dict(k=6, s=2, c=2, co=128, h=160, w=128, pad=2)), ("conv", dict(k=6, s=2, c=1, co=32, h=256, w=64, pad=2, no_bias=True)),
    # gather producer + tcgen05 (small Ci, >= 4096 output pixels)
    ("conv", dict(k=6, s=2, c=3, co=32, h=128, w=128)), ("conv", dict(k=3, s=1, c=8, co=24, h=70, w=66, padding=1)),
    ("conv", dict(k=3, s=2, c=5, co=17, h=130, w=140)),
    # channel counts that are not multiples of 32 on the tensor-core path: zero-padded K (TMA fill / padded copy), ragged N > 256
    ("conv", dict(k=1, s=1, c=58, co=58, h=40, w=40)), ("conv", dict(k=1, s=1, c=116, co=232, h=10, w=10)),
    ("conv", dict(k=1, s=1, c=232, co=464, h=10, w=10)), ("conv", dict(k=1, s=1, c=48, co=40, h=20, w=20)),
    ("conv", dict(k=1, s=1, c=464, co=300, h=12, w=12)), ("conv", dict(k=3, s=1, c=48, co=32, h=20, w=20)),
    ("conv", dict(k=3, s=2, c=24, co=40, h=40, w=40)), ("conv", dict(k=3, s=1, c=116, co=58, h=20, w=20, padding=1)),
    ("conv", dict(k=5, s=1, c=40, co=272, h=12, w=14)),
    # channel-innermost (--nhwc convention, conv2d_int8_nhwc_mxu) shapes on the tensor-core path: flat 1x1 tiles from the arena,
    # rectangular tiles with one 4-d TMA box per tap (OOB zero fill, traversal stride 2), the stem, ragged channel counts
    ("conv", dict(k=1, s=1, nhwc=True, c=32, co=64, h=20, w=20)), ("conv", dict(k=1, s=1, nhwc=True, c=128, co=512, h=8, w=8)),
    ("conv", dict(k=1, s=1, nhwc=True, c=64, co=32, h=16, w=24)), ("conv", dict(k=1, s=1, nhwc=True, c=256, co=255, h=20, w=20)),
    ("conv", dict(k=3, s=1, nhwc=True, c=32, co=32, h=20, w=20)), ("conv", dict(k=3, s=1, nhwc=True, c=64, co=255, h=13, w=11)),
    ("conv", dict(k=3, s=1, nhwc=True, c=32, co=48, h=40, w=40, padding=1)), ("conv", dict(k=3, s=2, nhwc=True, c=64, co=128, h=40, w=40)),
    ("conv", dict(k=3, s=2, nhwc=True, c=32, co=64, h=34, w=30, padding=1)), ("conv", dict(k=5, s=1, nhwc=True, c=32, co=32, h=20, w=20)),
    ("conv", dict(k=3, s=1, nhwc=True, c=128, co=128, h=40, w=40)), ("conv", dict(k=3, s=1, nhwc=True, c=96, co=16, h=9, w=50, no_bias=True)),
    ("conv", dict(k=6, s=2, nhwc=True, c=3, co=32, h=128, w=128, pad=2)), ("conv", dict(k=6, s=2, nhwc=True, c=4, co=48, h=128, w=160, pad=2, padding=1)),
    ("conv", dict(k=3, s=1, nhwc=True, c=256, co=512, h=20, w=20)),
]
MICRO = MICRO + MICRO_TC
