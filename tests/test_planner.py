"""Planner decisions (csrc/program.cpp) checked on the CPU through mars_b200_plan_describe: no device is touched.

What the reference decides per layer at run time (src/mars/mars_runtime.c:1161-1224) is compiled once into an op list; the
optimisation levels add fusion (2) and dead-store elision + concat forwarding (3).  These tests pin the decisions the measured
numbers rely on for the headline model (BASELINE configs[2] shape) and the level contract (levels 0-2 never drop or move a store)."""
import ctypes as C
import re

import pytest

from conftest import load_package

pkg = load_package()
lib = pkg.lib()
mf = pkg.marsfile


def plan(blob, arena, opt):
    buf = C.create_string_buffer(4 << 20)
    n = lib.mars_b200_plan_describe(blob, len(blob), arena, opt, buf, len(buf))
    assert 0 < n < len(buf)
    ops = []
    for line in buf.value.decode().splitlines():
        m = re.match(r"op\s+(\d+) layer\s+(\d+) (\S+)\s+(\S+)\s+impl=(\d) in=(-?\d+) out=(-?\d+) .*? n=(\d+) fused=(\d)(.*)$", line)
        assert m, line
        ops.append(dict(op=int(m.group(1)), layer=int(m.group(2)), kind=m.group(3), mode=m.group(4), impl=int(m.group(5)), in0=int(m.group(6)),
                        out=int(m.group(7)), n=int(m.group(8)), fused=int(m.group(9)), note=m.group(10)))
    return ops


@pytest.fixture(scope="module")
def headline():
    return mf.build_yolov5(width=0.5, size=640, seed=5).to_bytes()


def test_level0_keeps_the_exact_kernels_and_every_layer(headline):
    ops = plan(headline, mf.ARENA_YOLOV5S_INT8, 0)
    assert all(o["impl"] == 0 and o["fused"] == 0 for o in ops)
    assert sum(o["kind"] == "sigmoid_i8" for o in ops) == sum(o["kind"] == "mul_i8" for o in ops) > 50
    assert not any("FAIL" in o["mode"] for o in ops)


def test_level2_fuses_but_never_drops_or_moves_a_store(headline):
    ops = plan(headline, mf.ARENA_YOLOV5S_INT8, 2)
    convs = [o for o in ops if o["kind"] == "conv_i8_nchw"]
    assert sum(o["impl"] == 1 for o in convs) == len(convs) - 1  # all but the in-place 1x1 layer run on the tensor pipe
    assert sum(o["fused"] == 2 for o in convs) == 54             # every conv + sigmoid + mul chain but three (below), the in-place conv included
    assert not any(re.search(r" -[YSZ]\b|\+fwd|forwarded", o["note"]) for o in ops)  # whole-arena parity holds at levels 0-2
    assert sum(o["kind"] == "sigmoid_i8" for o in ops) == sum(o["kind"] == "mul_i8" for o in ops) == 3  # two-N-tile layers whose outputs overwrite their input are not fused


def test_level3_elides_forwards_and_trims(headline):
    ops = plan(headline, mf.ARENA_YOLOV5S_INT8, 3)
    fwd = [o for o in ops if "+fwd" in o["note"]]
    assert len(fwd) == 9
    assert sum("-Z" in o["note"] for o in fwd) >= 8           # the original store of a forwarded stream is dead
    assert sum("reads the forwarded copy" in o["note"] for o in ops) >= 5
    heads = [o for o in ops if "head written by the producing conv" in o["note"] or "written by the producing conv" in o["note"]]
    assert len(heads) == 9
    # an input copied in front of a periodic (in-place) input survives only in the bytes that input reads: 80 of 1 638 400
    per = [i for i, o in enumerate(ops) if o["kind"] == "concat_periodic"]
    assert per and all(ops[i - 1]["kind"] == "concat" and ops[i - 1]["n"] <= 160 for i in per if ops[i - 1]["layer"] == ops[i]["layer"])
    assert any(o["mode"] == "pixel-serial" and "+sigmoid+mul fused" in o["note"] for o in ops)
    assert not any("FAIL" in o["mode"] for o in ops)


def test_nhwc_and_f32_graphs_compile(headline):
    ops = plan(mf.build_yolov5(width=0.5, size=640, seed=5, nhwc=True).to_bytes(), mf.ARENA_YOLOV5S_INT8, 3)
    convs = [o for o in ops if o["kind"] == "conv_i8_nhwc"]
    assert convs and sum(o["impl"] == 1 for o in convs) >= len(convs) - 1
    ops = plan(mf.build_yolov5(width=0.25, size=160, seed=6, f32=True).to_bytes(), 32 << 20, 3)
    assert any(o["kind"] == "conv_f32_nchw" and o["impl"] == 2 for o in ops)


def test_bad_blobs_are_refused():
    buf = C.create_string_buffer(64)
    assert lib.mars_b200_plan_describe(b"\x00" * 256, 256, 0, 3, buf, 64) == 0
    assert lib.mars_b200_plan_describe(None, 0, 0, 3, buf, 64) == 0
