"""GPU: the CUDA path (through the C-ABI) against the oracle -- bit-exact over the WHOLE arena
for int8 models (run 1 and run 2, both arena modes), and layer by layer; float32 models bit-exact
too on the exact-order kernels.  On the reference's shipped files (staged by oracle/build_ref.sh)
also against the reference's committed golden outputs; where they are not staged, the tests run
on generated stand-ins (tests/util.py STAND_INS), which tie the CUDA path to the oracle and to
outputs recorded from this project, not to the reference."""
import os

import numpy as np
import pytest

from util import GOLDEN, GOLDEN_DIR, STANDIN_GOLDEN, first_diff, make_input, model_blob, numel, sha

pytestmark = pytest.mark.gpu

MODEL_CASES = [k for k, v in GOLDEN.items() if "model" in v]


def run_both(pkg, ob, blob, arena, x, runs=2, opt=None, depthwise=False):
    """opt <= 2: the whole arena must equal the oracle's after every run; opt 3 (dead stores
    elided): every model output must, over consecutive runs with DIFFERENT inputs (stale bytes of
    run k are inputs of run k+1, so this also checks the liveness analysis across runs)."""
    gm = pkg.MarsModel(blob, arena_bytes=arena)
    gm.set_f32_mode(0)  # bit-exact comparison: float32 convolutions on the exact-order control (default: tf32x3 tensor path)
    if opt is not None:
        gm.set_opt_level(opt)
    if depthwise:
        gm.set_depthwise_mode(1)
    om = ob.OracleModel(blob, arena_bytes=arena, depthwise=depthwise)
    whole = opt is not None and opt <= 2
    for run in range(runs if whole else runs + 2):
        xr = x if (whole or run == 0) else np.roll(x, 7919 * run)
        gm.set_input(xr)
        gm.run()
        om.set_input(xr)
        om.run()
        if whole:
            got = gm.arena_download()
            want = om.arena()[: got.size]
            at, cnt = first_diff(got, want)
            assert cnt == 0, "run %d: %d arena bytes differ, first at %d (weights end %d, buffer %d)" % (
                run + 1, cnt, at, gm.weights_size, gm.buffer_size)
        at, cnt = first_diff(gm.output_bytes(), om.output_bytes())
        assert cnt == 0, "run %d: %d output bytes differ, first at %d" % (run + 1, cnt, at)
    return gm, om


@pytest.mark.parametrize("opt", [0, 1, 2, 3])
@pytest.mark.parametrize("case", MODEL_CASES)
def test_shipped_models_whole_arena(pkg, ob, case, opt):
    """golden.json model cases: on the shipped file, output hash and detection list of the reference itself; on the stand-in,
    the output hash recorded from the oracle (tests/golden/standin.json: catches a change that moves the oracle and the CUDA
    path together) and the oracle's detection list"""
    g = GOLDEN[case]
    if case.startswith("yolov5n/f32"):
        pytest.skip("f32 sigmoid uses the device expf (tolerance path): covered by test_f32_model_layerwise")
    blob, shipped = model_blob(pkg, g["model"])
    om0 = ob.OracleModel(blob, arena_bytes=g["arena"])
    x = make_input(g["pattern"], numel(om0.tensor_desc(om0.input_index())))
    om0.close()
    gm, om = run_both(pkg, ob, blob, g["arena"], x, opt=opt)
    if opt <= 2:  # same input twice
        assert sha(gm.output_bytes()) == (g["run2"]["output_sha256"] if shipped else STANDIN_GOLDEN[case])
    if "dets" in g and opt <= 2:
        o = gm.output_bytes().view(np.int8)
        od = gm.output().desc
        kept = pkg.capi.nms(pkg.capi.parse_output(o, od.shape[1], od.scale))
        if shipped:
            want = np.load(os.path.join(GOLDEN_DIR, g["dets"]["file"]))
        else:
            oo = om.output_bytes().view(np.int8)
            want = ob.nms(ob.parse_output(oo, od.shape[1], om.tensor_desc(om.output_index()).scale))
        assert kept.tobytes() == want.tobytes()
    gm.close()
    om.close()


@pytest.mark.parametrize("opt", [0, 1])
@pytest.mark.parametrize("name,arena", [("yolov5n_int8.mars", 8 << 20), ("yolov5nu.mars", 8 << 20), ("tiny_160_int8.mars", 8 << 20)])
def test_layer_by_layer(pkg, ob, name, arena, opt):
    """each GPU layer is fed the oracle's exact bytes (isolates a divergence to one layer)"""
    blob, _ = model_blob(pkg, name)
    gm = pkg.MarsModel(blob, arena_bytes=arena)
    gm.set_opt_level(opt)
    om = ob.OracleModel(blob, arena_bytes=arena)
    rng = np.random.default_rng(4)
    x = rng.integers(-128, 128, size=numel(om.tensor_desc(om.input_index())), dtype=np.int8)
    om.set_input(x)
    W = om.weights_size
    nl = om.num_layers
    step = 1 if nl < 40 else 7  # every layer for small models, a stride for the big ones (plus hazards)
    hazard = {43, 110, 128, 139, 149, 169, 179, 189, 203, 211, 229}
    for i in range(nl):
        before = om.arena().copy()
        assert om.run_layer(i) == 0
        if i % step and i not in hazard:
            continue
        gm.mirror()[W:om.arena_bytes] = before[W:]
        gm.arena_upload()
        assert gm.run_layer(i) == 0, pkg.lib().mars_b200_last_error()
        got = gm.arena_download()
        at, cnt = first_diff(got, om.arena()[: got.size])
        assert cnt == 0, "layer %d: %d bytes differ, first at %d" % (i, cnt, at)
    gm.close()
    om.close()


def micro(pkg, kind, **kw):
    return pkg.marsfile.build_single_layer(kind, **kw).to_bytes()


from util import MICRO, MICRO_TC  # noqa: E402  (shared with the CPU pin of the restatement against the reference, tests/test_oracle.py)


@pytest.mark.parametrize("kind,kw", MICRO)
def test_micro_models(pkg, ob, kind, kw):
    blob = micro(pkg, kind, **kw)
    gm = pkg.MarsModel(blob)
    if (kind, kw) in MICRO_TC:  # a failed tensor-core plan would silently recompile on the direct kernels
        desc = gm.describe()
        assert " impl=1 rq=" in desc, "%r did not take the tensor-core path:\n%s" % (kw, desc)
    om = ob.OracleModel(blob)
    rng = np.random.default_rng(2)
    W = om.weights_size
    if kw.get("f32"):
        fill = rng.standard_normal((om.arena_bytes - W) // 4).astype(np.float32).view(np.uint8)
    else:
        fill = rng.integers(0, 256, size=om.arena_bytes - W, dtype=np.uint8)
    om.arena()[W:W + fill.size] = fill
    gm.mirror()[W:W + fill.size] = fill
    gm.arena_upload()
    om.run()
    for i in range(om.num_layers):
        assert gm.run_layer(i) == 0, pkg.lib().mars_b200_last_error()
    got = gm.arena_download()
    want = om.arena()[: got.size]
    if kind == "sigmoid" and kw.get("f32"):
        # device expf vs glibc expf: tolerance path (<= 1e-6 absolute on a [0,1] output)
        n = got.size // 4 * 4
        assert np.allclose(got[W:n].view(np.float32), want[W:n].view(np.float32), atol=1e-6, rtol=0, equal_nan=True)
    else:
        at, cnt = first_diff(got, want)
        assert cnt == 0, "%s %r: %d bytes differ, first at %d" % (kind, kw, cnt, at)
    gm.close()
    om.close()


def test_depthwise_modes(pkg, ob):
    blob = micro(pkg, "depthwise")
    for mode in (0, 1):
        gm = pkg.MarsModel(blob)
        gm.set_depthwise_mode(mode)
        om = ob.OracleModel(blob, depthwise=bool(mode))
        x = np.random.default_rng(8).integers(-128, 128, size=8 * 12 * 10, dtype=np.int8)
        gm.set_input(x)
        gm.run()
        om.set_input(x)
        om.run()
        assert np.array_equal(gm.arena_download(), om.arena()[: gm.arena_download().size])
        gm.close()
        om.close()


def test_unknown_layer_fails_like_the_reference(pkg):
    gm = pkg.MarsModel(micro(pkg, "fc"))
    with pytest.raises(pkg.capi.MarsError) as e:
        gm.run()
    assert e.value.code == -8
    gm.close()


@pytest.mark.parametrize("opt", [2, 3])
@pytest.mark.parametrize("width,size,arena,nhwc", [(0.125, 160, 8 << 20, False), (0.25, 320, 16 << 20, False), (0.5, 128, 8 << 20, False),
                                                   (0.5, 256, 8 << 20, False), (0.5, 256, 8 << 20, True), (0.25, 320, 16 << 20, True)])
def test_generated_yolov5_batch(pkg, ob, width, size, arena, nhwc, opt):
    """batch sharded over image slots == oracle per image (run + decode + NMS); nhwc = the compiler's --nhwc convention
    (channel-innermost activations, OHWI weights: conv2d_int8_nhwc_mxu, reference src/mars/mxu_conv.c:713-757)"""
    blob = pkg.marsfile.build_yolov5(width=width, size=size, seed=9, nhwc=nhwc).to_bytes()
    n = 5
    gm = pkg.MarsModel(blob, arena_bytes=arena, batch=n)
    gm.set_opt_level(opt)
    rng = np.random.default_rng(11)
    xs = rng.integers(-128, 128, size=(n, 3 * size * size), dtype=np.int8)
    gm.upload_inputs(0, n, xs, xs.shape[1])
    gm.step_resident(0, n, 0.45, True)
    outs = gm.download_outputs(0, n)
    dets, counts = gm.download_detections(0, n)
    # the same through the host-buffer pipeline (chunks of capacity/2)
    dets2 = np.zeros((n, 1000), dtype=pkg.capi.DET_DTYPE)
    counts2 = np.zeros(n, dtype=np.int32)
    for i in range(n):
        om = ob.OracleModel(blob, arena_bytes=arena)
        om.set_input(xs[i])
        om.run()
        assert np.array_equal(outs[i], om.output_bytes()), "image %d" % i
        if opt <= 2:
            got = gm.arena_download(i)
            at, cnt = first_diff(got, om.arena()[: got.size])
            assert cnt == 0, "image %d: %d arena bytes differ, first at %d" % (i, cnt, at)
        o = om.output_bytes().view(np.int8)
        d = ob.nms(ob.parse_output(o, o.size // 85, om.tensor_desc(om.output_index()).scale))
        assert counts[i] == len(d)
        assert dets[i, : len(d)].tobytes() == d.tobytes()
        om.close()
    gm.arena_clear()
    gm.detect_batch(n, xs, xs.shape[1], dets2, counts2)
    assert np.array_equal(counts, counts2)
    for i in range(n):
        assert dets[i, : counts[i]].tobytes() == dets2[i, : counts[i]].tobytes()
    gm.close()


@pytest.mark.parametrize("nhwc", [False, True])
def test_yolov5s_full_size(pkg, ob, nhwc):
    """BASELINE config 3 shape: yolov5s-shaped 640x640 int8; two consecutive batches through the
    same image slots (default opt level), output tensor + detections bit-exact vs the oracle fed
    the same image sequence per slot.  nhwc: the same graph in the compiler's --nhwc convention."""
    mf = pkg.marsfile
    blob = mf.build_yolov5(width=0.5, size=640, seed=5, nhwc=nhwc).to_bytes()
    n = 3
    gm = pkg.MarsModel(blob, arena_bytes=mf.ARENA_YOLOV5S_INT8, batch=n)
    oms = [ob.OracleModel(blob, arena_bytes=mf.ARENA_YOLOV5S_INT8) for _ in range(n)]
    for step in range(2):
        xs = np.stack([np.random.default_rng(1000 + step * n + b).integers(-128, 128, size=3 * 640 * 640, dtype=np.int8) for b in range(n)])
        gm.upload_inputs(0, n, xs, xs.shape[1])
        gm.step_resident(0, n, 0.45, True)
        outs = gm.download_outputs(0, n)
        dets, counts = gm.download_detections(0, n)
        for i, om in enumerate(oms):
            om.set_input(xs[i])
            om.run()
            at, cnt = first_diff(outs[i], om.output_bytes())
            assert cnt == 0, "step %d image %d: %d output bytes differ, first at %d" % (step, i, cnt, at)
            o = om.output_bytes().view(np.int8)
            d = ob.nms(ob.parse_output(o, 25200, om.tensor_desc(om.output_index()).scale))
            assert counts[i] == len(d) and dets[i, : len(d)].tobytes() == d.tobytes()
    desc = gm.describe()
    assert "fused" in desc
    gm.close()


def test_f32_model_layerwise(pkg, ob):
    """yolov5n.mars (shipped: fp16 payloads tagged f32, activations up to 4e11 -- garbage in, deterministic; stand-in: the
    generated float32 graph of the same layer types, synthetic weights): every layer is fed the oracle's exact bytes.  Conv / mul / add / concat / pool
    are bit-exact (reference accumulation order, no FMA); SIGMOID uses the device expf and is
    checked to <= 2 ulp-of-1 absolute (outputs lie in [0,1])."""
    blob, _ = model_blob(pkg, "yolov5n.mars")
    arena = 64 << 20
    gm = pkg.MarsModel(blob, arena_bytes=arena)
    gm.set_f32_mode(0)  # the exact-order control (the default is the tf32x3 tensor path, see test_f32_tensor_path_*)
    om = ob.OracleModel(blob, arena_bytes=arena)
    x = make_input("f32", numel(om.tensor_desc(om.input_index())))
    om.set_input(x)
    W = om.weights_size
    used = W + om.num_buffers * om.buffer_size
    checked = 0
    for i in range(om.num_layers):
        ltype = om.layer_desc(i).type
        before = om.arena()[:used].copy()
        assert om.run_layer(i) == 0
        if ltype == 0 and i % 4:  # every 4th conv (each upload moves 40 MB)
            continue
        if ltype not in (0, 9, 11, 12, 2, 10, 13):
            continue
        if ltype in (9, 12) and i % 6:
            continue
        gm.mirror()[W:used] = before[W:]
        gm.arena_upload()
        assert gm.run_layer(i) == 0
        got = gm.arena_download()
        want = om.arena()[: got.size]
        if ltype == 9:
            n4 = (got.size - W) // 4 * 4
            a, b = got[W:W + n4].view(np.float32), want[W:W + n4].view(np.float32)
            ok = (a == b) | (np.abs(a - b) <= 2.5e-7) | (np.isnan(a) & np.isnan(b))
            assert ok.all(), "layer %d sigmoid: max abs err %g" % (i, np.nanmax(np.abs(a - b)))
        else:
            at, cnt = first_diff(got, want)
            assert cnt == 0, "layer %d (type %d): %d bytes differ, first at %d" % (i, ltype, cnt, at)
        checked += 1
    assert checked > 40
    gm.close()
    om.close()


@pytest.mark.parametrize("depthwise", [False, True])
@pytest.mark.parametrize("opt", [1, 3])
def test_generated_nanodet_like(pkg, ob, depthwise, opt):
    """BASELINE config 5 shape (synthetic NanoDet-m-like graph, 320x320 int8): depthwise + pointwise blocks, concat,
    upsample, 1x1 heads.  depthwise=False is the reference's semantics (DEPTHWISE_CONV2D is a no-op,
    src/mars/mars_runtime.c:1168-1170); True is the restated depthwise (parity unpinned, oracle restatement)."""
    blob = pkg.marsfile.build_nanodet_like(size=320, seed=7).to_bytes()
    n = 3
    gm = pkg.MarsModel(blob, arena_bytes=16 << 20, batch=n)
    gm.set_opt_level(opt)
    gm.set_depthwise_mode(1 if depthwise else 0)
    oms = [ob.OracleModel(blob, arena_bytes=16 << 20, depthwise=depthwise) for _ in range(n)]
    for step in range(2):  # two frames per stream through the same slots (stale bytes carry over, as in the reference)
        xs = np.stack([np.random.default_rng(s * 1_000_003 + step).integers(-128, 128, size=3 * 320 * 320, dtype=np.int8) for s in range(n)])
        gm.upload_inputs(0, n, xs, xs.shape[1])
        gm.run_resident(0, n)
        outs = gm.download_outputs(0, n)
        for i, om in enumerate(oms):
            om.set_input(xs[i])
            om.run()
            at, cnt = first_diff(outs[i], om.output_bytes())
            assert cnt == 0, "frame %d stream %d: %d output bytes differ, first at %d" % (step, i, cnt, at)
            if opt <= 2:
                got = gm.arena_download(i)
                at, cnt = first_diff(got, om.arena()[: got.size])
                assert cnt == 0, "frame %d stream %d: %d arena bytes differ, first at %d" % (step, i, cnt, at)
    gm.close()


def test_generated_yolov5_f32_within_tolerance(pkg, ob):
    """BASELINE config 4 shape (synthetic yolov5-shaped float32 model) on the exact-order control (f32 mode 0): convolutions
    run in the reference's accumulation order, SIGMOID uses the device expf -> logits within 1e-3 relative of the
    reference's (north_star tolerance), same NaN pattern (the head's output tensor holds stale work-buffer bytes, SURVEY B.2)."""
    blob = pkg.marsfile.build_yolov5(width=0.25, size=160, seed=6, f32=True).to_bytes()
    arena = 64 << 20
    gm = pkg.MarsModel(blob, arena_bytes=arena)
    gm.set_f32_mode(0)
    om = ob.OracleModel(blob, arena_bytes=arena)
    x = np.random.default_rng(2).random(3 * 160 * 160).astype(np.float32)
    for run in range(2):
        gm.set_input(x)
        gm.run()
        om.set_input(x)
        om.run()
        a, b = gm.output_bytes().view(np.float32), om.output_bytes().view(np.float32)
        assert np.array_equal(np.isnan(a), np.isnan(b))
        fin = np.isfinite(b)
        assert fin.any() and np.array_equal(np.isfinite(a), fin)
        rel = np.abs(a[fin] - b[fin]) / np.maximum(np.abs(b[fin]), 1e-6)
        assert rel.max() <= 1e-3, "run %d: max relative error %g" % (run, rel.max())
    gm.close()
    om.close()


F32_TOL = {1: 5e-3, 2: 2e-5}  # max |gpu - ref| / max |ref| per layer: plain tf32 / tf32x3 (north_star: <= 1e-3 on the logits)


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("kw", [dict(k=3, s=1, c=32, co=32, h=40, w=40), dict(k=1, s=1, c=64, co=128, h=40, w=40), dict(k=3, s=2, c=16, co=48, h=64, w=64),
                                dict(k=6, s=2, c=3, co=32, h=128, w=128, pad=2), dict(k=3, s=1, c=40, co=255, h=26, w=22), dict(k=1, s=1, c=256, co=512, h=20, w=20),
                                dict(k=3, s=1, c=128, co=300, h=20, w=20, padding=1), dict(k=5, s=1, c=8, co=16, h=48, w=48, no_bias=True)])
def test_f32_tensor_path_micro(pkg, ob, kw, mode):
    """conv2d_float32_mxu (reference src/mars/mxu_conv.c:673-710) on tcgen05 kind::tf32: mode 2 (operand hi/lo split, three MMAs)
    reproduces the reference's fp32 result to summation-order noise, mode 1 (plain tf32) to ~1e-3; mode 0 is bit-exact"""
    blob = micro(pkg, "conv", f32=True, **kw)
    om = ob.OracleModel(blob)
    W = om.weights_size
    fill = np.random.default_rng(2).standard_normal((om.arena_bytes - W) // 4).astype(np.float32).view(np.uint8)
    om.arena()[W:W + fill.size] = fill
    om.run()
    want = om.output_bytes().view(np.float32)
    for m in (mode, 0):
        gm = pkg.MarsModel(blob)
        gm.set_f32_mode(m)
        gm.set_opt_level(3)
        gm.mirror()[W:W + fill.size] = fill
        gm.arena_upload()
        assert gm.run_layer(0) == 0
        got_arena = gm.arena_download()
        off = om.tensor_offset(om.output_index())
        got = got_arena[off: off + want.nbytes].view(np.float32)
        if m == 0:
            assert np.array_equal(got, want)
        else:
            assert "conv_f32" in gm.describe() and " impl=2 " in gm.describe(), "the layer did not take the tensor-core path"
            err = np.abs(got - want).max() / np.abs(want).max()
            assert err <= F32_TOL[m], "mode %d: max error %g of max |ref|" % (m, err)
        gm.close()
    om.close()


@pytest.mark.parametrize("mode", [1, 2])
def test_f32_tensor_path_yolov5s_layerwise(pkg, ob, mode):
    """BASELINE configs[3] at its stated size: the yolov5s-shaped float32 graph at 640x640.  Every convolution is fed the
    restatement's exact input bytes (the graph as the reference executes it turns to byte garbage behind SPPF / upsample --
    maxpool, upsample and concat index float tensors as bytes, SURVEY C.4 -- so an end-to-end float comparison is only
    meaningful per layer): outputs within F32_TOL of the reference's, layers whose inputs hold NaN / Inf excluded."""
    mf = pkg.marsfile
    blob = mf.build_yolov5(width=0.5, size=640, seed=6, f32=True).to_bytes()
    arena = mf.ARENA_YOLOV5S_F32
    gm = pkg.MarsModel(blob, arena_bytes=arena)
    gm.set_f32_mode(mode)
    om = ob.OracleModel(blob, arena_bytes=arena)
    x = np.random.default_rng(6).random(3 * 640 * 640, dtype=np.float32)
    om.set_input(x.view(np.int8))
    W = om.weights_size
    used = W + om.num_buffers * om.buffer_size
    desc = gm.describe()
    checked, worst = 0, 0.0
    for i in range(om.num_layers):
        ltype = om.layer_desc(i).type
        before = om.arena()[:used].copy()
        assert om.run_layer(i) == 0
        if ltype != 0 or (checked >= 6 and i % 5):  # the first convs, then every fifth layer (each upload moves ~40 MB)
            continue
        if ("layer %3d conv_f32_nchw" % i) not in desc:
            continue
        oi = om.layer_desc(i).output_tensor_ids[0]
        off, n = om.tensor_offset(oi), numel(om.tensor_desc(oi))
        want = om.arena()[off: off + 4 * n].view(np.float32)
        ii = om.layer_desc(i).input_tensor_ids[0]
        ioff, inn = om.tensor_offset(ii), numel(om.tensor_desc(ii))
        if not np.isfinite(before[ioff: ioff + 4 * inn].view(np.float32)).all() or not np.isfinite(want).all():
            continue
        gm.mirror()[W:used] = before[W:]
        gm.arena_upload()
        assert gm.run_layer(i) == 0
        got = gm.arena_download()[off: off + 4 * n].view(np.float32)
        err = float(np.abs(got - want).max() / max(np.abs(want).max(), 1e-30))
        worst = max(worst, err)
        assert err <= F32_TOL[mode], "layer %d: max error %g of max |ref|" % (i, err)
        checked += 1
    assert checked >= 8, "only %d convolution layers had finite operands" % checked
    print("f32 mode %d: %d conv layers, worst error %.3g of max |ref|" % (mode, checked, worst))
    gm.close()
    om.close()


def test_f32_tensor_path_end_to_end_chain(pkg, ob):
    """a float32 graph without byte-indexed layers (three valid 3x3 convs + ReLU, the tiny_160_f32 shape at 320 px) end to end:
    logits within 1e-3 relative (north_star) on the default tf32x3 path and on plain tf32"""
    blob = pkg.marsfile.build_tiny(size=320, seed=11, f32=True).to_bytes()
    _f32_end_to_end(pkg, ob, blob, np.random.default_rng(3).random(3 * 320 * 320, dtype=np.float32))


def test_f32_tensor_path_shipped_tiny_160_f32(pkg, ob):
    """the shipped tiny_160_f32.mars (or its stand-in) through mars_run on the default float32 path"""
    blob, _ = model_blob(pkg, "tiny_160_f32.mars")
    _f32_end_to_end(pkg, ob, blob, make_input("f32", 3 * 160 * 160))


def _f32_end_to_end(pkg, ob, blob, x):
    arena = 64 << 20
    om = ob.OracleModel(blob, arena_bytes=arena)
    om.set_input(x.view(np.int8))
    om.run()
    want = om.output_bytes().view(np.float32)
    for mode, tol in ((2, 1e-5), (1, 1e-3)):
        gm = pkg.MarsModel(blob, arena_bytes=arena)
        gm.set_f32_mode(mode)
        gm.set_input(x.view(np.int8))
        gm.run()
        got = gm.output_bytes().view(np.float32)
        err = float(np.abs(got - want).max() / np.abs(want).max())
        assert err <= tol, "mode %d: max error %g of max |logit|" % (mode, err)
        gm.close()
    om.close()


def test_submit_wait_batches_match_the_synchronous_path(pkg, ob):
    """mars_b200_submit_batch / wait_batch (two halves of the slot pool, copies overlapping kernels) give the same
    detection lists as the oracle, batch after batch, including a short last batch"""
    blob = pkg.marsfile.build_yolov5(width=0.125, size=160, seed=9).to_bytes()
    half, total = 3, 8
    gm = pkg.MarsModel(blob, arena_bytes=8 << 20, batch=2 * half)
    rng = np.random.default_rng(21)
    xs = rng.integers(-128, 128, size=(total, 3 * 160 * 160), dtype=np.int8)
    want = []
    for i in range(total):
        om = ob.OracleModel(blob, arena_bytes=8 << 20)
        om.set_input(xs[i])
        om.run()
        o = om.output_bytes().view(np.int8)
        want.append(ob.nms(ob.parse_output(o, o.size // 85, om.tensor_desc(om.output_index()).scale)))
        om.close()
    dets = [np.zeros((half, 1000), dtype=pkg.capi.DET_DTYPE) for _ in range(2)]
    counts = [np.zeros(half, dtype=np.int32) for _ in range(2)]
    batches = [(s, min(half, total - s)) for s in range(0, total, half)]

    def check(k):
        s, n = batches[k]
        gm.wait_batch(k & 1)
        for i in range(n):
            w = want[s + i]
            assert counts[k & 1][i] == len(w) and dets[k & 1][i, : len(w)].tobytes() == w.tobytes(), "batch %d image %d" % (k, i)

    for k, (s, n) in enumerate(batches):
        if k >= 2:
            check(k - 2)  # the half is reused: its previous batch must have been collected
        gm.submit_batch(k & 1, n, xs[s:s + n], xs.shape[1], dets[k & 1], counts[k & 1])
    for k in range(max(0, len(batches) - 2), len(batches)):
        check(k)
    with pytest.raises(pkg.capi.MarsError):
        gm.submit_batch(0, half + 1, xs, xs.shape[1], dets[0], counts[0])
    gm.close()


def test_enqueue_only_step_equals_the_synchronous_step(pkg):
    """mars_b200_enqueue_step_resident (no host synchronisation; the caller waits on the compute stream) leaves the same outputs and
    detection records as mars_b200_step_resident -- first plain launches, then the captured graph"""
    blob = pkg.marsfile.build_yolov5(width=0.125, size=160, seed=9).to_bytes()
    gm = pkg.MarsModel(blob, arena_bytes=8 << 20, batch=3)
    xs = np.random.default_rng(33).integers(-128, 128, size=(3, 3 * 160 * 160), dtype=np.int8)
    gm.upload_inputs(0, 3, xs, xs.shape[1])
    gm.step_resident(0, 3, 0.45, True)
    want_out = gm.download_outputs(0, 3).copy()
    wd, wc = gm.download_detections(0, 3)
    wd, wc = wd.copy(), wc.copy()
    for _ in range(3):  # 1st: plain, 2nd: capture, 3rd: replay
        gm.upload_inputs(0, 3, xs, xs.shape[1])
        gm.enqueue_step_resident(0, 3, 0.45, True)
        got_out = gm.download_outputs(0, 3)  # synchronous copies on the same stream order behind the enqueued step
        gd, gc = gm.download_detections(0, 3)
        assert np.array_equal(got_out, want_out)
        assert np.array_equal(gc, wc)
        for i in range(3):
            assert gd[i, :gc[i]].tobytes() == wd[i, :wc[i]].tobytes()
    gm.close()
