"""GPU: every requantisation variant of the tcgen05 int8 conv epilogue (csrc/conv_tc.cu, select_requant: RQ 0 general float with
the x86 overflow rule, RQ 1 fast float, RQ 2 float half-up, RQ 3 integer form) on the crafted models of tests/requant_ref.py, whose
inputs put the accumulators on every step of r, on the negative ties, at the range ends and across the int32 wrap.

Each case runs at batch 3 (a different pixel permutation per slot) through upload_inputs / run_resident at opt 2 (SiLU fold and
producer-written side copies), opt 3 (dead-store elision) and opt 0 (the direct kernels' requantisation), with strict mode on, so
a failed tensor-core plan fails the case instead of falling back.  Checked: the conv's bytes against the numpy reference, the
output (at opt <= 2 the whole arena of every slot) against the oracle, and the planner's " impl=1 rq=N" line for the conv.

Combinations the planner cannot produce are not in the matrix: the gather producer takes at most 256 output channels and the
space-to-depth stem at most 128 (so neither has Co 300, nor the stem Co 255); a SiLU after a 1x1 NCHW conv with two N tiles
(Co 300) is not folded (its fused outputs would overwrite input pixels another N tile still reads), so that case runs the
sigmoid and mul as their own ops.  EPI 16 (one 256-wide N tile, 16 epilogue warps) is Co 255 off the gather path.

The planner does not fold a conv's RELU activation into the epilogue: it runs as a byte-ReLU op of its own over the conv's output
(reference src/mars/mars_runtime.c:700-707).  So the ReLU cases check the plain requantised bytes after that op, the word table
(TAB) is reached through the folded SiLU only, and the 1x1 -> 3x3 chains are plain: a byte-ReLU op between the two convs is the
last writer of the 3x3's input, and the planner links a producer-written copy only to a tensor-core conv."""
import os

import numpy as np
import pytest

import requant_ref as R
from util import first_diff

pytestmark = pytest.mark.gpu

COVERED = {}  # case name -> set of (rq, table) cells and column names it exercised


@pytest.fixture(scope="module", autouse=True)
def strict(pkg):
    lib = pkg.lib()
    lib.mars_b200_set_strict(1)
    yield
    lib.mars_b200_set_strict(1 if os.environ.get("MARS_STRICT", "0") not in ("", "0") else 0)


def conv_line(desc, layer):
    for line in desc.splitlines():
        if (" layer %3d conv_i8_" % layer) in line:
            return line
    raise AssertionError("no conv line for layer %d:\n%s" % (layer, desc))


@pytest.mark.parametrize("case", R.CASES, ids=lambda c: c.name)
def test_requant_variant(pkg, ob, case):
    blob = case.marsfile(pkg.marsfile).to_bytes()
    xs, _ = case.slot_inputs(3)
    n = len(xs)
    flat = np.stack([case.to_bytes_layout(x) for x in xs])
    refs = [case.reference(x) for x in xs]
    oms = []
    for i in range(n):
        om = ob.OracleModel(blob)
        om.set_input(flat[i])
        om.run()
        oms.append(om)
    out_is_y = case.act != R.ACT_SILU
    cells = set()
    for opt in (2, 3, 0):
        gm = pkg.MarsModel(blob, batch=n)
        gm.set_opt_level(opt)
        desc = gm.describe()
        if opt:
            line = conv_line(desc, 0)
            assert " impl=1 rq=%d " % case.rq in line, "%s opt %d: %s" % (case.name, opt, line)
            if case.chain:
                assert " impl=1 rq=" in conv_line(desc, 1), desc
                if opt >= 2:
                    assert "+copy" in line, line
                    cells.add("side")
            fused = " fused=2 " in line
            if case.act == R.ACT_SILU and opt >= 2 and not (case.layout == "nchw1" and case.convs[0].co > 256):
                assert fused, line
            if case.act == R.ACT_RELU:
                assert " byte_relu " in desc.splitlines()[desc.splitlines().index(line) + 1], desc
            cells.add((case.rq, fused))  # the epilogue reads the word table exactly when followers are folded into it
        else:
            assert " rq=" not in desc
        gm.upload_inputs(0, n, flat, flat.shape[1])
        gm.run_resident(0, n)
        outs = gm.download_outputs(0, n)
        for i, om in enumerate(oms):
            want = om.output_bytes()
            at, cnt = first_diff(outs[i][: want.size], want)
            assert cnt == 0, "%s opt %d slot %d: %d output bytes differ from the oracle, first at %d" % (case.name, opt, i, cnt, at)
            if out_is_y:
                y = refs[i][-1][1]
                got = case.from_layout(outs[i], *y.shape)
                assert np.array_equal(got, y), "%s opt %d slot %d: %d bytes differ from the numpy reference" % (case.name, opt, i, int((got != y).sum()))
            if opt <= 2:
                arena = gm.arena_download(i)
                at, cnt = first_diff(arena, om.arena()[: arena.size])
                assert cnt == 0, "%s opt %d slot %d: %d arena bytes differ from the oracle, first at %d" % (case.name, opt, i, cnt, at)
                for (t, y), yid in zip(refs[i], case.y_ids):  # every conv's stored bytes, the SiLU's Y stream included
                    off = gm.tensor_offset(yid)
                    got = case.from_layout(arena[off: off + y.size], *y.shape)
                    assert np.array_equal(got, y), "%s opt %d slot %d tensor %d differs from the numpy reference" % (case.name, opt, i, yid)
        gm.close()
    for om in oms:
        om.close()
    co = case.convs[0].co
    if case.nhwc:
        cells.add("nhwc")
    if co == 255 and case.layout != "gather":
        cells.add("epi16")
    if co % 16:
        cells.add("ragged")
    if co > 256:
        cells.add("two N tiles")
    cells.add(case.layout)
    COVERED[case.name] = cells


def test_every_variant_and_column_was_exercised():
    """all four variants with and without the word table, and the NHWC, EPI 16, ragged, two-N-tile and side-output columns"""
    if len(COVERED) < len(R.CASES):
        pytest.skip("runs after the whole case matrix (%d of %d cases ran)" % (len(COVERED), len(R.CASES)))
    seen = set().union(*COVERED.values())
    want = {(rq, tab) for rq in range(4) for tab in (False, True)} | {"nhwc", "epi16", "ragged", "two N tiles", "side"} | set(R.LAYOUTS)
    assert want <= seen, sorted(map(str, want - seen))
    print("requantisation cells: %s" % sorted(str(c) for c in seen))
