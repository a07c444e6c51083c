"""CPU: the numpy requantisation reference (tests/requant_ref.py) against the library's restatement of the reference, the sweep
generator against its own claims, the variant each crafted model selects, and the oracle against the numpy reference on every
crafted model.  No GPU needed; tests/test_gpu_requant.py runs the same models on the tensor-core kernels."""
import ctypes as C

import numpy as np
import pytest

import requant_ref as R
from conftest import load_package

lib = load_package().lib()

EDGE_SCALES = [0.013, 2.0 ** -10, 0.000528381613548845, 0.0002641908067744225, 0.6, 1.0, 3.0, -0.0012345, 1e9, -1e9, 3e38,
               float("inf"), float("-inf"), float("nan"), 0.0, -0.0, 1e-45]


def lib_ref(t, cs):
    return np.array([lib.mars_b200_requant_ref(int(v), C.c_float(cs)) for v in t], dtype=np.int64)


@pytest.mark.parametrize("cs", EDGE_SCALES)
def test_numpy_requant_equals_the_library_reference(cs):
    """overflow (h >= 2^31 -> -128, h <= -2^31 - 256 -> -128), NaN (0 * inf, NaN scale), +-inf, exact ties and the int32 ends"""
    rng = np.random.default_rng(7)
    t = [rng.integers(-2 ** 31, 2 ** 31, size=600), np.array([-2 ** 31, -2 ** 31 + 1, -1, 0, 1, 2 ** 31 - 2, 2 ** 31 - 1])]
    c = np.float32(cs)
    if np.isfinite(c) and c != 0:
        t.append(R.negative_ties(c, -2 ** 31, 2 ** 31 - 1))
        t.append(np.clip(np.round(np.arange(-130, 131) / float(c)), -2 ** 31, 2 ** 31 - 1).astype(np.int64) + rng.integers(-2, 3, size=261))
        big = np.clip(np.round(np.array([2.0 ** 31, -(2.0 ** 31) - 256, -(2.0 ** 31)]) / float(c)), -2 ** 31, 2 ** 31 - 1).astype(np.int64)
        t.append((big[:, None] + np.arange(-3, 4)[None, :]).ravel())
    t = np.clip(np.concatenate(t), -2 ** 31, 2 ** 31 - 1)
    assert np.array_equal(R.requant(t, cs), lib_ref(t, cs))


def test_x86_overflow_rule_is_the_reference():
    # positive overflow and NaN give -128 (INT_MIN clamped), not 127: fl(1 * 1e9) + 0.5 < 2^31 saturates to 127, 3e9 does not
    assert R.requant(np.array([1, 3, 0, -1, -3]), 1e9).tolist() == [127, -128, 0, -128, -128]
    assert R.requant(np.array([1, 0, -1]), float("inf")).tolist() == [-128, -128, -128]
    assert R.requant(np.array([1, 0, -1]), float("nan")).tolist() == [-128, -128, -128]
    assert lib.mars_b200_requant_ref(3, C.c_float(1e9)) == -128


def test_int32_wrap_of_accumulator_plus_bias():
    rng = np.random.default_rng(3)
    acc = rng.integers(-5_000_000, 5_000_000, size=1000)
    b = rng.choice([2 ** 31 - 1000, -2 ** 31 + 1000, 12345], size=1000)
    want = (acc.astype(np.int32).view(np.uint32) + b.astype(np.int32).view(np.uint32)).view(np.int32)  # what the executor's uint32 sum gives
    assert np.array_equal(R.wrap32(acc + b), want.astype(np.int64))


def test_solve_pixels_reaches_the_whole_range():
    for ci in (4, 8, 32, 288):
        n1 = ci - 1
        amax, amin = 127 + 127 * 127 * n1, -128 - 127 * 128 * n1
        A = np.concatenate([np.array([amin, amin + 1, -1, 0, 1, amax - 1, amax]), np.random.default_rng(ci).integers(amin, amax + 1, 500)])
        v = R.solve_pixels(A, ci)
        assert (v[:, 0] + 127 * v[:, 1:].sum(1) == A).all()


@pytest.mark.parametrize("case", R.CASES, ids=lambda c: c.name)
def test_case_selects_its_variant(case):
    """the variant each crafted model names is what the library's selection gives for its scale and accumulator bound"""
    cv = case.convs[0]
    assert lib.mars_b200_requant_variant(C.c_float(cv.cs), C.c_longlong(cv.bound)) == case.rq, (float(cv.cs), cv.bound)


def _reached(case):
    xs, claims = case.slot_inputs(3)
    ts = [case.reference(x)[0][0] for x in xs]
    return xs, claims, ts


@pytest.mark.parametrize("case", R.CASES, ids=lambda c: c.name)
def test_sweep_reaches_what_it_claims(case):
    """every claimed accumulator value (steps -2 .. +1, negative ties, -1 / 0 / 1, range ends) occurs in its channel, on every slot;
    every step of r inside the channel's range is claimed; the claimed ties are ties"""
    xs, claims, ts = _reached(case)
    cv = case.convs[0]
    for c, want in claims.items():
        for t in ts:
            got = np.unique(t[c])
            assert np.isin(want, got).all(), "channel %d misses %s" % (c, want[~np.isin(want, got)][:8])
    if case.random_w:
        return
    for c in claims:
        assert np.array_equal(np.sort(ts[0][c].ravel()), np.sort(ts[1][c].ravel()))  # slots permute pixels only
    n1 = case.ci - 1
    amax, amin = 127 + 127 * 127 * n1, -128 - 127 * 128 * n1
    for c, sign in ((0, 1), (1, -1)):
        b = int(cv.bias[c])
        f = lambda A: R.requant(R.wrap32(sign * np.asarray(A) + b), cv.cs)  # noqa: E731
        steps = R.change_points(f, amin, amax)
        if steps.size * 4 + 300 < ts[0][c].size // 2:  # the pixel budget held the whole list
            assert np.isin(R.wrap32(sign * steps + b), claims[c]).all()
            assert np.isin(R.wrap32(sign * (steps - 1) + b), claims[c]).all()
        # every change point is real: the value differs from its neighbour's
        assert (f(steps) != f(steps - 1)).all()
    ties = R.negative_ties(cv.cs, int(claims[0].min()), int(claims[0].max()))
    with np.errstate(all="ignore"):
        sc = ties.astype(np.float32) * np.float32(cv.cs)
    assert ((sc == -np.nextafter(np.float32(0.5), np.float32(0))) | (sc + np.float32(0.5) == np.floor(sc + np.float32(0.5)))).all()
    if case.rq == 2:
        assert ties.size == 0, "RQ 2 was selected although the range holds negative ties"


def test_sweeps_reach_ties_and_steps_where_the_variants_differ():
    """the sweep reaches negative ties for the float variants that round them away from zero, and all 255 steps at some scale"""
    n_ties = {0: 0, 1: 0, 3: 0}
    full = False
    for case in R.CASES:
        if case.random_w or case.rq == 2:
            continue
        _, claims = case.sweep()
        cv = case.convs[0]
        for c in claims:
            n_ties[case.rq] += R.negative_ties(cv.cs, int(claims[c].min()), int(claims[c].max())).size
            r = R.requant(claims[c], cv.cs)
            full = full or np.unique(r).size == 256
    assert n_ties[0] > 0 and n_ties[1] > 0 and n_ties[3] > 0, n_ties
    assert full


@pytest.mark.parametrize("case", R.CASES, ids=lambda c: c.name)
def test_oracle_equals_numpy_reference(ob, case):
    """the oracle (C restatement of the reference) produces the numpy reference's bytes for every conv of every crafted model"""
    blob = case.marsfile(load_package().marsfile).to_bytes()
    xs, _ = case.slot_inputs(2)
    for x in xs:
        om = ob.OracleModel(blob)
        om.set_input(case.to_bytes_layout(x))
        om.run()
        for (t, y), yid in zip(case.reference(x), case.y_ids):
            off = om.tensor_offset(yid)
            got = case.from_layout(om.arena()[off: off + y.size], *y.shape)
            assert np.array_equal(got, y), "%s tensor %d: %d bytes differ" % (case.name, yid, int((got != y).sum()))
        om.close()
