"""Independent numpy reference of the int8 convolution with its requantisation, and crafted models that drive every
requantisation variant of the tcgen05 conv epilogue (csrc/conv_tc.cu, select_requant) onto its edges.

Reference arithmetic (src/mars/mxu_conv.c:642-669 NCHW, :726-756 NHWC; the oracle's mo_requant_conv):
  acc = sum of int8 x int8 products over the taps inside the input (padding skips taps), in int64 here;
  t   = int32 wrap of acc + bias, the bias read as the raw int32 bytes of the bias tensor;
  sc  = fl((float)t * cs), h = fl(sc + (sc >= 0 ? 0.5f : -0.5f)), one float32 rounding per operation;
  r   = clamp((int32)h) with the x86 cvttss2si rule: NaN and h outside (-2^31 - 256, 2^31) give INT_MIN, hence -128;
  then the byte ReLU (negative bytes -> 0) when the layer's activation is RELU.
cs = fl(fl(in_scale * w_scale) / out_scale); the crafted models use in_scale = out_scale = 1, so cs is the weight scale.

The sweep generator finds, for a scale and an accumulator range, every step of r (by bisection over a grid), every negative
exact tie -(n + 0.5) and -pred(0.5) of fl(t * cs), and solves for int8 input pixels whose accumulators hit the steps -2 .. +1,
the ties, -1 / 0 / 1 and both ends of the range."""
import struct

import numpy as np

F32 = np.float32
INT_MIN = -(1 << 31)


# ---- arithmetic --------------------------------------------------------------------------------------------------------
def wrap32(v):
    """two's-complement int32 wrap of int64 values"""
    return ((np.asarray(v, dtype=np.int64) + (1 << 31)) % (1 << 32)) - (1 << 31)


def conv_scale(in_scale, w_scale, out_scale):
    with np.errstate(all="ignore"):
        return F32(F32(F32(in_scale) * F32(w_scale)) / F32(out_scale))


def requant(t, cs):
    """r(t) of the reference for int32 values t (int64 array), as int64 in [-128, 127]"""
    t = np.asarray(t, dtype=np.int64)
    cs = F32(cs)
    with np.errstate(all="ignore"):
        sc = t.astype(F32) * cs
        h = sc + np.where(sc >= 0, F32(0.5), F32(-0.5))
        ok = (h > F32(-2147483904.0)) & (h < F32(2147483648.0))
        r = np.where(ok, np.trunc(np.where(ok, h, F32(0)).astype(np.float64)), float(INT_MIN)).astype(np.int64)
    return np.clip(r, -128, 127)


def conv_acc(x, w, s, pt, pl, oh, ow):
    """int64 accumulators [Co, oh, ow] of x (C, H, W) with w (Co, C, kh, kw): output (y, x), tap (ky, kx) reads input
    (y*s - pt + ky, x*s - pl + kx) when it lies inside the image.  Products and sums are exact in float64 (|sum| < 2^53)."""
    C, H, W = x.shape
    co, _, kh, kw = w.shape
    # zero border wide enough for every tap: a skipped tap and a zero input contribute the same nothing
    PT, PL = max(pt, 0), max(pl, 0)
    PB, PR = max(0, (oh - 1) * s - pt + kh - H), max(0, (ow - 1) * s - pl + kw - W)
    xp = np.zeros((C, H + PT + PB, W + PL + PR), dtype=np.float64)
    xp[:, PT:PT + H, PL:PL + W] = x
    acc = np.zeros((co, oh, ow), dtype=np.float64)
    wf = w.astype(np.float64)
    for ky in range(kh):
        for kx in range(kw):
            if not wf[:, :, ky, kx].any():
                continue
            y0, x0 = PT - pt + ky, PL - pl + kx
            patch = xp[:, y0: y0 + (oh - 1) * s + 1: s, x0: x0 + (ow - 1) * s + 1: s]
            acc += np.tensordot(wf[:, :, ky, kx], patch, axes=(1, 0))
    return acc.astype(np.int64)


# ---- crafted models ------------------------------------------------------------------------------------------------------
ACT_PLAIN, ACT_RELU, ACT_SILU = "plain", "relu", "silu"

# layout -> (nhwc, k, stride, ci, h, w): the tensor-core mode each one takes
#   nchw1: 1x1 straight from the NCHW planes (TMA); nchw3: 3x3 over the padded channel-innermost copy (halo loads);
#   nhwc1: 1x1 flat tiles from the channel-innermost arena tensor; nhwc3: 3x3 rect tiles, one 4-d TMA box per tap;
#   gather: 3x3 over 8 channels, K rows built in shared memory; stem: 6x6 stride 2 over 4 channels (space-to-depth copy)
LAYOUTS = {
    "nchw1": (False, 1, 1, 32, 48, 64), "nchw3": (False, 3, 1, 32, 48, 64),
    "nhwc1": (True, 1, 1, 32, 48, 64), "nhwc3": (True, 3, 1, 32, 48, 64),
    "gather": (False, 3, 1, 8, 70, 64), "stem": (False, 6, 2, 4, 128, 128),
}


class ConvSpec:
    """one int8 conv of a crafted model: OIHW weights, raw int32 biases, weight scale, activation"""

    def __init__(self, w, bias, ws, act, s, same):
        self.w, self.bias, self.ws, self.act, self.s, self.same = w, np.asarray(bias, dtype=np.int64), ws, act, s, same
        self.co, self.ci, self.k = w.shape[0], w.shape[1], w.shape[2]

    @property
    def cs(self):
        return conv_scale(1.0, self.ws, 1.0)

    @property
    def bound(self):
        """max over output channels of 128 * sum |w| + |bias| (what the planner computes, csrc/conv_tc.cu acc_bound)"""
        return int((128 * np.abs(self.w.astype(np.int64)).reshape(self.co, -1).sum(1) + np.abs(wrap32(self.bias))).max())

    def geometry(self, h, w):
        """(oh, ow, pt, pl) as the executor derives them: SAME -> centred pads, anything else -> no padding"""
        p = self.k // 2 if self.k != 6 else 2
        oh, ow = (h + 2 * p - self.k) // self.s + 1, (w + 2 * p - self.k) // self.s + 1
        if not self.same:
            return oh, ow, 0, 0
        return oh, ow, ((oh - 1) * self.s + self.k - h) // 2, ((ow - 1) * self.s + self.k - w) // 2

    def forward(self, x):
        """x (C, H, W) int -> (t [Co, oh, ow] int32 values, output bytes as int8 [Co, oh, ow])"""
        oh, ow, pt, pl = self.geometry(x.shape[1], x.shape[2])
        t = wrap32(conv_acc(x, self.w, self.s, pt, pl, oh, ow) + self.bias[:, None, None])
        r = requant(t, self.cs)
        if self.act == ACT_RELU:
            r = np.maximum(r, 0)
        return t, r.astype(np.int8)


class Case:
    """A crafted model: one conv (optionally followed by Sigmoid + Mul, the compiler's SiLU) or a 1x1 -> 3x3 chain.
    rq: the variant the planner must select for the first conv."""

    def __init__(self, name, rq, layout, co, act, ws, bias0=700, ci=None, random_w=False, chain=False, seed=0):
        self.name, self.rq, self.layout, self.act, self.chain = name, rq, layout, act, chain
        nhwc, k, s, ci0, h, w = LAYOUTS[layout]
        self.nhwc, self.h, self.w = nhwc, h, w
        self.ci = ci or ci0
        rng = np.random.default_rng(seed)
        same = k > 1
        wt = np.zeros((co, self.ci, k, k), dtype=np.int8)
        if random_w:
            # random magnitudes on every tap; the sign depends on (co, ci) only, so inputs matched to channel 0's signs reach
            # +127 * sum|w| and -128 * sum|w| on the interior pixels
            mag = rng.integers(1, 128, size=(co, self.ci, k, k))
            sgn = np.where(rng.random((co, self.ci)) < 0.5, -1, 1)
            wt[:] = (mag * sgn[:, :, None, None]).astype(np.int8)
        else:
            # one weight row (1, 127, ..., 127) on a single tap, negated on odd channels: t = +-A + bias with A = x0 + 127 * sum x_i
            row = np.full(self.ci, 127, dtype=np.int64)
            row[0] = 1
            sign = np.where(np.arange(co) % 2 == 0, 1, -1)
            conv0 = ConvSpec(wt, np.zeros(co), ws, act, s, same)
            _, _, pt, pl = conv0.geometry(h, w)
            # tap (pt, pl) maps output (y, x) to input (y*s, x*s): always inside the image
            wt[:, :, pt, pl] = (sign[:, None] * row[None, :]).astype(np.int8)
        if isinstance(bias0, (list, tuple)):
            bias = np.array([bias0[c % len(bias0)] for c in range(co)], dtype=np.int64)
        else:  # small per-channel spread around +-bias0: P pixels x Co channels give many distinct t
            bias = np.array([(bias0 if c % 2 == 0 else -bias0) + (c // 2) % 7 - 3 for c in range(co)], dtype=np.int64)
        self.convs = [ConvSpec(wt, bias, ws, act, s, same)]
        if chain:  # second conv: 3x3 over the first's output (its epilogue writes this conv's channel-innermost copy)
            w2 = rng.integers(-127, 128, size=(48, co, 3, 3), dtype=np.int8)
            self.convs.append(ConvSpec(w2, rng.integers(-1500, 1501, size=48), 0.0011, ACT_PLAIN, 1, True))
        self.random_w = random_w
        self.seed = seed

    # ---- the .mars file --------------------------------------------------------------------------------------------------
    def marsfile(self, mf):
        m = mf.MarsFile()
        fmt = mf.FMT_NHWC if self.nhwc else mf.FMT_NCHW

        def shape(c, h, w):
            return [1, h, w, c] if self.nhwc else [1, c, h, w]

        x = m.add_tensor("x", mf.DT_I8, fmt, shape(self.ci, self.h, self.w), 1.0)
        m.inputs = [x]
        self.y_ids = []
        cur, (c, h, w) = x, (self.ci, self.h, self.w)
        for i, cv in enumerate(self.convs):
            wt = np.ascontiguousarray(cv.w.transpose(0, 2, 3, 1)) if self.nhwc else cv.w
            wid = m.add_tensor("w%d" % i, mf.DT_I8, mf.FMT_OHWI if self.nhwc else mf.FMT_OIHW, list(wt.shape), cv.ws, wt.tobytes())
            bid = m.add_tensor("b%d" % i, mf.DT_F32, mf.FMT_NCHW, [cv.co], 1.0, wrap32(cv.bias).astype("<i4").tobytes())
            oh, ow, _, _ = cv.geometry(h, w)
            y = m.add_tensor("y%d" % i, mf.DT_I8, fmt, shape(cv.co, oh, ow), 1.0)
            pad = cv.k // 2 if cv.k != 6 else 2
            params = struct.pack("<15I", cv.k, cv.k, cv.s, cv.s, 1, 1, mf.PAD_SAME if cv.same else mf.PAD_VALID, pad, pad, pad, pad, 1,
                                 mf.ACT_RELU if cv.act == ACT_RELU else mf.ACT_NONE, wid, bid)
            m.add_layer(mf.L_CONV, [cur], [y], params)
            self.y_ids.append(y)
            cur, (c, h, w) = y, (cv.co, oh, ow)
        m.outputs = [cur]
        if self.act == ACT_SILU:
            sg = m.add_tensor("sig", mf.DT_I8, fmt, shape(c, h, w), 1.0 / 127.0)
            m.add_layer(mf.L_SIGMOID, [cur], [sg])
            mu = m.add_tensor("mul", mf.DT_I8, fmt, shape(c, h, w), 1.0)
            m.add_layer(mf.L_MUL, [cur, sg], [mu])
            m.outputs = [mu]
        return m

    # ---- inputs ----------------------------------------------------------------------------------------------------------
    def sweep(self):
        """(input (C, H, W) int8 of slot 0, claims): claims[c] = the t values channel c (0: weight sign +, 1: -) must reach"""
        cv = self.convs[0]
        oh, ow, _, _ = cv.geometry(self.h, self.w)
        rng = np.random.default_rng(self.seed + 1)
        x = rng.integers(-128, 128, size=(self.ci, self.h, self.w)).astype(np.int64)
        if self.random_w:
            pos = cv.w[0, :, 0, 0] > 0
            hi_px, lo_px = np.where(pos, 127, -128), np.where(pos, -128, 127)
            top = self.h * 2 // 5
            x[:, :top] = hi_px[:, None, None]
            x[:, self.h - top:] = lo_px[:, None, None]
            w0 = cv.w[0].astype(np.int64).sum(axis=(1, 2))
            return x.astype(np.int8), {0: np.array([int(w0 @ hi_px) + int(cv.bias[0]), int(w0 @ lo_px) + int(cv.bias[0])])}
        n1 = self.ci - 1
        amax, amin = 127 + 127 * 127 * n1, -128 - 127 * 128 * n1
        npix = oh * ow
        A = rng.integers(amin, amax + 1, size=npix)
        claims = {}
        at = 0
        for c, sign in ((0, 1), (1, -1)):
            b = int(cv.bias[c])
            a_list = sweep_targets(cv.cs, sign, b, amin, amax)[: npix // 2]
            A[at: at + a_list.size] = a_list
            at += a_list.size
            claims[c] = np.unique(wrap32(sign * a_list + b))
        vec = solve_pixels(A, self.ci)  # (npix, ci): the single weighted tap reads input pixel (y*s, x*s) for output (y, x)
        ys, xs = np.divmod(np.arange(npix), ow)
        x[:, ys * cv.s, xs * cv.s] = vec.T
        return x.astype(np.int8), claims

    def slot_inputs(self, n=3):
        """n input images (C, H, W): slot 0 the sweep, slot i its output pixels permuted (the same multiset of t per channel; random
        weights: the columns rotated)"""
        x0, claims = self.sweep()
        xs = [x0]
        cv = self.convs[0]
        oh, ow, _, _ = cv.geometry(self.h, self.w)
        for i in range(1, n):
            if self.random_w:  # every tap is weighted: keep the sign-matched bands whole, move the columns
                xs.append(np.roll(x0, 7 * i, axis=2))
                continue
            perm = np.random.default_rng(100 + i).permutation(oh * ow)
            xi = x0.copy()
            ys, xs_ = np.divmod(np.arange(oh * ow), ow)
            py, px = ys * cv.s, xs_ * cv.s
            xi[:, py, px] = x0[:, py[perm], px[perm]]
            xs.append(xi)
        return xs, claims

    def to_bytes_layout(self, x):
        """(C, H, W) -> the model's input tensor bytes"""
        return np.ascontiguousarray(x.transpose(1, 2, 0) if self.nhwc else x).reshape(-1).astype(np.int8)

    def from_layout(self, flat, c, h, w):
        a = np.asarray(flat).view(np.int8)[: c * h * w]
        return a.reshape(h, w, c).transpose(2, 0, 1) if self.nhwc else a.reshape(c, h, w)

    def reference(self, x):
        """[(t, y)] of every conv for input x (C, H, W)"""
        out = []
        cur = x.astype(np.int64)
        for cv in self.convs:
            t, y = cv.forward(cur)
            out.append((t, y))
            cur = y.astype(np.int64)
        return out


def solve_pixels(A, ci):
    """int8 channel vectors v (len(A), ci) with v0 + 127 * sum(v1..) == A (A within [-128 - 127*128*(ci-1), 127 + 127*127*(ci-1)])"""
    A = np.asarray(A, dtype=np.int64)
    n1 = ci - 1
    S = np.clip(np.floor_divide(A + 63, 127), -128 * n1, 127 * n1)
    x0 = A - 127 * S
    S = np.where(x0 > 127, S + 1, np.where(x0 < -128, S - 1, S))
    S = np.clip(S, -128 * n1, 127 * n1)
    x0 = A - 127 * S
    assert ((x0 >= -128) & (x0 <= 127)).all(), "accumulator target out of reach"
    q, r = np.divmod(S, n1)
    v = np.empty((A.size, ci), dtype=np.int64)
    v[:, 0] = x0
    v[:, 1:] = q[:, None] + (np.arange(n1)[None, :] < r[:, None])
    assert ((v >= -128) & (v <= 127)).all() and (v[:, 0] + 127 * v[:, 1:].sum(1) == A).all()
    return v


def change_points(f, lo, hi, grid=4097):
    """every integer u in (lo, hi] with f(u) != f(u - 1), for f monotone between the points of an even grid (vectorised bisection)"""
    g = np.unique(np.linspace(lo, hi, grid).round().astype(np.int64))
    a, b = g[:-1], g[1:]
    out = []
    while a.size:
        keep = f(a) != f(b)
        a, b = a[keep], b[keep]
        unit = (b - a) == 1
        out.append(b[unit])
        a, b = a[~unit], b[~unit]
        mid = a + (b - a) // 2
        a, b = np.concatenate([a, mid]), np.concatenate([mid, b])
    return np.unique(np.concatenate(out)) if out else np.zeros(0, dtype=np.int64)


def negative_ties(cs, lo, hi):
    """every t in [lo, hi] whose fl(t * cs) is -(n + 0.5) (n = 0..127) or -pred(0.5)"""
    cs = F32(cs)
    if not np.isfinite(cs) or cs == 0:
        return np.zeros(0, dtype=np.int64)
    ties = [-np.nextafter(F32(0.5), F32(0))] + [-(F32(n) + F32(0.5)) for n in range(128)]
    found = []
    for c in ties:
        t0 = float(c) / float(cs)
        if t0 < lo - 8 or t0 > hi + 8:
            continue
        ulp = float(np.spacing(abs(c)))
        span = min(int(2 * ulp / abs(float(cs))) + 3, 1 << 16)
        t = np.arange(int(round(t0)) - span, int(round(t0)) + span + 1, dtype=np.int64)
        t = t[(t >= lo) & (t <= hi)]
        with np.errstate(all="ignore"):
            found.append(t[t.astype(F32) * cs == c])
    return np.unique(np.concatenate(found)) if found else np.zeros(0, dtype=np.int64)


def sweep_targets(cs, sign, bias, amin, amax):
    """values A of the pixel sum for the channel t = wrap32(sign * A + bias): the range ends, t = -1 / 0 / 1, every negative tie,
    and u - 2 .. u + 1 around every step u of r(t(A)) over [amin, amax].  Ends and ties come first (they are kept when the pixel
    budget truncates the list)."""
    def f(A):
        return requant(wrap32(sign * np.asarray(A, dtype=np.int64) + bias), cs)

    def a_of_t(t):  # every A in range with wrap32(sign * A + bias) == t
        t = np.asarray(t, dtype=np.int64)
        out = [sign * (t - bias + j * (1 << 32)) for j in (-1, 0, 1)]
        a = np.concatenate(out)
        return a[(a >= amin) & (a <= amax)]

    tlo, thi = sorted((sign * amin + bias, sign * amax + bias))
    ends = np.array([amin, amax], dtype=np.int64)
    small = a_of_t(np.array([-1, 0, 1]))
    ties = a_of_t(negative_ties(cs, max(tlo, -(1 << 31)), min(thi, (1 << 31) - 1)))
    steps = change_points(f, amin, amax)
    around = (steps[:, None] + np.arange(-2, 2)[None, :]).ravel()
    around = around[(around >= amin) & (around <= amax)]
    seen, out = set(), []
    for v in np.concatenate([ends, small, ties, around]).tolist():
        if v not in seen:
            seen.add(v)
            out.append(v)
    return np.array(out, dtype=np.int64)


# ---- the case matrix -----------------------------------------------------------------------------------------------------
# Scales per variant and layout.  select_requant (csrc/conv_tc.cu) picks the variant from the scale and the accumulator bound
# 128 * sum|w| + |bias|: one weighted tap of (1, 127, ..., 127) gives 504 064 + |bias| over 32 channels, 4 665 600 + |bias| over
# 288, 113 920 over the gather's 8 and 48 896 over the stem's 4.  The CPU suite checks every case's variant against the library.
SCALE = {
    3: {"*": 0.013},
    2: {"*": 1.0},
    1: {"*": 0.000528381613548845, "gather": 0.00105676322709769, "stem": 0.0021},
    0: {"*": 0.0002641908067744225, "gather": 0.013, "stem": 0.013},
}
CI288 = {"nchw1", "nchw3", "nhwc1", "nhwc3"}  # RQ 0 by an accumulator bound >= 2^22
WRAP_BIAS = [(1 << 31) - 700, -(1 << 31) + 700]  # acc + bias wraps around int32 (and the bound is >= 2^22)
COS = [48, 40, 255, 300]  # one 16-column unit set, a ragged unit, EPI 16 (one 256-wide N tile), two N tiles (ragged last)


def _co_ok(layout, co, rq):
    if layout == "gather":
        return co <= 256  # the gather producer takes one N tile of at most 256 columns
    if layout == "stem":
        return co <= 128  # the space-to-depth stem: at most 128 output channels
    if rq == 0 and layout in ("nchw3", "nhwc3"):
        return co <= 48  # keeps the 288-channel 3x3 references cheap; the wider columns run on the 1x1 layouts
    return True


def make_cases():
    cases = []
    for rq in (3, 2, 1, 0):
        k = 0
        for act in (ACT_PLAIN, ACT_RELU, ACT_SILU):
            for layout in LAYOUTS:
                while not _co_ok(layout, COS[k % 4], rq):
                    k += 1
                co = COS[k % 4]
                k += 1
                ws = SCALE[rq].get(layout, SCALE[rq]["*"])
                ci = 288 if (rq == 0 and layout in CI288) else None
                bias = WRAP_BIAS if (rq == 0 and layout not in CI288) else 700
                cases.append(Case("rq%d-%s-%s-co%d" % (rq, layout, act, co), rq, layout, co, act, ws, bias0=bias, ci=ci, seed=len(cases)))
    extra = [  # more scales on the 1x1 NCHW layout
        (3, 2.0 ** -10, 700, ACT_PLAIN), (3, 0.013, 1_290_000_000, ACT_PLAIN), (3, 0.0123, 1500, ACT_RELU),
        (2, 0.6, 700, ACT_PLAIN), (2, 0.8, 700, ACT_RELU), (2, 3.0, 700, ACT_SILU), (2, -0.0012345, 700, ACT_PLAIN),
        (2, -0.0012345, 700, ACT_SILU), (1, 0.00105676322709769, 700, ACT_PLAIN), (1, 0.000528381613548845, 1500, ACT_SILU),
        (0, 1e9, 700, ACT_PLAIN), (0, float("inf"), 700, ACT_RELU), (0, float("nan"), 700, ACT_PLAIN), (0, 1e9, 700, ACT_SILU),
        (0, 0.000528381613548845, WRAP_BIAS, ACT_RELU),
    ]
    for i, (rq, ws, bias, act) in enumerate(extra):
        co = COS[i % 4]
        cases.append(Case("rq%d-nchw1-%s-co%d-cs%g%s" % (rq, act, co, ws, "-wrap" if isinstance(bias, list) else "-b%d" % bias), rq, "nchw1",
                          co, act, ws, bias0=bias, seed=100 + i))
    # one random-weight case per layout (every tap weighted, inputs sign-matched to channel 0: the true accumulator extremes)
    for i, (layout, rq, ws) in enumerate([("nchw1", 3, 0.0004), ("nchw3", 1, 0.000528381613548845), ("nhwc1", 2, 1.0),
                                          ("nhwc3", 3, 0.00012), ("gather", 1, 0.0021), ("stem", 3, 0.00012)]):
        co = [48, 40, 255, 48, 40, 48][i]
        cases.append(Case("rand-rq%d-%s-co%d" % (rq, layout, co), rq, layout, co, [ACT_PLAIN, ACT_RELU, ACT_SILU][i % 3], ws, bias0=1500,
                          random_w=True, seed=200 + i))
    # 1x1 -> 3x3 chains: the 1x1's epilogue writes the 3x3's channel-innermost copy (side output).  Plain only: a ReLU on the 1x1
    # is a byte-ReLU op of its own that rewrites the 1x1's output, and the planner links a copy only to the last writer of a tensor
    for i, (rq, ws) in enumerate([(3, 0.013), (2, 1.0), (1, 0.000528381613548845), (0, 1e9)]):
        cases.append(Case("chain-rq%d" % rq, rq, "nchw1", 64, ACT_PLAIN, ws, seed=300 + i, chain=True))
    return cases


CASES = make_cases()
