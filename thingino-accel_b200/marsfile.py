"""marsfile.py -- reader/writer for `.mars` files and deterministic synthetic-model builders.

Three of the five models BASELINE.json names (yolov5s_int8, yolov5s_float32, nanodet_320) are
absent from the reference checkout (.MISSING_LARGE_BLOBS), and its ONNX->.mars compiler is Rust
(not buildable here).  This module writes files that follow the compiler's layout conventions
(reference mars-compiler/src/main.rs:611-916,1463-1522; mars_format.rs:93-397;
tools/mars_gen_test.py) so that the reference runtime and this library load them identically:

  header(76) | tensor descriptors (124 each) | layer descriptors (112 each) | weight blob

  * tensors in creation order: input; per conv: weight, bias, conv output; per SiLU: Sigmoid
    output, Mul output -- the round-robin work-buffer planner depends on that order;
  * conv padding field EXPLICIT with the ONNX pads for k>1 (ignored by the executor!), VALID
    for 1x1; activation NONE; SiLU as separate SIGMOID + MUL layers;
  * weights 4-byte aligned in the blob; weights_offset = 76 + 124*T + 112*L.

`build_yolov5(width=0.25)` reproduces the layer/tensor tables of the shipped
models/yolov5n_int8.mars one for one (checked by tests/test_marsfile.py); width=0.5 is the
yolov5s-shaped model used as the headline workload.  WEIGHTS ARE SYNTHETIC (seeded RNG).
"""
import struct

import numpy as np

MAGIC = 0x5352414D
DT_F32, DT_I32, DT_I16, DT_I8, DT_U8, DT_U4 = 0, 1, 2, 3, 4, 5
FMT_NCHW, FMT_NDHWC32, FMT_HWIO, FMT_NMHWSOIB2, FMT_NMC32, FMT_D1, FMT_OHWI, FMT_NHWC, FMT_OIHW = range(9)
(L_CONV, L_DW, L_MAXPOOL, L_AVGPOOL, L_GAP, L_RELU, L_RELU6, L_LEAKY, L_SILU, L_SIGMOID, L_CONCAT, L_ADD, L_MUL,
 L_UPSAMPLE, L_RESHAPE, L_SOFTMAX, L_FC, L_TRANSPOSE, L_BATCHNORM) = range(19)
PAD_VALID, PAD_SAME, PAD_EXPLICIT = 0, 1, 2
ACT_NONE, ACT_RELU = 0, 1
NO_ID = 0xFFFFFFFF
LAYER_NAMES = {L_CONV: "conv", L_DW: "depthwise", L_MAXPOOL: "maxpool", L_AVGPOOL: "avgpool", L_GAP: "gap",
               L_RELU: "relu", L_RELU6: "relu6", L_LEAKY: "leaky", L_SILU: "silu", L_SIGMOID: "sigmoid",
               L_CONCAT: "concat", L_ADD: "add", L_MUL: "mul", L_UPSAMPLE: "upsample", L_RESHAPE: "reshape",
               L_SOFTMAX: "softmax", L_FC: "fc", L_TRANSPOSE: "transpose", L_BATCHNORM: "batchnorm"}
DTYPE_SIZE = {DT_F32: 4, DT_I32: 4, DT_I16: 2, DT_I8: 1, DT_U8: 1, DT_U4: 1}


class Tensor:
    def __init__(self, tid, name, dtype, fmt, shape, scale=1.0, zero_point=0, data=None):
        self.id, self.name, self.dtype, self.format = tid, name, dtype, fmt
        self.shape, self.scale, self.zero_point = list(shape), float(scale), int(zero_point)
        self.data = data  # bytes for weight tensors, None for runtime tensors
        self.data_offset = 0
        self.data_size = 0

    def pack(self):
        shape = (self.shape + [0] * 6)[:6]
        return struct.pack("<I60siiI6iQQfi", self.id, self.name.encode()[:59], self.dtype, self.format,
                           len(self.shape), *shape, self.data_offset, self.data_size, np.float32(self.scale),
                           self.zero_point)

    @property
    def numel(self):
        n = 1
        for d in self.shape:
            n *= max(d, 0)
        return n


class Layer:
    def __init__(self, lid, ltype, inputs, outputs, params=b""):
        self.id, self.type, self.inputs, self.outputs = lid, ltype, list(inputs), list(outputs)
        self.params = bytes(params)

    def pack(self):
        ins = (self.inputs + [0] * 4)[:4]
        outs = (self.outputs + [0] * 4)[:4]
        return struct.pack("<IiII4I4I64s", self.id, self.type, len(self.inputs), len(self.outputs), *ins, *outs,
                           self.params.ljust(64, b"\0"))

    def conv_params(self):
        k = struct.unpack("<15I", self.params[:60])
        return dict(zip(("kh", "kw", "sh", "sw", "dh", "dw", "padding", "pt", "pb", "pl", "pr", "groups", "act",
                         "weight", "bias"), k))


class MarsFile:
    """In-memory .mars model: tensor table, layer table, weight blob."""

    def __init__(self):
        self.tensors, self.layers = [], []
        self.inputs, self.outputs = [], []
        self.version = (1, 0)
        self.flags = 0

    # ---- building -------------------------------------------------------------
    def add_tensor(self, name, dtype, fmt, shape, scale=1.0, data=None):
        t = Tensor(len(self.tensors), name, dtype, fmt, shape, scale, 0, data)
        self.tensors.append(t)
        return t.id

    def add_layer(self, ltype, inputs, outputs, params=b""):
        self.layers.append(Layer(len(self.layers), ltype, inputs, outputs, params))
        return len(self.layers) - 1

    # ---- serialisation --------------------------------------------------------
    def to_bytes(self):
        blob = bytearray()
        for t in self.tensors:
            if t.data is not None:
                while len(blob) % 4:  # reference mars-compiler/src/main.rs:611-619
                    blob.append(0)
                t.data_offset, t.data_size = len(blob), len(t.data)
                blob += t.data
            else:
                t.data_offset = t.data_size = 0
        woff = 76 + 124 * len(self.tensors) + 112 * len(self.layers)
        ins = (self.inputs + [NO_ID] * 4)[:4]
        outs = (self.outputs + [NO_ID] * 4)[:4]
        hdr = struct.pack("<IHHIIIIIQQ4I4I", MAGIC, self.version[0], self.version[1], self.flags, len(self.layers),
                          len(self.tensors), len(self.inputs), len(self.outputs), woff, len(blob), *ins, *outs)
        assert len(hdr) == 76
        return hdr + b"".join(t.pack() for t in self.tensors) + b"".join(l.pack() for l in self.layers) + bytes(blob)

    def save(self, path):
        with open(path, "wb") as f:
            f.write(self.to_bytes())

    @staticmethod
    def from_bytes(b):
        (magic, vmaj, vmin, flags, nl, nt, ni, no, woff, wsize) = struct.unpack_from("<IHHIIIIIQQ", b, 0)
        if magic != MAGIC:
            raise ValueError("bad magic")
        m = MarsFile()
        m.version, m.flags = (vmaj, vmin), flags
        ids = struct.unpack_from("<8I", b, 44)
        m.inputs, m.outputs = list(ids[:ni]), list(ids[4:4 + no])
        off = 76
        for _ in range(nt):
            f = struct.unpack_from("<I60siiI6iQQfi", b, off)
            off += 124
            t = Tensor(f[0], f[1].split(b"\0")[0].decode(errors="replace"), f[2], f[3], list(f[5:5 + min(f[4], 6)]),
                       f[13], f[14])
            t.data_offset, t.data_size = f[11], f[12]
            if t.data_size:
                t.data = bytes(b[woff + t.data_offset: woff + t.data_offset + t.data_size])
            m.tensors.append(t)
        for _ in range(nl):
            f = struct.unpack_from("<IiII4I4I64s", b, off)
            off += 112
            m.layers.append(Layer(f[0], f[1], f[4:4 + min(f[2], 4)], f[8:8 + min(f[3], 4)], f[12]))
        m.weights_size = wsize
        return m

    @staticmethod
    def load(path):
        with open(path, "rb") as f:
            return MarsFile.from_bytes(f.read())

    # ---- analysis -------------------------------------------------------------
    def conv_macs(self):
        """Sum over CONV2D layers of Co*Ho*Wo*Ci*kh*kw (SURVEY 8d), from the descriptors."""
        by_id = {t.id: t for t in self.tensors}
        total = 0
        for l in self.layers:
            if l.type != L_CONV:
                continue
            p = l.conv_params()
            i, o = by_id.get(l.inputs[0]), by_id.get(l.outputs[0])
            if i is None or o is None or len(i.shape) < 4 or len(o.shape) < 4:
                continue
            if i.format == FMT_NHWC:
                ci, (co, oh, ow) = i.shape[3], (o.shape[3], o.shape[1], o.shape[2])
            else:
                ci, (co, oh, ow) = i.shape[1], (o.shape[1], o.shape[2], o.shape[3])
            total += max(co, 0) * max(oh, 0) * max(ow, 0) * max(ci, 0) * p["kh"] * p["kw"]
        return total

    def layer_bytes(self):
        """(conv_bytes, other_bytes) per image as the reference executes them (SURVEY 8d):
        conv in+out+w; sigmoid/relu 2n; mul/add 3n; pool/concat/upsample read+write."""
        by_id = {t.id: t for t in self.tensors}
        conv = other = 0
        for l in self.layers:
            ts = [by_id.get(i) for i in l.inputs]
            o = by_id.get(l.outputs[0]) if l.outputs else None
            if l.type == L_CONV:
                p = l.conv_params()
                w = by_id.get(p["weight"])
                if ts[0] is None or o is None or w is None:
                    continue
                es = DTYPE_SIZE[ts[0].dtype]
                conv += (ts[0].numel + o.numel) * es + w.numel * es
            elif l.type in (L_SIGMOID, L_RELU, L_RELU6, L_LEAKY, L_BATCHNORM):
                if ts and ts[0] is not None:
                    other += 2 * ts[0].numel * DTYPE_SIZE[ts[0].dtype]
            elif l.type in (L_ADD, L_MUL):
                if ts and ts[0] is not None:
                    other += 3 * ts[0].numel * DTYPE_SIZE[ts[0].dtype]
            elif l.type in (L_MAXPOOL, L_UPSAMPLE):
                if ts and ts[0] is not None and o is not None:
                    other += ts[0].numel + o.numel
            elif l.type == L_CONCAT and o is not None:
                other += 2 * o.numel
        return conv, other


# --------------------------------------------------------------------------------------
# builders
# --------------------------------------------------------------------------------------
def _conv_params(k, s, pad, w_id, b_id, padding=None, act=ACT_NONE, groups=1):
    if padding is None:
        padding = PAD_EXPLICIT if k > 1 else PAD_VALID  # what the compiler emits (main.rs:897-901)
    return struct.pack("<15I", k, k, s, s, 1, 1, padding, pad, pad, pad, pad, groups, act, w_id, b_id)


class _Builder:
    """Emits tensors/layers in the order mars-compiler does for a YOLOv5-style ONNX graph."""

    def __init__(self, seed, f32=False, nhwc=False, act_scale=0.05, sig_scale=1.0 / 127.0):
        self.m = MarsFile()
        self.rng = np.random.default_rng(seed)
        self.f32, self.nhwc = f32, nhwc
        self.act_scale, self.sig_scale = act_scale, sig_scale
        self.adt = DT_F32 if f32 else DT_I8
        self.afmt = FMT_NHWC if nhwc else FMT_NCHW
        self.shape = {}  # tensor id -> (c, h, w)

    def ashape(self, c, h, w):
        return [1, h, w, c] if self.nhwc else [1, c, h, w]

    def rt(self, name, c, h, w, scale=None):
        tid = self.m.add_tensor(name, self.adt, self.afmt, self.ashape(c, h, w), self.act_scale if scale is None else scale)
        self.shape[tid] = (c, h, w)
        return tid

    def weights(self, name, co, ci, k, in_rms=24.0, out_rms=28.0):
        """int8: uniform [-127,127] values, per-tensor scale chosen so that the requantised output
        neither saturates nor collapses (cs = in_scale*w_scale/out_scale); f32: N(0, 1/K)."""
        K = ci * k * k
        if self.f32:
            w = (self.rng.standard_normal((co, ci, k, k)) / np.sqrt(K)).astype(np.float32)
            b = (self.rng.standard_normal(co) * 0.1).astype(np.float32)
            wscale = 1.0
        else:
            w = self.rng.integers(-127, 128, size=(co, ci, k, k), dtype=np.int8)
            b = self.rng.integers(-1500, 1501, size=co).astype(np.int32)  # read as int32[Co] by the executor
            cs = out_rms / (np.sqrt(K) * 73.6 * in_rms)
            wscale = float(np.float32(cs))  # in_scale == out_scale for conv in/out tensors
        if self.nhwc:
            w = np.ascontiguousarray(w.transpose(0, 2, 3, 1))  # OIHW -> OHWI (mars_format.rs:407-434)
            wshape, wfmt = [co, k, k, ci], FMT_OHWI
        else:
            wshape, wfmt = [co, ci, k, k], FMT_OIHW
        wid = self.m.add_tensor(name + ".weight", self.adt, wfmt, wshape, wscale, w.tobytes())
        bid = self.m.add_tensor(name + ".bias", DT_F32, FMT_NCHW, [co], 1.0, b.tobytes())
        return wid, bid

    def conv(self, wname, oname, x, co, k, s, act=True, in_rms=24.0):
        ci, h, w = self.shape[x]
        pad = k // 2 if k != 6 else 2
        ho, wo = (h + 2 * pad - k) // s + 1, (w + 2 * pad - k) // s + 1
        wid, bid = self.weights(wname, co, ci, k, in_rms=in_rms)
        y = self.rt(oname + "/Conv_output_0", co, ho, wo)
        self.m.add_layer(L_CONV, [x], [y], _conv_params(k, s, pad, wid, bid))
        return y

    def silu(self, base, y):
        c, h, w = self.shape[y]
        sg = self.rt(base + "/Sigmoid_output_0", c, h, w, scale=self.sig_scale)
        self.m.add_layer(L_SIGMOID, [y], [sg])
        mu = self.rt(base + "/Mul_output_0", c, h, w)
        self.m.add_layer(L_MUL, [y, sg], [mu])
        return mu

    def cbs(self, mod, path, x, co, k, s, in_rms=24.0):
        """Conv + SiLU block named like the ONNX export of a YOLOv5 `Conv` module."""
        y = self.conv(mod + ".conv", path + "/conv", x, co, k, s, in_rms=in_rms)
        return self.silu(path + "/act", y)

    def c3(self, idx, x, c2, n, shortcut):
        mod, path = "model.%d" % idx, "/model.%d" % idx
        c_ = c2 // 2
        a = self.cbs(mod + ".cv1", path + "/cv1", x, c_, 1, 1)
        for i in range(n):
            b1 = self.cbs("%s.m.%d.cv1" % (mod, i), "%s/m/m.%d/cv1" % (path, i), a, c_, 1, 1)
            b2 = self.cbs("%s.m.%d.cv2" % (mod, i), "%s/m/m.%d/cv2" % (path, i), b1, c_, 3, 1)
            if shortcut:
                s = self.rt("%s/m/m.%d/Add_output_0" % (path, i), c_, *self.shape[a][1:])
                self.m.add_layer(L_ADD, [a, b2], [s])
                a = s
            else:
                a = b2
        b = self.cbs(mod + ".cv2", path + "/cv2", x, c_, 1, 1)
        cat = self.concat(path + "/Concat_output_0", [a, b])
        return self.cbs(mod + ".cv3", path + "/cv3", cat, c2, 1, 1)

    def concat(self, name, xs, axis=1):
        c = sum(self.shape[x][0] for x in xs)
        _, h, w = self.shape[xs[0]]
        y = self.rt(name, c, h, w)
        self.m.add_layer(L_CONCAT, xs, [y], struct.pack("<2I", 3 if self.nhwc else axis, len(xs)))
        return y

    def sppf(self, idx, x, c2):
        mod, path = "model.%d" % idx, "/model.%d" % idx
        c_ = self.shape[x][0] // 2
        a = self.cbs(mod + ".cv1", path + "/cv1", x, c_, 1, 1)
        pools = [a]
        for i in range(3):
            p = self.rt("%s/m%s/MaxPool_output_0" % (path, "" if i == 0 else "_%d" % i), *self.shape[a])
            self.m.add_layer(L_MAXPOOL, [pools[-1]], [p], struct.pack("<9I", 5, 5, 1, 1, PAD_EXPLICIT, 2, 2, 2, 2))
            pools.append(p)
        cat = self.concat(path + "/Concat_output_0", pools)
        return self.cbs(mod + ".cv2", path + "/cv2", cat, c2, 1, 1)

    def upsample(self, idx, x):
        c, h, w = self.shape[x]
        y = self.rt("/model.%d/Resize_output_0" % idx, c, 2 * h, 2 * w)
        self.m.add_layer(L_UPSAMPLE, [x], [y], struct.pack("<3I", 2, 2, 0))
        return y


def _sfx(base, i):
    return base + ("" if i == 0 else "_%d" % i)


def build_yolov5(width=0.5, depth=0.33, size=640, seed=5, f32=False, nhwc=False, nc=80):
    """YOLOv5 v6 graph (width 0.25 = n, 0.5 = s) as mars-compiler emits it, synthetic weights."""
    ch = lambda c: int(np.ceil(c * width / 8) * 8)
    rep = lambda n: max(round(n * depth), 1)
    b = _Builder(seed, f32=f32, nhwc=nhwc)
    m = b.m
    x = m.add_tensor("images", b.adt, b.afmt, b.ashape(3, size, size), 1.0 if not f32 else 1.0)
    b.shape[x] = (3, size, size)
    m.inputs = [x]
    # the int8 input is pixel-128 in [-128,127]: rms ~74
    x0 = b.cbs("model.0", "/model.0", x, ch(64), 6, 2, in_rms=74.0)
    x1 = b.cbs("model.1", "/model.1", x0, ch(128), 3, 2)
    x2 = b.c3(2, x1, ch(128), rep(3), True)
    x3 = b.cbs("model.3", "/model.3", x2, ch(256), 3, 2)
    x4 = b.c3(4, x3, ch(256), rep(6), True)
    x5 = b.cbs("model.5", "/model.5", x4, ch(512), 3, 2)
    x6 = b.c3(6, x5, ch(512), rep(9), True)
    x7 = b.cbs("model.7", "/model.7", x6, ch(1024), 3, 2)
    x8 = b.c3(8, x7, ch(1024), rep(3), True)
    x9 = b.sppf(9, x8, ch(1024))
    x10 = b.cbs("model.10", "/model.10", x9, ch(512), 1, 1)
    x11 = b.upsample(11, x10)
    x12 = b.concat("/model.12/Concat_output_0", [x11, x6])
    x13 = b.c3(13, x12, ch(512), rep(3), False)
    x14 = b.cbs("model.14", "/model.14", x13, ch(256), 1, 1)
    x15 = b.upsample(15, x14)
    x16 = b.concat("/model.16/Concat_output_0", [x15, x4])
    x17 = b.c3(17, x16, ch(256), rep(3), False)
    x18 = b.cbs("model.18", "/model.18", x17, ch(256), 3, 2)
    x19 = b.concat("/model.19/Concat_output_0", [x18, x14])
    x20 = b.c3(20, x19, ch(512), rep(3), False)
    x21 = b.cbs("model.21", "/model.21", x20, ch(512), 3, 2)
    x22 = b.concat("/model.22/Concat_output_0", [x21, x10])
    x23 = b.c3(23, x22, ch(1024), rep(3), False)
    # Detect head.  The compiler drops Split/Pow/Constant nodes (main.rs:96-97) and leaves their
    # tensors with all-zero shapes, so every layer after the three head convs iterates zero
    # elements and `output0` exposes whatever its work buffer holds (SURVEY Appendix B.2).
    no = 3 * (nc + 5)
    zero = lambda name, last=0: m.add_tensor(name, b.adt, b.afmt, [0, 0, 0, last], b.act_scale)
    finals = []
    for li, feat in enumerate((x17, x20, x23)):
        p = "/model.24/"
        y = b.conv("model.24.m.%d" % li, "/model.24/m.%d" % li, feat, no, 1, 1)
        # rename to the ONNX names of the raw nn.Conv2d heads (no ".conv" infix)
        m.tensors[y - 2].name = "model.24.m.%d.weight" % li
        m.tensors[y - 1].name = "model.24.m.%d.bias" % li
        r0 = zero(p + _sfx("Reshape", 2 * li) + "_output_0")
        m.add_layer(L_RESHAPE, [y], [r0], struct.pack("<6iI", 0, 0, 0, 0, 0, 0, 4))
        t0 = zero(p + _sfx("Transpose", li) + "_output_0", 1)
        m.add_layer(L_SOFTMAX, [r0], [t0], struct.pack("<7I", 0, 1, 3, 4, 2, 0, 5))  # Transpose written as type 15
        s0 = zero(p + _sfx("Sigmoid", li) + "_output_0", 1)
        m.add_layer(L_SIGMOID, [t0], [s0])
        sp0 = zero(p + _sfx("Split", li) + "_output_0")
        c1 = zero(p + "Constant_%d_output_0" % (8 * li + 1))
        mu0 = zero(p + _sfx("Mul", 4 * li) + "_output_0")
        m.add_layer(L_MUL, [sp0, c1], [mu0])
        c2 = zero(p + "Constant_%d_output_0" % (8 * li + 2))
        ad = zero(p + _sfx("Add", li) + "_output_0")
        m.add_layer(L_ADD, [mu0, c2], [ad])
        c3 = zero(p + "Constant_%d_output_0" % (8 * li + 3))
        mu1 = zero(p + _sfx("Mul", 4 * li + 1) + "_output_0")
        m.add_layer(L_MUL, [ad, c3], [mu1])
        sp1 = zero(p + _sfx("Split", li) + "_output_1")
        c4 = zero(p + "Constant_%d_output_0" % (8 * li + 4))
        mu2 = zero(p + _sfx("Mul", 4 * li + 2) + "_output_0")
        m.add_layer(L_MUL, [sp1, c4], [mu2])
        pw = zero(p + _sfx("Pow", li) + "_output_0")
        c6 = zero(p + "Constant_%d_output_0" % (8 * li + 6))
        mu3 = zero(p + _sfx("Mul", 4 * li + 3) + "_output_0")
        m.add_layer(L_MUL, [pw, c6], [mu3])
        sp2 = zero(p + _sfx("Split", li) + "_output_2")
        cc = zero(p + _sfx("Concat", li) + "_output_0")
        m.add_layer(L_CONCAT, [mu1, mu3, sp2], [cc], struct.pack("<2I", 3, 3))
        r1 = zero(p + _sfx("Reshape", 2 * li + 1) + "_output_0")
        m.add_layer(L_RESHAPE, [cc], [r1], struct.pack("<6iI", 0, 0, 0, 0, 0, 0, 4))
        finals.append(r1)
    npred = 3 * sum((size // s) ** 2 for s in (8, 16, 32))
    out = m.add_tensor("output0", b.adt, b.afmt, [1, npred, nc + 5], b.act_scale)
    m.add_layer(L_CONCAT, finals, [out], struct.pack("<2I", 1, 3))
    m.outputs = [out]
    return m


def build_tiny(size=160, seed=11, f32=False, relu_layers=True, chans=(16, 32, 64)):
    """tiny_160-shaped chain: three valid 3x3 convs with ReLU layers between (SURVEY B.2)."""
    b = _Builder(seed, f32=f32)
    m = b.m
    x = m.add_tensor("input", b.adt, b.afmt, b.ashape(3, size, size), 1.0)
    b.shape[x] = (3, size, size)
    m.inputs = [x]
    cur, rms = x, 74.0
    for i, co in enumerate(chans):
        ci, h, w = b.shape[cur]
        wid, bid = b.weights("conv%d" % i, co, ci, 3, in_rms=rms)
        y = b.rt("conv%d_out" % i, co, h - 2, w - 2)
        m.add_layer(L_CONV, [cur], [y], _conv_params(3, 1, 0, wid, bid, padding=PAD_VALID))
        cur, rms = y, 24.0
        if relu_layers and i + 1 < len(chans):
            r = b.rt("relu%d_out" % i, co, h - 2, w - 2)
            m.add_layer(L_RELU, [cur], [r])
            cur = r
    m.outputs = [cur]
    return m


def build_nanodet_like(size=320, seed=7, width=1.0, nhwc=False, nc=80, reg_max=7, levels=3):
    """NanoDet-m-shaped graph (ShuffleNetV2-style stem, depthwise 3x3 + pointwise 1x1 blocks,
    concat, 2x nearest upsample, 1x1 heads).  The reference has no NanoDet file or code; its
    DEPTHWISE_CONV2D layer is a no-op (src/mars/mars_runtime.c:1168-1170), which this library
    reproduces by default (mars_b200_set_depthwise_mode(1) = restated depthwise).
    Each head "/head{k}.out/Conv_output_0" is the shared classification + regression conv of a GFL
    head: nc + 4 (reg_max + 1) channels at stride 8 << k.  levels=4 adds a stride-64 level
    (NanoDet-Plus) behind the other three, fed by a stride-2 depthwise block on the last head's
    features.  nhwc=True lays every activation out as [1, h, w, c] (the depthwise weights as OHWI
    [c, 3, 3, 1], the same bytes)."""
    assert levels in (3, 4)
    b = _Builder(seed, nhwc=nhwc)
    m = b.m
    c = lambda v: int(v * width)
    x = m.add_tensor("data", b.adt, b.afmt, b.ashape(3, size, size), 1.0)
    b.shape[x] = (3, size, size)
    m.inputs = [x]

    def relu(name, y):
        r = b.rt(name, *b.shape[y])
        m.add_layer(L_LEAKY, [y], [r])
        return r

    def dw(name, xin, s):
        ci, h, w = b.shape[xin]
        wt = b.rng.integers(-127, 128, size=(ci, 1, 3, 3), dtype=np.int8)
        bs = b.rng.integers(-500, 501, size=ci).astype(np.int32)
        wfmt, wshape = (FMT_OHWI, [ci, 3, 3, 1]) if nhwc else (FMT_OIHW, [ci, 1, 3, 3])
        wid = m.add_tensor(name + ".weight", DT_I8, wfmt, wshape, float(np.float32(28.0 / (3 * 73.6 * 24.0))), wt.tobytes())
        bid = m.add_tensor(name + ".bias", DT_F32, FMT_NCHW, [ci], 1.0, bs.tobytes())
        y = b.rt(name + "_out", ci, (h + 2 - 3) // s + 1, (w + 2 - 3) // s + 1)
        m.add_layer(L_DW, [xin], [y], _conv_params(3, s, 1, wid, bid, padding=PAD_EXPLICIT, groups=ci))
        return y

    def pw(name, xin, co):
        y = b.conv(name, "/" + name, xin, co, 1, 1)
        return relu("/" + name + "/act", y)

    s0 = relu("/stem/act", b.conv("stem", "/stem", x, c(24), 3, 2, in_rms=74.0))
    p0 = b.rt("/stem/pool", *((b.shape[s0][0],) + tuple(v // 2 for v in b.shape[s0][1:])))
    m.add_layer(L_MAXPOOL, [s0], [p0], struct.pack("<9I", 2, 2, 2, 2, PAD_VALID, 0, 0, 0, 0))
    feats, cur = [], p0
    for si, (co, n) in enumerate(((c(116), 4), (c(232), 8), (c(464), 4))):
        cur = pw("stage%d.down.pw" % si, dw("stage%d.down.dw" % si, cur, 2), co)
        for i in range(n - 1):
            a = pw("stage%d.%d.pw1" % (si, i), cur, co // 2)
            d = dw("stage%d.%d.dw" % (si, i), a, 1)
            e = pw("stage%d.%d.pw2" % (si, i), d, co // 2)
            cur = b.concat("/stage%d.%d/Concat" % (si, i), [a, e])
        feats.append(cur)
    f = [pw("fpn.lat%d" % i, t, c(96)) for i, t in enumerate(feats)]
    u1 = b.upsample(101, f[2])
    t1 = b.rt("/fpn/add1", *b.shape[f[1]])
    m.add_layer(L_ADD, [u1, f[1]], [t1])
    u0 = b.upsample(102, t1)
    t0 = b.rt("/fpn/add0", *b.shape[f[0]])
    m.add_layer(L_ADD, [u0, f[0]], [t0])
    outs, chans = [], nc + 4 * (reg_max + 1)
    for i, t in enumerate((t0, t1, f[2])):
        h1 = pw("head%d.pw" % i, dw("head%d.dw" % i, t, 1), c(96))
        outs.append(b.conv("head%d.out" % i, "/head%d.out" % i, h1, chans, 1, 1))
    if levels == 4:
        t3 = pw("fpn.extra.pw", dw("fpn.extra.dw", h1, 2), c(96))
        h1 = pw("head3.pw", dw("head3.dw", t3, 1), c(96))
        outs.append(b.conv("head3.out", "/head3.out", h1, chans, 1, 1))
    m.outputs = [outs[0]]
    return m


def build_single_layer(kind, **kw):
    """1-3 layer micro-models for kernels no shipped file exercises (SURVEY B.4)."""
    seed = kw.get("seed", 3)
    f32 = kw.get("f32", False)
    nhwc = kw.get("nhwc", False)
    b = _Builder(seed, f32=f32, nhwc=nhwc, act_scale=kw.get("act_scale", 0.05))
    m = b.m
    c, h, w = kw.get("c", 8), kw.get("h", 12), kw.get("w", 10)
    x = m.add_tensor("x", b.adt, b.afmt, b.ashape(c, h, w), kw.get("in_scale", 0.05))
    b.shape[x] = (c, h, w)
    m.inputs = [x]
    if kind == "conv":
        k, s, co = kw.get("k", 3), kw.get("s", 1), kw.get("co", 16)
        padding = kw.get("padding", PAD_EXPLICIT)
        pad = kw.get("pad", k // 2)
        if padding == PAD_VALID:
            ho, wo = (h - k) // s + 1, (w - k) // s + 1
        else:
            ho, wo = (h + 2 * pad - k) // s + 1, (w + 2 * pad - k) // s + 1
        wid, bid = b.weights("w", co, c, k, in_rms=60.0)
        if kw.get("no_bias"):
            bid = NO_ID
        y = b.rt("y", co, ho, wo)
        m.add_layer(L_CONV, [x], [y], _conv_params(k, s, pad, wid, bid, padding=padding, act=kw.get("act", ACT_NONE)))
    elif kind in ("sigmoid", "relu", "relu6", "leaky"):
        y = b.rt("y", c, h, w, scale=kw.get("out_scale", 1.0 / 127.0 if kind == "sigmoid" else 0.05))
        m.add_layer({"sigmoid": L_SIGMOID, "relu": L_RELU, "relu6": L_RELU6, "leaky": L_LEAKY}[kind], [x], [y])
    elif kind in ("add", "mul"):
        x2 = m.add_tensor("x2", b.adt, b.afmt, b.ashape(c, h, w), kw.get("in2_scale", 0.02))
        b.shape[x2] = (c, h, w)
        m.inputs = [x, x2]
        y = b.rt("y", c, h, w, scale=kw.get("out_scale", 0.07))
        m.add_layer(L_ADD if kind == "add" else L_MUL, [x, x2], [y])
    elif kind == "maxpool":
        k, s = kw.get("k", 2), kw.get("s", 2)
        # the executor indexes shape[1..3] as H, W, C whatever the tag
        sh = m.tensors[x].shape
        oh, ow = (sh[1] - k) // s + 1, (sh[2] - k) // s + 1
        y = m.add_tensor("y", b.adt, b.afmt, [1, oh, ow, sh[3]], 0.05)
        m.add_layer(L_MAXPOOL, [x], [y], struct.pack("<9I", k, k, s, s, PAD_VALID, 0, 0, 0, 0))
    elif kind == "upsample":
        sc = kw.get("scale", 2)
        sh = m.tensors[x].shape
        y = m.add_tensor("y", b.adt, b.afmt, [1, sh[1] * sc, sh[2] * sc, sh[3]], 0.05)
        m.add_layer(L_UPSAMPLE, [x], [y], struct.pack("<3I", 0 if kw.get("ratio_fallback") else sc,
                                                      0 if kw.get("ratio_fallback") else sc, 0))
    elif kind == "concat":
        n = kw.get("n", 4)
        xs = [x]
        for i in range(1, n):
            t = m.add_tensor("x%d" % i, b.adt, b.afmt, m.tensors[x].shape, 0.05)
            xs.append(t)
        sh = m.tensors[x].shape
        y = m.add_tensor("y", b.adt, b.afmt, [1, sh[1], sh[2], sh[3] * n], 0.05)
        m.inputs = xs
        m.add_layer(L_CONCAT, xs, [y], struct.pack("<2I", 3, n))
    elif kind == "batchnorm":
        sc = (b.rng.standard_normal(c) * 0.5 + 1.0).astype(np.float32)
        bi = (b.rng.standard_normal(c) * 0.3).astype(np.float32)
        sid = m.add_tensor("bn.scale", DT_F32, FMT_NCHW, [c], 1.0, sc.tobytes())
        bid = m.add_tensor("bn.bias", DT_F32, FMT_NCHW, [c], 1.0, bi.tobytes())
        y = b.rt("y", c, h, w, scale=kw.get("out_scale", 0.06))
        m.add_layer(L_BATCHNORM, [x, sid, bid], [y])
    elif kind == "depthwise":
        wt = b.rng.integers(-127, 128, size=(c, 1, 3, 3), dtype=np.int8)
        bs = b.rng.integers(-500, 501, size=c).astype(np.int32)
        wid = m.add_tensor("w", DT_I8, FMT_OIHW, [c, 1, 3, 3], 0.002, wt.tobytes())
        bid = m.add_tensor("b", DT_F32, FMT_NCHW, [c], 1.0, bs.tobytes())
        y = b.rt("y", c, h, w)
        m.add_layer(L_DW, [x], [y], _conv_params(3, 1, 1, wid, bid, padding=PAD_EXPLICIT, groups=c))
    elif kind == "fc":
        y = b.rt("y", c, h, w)
        m.add_layer(L_FC, [x], [y])
    else:
        raise ValueError(kind)
    m.outputs = [len(m.tensors) - 1] if kind not in ("batchnorm",) else [y]
    if kind in ("conv", "depthwise", "fc", "sigmoid", "relu", "relu6", "leaky", "add", "mul"):
        m.outputs = [y]
    return m


# arena sizes the synthetic models need (the reference literal is 8 MiB, src/mars/mars_runtime.c:209)
ARENA_YOLOV5S_INT8 = 32 << 20
ARENA_YOLOV5S_F32 = 128 << 20
