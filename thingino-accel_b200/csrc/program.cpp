/*
 * program.cpp -- compiles a .mars layer table into a list of device ops.
 *
 * This is the host-side replacement of the reference's execute_layer() switch
 * (src/mars/mars_runtime.c:1161-1224): what the reference decides per layer at run
 * time (tensor lookup, dimension extraction, SAME-only padding, kernel choice) is
 * decided once here, together with the two analyses the reference does not need
 * because it runs on one thread:
 *   - hazard analysis: which layers alias their own inputs through the planner's
 *     round-robin work buffers and must keep the reference's loop order to stay
 *     byte-exact (SURVEY §7.2, Appendix C);
 *   - observability analysis + fusion (opt_level >= 1): which writes are dead and
 *     which following int8 unary layers fold into a producer's epilogue.
 */
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <cmath>

#include "conv_tc.h"
#include "conv_tf32.h"
#include "mars_internal.h"

namespace marsb200 {

/* ---- arithmetic contracts evaluated on the host (tables) ------------------ */
/* (int32_t)float as x86-64 cvttss2si does it: NaN / out of range -> INT_MIN (SURVEY A.1) */
static inline int32_t f2i_x86(float v) {
    if (!(v > -2147483904.0f && v < 2147483648.0f)) return INT32_MIN;
    return (int32_t)v;
}
static inline int8_t clamp_i8(int32_t r) { return (int8_t)(r > 127 ? 127 : (r < -128 ? -128 : r)); }

static int pool_add(Program *p, const int8_t lut[256]) {
    /* de-duplicate identical tables */
    for (size_t o = 0; o + 256 <= p->const_pool.size(); o += 256)
        if (memcmp(&p->const_pool[o], lut, 256) == 0) return (int)o;
    size_t o = p->const_pool.size();
    p->const_pool.resize(o + 256);
    memcpy(&p->const_pool[o], lut, 256);
    return (int)o;
}

/* expf is the host libm's, the same one the reference would call (this file is compiled without FP contraction) */
void build_sigmoid_table(float scale, float sig[256]) {
    for (int v = -128; v < 128; v++) {
        volatile float x = (float)v * scale;
        volatile float e = expf(-x);
        volatile float den = 1.0f + e;
        volatile float r = 1.0f / den;
        sig[v + 128] = r;
    }
}

void build_gfl_exp_table(float scale, float e[256]) {
    for (int d = 0; d < 256; d++) {
        volatile float x = (float)d * scale;
        volatile float r = expf(-x);
        e[d] = r;
    }
}

/* reference src/mars/mars_runtime.c:752-768 tabulated over the 256 possible inputs */
static void build_sigmoid_lut(float in_scale, float out_scale_raw, int8_t lut[256]) {
    float os = out_scale_raw > 0 ? out_scale_raw : 1.0f;
    float sig[256];
    build_sigmoid_table(in_scale, sig);
    for (int v = -128; v < 128; v++) {
        volatile float t = sig[v + 128] / os;
        volatile float u = t + 0.5f;
        lut[v + 128] = clamp_i8(f2i_x86(u));
    }
}

/* reference src/mars/mars_runtime.c:1072-1085 */
static void build_relu_lut(int leaky, int8_t lut[256]) {
    for (int v = -128; v < 128; v++) {
        if (v > 0) lut[v + 128] = (int8_t)v;
        else if (leaky) {
            volatile float t = (float)v * 0.01f;
            int32_t q = f2i_x86(t);
            lut[v + 128] = (int8_t)(q < -128 ? -128 : q);
        } else lut[v + 128] = 0;
    }
}

static bool overlap(int64_t a0, int64_t a1, int64_t b0, int64_t b1) { return a0 < a1 && b0 < b1 && a0 < b1 && b0 < a1; }

static uint64_t numel_of(const mars_tensor_t &t) {
    uint64_t n = 1;
    for (uint32_t i = 0; i < t.ndims && i < MARS_MAX_DIMS; i++) n *= (uint64_t)(t.shape[i] < 0 ? 0 : t.shape[i]);
    return n;
}

struct Ctx {
    const mars_header_t &h;
    const mars_runtime_tensor_t *tensors;
    const std::vector<size_t> &toff;
    int64_t W, A;
    Program *prog;
    int find(uint32_t id) const { return find_tensor(h, tensors, id); }
    int64_t off(int idx) const { return (int64_t)toff[idx]; }
    const mars_tensor_t &desc(int idx) const { return tensors[idx].desc; }
};

static Op fail_op(int layer, mars_error_t err, const char *why) {
    Op o;
    o.kind = OP_NOP;
    o.layer = layer;
    o.mode = -(int)err + 1000; /* >= 1000: run stops here and returns -(mode-1000) */
    o.note = why;
    return o;
}

/* true when [lo,hi) crosses the weights/slot boundary */
static bool straddles(const Ctx &c, int64_t lo, int64_t hi) { return lo < hi && lo < c.W && hi > c.W; }

static mars_error_t check_write(const Ctx &c, int layer, int64_t lo, int64_t hi) {
    if (lo >= hi) return MARS_OK;
    if (lo < c.W) {
        set_last_error("layer %d writes into the weight blob (arena offset %lld < %lld): unsupported, weights are shared by all images",
                       layer, (long long)lo, (long long)c.W);
        return MARS_ERR_INVALID_LAYER;
    }
    if (hi > c.A) {
        set_last_error("layer %d writes past the arena end (%lld > %lld); the reference would corrupt its heap here",
                       layer, (long long)hi, (long long)c.A);
        return MARS_ERR_INVALID_LAYER;
    }
    c.prog->max_extent = std::max(c.prog->max_extent, (size_t)hi); /* the image slot is sized to the furthest access */
    return MARS_OK;
}
static mars_error_t check_read(const Ctx &c, int layer, int64_t lo, int64_t hi) {
    if (lo >= hi) return MARS_OK;
    if (lo < 0 || hi > c.A) {
        set_last_error("layer %d reads outside the arena [%lld,%lld) (arena %lld bytes)", layer, (long long)lo,
                       (long long)hi, (long long)c.A);
        return MARS_ERR_INVALID_LAYER;
    }
    c.prog->max_extent = std::max(c.prog->max_extent, (size_t)hi);
    return MARS_OK;
}

/* Conv in place (output range overlaps input range), NCHW: decide whether one launch per
 * output channel reproduces the reference's oc-outermost loop (src/mars/mxu_conv.c:642-669)
 * exactly.  cross: some pixel's write is read by a different pixel of the same pass;
 * later_reads_earlier: ... by a LATER pixel (then even a staged pass differs). */
static void conv_pass_analysis(const Op &o, int es, bool *cross, bool *later_reads_earlier, bool *misaligned) {
    *cross = *later_reads_earlier = *misaligned = false;
    const int64_t Po = (int64_t)o.oh * o.ow, Pi = (int64_t)o.ih * o.iw;
    for (int oc = 0; oc < o.oc; oc++) {
        int64_t wlo = o.out + (int64_t)oc * Po * es, whi = wlo + Po * es;
        for (int ic = 0; ic < o.ic; ic++) {
            int64_t rlo = o.in0 + (int64_t)ic * Pi * es, rhi = rlo + Pi * es;
            if (!overlap(wlo, whi, rlo, rhi)) continue;
            for (int oh = 0; oh < o.oh; oh++)
                for (int ow = 0; ow < o.ow; ow++) {
                    int64_t pp = (int64_t)oh * o.ow + ow;
                    for (int y = 0; y < o.kh; y++) {
                        int ih = oh * o.sh - o.pt + y;
                        if (ih < 0 || ih >= o.ih) continue;
                        for (int x = 0; x < o.kw; x++) {
                            int iw = ow * o.sw - o.pl + x;
                            if (iw < 0 || iw >= o.iw) continue;
                            int64_t r = rlo + ((int64_t)ih * o.iw + iw) * es;
                            if (r + es <= wlo || r >= whi) continue;
                            if ((r - wlo) % es) { *misaligned = true; return; }
                            int64_t p = (r - wlo) / es;
                            if (p != pp) *cross = true;
                            if (p < pp) *later_reads_earlier = true;
                        }
                    }
                }
        }
    }
}

/* NHWC conv in place: loop order oh, ow, oc (src/mars/mxu_conv.c:726-756).  Thread-per-pixel
 * with the oc loop kept sequential inside the thread is exact iff no pixel reads a byte that a
 * different pixel writes. */
static bool nhwc_pixel_private(const Op &o) {
    for (int oh = 0; oh < o.oh; oh++)
        for (int ow = 0; ow < o.ow; ow++) {
            int64_t wlo = o.out + ((int64_t)oh * o.ow + ow) * o.oc, whi = wlo + o.oc;
            (void)whi;
            for (int y = 0; y < o.kh; y++) {
                int ih = oh * o.sh - o.pt + y;
                if (ih < 0 || ih >= o.ih) continue;
                for (int x = 0; x < o.kw; x++) {
                    int iw = ow * o.sw - o.pl + x;
                    if (iw < 0 || iw >= o.iw) continue;
                    int64_t rlo = o.in0 + ((int64_t)ih * o.iw + iw) * o.ic, rhi = rlo + o.ic;
                    /* which output pixels' byte ranges does [rlo,rhi) touch? */
                    int64_t olo = o.out, ohi = o.out + (int64_t)o.oh * o.ow * o.oc;
                    if (!overlap(rlo, rhi, olo, ohi)) continue;
                    int64_t first = (std::max(rlo, olo) - o.out) / o.oc, last = (std::min(rhi, ohi) - 1 - o.out) / o.oc;
                    int64_t me = (int64_t)oh * o.ow + ow;
                    if (first != me || last != me) return false;
                }
            }
        }
    return true;
}

static mars_error_t compile_conv(Ctx &c, int li, const mars_layer_t &L, int depthwise) {
    const mars_conv_params_t &p = L.params.conv;
    int ii = c.find(L.input_tensor_ids[0]), oi = c.find(L.output_tensor_ids[0]);
    int wi = c.find(p.weight_tensor_id), bi = c.find(p.bias_tensor_id);
    if (ii < 0 || oi < 0 || wi < 0) { /* reference src/mars/mars_runtime.c:524,535,546 */
        c.prog->ops.push_back(fail_op(li, MARS_ERR_INVALID_TENSOR, "conv: tensor id not found"));
        return MARS_OK;
    }
    const mars_tensor_t &it = c.desc(ii), &ot = c.desc(oi), &wt = c.desc(wi);
    Op o;
    o.layer = li;
    bool in_nhwc = it.format == MARS_FORMAT_NHWC, out_nhwc = ot.format == MARS_FORMAT_NHWC;
    if (in_nhwc) { o.ih = it.shape[1]; o.iw = it.shape[2]; o.ic = it.shape[3]; }
    else { o.ic = it.shape[1]; o.ih = it.shape[2]; o.iw = it.shape[3]; }
    if (out_nhwc) { o.oh = ot.shape[1]; o.ow = ot.shape[2]; o.oc = ot.shape[3]; }
    else { o.oc = ot.shape[1]; o.oh = ot.shape[2]; o.ow = ot.shape[3]; }
    o.kh = (int)p.kernel_h; o.kw = (int)p.kernel_w; o.sh = (int)p.stride_h; o.sw = (int)p.stride_w;
    if (p.padding == MARS_PAD_SAME) { /* :591-598; EXPLICIT pads are ignored by the reference */
        o.pt = ((o.oh - 1) * o.sh + o.kh - o.ih) / 2;
        o.pl = ((o.ow - 1) * o.sw + o.kw - o.iw) / 2;
    }
    if (depthwise && p.padding == MARS_PAD_EXPLICIT) { o.pt = (int)p.pad_top; o.pl = (int)p.pad_left; }
    bool is_float = it.dtype == MARS_DTYPE_FLOAT32;
    int es = is_float ? 4 : 1;
    o.in0 = c.off(ii); o.out = c.off(oi); o.w = c.off(wi); o.bias = bi >= 0 ? c.off(bi) : -1;
    if (o.kh < 0 || o.kw < 0 || o.sh < 0 || o.sw < 0) {
        set_last_error("layer %d: conv kernel/stride out of range", li);
        return MARS_ERR_INVALID_LAYER;
    }
    bool empty = o.oc <= 0 || o.oh <= 0 || o.ow <= 0;
    int64_t nout = empty ? 0 : (int64_t)o.oc * o.oh * o.ow;
    int64_t nin = (o.ic > 0 && o.ih > 0 && o.iw > 0) ? (int64_t)o.ic * o.ih * o.iw : 0;
    int64_t icp = o.ic > 0 ? o.ic : 0;
    int64_t wbytes = depthwise ? (int64_t)(o.oc > 0 ? o.oc : 0) * o.kh * o.kw * es
                               : (int64_t)(o.oc > 0 ? o.oc : 0) * icp * o.kh * o.kw * es;
    if (!empty) {
        if (depthwise) {
            if (is_float) { c.prog->ops.push_back(fail_op(li, MARS_ERR_INVALID_LAYER, "restated depthwise: int8 only")); return MARS_OK; }
            o.kind = OP_DW_I8;
            o.coff = in_nhwc ? 1 : 0; /* layout flag for the depthwise kernels */
        } else o.kind = is_float ? OP_CONV_F32_NCHW : (in_nhwc ? OP_CONV_I8_NHWC : OP_CONV_I8_NCHW);
        if (!is_float) {
            volatile float prod = it.scale * wt.scale; /* reference src/mars/mxu_conv.c:639 */
            o.f0 = prod / ot.scale;
        }
        o.wlo = o.out; o.whi = o.out + nout * es;
        mars_error_t e;
        if ((e = check_write(c, li, o.wlo, o.whi))) return e;
        /* the kernels only touch taps inside the input plane, so the read extent is the tensor */
        if (nin && (o.kh > 0 && o.kw > 0) && (e = check_read(c, li, o.in0, o.in0 + nin * es))) return e;
        if (nin && (e = check_read(c, li, o.w, o.w + wbytes))) return e;
        if (o.bias >= 0 && (e = check_read(c, li, o.bias, o.bias + 4 * (int64_t)o.oc))) return e;
        o.xlat = straddles(c, o.in0, o.in0 + nin * es) || straddles(c, o.w, o.w + wbytes) ||
                 (o.bias >= 0 && straddles(c, o.bias, o.bias + 4 * (int64_t)o.oc));
        bool haz_in = nin && overlap(o.wlo, o.whi, o.in0, o.in0 + nin * es);
        bool haz_w = overlap(o.wlo, o.whi, o.w, o.w + wbytes) ||
                     (o.bias >= 0 && overlap(o.wlo, o.whi, o.bias, o.bias + 4 * (int64_t)o.oc));
        if (haz_w || (haz_in && depthwise)) {
            o.mode = EXEC_SERIAL;
            o.note = "output aliases weights/bias: literal order";
        } else if (haz_in) {
            if (o.kind == OP_CONV_I8_NHWC) {
                o.mode = nhwc_pixel_private(o) ? EXEC_PIXEL_SERIAL : EXEC_SERIAL;
                o.note = "in-place NHWC conv";
            } else {
                /* 1x1 in place on its own planes, channel vector + weights fit shared memory: per-pixel serial */
                const bool pix_serial = !is_float && !depthwise && o.kh == 1 && o.kw == 1 && o.sh == 1 && o.sw == 1 && o.pt == 0 &&
                                        o.pl == 0 && o.out == o.in0 && o.oh == o.ih && o.ow == o.iw && o.ic % 4 == 0 && !o.xlat &&
                                        o.w < c.W && (o.bias < 0 || o.bias + 4 * (int64_t)o.oc <= c.W) &&
                                        (size_t)o.ic * 128 + (size_t)o.oc * o.ic <= 160 * 1024;
                if (pix_serial) {
                    o.mode = EXEC_PIXEL_SERIAL;
                    o.note = "in-place NCHW 1x1 conv: per-pixel serial over output channels";
                    c.prog->ops.push_back(o);
                    goto conv_done;
                }
                bool cross, lre, mis;
                conv_pass_analysis(o, es, &cross, &lre, &mis);
                if (mis || lre) o.mode = EXEC_SERIAL;
                else if (cross) {
                    o.mode = EXEC_OC_PASSES_SCRATCH;
                    c.prog->scratch_bytes = std::max(c.prog->scratch_bytes, (size_t)((int64_t)o.oh * o.ow * es));
                } else o.mode = EXEC_OC_PASSES;
                o.note = "in-place NCHW conv: sequential over output channels";
            }
        }
        c.prog->ops.push_back(o);
    }
conv_done:
    if (p.activation == MARS_ACT_RELU) { /* :700-707: signed-byte clamp of the first oh*ow*oc BYTES */
        int64_t total = (int64_t)o.oh * o.ow * o.oc;
        if (total > 0 && o.oh > 0 && o.ow > 0) {
            Op r;
            r.kind = OP_BYTE_RELU; r.layer = li; r.out = o.out; r.in0 = o.out; r.n = (uint64_t)total;
            r.wlo = r.out; r.whi = r.out + total;
            mars_error_t e;
            if ((e = check_write(c, li, r.wlo, r.whi))) return e;
            c.prog->ops.push_back(r);
        }
    }
    return MARS_OK;
}

/* flat unary / binary layers */
static mars_error_t compile_eltwise(Ctx &c, int li, const mars_layer_t &L) {
    int type = (int)L.type;
    bool binary = type == MARS_LAYER_ADD || type == MARS_LAYER_MUL;
    int ai = c.find(L.input_tensor_ids[0]), bi = binary ? c.find(L.input_tensor_ids[1]) : -1;
    int oi = c.find(L.output_tensor_ids[0]);
    if (ai < 0 || oi < 0 || (binary && bi < 0)) {
        c.prog->ops.push_back(fail_op(li, MARS_ERR_INVALID_TENSOR, "eltwise: tensor id not found"));
        return MARS_OK;
    }
    const mars_tensor_t &at = c.desc(ai), &ot = c.desc(oi);
    Op o;
    o.layer = li;
    o.n = numel_of(at); /* numel always from input A (reference :788-791 etc.) */
    if (o.n == 0) return MARS_OK;
    bool is_float = at.dtype == MARS_DTYPE_FLOAT32;
    int es = is_float ? 4 : 1;
    o.in0 = c.off(ai); o.in1 = binary ? c.off(bi) : -1; o.out = c.off(oi);
    switch (type) {
        case MARS_LAYER_SIGMOID:
            if (is_float) o.kind = OP_SIGMOID_F32;
            else {
                int8_t lut[256];
                build_sigmoid_lut(at.scale, ot.scale, lut);
                o.kind = OP_SIGMOID_I8; o.lut = pool_add(c.prog, lut);
            }
            break;
        case MARS_LAYER_RELU: case MARS_LAYER_RELU6: case MARS_LAYER_LEAKY_RELU:
            if (is_float) { o.kind = OP_RELU_F32; o.f0 = type == MARS_LAYER_LEAKY_RELU ? 0.01f : 0.0f; }
            else {
                int8_t lut[256];
                build_relu_lut(type == MARS_LAYER_LEAKY_RELU, lut);
                o.kind = OP_RELU_I8; o.lut = pool_add(c.prog, lut);
            }
            break;
        case MARS_LAYER_ADD: case MARS_LAYER_MUL: {
            const mars_tensor_t &bt = c.desc(bi);
            if (is_float) o.kind = type == MARS_LAYER_ADD ? OP_ADD_F32 : OP_MUL_F32;
            else {
                o.kind = type == MARS_LAYER_ADD ? OP_ADD_I8 : OP_MUL_I8;
                float so = ot.scale > 0 ? ot.scale : 1.0f;
                o.f0 = at.scale; o.f1 = bt.scale;
                volatile float inv = 1.0f / so; /* reference :825, :892 */
                o.f2 = inv;
            }
            break;
        }
    }
    int64_t bytes = (int64_t)o.n * es;
    o.wlo = o.out; o.whi = o.out + bytes;
    mars_error_t e;
    if ((e = check_write(c, li, o.wlo, o.whi))) return e;
    if ((e = check_read(c, li, o.in0, o.in0 + bytes))) return e;
    if (binary && (e = check_read(c, li, o.in1, o.in1 + bytes))) return e;
    o.xlat = straddles(c, o.in0, o.in0 + bytes) || (binary && straddles(c, o.in1, o.in1 + bytes));
    /* same base = each element reads then writes its own position: order-free.  A shifted
     * overlap makes the reference's ascending loop observable -> literal order. */
    if ((o.in0 != o.out && overlap(o.wlo, o.whi, o.in0, o.in0 + bytes)) ||
        (binary && o.in1 != o.out && overlap(o.wlo, o.whi, o.in1, o.in1 + bytes))) {
        o.mode = EXEC_SERIAL;
        o.note = "shifted in/out overlap: literal order";
    }
    c.prog->ops.push_back(o);
    return MARS_OK;
}

static mars_error_t compile_batchnorm(Ctx &c, int li, const mars_layer_t &L) {
    int ii = c.find(L.input_tensor_ids[0]), si = c.find(L.input_tensor_ids[1]);
    int bi = c.find(L.input_tensor_ids[2]), oi = c.find(L.output_tensor_ids[0]);
    if (ii < 0 || oi < 0) {
        c.prog->ops.push_back(fail_op(li, MARS_ERR_INVALID_TENSOR, "batchnorm: tensor id not found"));
        return MARS_OK;
    }
    const mars_tensor_t &it = c.desc(ii), &ot = c.desc(oi);
    Op o;
    o.layer = li;
    int n = it.shape[0] > 0 ? it.shape[0] : 1, ch = it.shape[1] > 0 ? it.shape[1] : 1;
    int h = it.shape[2] > 0 ? it.shape[2] : 1, w = it.shape[3] > 0 ? it.shape[3] : 1;
    bool is_float = it.dtype == MARS_DTYPE_FLOAT32;
    int es = is_float ? 4 : 1;
    o.kind = is_float ? OP_BN_F32 : OP_BN_I8;
    o.ic = ch; o.ih = h; o.iw = w; o.oc = n;
    o.n = (uint64_t)n * ch * h * w;
    o.in0 = c.off(ii); o.out = c.off(oi); o.in1 = si >= 0 ? c.off(si) : -1; o.in2 = bi >= 0 ? c.off(bi) : -1;
    o.f0 = it.scale > 0 ? it.scale : 1.0f; /* :1135 */
    o.f1 = ot.scale > 0 ? ot.scale : 1.0f; /* :1136 */
    int64_t bytes = (int64_t)o.n * es;
    o.wlo = o.out; o.whi = o.out + bytes;
    mars_error_t e;
    if ((e = check_write(c, li, o.wlo, o.whi))) return e;
    if ((e = check_read(c, li, o.in0, o.in0 + bytes))) return e;
    if (o.in1 >= 0 && (e = check_read(c, li, o.in1, o.in1 + 4 * (int64_t)ch))) return e;
    if (o.in2 >= 0 && (e = check_read(c, li, o.in2, o.in2 + 4 * (int64_t)ch))) return e;
    o.xlat = straddles(c, o.in0, o.in0 + bytes) || (o.in1 >= 0 && straddles(c, o.in1, o.in1 + 4 * (int64_t)ch)) ||
             (o.in2 >= 0 && straddles(c, o.in2, o.in2 + 4 * (int64_t)ch));
    if ((o.in0 != o.out && overlap(o.wlo, o.whi, o.in0, o.in0 + bytes)) ||
        (o.in1 >= 0 && overlap(o.wlo, o.whi, o.in1, o.in1 + 4 * (int64_t)ch)) ||
        (o.in2 >= 0 && overlap(o.wlo, o.whi, o.in2, o.in2 + 4 * (int64_t)ch))) {
        o.mode = EXEC_SERIAL;
        o.note = "batchnorm output aliases an operand: literal order";
    }
    c.prog->ops.push_back(o);
    return MARS_OK;
}

/* maxpool / upsample: NHWC indexing of shape[1..3] whatever the tag (SURVEY C.4) */
static mars_error_t compile_spatial(Ctx &c, int li, const mars_layer_t &L) {
    int ii = c.find(L.input_tensor_ids[0]), oi = c.find(L.output_tensor_ids[0]);
    if (ii < 0 || oi < 0) {
        c.prog->ops.push_back(fail_op(li, MARS_ERR_INVALID_TENSOR, "pool/upsample: tensor id not found"));
        return MARS_OK;
    }
    const mars_tensor_t &it = c.desc(ii), &ot = c.desc(oi);
    Op o;
    o.layer = li;
    o.ih = it.shape[1]; o.iw = it.shape[2]; o.ic = it.shape[3]; o.oh = ot.shape[1]; o.ow = ot.shape[2];
    o.oc = o.ic;
    o.in0 = c.off(ii); o.out = c.off(oi);
    if (o.oh <= 0 || o.ow <= 0 || o.ic <= 0) return MARS_OK;
    if ((int)L.type == MARS_LAYER_MAXPOOL) {
        const mars_pool_params_t &p = L.params.pool;
        o.kind = OP_MAXPOOL;
        o.kh = (int)p.kernel_h; o.kw = (int)p.kernel_w; o.sh = (int)p.stride_h; o.sw = (int)p.stride_w;
        if (o.kh < 0 || o.kw < 0 || o.sh < 0 || o.sw < 0) { set_last_error("layer %d: pool params out of range", li); return MARS_ERR_INVALID_LAYER; }
    } else {
        const mars_upsample_params_t &p = L.params.upsample;
        o.kind = OP_UPSAMPLE;
        if ((p.scale_h == 0 && o.ih == 0) || (p.scale_w == 0 && o.iw == 0)) {
            c.prog->ops.push_back(fail_op(li, MARS_ERR_INVALID_LAYER, "upsample: the reference divides by zero here"));
            return MARS_OK;
        }
        o.sh = p.scale_h > 0 ? (int)p.scale_h : o.oh / o.ih; /* :1020-1021 */
        o.sw = p.scale_w > 0 ? (int)p.scale_w : o.ow / o.iw;
        if (o.sh == 0 || o.sw == 0) {
            c.prog->ops.push_back(fail_op(li, MARS_ERR_INVALID_LAYER, "upsample: zero scale (division by zero in the reference)"));
            return MARS_OK;
        }
    }
    int64_t nin = (o.ih > 0 && o.iw > 0) ? (int64_t)o.ih * o.iw * o.ic : 0, nout = (int64_t)o.oh * o.ow * o.ic;
    o.wlo = o.out; o.whi = o.out + nout;
    mars_error_t e;
    if ((e = check_write(c, li, o.wlo, o.whi))) return e;
    if ((e = check_read(c, li, o.in0, o.in0 + nin))) return e;
    if (o.kind == OP_UPSAMPLE && nin == 0) { /* ih clamps to in_h-1 < 0: the reference reads before the tensor */
        c.prog->ops.push_back(fail_op(li, MARS_ERR_INVALID_LAYER, "upsample of an empty input"));
        return MARS_OK;
    }
    o.xlat = straddles(c, o.in0, o.in0 + nin);
    if (overlap(o.wlo, o.whi, o.in0, o.in0 + nin)) {
        o.mode = EXEC_SERIAL;
        o.note = "in-place pool/upsample: literal order";
    }
    c.prog->ops.push_back(o);
    return MARS_OK;
}

static mars_error_t compile_concat(Ctx &c, int li, const mars_layer_t &L) {
    int oi = c.find(L.output_tensor_ids[0]);
    if (oi < 0) {
        c.prog->ops.push_back(fail_op(li, MARS_ERR_INVALID_TENSOR, "concat: output id not found"));
        return MARS_OK;
    }
    const mars_tensor_t &ot = c.desc(oi);
    int OH = ot.shape[1], OW = ot.shape[2], OC = ot.shape[3];
    int coff = 0;
    uint32_t nin = L.num_inputs > 4 ? 4 : L.num_inputs;
    const size_t first_op = c.prog->ops.size();
    for (uint32_t n = 0; n < nin; n++) {
        int ii = c.find(L.input_tensor_ids[n]);
        if (ii < 0) continue; /* :980: skipped inputs do not advance the channel offset */
        int IC = c.desc(ii).shape[3];
        if (OH > 0 && OW > 0 && IC > 0) {
            Op o;
            o.layer = li; o.kind = OP_CONCAT;
            o.oh = OH; o.ow = OW; o.oc = OC; o.ic = IC; o.coff = coff;
            o.in0 = c.off(ii); o.out = c.off(oi);
            int64_t npix = (int64_t)OH * OW, len = npix * IC;
            int64_t wlo = o.out + coff, whi = o.out + (npix - 1) * OC + coff + IC;
            if (OC < 0) { set_last_error("layer %d: concat with negative channel count", li); return MARS_ERR_INVALID_LAYER; }
            o.wlo = wlo; o.whi = whi; o.n = (uint64_t)len;
            mars_error_t e;
            if ((e = check_write(c, li, wlo, whi))) return e;
            if ((e = check_read(c, li, o.in0, o.in0 + len))) return e;
            o.xlat = straddles(c, o.in0, o.in0 + len);
            if (overlap(wlo, whi, o.in0, o.in0 + len)) {
                if (o.in0 == o.out && IC == OC) {
                    /* out_idx - in_idx == coff for every element (SURVEY C.4b) */
                    if (coff == 0) o.kind = OP_NOP; /* self copy */
                    else { o.kind = OP_CONCAT_PERIODIC; o.note = "in-place concat: periodic replication"; }
                } else {
                    o.mode = EXEC_SERIAL;
                    o.note = "overlapping concat with varying shift: literal order";
                }
            }
            if (o.kind != OP_NOP) c.prog->ops.push_back(o);
        }
        coff += IC;
    }
    /* With NCHW-shaped descriptors every input is a flat copy shifted by its channel offset (SURVEY C.4), and each
     * later input overwrites all but the first bytes of the earlier ones.  Those overwritten bytes are dead inside the
     * layer (no later input of a hazard-free copy reads the output), so the earlier copies shrink to the slivers that
     * survive; the arena after the layer is unchanged. */
    int64_t later_lo = -1, later_hi = -1;
    for (size_t k = c.prog->ops.size(); k-- > first_op;) {
        Op &o = c.prog->ops[k];
        if ((o.kind != OP_CONCAT && o.kind != OP_CONCAT_PERIODIC) || o.mode != EXEC_PARALLEL || o.ic != o.oc || o.xlat) break;
        const int64_t lo = o.wlo, hi = o.wlo + (int64_t)o.n;
        /* an in-place (periodic) input reads only out[0, coff) -- bytes in front of its own writes, which the trimmed copies
         * below keep -- and overwrites [out + coff, out + coff + n) like any other input; it is not trimmed itself */
        if (o.kind == OP_CONCAT && later_lo >= 0 && later_lo > lo && later_lo < hi && later_hi >= hi) {
            o.n = (uint64_t)(later_lo - lo);
            o.whi = later_lo;
            o.note = "concat input trimmed to the bytes later inputs do not overwrite";
        }
        later_lo = later_lo < 0 ? lo : std::min(later_lo, lo);
        later_hi = std::max(later_hi, hi);
    }
    return MARS_OK;
}


/* ---- detection heads (mars_b200_set_yolo_heads, mars_b200_set_gfl_heads) -------------------------------------------------
 * The compiler drops the Split / Pow / Constant nodes of the Detect block, so everything after the three head convolutions runs
 * over zero elements and output0 holds stale bytes (SURVEY Appendix B.2).  The detections are in the raw head convolutions
 * [1, 3 (5 + nc), gh, gw] (or [1, gh, gw, 3 (5 + nc)] with --nhwc).  A NanoDet graph keeps its GFL heads the same way:
 * [1, nc + 4 (reg_max + 1), gh, gw] per level, of which at most one is a model output.  The planner's round-robin buffers let later
 * layers overwrite a head, so each head is decoded by an op placed right after the op that completes it. */
static const int YOLO_STRIDES[3] = {8, 16, 32};
static const int GFL_STRIDES[4] = {8, 16, 32, 64};

/* geometry of a head candidate: int8 [1,C,gh,gw] / [1,gh,gw,C] whose channel count C passes `channels_ok(C, hd, why)` (which sets
 * hd->nc) and whose grid divides the network input by one of strides[0..ns).  Returns false when the tensor does not have that
 * shape; *why (optional) says what is wrong */
template <class ChannelRule>
static bool head_geometry(const mars_header_t &h, const mars_runtime_tensor_t *tensors, int ti, HeadTensor *hd, const char **why,
                          const int *strides, int ns, const char *grid_why, ChannelRule channels_ok) {
    static const char *dummy;
    const char *&w = why ? *why : dummy;
    const mars_tensor_t &d = tensors[ti].desc;
    if (d.dtype != MARS_DTYPE_INT8 || d.ndims != 4 || d.shape[0] != 1) { w = "is not an int8 [1,C,gh,gw] / [1,gh,gw,C] tensor"; return false; }
    hd->nhwc = d.format == MARS_FORMAT_NHWC;
    hd->channels = hd->nhwc ? d.shape[3] : d.shape[1];
    hd->gh = hd->nhwc ? d.shape[1] : d.shape[2];
    hd->gw = hd->nhwc ? d.shape[2] : d.shape[3];
    if (!channels_ok(hd->channels, hd, &w)) return false;
    hd->scale = d.scale;
    const uint32_t ii = h.num_inputs ? h.input_tensor_ids[0] : 0xFFFFFFFFu;
    if (ii >= h.num_tensors) { w = "belongs to a model without an input tensor"; return false; }
    const mars_tensor_t &in = tensors[ii].desc;
    const bool in_nhwc = in.format == MARS_FORMAT_NHWC;
    const int H = in_nhwc ? in.shape[1] : in.shape[2], W = in_nhwc ? in.shape[2] : in.shape[3];
    hd->stride = 0;
    if (hd->gh > 0 && hd->gw > 0 && H % hd->gh == 0 && W % hd->gw == 0 && H / hd->gh == W / hd->gw)
        for (int k = 0; k < ns; k++) if (H / hd->gh == strides[k]) hd->stride = strides[k];
    if (!hd->stride) { w = grid_why; return false; }
    return true;
}

static bool yolo_geometry(const mars_header_t &h, const mars_runtime_tensor_t *tensors, int ti, HeadTensor *hd, const char **why) {
    return head_geometry(h, tensors, ti, hd, why, YOLO_STRIDES, 3, "has a grid that is not the input size divided by 8, 16 or 32",
                         [](int C, HeadTensor *t, const char **w) {
                             if (C < 18 || C % 3) { *w = "does not have 3 * (5 + nc) channels (nc >= 1)"; return false; }
                             t->nc = C / 3 - 5;
                             return true;
                         });
}

static bool gfl_geometry(const mars_header_t &h, const mars_runtime_tensor_t *tensors, int ti, HeadTensor *hd, const char **why, int nc,
                         int reg_max) {
    return head_geometry(h, tensors, ti, hd, why, GFL_STRIDES, 4, "has a grid that is not the input size divided by 8, 16, 32 or 64",
                         [nc, reg_max](int C, HeadTensor *t, const char **w) {
                             if (C != nc + 4 * (reg_max + 1)) { *w = "does not have nc + 4 * (reg_max + 1) channels"; return false; }
                             t->nc = nc;
                             return true;
                         });
}

/* the last CONV2D layer that writes tensor `id`, or -1 */
static int producing_conv(const mars_header_t &h, const mars_runtime_layer_t *layers, uint32_t id) {
    for (uint32_t i = h.num_layers; i-- > 0;)
        if ((int)layers[i].desc.type == MARS_LAYER_CONV2D && layers[i].desc.num_outputs >= 1 && layers[i].desc.output_tensor_ids[0] == id) return (int)i;
    return -1;
}

/* true when a layer that computes something (not one of the reference's no-op layer types) reads tensor `id` */
static bool read_by_compute(const mars_header_t &h, const mars_runtime_layer_t *layers, uint32_t id) {
    for (uint32_t i = 0; i < h.num_layers; i++) {
        const mars_layer_t &L = layers[i].desc;
        const int t = (int)L.type;
        if (t == MARS_LAYER_RESHAPE || t == MARS_LAYER_TRANSPOSE || t == MARS_LAYER_SOFTMAX || t == MARS_LAYER_SILU || t == MARS_LAYER_AVGPOOL) continue;
        for (uint32_t k = 0; k < L.num_inputs && k < 4; k++)
            if (L.input_tensor_ids[k] == id) return true;
    }
    return false;
}

/* true for a 1x1 CONV2D without activation whose output no compute layer reads: what a detection head conv looks like */
static bool head_conv(const mars_header_t &h, const mars_runtime_layer_t *layers, const mars_layer_t &L) {
    if ((int)L.type != MARS_LAYER_CONV2D || L.num_outputs < 1) return false;
    const mars_conv_params_t &p = L.params.conv;
    return p.kernel_h == 1 && p.kernel_w == 1 && p.activation == MARS_ACT_NONE && !read_by_compute(h, layers, L.output_tensor_ids[0]);
}

int find_yolo_heads(const mars_header_t &h, const mars_runtime_tensor_t *tensors, const mars_runtime_layer_t *layers, uint32_t *ids, int cap) {
    /* A Detect head is a 1x1 conv without activation whose output only the dropped decode layers read.  The last such conv fixes
     * nc; each stride then takes its last conv of that channel count. */
    int nc = -1, found[3] = {-1, -1, -1};
    for (uint32_t i = h.num_layers; i-- > 0;) {
        const mars_layer_t &L = layers[i].desc;
        if (!head_conv(h, layers, L)) continue;
        const int ti = find_tensor(h, tensors, L.output_tensor_ids[0]);
        HeadTensor hd;
        if (ti < 0 || !yolo_geometry(h, tensors, ti, &hd, nullptr)) continue;
        if (nc < 0) nc = hd.nc;
        if (hd.nc != nc) continue;
        for (int k = 0; k < 3; k++)
            if (hd.stride == YOLO_LEVELS[k].stride && found[k] < 0) found[k] = (int)i;
    }
    if (found[0] < 0 || found[1] < 0 || found[2] < 0) return 0;
    for (int k = 0; k < 3 && k < cap; k++) if (ids) ids[k] = layers[found[k]].desc.output_tensor_ids[0];
    return 3;
}

int find_gfl_heads(const mars_header_t &h, const mars_runtime_tensor_t *tensors, const mars_runtime_layer_t *layers, int nc, int reg_max,
                   uint32_t *ids, int cap) {
    if (nc < 1 || reg_max < 1 || reg_max > 16) return 0;
    int found[4] = {-1, -1, -1, -1};
    for (uint32_t i = h.num_layers; i-- > 0;) {
        const mars_layer_t &L = layers[i].desc;
        if (!head_conv(h, layers, L)) continue;
        const int ti = find_tensor(h, tensors, L.output_tensor_ids[0]);
        HeadTensor hd;
        if (ti < 0 || !gfl_geometry(h, tensors, ti, &hd, nullptr, nc, reg_max)) continue;
        for (int k = 0; k < 4; k++)
            if (hd.stride == GFL_STRIDES[k] && found[k] < 0) found[k] = (int)i;
    }
    if (found[0] < 0 || found[1] < 0 || found[2] < 0) return 0;
    const int n = found[3] < 0 ? 3 : 4;
    for (int k = 0; k < n && k < cap; k++) if (ids) ids[k] = layers[found[k]].desc.output_tensor_ids[0];
    return n;
}

/* the checks both setters make on n resolved heads: conv output, geometry (`geometry(ti, hd, why)`), scale, arena placement, level
 * order and each level's stride (strides[k]) */
template <class Geometry>
static mars_error_t resolve_heads(const char *what, const mars_header_t &h, const mars_runtime_tensor_t *tensors,
                                  const mars_runtime_layer_t *layers, const std::vector<size_t> &toff, size_t weights_size,
                                  const uint32_t *ids, int n, const int *strides, Geometry geometry, std::vector<HeadTensor> *out) {
    for (int k = 0; k < n; k++) {
        HeadTensor hd;
        hd.id = ids[k];
        hd.tensor = find_tensor(h, tensors, ids[k]);
        hd.layer = hd.tensor < 0 ? -1 : producing_conv(h, layers, ids[k]);
        const char *why = "";
        if (hd.layer < 0) {
            set_last_error("%s: head %d (tensor id %u) is not the output of a CONV2D layer", what, k, ids[k]);
            return MARS_ERR_INVALID_TENSOR;
        }
        if (!geometry(hd.tensor, &hd, &why)) {
            set_last_error("%s: head %d (tensor id %u) %s", what, k, ids[k], why);
            return MARS_ERR_INVALID_TENSOR;
        }
        if (k > 0 && hd.channels != (*out)[0].channels) {
            set_last_error("%s: head %d (tensor id %u) has %d channels, head 0 has %d: the channel count must be the same", what, k, ids[k],
                           hd.channels, (*out)[0].channels);
            return MARS_ERR_INVALID_TENSOR;
        }
        if (!(hd.scale > 0.0f) || !std::isfinite(hd.scale)) { /* the decodes need a monotone dequantisation */
            set_last_error("%s: head %d (tensor id %u) has scale %g; the decode needs a finite scale > 0", what, k, ids[k], (double)hd.scale);
            return MARS_ERR_INVALID_TENSOR;
        }
        if (toff[hd.tensor] < weights_size) {
            set_last_error("%s: head %d (tensor id %u) lives in the weight blob", what, k, ids[k]);
            return MARS_ERR_INVALID_TENSOR;
        }
        out->push_back(hd);
    }
    const std::vector<HeadTensor> &v = *out;
    for (int k = 1; k < n; k++)
        if (v[k].layer <= v[k - 1].layer) {
            set_last_error("%s: head %d (layer %d) is not produced after head %d (layer %d): heads are decoded in level order", what,
                           k, v[k].layer, k - 1, v[k - 1].layer);
            return MARS_ERR_INVALID_TENSOR;
        }
    for (int k = 0; k < n; k++)
        if (v[k].stride != strides[k]) {
            set_last_error("%s: head %d (tensor id %u) has stride %d; level %d needs stride %d", what, k, ids[k], v[k].stride, k, strides[k]);
            return MARS_ERR_INVALID_TENSOR;
        }
    return MARS_OK;
}

mars_error_t resolve_yolo_heads(const mars_header_t &h, const mars_runtime_tensor_t *tensors, const mars_runtime_layer_t *layers,
                                const std::vector<size_t> &toff, size_t weights_size, const uint32_t *ids, int n, std::vector<HeadTensor> *out) {
    out->clear();
    if (n != 3) {
        set_last_error("set_yolo_heads: %d heads given; a YOLOv5 Detect block has 3 (n = 0 switches the decode off)", n);
        return MARS_ERR_INVALID_TENSOR;
    }
    return resolve_heads("set_yolo_heads", h, tensors, layers, toff, weights_size, ids, n, YOLO_STRIDES,
                         [&](int ti, HeadTensor *hd, const char **why) { return yolo_geometry(h, tensors, ti, hd, why); }, out);
}

mars_error_t check_gfl_params(int nc, int reg_max, int centre, float conf) {
    if (nc < 1) { set_last_error("set_gfl_heads: nc = %d; a GFL head has at least one class", nc); return MARS_ERR_INVALID_TENSOR; }
    if (reg_max < 1 || reg_max > 16) {
        set_last_error("set_gfl_heads: reg_max = %d is outside 1..16", reg_max);
        return MARS_ERR_INVALID_TENSOR;
    }
    if (centre != MARS_B200_GFL_CENTRE_HALF && centre != MARS_B200_GFL_CENTRE_CORNER) {
        set_last_error("set_gfl_heads: centre = %d is not MARS_B200_GFL_CENTRE_HALF or MARS_B200_GFL_CENTRE_CORNER", centre);
        return MARS_ERR_INVALID_TENSOR;
    }
    if (!std::isfinite(conf)) { set_last_error("set_gfl_heads: conf_thresh %g is not finite", (double)conf); return MARS_ERR_INVALID_TENSOR; }
    return MARS_OK;
}

mars_error_t resolve_gfl_heads(const mars_header_t &h, const mars_runtime_tensor_t *tensors, const mars_runtime_layer_t *layers,
                               const std::vector<size_t> &toff, size_t weights_size, const uint32_t *ids, int n, int nc, int reg_max,
                               int centre, float conf, std::vector<HeadTensor> *out) {
    out->clear();
    mars_error_t e = check_gfl_params(nc, reg_max, centre, conf);
    if (e != MARS_OK) return e;
    if (n != 3 && n != 4) {
        set_last_error("set_gfl_heads: %d heads given; a GFL head has 3 or 4 levels (n = 0 switches the decode off)", n);
        return MARS_ERR_INVALID_TENSOR;
    }
    return resolve_heads("set_gfl_heads", h, tensors, layers, toff, weights_size, ids, n, GFL_STRIDES,
                         [&](int ti, HeadTensor *hd, const char **why) { return gfl_geometry(h, tensors, ti, hd, why, nc, reg_max); }, out);
}

/* one OP_YOLO_HEAD / OP_GFL_HEAD behind the last op of each head's layer (its conv, or the byte-ReLU that follows it), with the
 * head's tables */
static mars_error_t insert_heads(Ctx &c, const HeadSet &hs) {
    std::vector<Op> &ops = c.prog->ops;
    const bool gfl = hs.kind == HEADS_GFL;
    const mars_tensor_t &in = c.tensors[c.h.input_tensor_ids[0]].desc; /* checked by the setters */
    const bool in_nhwc = in.format == MARS_FORMAT_NHWC;
    for (size_t k = hs.heads.size(); k-- > 0;) {
        const HeadTensor &hd = hs.heads[k];
        size_t at = 0;
        for (size_t i = ops.size(); i-- > 0;)
            if (ops[i].layer == hd.layer) { at = i + 1; break; }
        if (!at) { set_last_error("detection head %zu: layer %d compiled to no device op", k, hd.layer); return MARS_ERR_INVALID_TENSOR; }
        Op o;
        o.kind = gfl ? OP_GFL_HEAD : OP_YOLO_HEAD;
        o.layer = hd.layer;
        o.in0 = c.off(hd.tensor);
        o.oc = hd.channels; o.oh = hd.gh; o.ow = hd.gw;
        o.sh = o.sw = hd.stride;
        o.n = (uint64_t)o.oc * hd.gh * hd.gw;
        o.f0 = hs.conf; o.f1 = hd.scale;
        o.head_level = (int)k; o.head_nc = hd.nc; o.head_nhwc = hd.nhwc;
        mars_error_t e;
        if ((e = check_read(c, hd.layer, o.in0, o.in0 + (int64_t)o.n))) return e;
        float tab[512];
        build_sigmoid_table(hd.scale, tab);
        if (gfl) build_gfl_exp_table(hd.scale, tab + 256);
        const size_t bytes = (gfl ? 512 : 256) * sizeof(float);
        o.lut = (int)c.prog->const_pool.size(); /* 256-byte units, float-aligned */
        c.prog->const_pool.resize(c.prog->const_pool.size() + bytes);
        memcpy(&c.prog->const_pool[o.lut], tab, bytes);
        char note[192];
        if (gfl) {
            o.head_reg_max = hs.reg_max;
            o.f2 = hs.centre == MARS_B200_GFL_CENTRE_HALF ? 0.5f : 0.0f;
            o.ih = in_nhwc ? in.shape[1] : in.shape[2];
            o.iw = in_nhwc ? in.shape[2] : in.shape[3];
            snprintf(note, sizeof note, "level %zu stride %d nc %d reg_max %d %s centre %s conf %g: decodes [in, in+n), the head store is kept",
                     k, hd.stride, hd.nc, hs.reg_max, hd.nhwc ? "nhwc" : "nchw", hs.centre == MARS_B200_GFL_CENTRE_HALF ? "half" : "corner",
                     (double)hs.conf);
        } else {
            snprintf(note, sizeof note, "level %zu stride %d nc %d %s conf %g: decodes [in, in+n), the head store is kept", k, hd.stride, hd.nc,
                     hd.nhwc ? "nhwc" : "nchw", (double)hs.conf);
        }
        o.note = note;
        ops.insert(ops.begin() + (ptrdiff_t)at, o);
    }
    return MARS_OK;
}

/* ---- opt_level >= 1: route hazard-free GEMM-shaped convs to the tcgen05 kernel ---------- */
static void select_tensor_core_convs(Program *p, int f32_mode) {
    for (auto &o : p->ops)
        if (o.kind == OP_CONV_F32_NCHW && tf32_supported(o, f32_mode)) o.impl = CONV_TC_F32;
    for (auto &o : p->ops)
        if ((o.kind == OP_CONV_I8_NCHW || o.kind == OP_CONV_I8_NHWC) && o.mode == EXEC_PARALLEL && !o.xlat && tc_supported(o)) o.impl = CONV_TC_NCHW;
}

/* reference src/mars/mars_runtime.c:818-835 for one (a, b) byte pair */
static int8_t mul_point(int a, int b, float sa, float sb, float inv) {
    volatile float va = (float)a * sa;
    volatile float vb = (float)b * sb;
    volatile float y = va * vb;
    volatile float t = y * inv;
    volatile float u = t + 0.5f;
    return clamp_i8(f2i_x86(u));
}

/* ---- opt_level >= 2: fold SIGMOID + MUL (the compiler's SiLU) into the conv epilogue ------
 * Y = conv output byte, S = sigmoid_table[Y], Z = mul(Y, S): both followers are pure functions
 * of the one byte Y, so the epilogue needs two 256-entry tables.  Legal only when the fused
 * write order cannot be observed through the planner's buffer aliasing:
 *   - S must not live in Y's buffer (the MUL would then read S where it expects Y);
 *   - S / Z may overwrite the conv's own INPUT buffer (they usually do, round-robin) only if
 *     the kernel reads its input from a private copy (3x3, stride 2) or every CTA reads exactly
 *     the pixels it later writes (1x1 with a single N tile). */
static void fuse_silu(Program *p, int64_t W) {
    std::vector<Op> &ops = p->ops;
    for (size_t i = 0; i + 2 < ops.size(); i++) {
        Op &c = ops[i];
        /* the in-place 1x1 conv on its own planes (register kernel, kernels_fast.cuh): same fusion, the kernel keeps the pixel's
         * channel vector in registers, so S and Z may go anywhere outside the conv's planes, weights and bias */
        const bool inplace_reg = c.kind == OP_CONV_I8_NCHW && c.impl == CONV_DIRECT && c.mode == EXEC_PIXEL_SERIAL && !c.post_relu && !c.xlat &&
                                 (c.ic == 32 || c.ic == 64 || c.ic == 128) && c.w >= 0 && (c.w & 3) == 0 && c.w + (int64_t)c.oc * c.ic <= W &&
                                 (size_t)c.oc * (c.ic / 4 + 1) * 4 <= 160 * 1024; /* = inplace_reg_ok (kernels_fast.cuh) */
        if (inplace_reg) {
            Op &s = ops[i + 1], &m = ops[i + 2];
            const int64_t numel = (int64_t)c.oc * c.oh * c.ow;
            if (s.kind != OP_SIGMOID_I8 || s.mode != EXEC_PARALLEL || s.xlat || m.kind != OP_MUL_I8 || m.mode != EXEC_PARALLEL || m.xlat) continue;
            if (s.in0 != c.out || (int64_t)s.n != numel || (int64_t)m.n != numel) continue;
            const bool y_first = m.in0 == c.out && m.in1 == s.out, s_first = m.in0 == s.out && m.in1 == c.out;
            if (!y_first && !s_first) continue;
            const int64_t x0 = c.in0, x1 = c.in0 + (int64_t)c.ic * c.ih * c.iw;
            if (s.out < W || m.out < W || s.out == m.out || overlap(s.out, s.out + numel, x0, x1) || overlap(m.out, m.out + numel, x0, x1) ||
                overlap(s.out, s.out + numel, m.out, m.out + numel)) continue;
            int8_t lut[256];
            const int8_t *sig = reinterpret_cast<const int8_t *>(&p->const_pool[s.lut]);
            for (int y = -128; y < 128; y++) {
                int sv = sig[y + 128];
                lut[y + 128] = y_first ? mul_point(y, sv, m.f0, m.f1, m.f2) : mul_point(sv, y, m.f0, m.f1, m.f2);
            }
            c.lut_s = s.lut; c.lut_z = pool_add(p, lut);
            c.out_s = s.out; c.out_z = m.out; c.store_y = true; c.fused_layers = 2;
            c.whi = std::max(c.whi, std::max(s.whi, m.whi));
            c.note += " +sigmoid+mul fused";
            s.kind = OP_NOP; s.note = "folded into the in-place conv"; m.kind = OP_NOP; m.note = "folded into the in-place conv";
            continue;
        }
        if (c.impl != CONV_TC_NCHW || (c.kind != OP_CONV_I8_NCHW && c.kind != OP_CONV_I8_NHWC) || c.post_relu) continue;
        Op &s = ops[i + 1], &m = ops[i + 2];
        if (s.kind != OP_SIGMOID_I8 || s.mode != EXEC_PARALLEL || s.xlat) continue;
        if (m.kind != OP_MUL_I8 || m.mode != EXEC_PARALLEL || m.xlat) continue;
        const int64_t numel = (int64_t)c.oc * c.oh * c.ow;
        if (s.in0 != c.out || (int64_t)s.n != numel || (int64_t)m.n != numel) continue;
        const bool y_first = m.in0 == c.out && m.in1 == s.out, s_first = m.in0 == s.out && m.in1 == c.out;
        if (!y_first && !s_first) continue;
        if (s.out == c.out) continue;
        if (s.out < W || m.out < W) continue;
        const int64_t x0 = c.in0, x1 = c.in0 + (int64_t)c.ic * c.ih * c.iw;
        const bool touches_input = overlap(s.out, s.out + numel, x0, x1) || overlap(m.out, m.out + numel, x0, x1);
        if (touches_input) {
            const bool same_tile = c.kh == 1 && c.kw == 1 && tc_n_tiles(c.oc) == 1 && c.oh == c.ih && c.ow == c.iw &&
                                   (s.out == c.in0 || !overlap(s.out, s.out + numel, x0, x1)) &&
                                   (m.out == c.in0 || !overlap(m.out, m.out + numel, x0, x1));
            /* several N tiles (Co > 256): a CTA's outputs would overwrite input pixels the other N tile's CTAs still read */
            if (!tc_uses_copy(c) && !same_tile) continue;
        }
        /* neither follower may clobber the weights or the bias the kernel is still reading: both live below W */
        int8_t lut[256];
        const int8_t *sig = reinterpret_cast<const int8_t *>(&p->const_pool[s.lut]);
        for (int y = -128; y < 128; y++) {
            int sv = sig[y + 128];
            lut[y + 128] = y_first ? mul_point(y, sv, m.f0, m.f1, m.f2) : mul_point(sv, y, m.f0, m.f1, m.f2);
        }
        c.lut_s = s.lut;
        c.lut_z = pool_add(p, lut);
        c.out_s = s.out == m.out ? -1 : s.out; /* an in-place MUL replaces S */
        c.out_z = m.out;
        c.store_y = c.out != m.out;
        c.fused_layers = 2;
        c.whi = std::max(c.whi, std::max(s.whi, m.whi));
        c.note = "conv+sigmoid+mul fused";
        s.kind = OP_NOP; s.note = "folded into the conv epilogue";
        m.kind = OP_NOP; m.note = "folded into the conv epilogue";
    }
}


/* ---- opt_level >= 2: producer-written channel-innermost copies for kxk tensor-core convs ------------------- */
static bool op_writes(const Op &o, int64_t lo, int64_t hi) {
    if (o.kind == OP_NOP || o.mode >= 1000) return false;
    if (o.kind == OP_CONV_I8_NCHW || o.kind == OP_CONV_I8_NHWC || o.kind == OP_CONV_F32_NCHW || o.kind == OP_DW_I8) {
        const int64_t numel = (int64_t)o.oc * o.oh * o.ow, es = o.kind == OP_CONV_F32_NCHW ? 4 : 1;
        return (o.store_y && overlap(o.out, o.out + numel * es, lo, hi)) || (o.out_s >= 0 && overlap(o.out_s, o.out_s + numel, lo, hi)) ||
               (o.out_z >= 0 && o.store_z && overlap(o.out_z, o.out_z + numel, lo, hi)) || (o.fwd_out >= 0 && overlap(o.fwd_out, o.fwd_out + numel, lo, hi));
    }
    return overlap(o.wlo, o.whi, lo, hi);
}

static void link_nhwc_copies(Program *p) {
    std::vector<Op> &ops = p->ops;
    size_t total = 0;
    for (size_t j = 0; j < ops.size(); j++) {
        Op &c = ops[j];
        if (c.impl != CONV_TC_NCHW || !tc_linkable(c)) continue;
        const int64_t numel = (int64_t)c.ic * c.ih * c.iw, lo = c.in0, hi = c.in0 + numel;
        for (size_t i = j; i-- > 0;) {
            Op &o = ops[i];
            if (!op_writes(o, lo, hi)) continue;
            /* o is the last op that touches the consumer's input: link iff it is a tensor-core conv whose final value
             * over exactly that range is one of its output streams */
            if (o.impl != CONV_TC_NCHW || o.kind != OP_CONV_I8_NCHW || o.mode != EXEC_PARALLEL || o.nhwc_consumer >= 0) break;
            if (o.oc != c.ic || o.oh != c.ih || o.ow != c.iw) break;
            int stream = -1;
            if (o.fused_layers > 0) {
                if (o.out_z == lo) stream = 0;
                else if (o.out_s == lo && !overlap(o.out_z, o.out_z + numel, lo, hi)) stream = 1;
                else if (o.out == lo && o.store_y && !overlap(o.out_z, o.out_z + numel, lo, hi) &&
                         !(o.out_s >= 0 && overlap(o.out_s, o.out_s + numel, lo, hi))) stream = 2;
            } else if (o.out == lo) stream = 2;
            if (stream < 0) break;
            o.nhwc_consumer = (int)j; o.nhwc_stream = stream;
            c.copy_from = (int)i; c.copy_off = (int64_t)total;
            total += (tc_scratch_need(c) + 1023) & ~(size_t)1023;
            o.note += " +copy"; c.note += " <copy";
            break;
        }
    }
    p->linked_bytes = total;
}

/* ---- opt_level >= 3: concat forwarding ---------------------------------------------------------------
 * With NCHW-shaped descriptors a concat input is a flat copy (SURVEY C.4): out[coff + t] = in[t].  When the head of that source
 * range is exactly one output stream of the tensor-core conv that wrote it last, and nothing between that conv and the concat
 * touches the destination bytes, the conv's epilogue writes the stream to its destination as well (Op::fwd_out) and the concat
 * copies only what follows the stream.  Dead-store elision afterwards drops the conv's original store when nothing else reads it,
 * so the forwarded bytes cost no extra store and save one read and one write.  Model outputs are unchanged; the intermediate
 * arena differs from the reference's only in dead bytes (opt level 3 promises outputs, levels 0-2 the whole arena). */
struct Access;
static void op_access(const Op &o, Access *a);
static void forward_concat_inputs(Program *p);

/* ---- opt_level >= 3: dead-store elision in fused epilogues (SURVEY C.6) ------------------
 * Backward liveness over byte intervals of the image slot.  A byte is live after op i when some
 * later op -- or op 0.. of the NEXT run on the same slot (work buffers are never cleared), or the
 * host through a model output's work buffer -- may read it before it is unconditionally
 * overwritten.  Reads are over-approximated, kills are exact.  Only the extra stores of a fused
 * conv (its pre-activation Y and the sigmoid S) are ever dropped; every layer's arithmetic runs. */
struct IvSet {
    std::vector<std::pair<int64_t, int64_t>> v; /* sorted, disjoint, non-empty [lo,hi) */
    void add(int64_t a, int64_t b) {
        if (a >= b) return;
        std::vector<std::pair<int64_t, int64_t>> r;
        size_t i = 0;
        while (i < v.size() && v[i].second < a) r.push_back(v[i++]);
        while (i < v.size() && v[i].first <= b) { a = std::min(a, v[i].first); b = std::max(b, v[i].second); i++; }
        r.emplace_back(a, b);
        while (i < v.size()) r.push_back(v[i++]);
        v.swap(r);
    }
    void sub(int64_t a, int64_t b) {
        if (a >= b) return;
        std::vector<std::pair<int64_t, int64_t>> r;
        for (auto &iv : v) {
            if (iv.second <= a || iv.first >= b) { r.push_back(iv); continue; }
            if (iv.first < a) r.emplace_back(iv.first, a);
            if (iv.second > b) r.emplace_back(b, iv.second);
        }
        v.swap(r);
    }
    bool hits(int64_t a, int64_t b) const {
        for (auto &iv : v) if (a < iv.second && iv.first < b && a < b) return true;
        return false;
    }
    bool operator==(const IvSet &o) const { return v == o.v; }
};

struct Access { std::vector<std::pair<int64_t, int64_t>> reads, kills; };

static int elem_size(int kind) {
    switch (kind) {
        case OP_CONV_F32_NCHW: case OP_SIGMOID_F32: case OP_MUL_F32: case OP_ADD_F32: case OP_RELU_F32: case OP_BN_F32: return 4;
        default: return 1;
    }
}

static void op_access(const Op &o, Access *a) {
    a->reads.clear(); a->kills.clear();
    if (o.mode >= 1000) return;
    const int64_t es = elem_size(o.kind);
    auto R = [&](int64_t lo, int64_t n) { if (lo >= 0 && n > 0) a->reads.emplace_back(lo, lo + n); };
    auto K = [&](int64_t lo, int64_t n) { if (lo >= 0 && n > 0) a->kills.emplace_back(lo, lo + n); };
    switch (o.kind) {
        case OP_CONV_I8_NCHW: case OP_CONV_I8_NHWC: case OP_CONV_F32_NCHW: case OP_DW_I8: {
            const int64_t numel = (int64_t)o.oc * o.oh * o.ow;
            if (o.copy_from < 0) R(o.in0, (int64_t)o.ic * o.ih * o.iw * es); /* else: reads the producer-written copy */
            R(o.w, (int64_t)o.oc * (o.kind == OP_DW_I8 ? 1 : o.ic) * o.kh * o.kw * es);
            if (o.bias >= 0) R(o.bias, 4 * (int64_t)o.oc);
            if (o.store_y) K(o.out, numel * es);
            if (o.out_s >= 0) K(o.out_s, numel);
            if (o.out_z >= 0 && o.store_z) K(o.out_z, numel);
            if (o.fwd_out >= 0) K(o.fwd_out, numel);
            break;
        }
        case OP_BYTE_RELU: R(o.out, (int64_t)o.n); break;
        case OP_SIGMOID_I8: case OP_SIGMOID_F32: case OP_RELU_I8: case OP_RELU_F32: case OP_LUT_I8:
            R(o.in0, (int64_t)o.n * es); K(o.out, (int64_t)o.n * es); break;
        case OP_MUL_I8: case OP_ADD_I8: case OP_MUL_F32: case OP_ADD_F32:
            R(o.in0, (int64_t)o.n * es); R(o.in1, (int64_t)o.n * es); K(o.out, (int64_t)o.n * es); break;
        case OP_BN_I8: case OP_BN_F32:
            R(o.in0, (int64_t)o.n * es); R(o.in1, 4 * (int64_t)o.ic); R(o.in2, 4 * (int64_t)o.ic); K(o.out, (int64_t)o.n * es); break;
        case OP_MAXPOOL: case OP_UPSAMPLE:
            R(o.in0, (int64_t)o.ih * o.iw * o.ic); K(o.out, (int64_t)o.oh * o.ow * o.ic); break;
        case OP_CONCAT:
            R(o.in0, (int64_t)o.n);
            if (o.ic == o.oc) K(o.out + o.coff, (int64_t)o.n); /* strided writes kill nothing (conservative) */
            break;
        case OP_CONCAT_PERIODIC: R(o.out, o.coff); K(o.out + o.coff, (int64_t)o.n); break;
        case OP_YOLO_HEAD: case OP_GFL_HEAD: R(o.in0, (int64_t)o.n); break; /* keeps the head conv's store alive through dead-store elision */
        default: break;
    }
}

static void forward_concat_inputs(Program *p) {
    std::vector<Op> &ops = p->ops;
    Access a;
    for (size_t j = 0; j < ops.size(); j++) {
        Op &c = ops[j];
        if (c.kind != OP_CONCAT || c.mode != EXEC_PARALLEL || c.ic != c.oc || c.xlat || c.n < 4096) continue;
        const int64_t src = c.in0, n = (int64_t)c.n, dst = c.out + c.coff;
        for (size_t i = j; i-- > 0;) {
            Op &o = ops[i];
            if (!op_writes(o, src, src + n)) continue;
            /* o = the last op that writes any byte the concat reads */
            if (o.impl != CONV_TC_NCHW || o.kind != OP_CONV_I8_NCHW || o.mode != EXEC_PARALLEL || o.fwd_out >= 0) break;
            const int64_t numel = (int64_t)o.oc * o.oh * o.ow;
            if (numel > n || numel < 4096) break;
            const bool zs = o.fused_layers > 0 && o.out_z >= 0 && o.store_z, ss = o.fused_layers > 0 && o.out_s >= 0, ys = o.store_y;
            int stream = -1;
            if (zs && o.out_z == src) stream = 0;
            else if (ss && o.out_s == src) stream = 1;
            else if (ys && o.out == src) stream = 2;
            if (stream < 0) break;
            /* the op's other stored streams must leave the stream's bytes alone (the epilogue's store order is unspecified) */
            if ((stream != 0 && zs && overlap(o.out_z, o.out_z + numel, src, src + numel)) || (stream != 1 && ss && overlap(o.out_s, o.out_s + numel, src, src + numel)) ||
                (stream != 2 && ys && overlap(o.out, o.out + numel, src, src + numel))) break;
            if ((int)zs + (int)ss + (int)ys >= 3) break; /* no table byte left for a fourth stream */
            /* the destination: not read or written by the conv itself nor by anything up to the concat */
            bool clash = false;
            for (size_t k = i; k < j && !clash; k++) {
                const Op &q = ops[k];
                if (q.kind == OP_NOP) continue;
                if (op_writes(q, dst, dst + numel)) clash = true;
                op_access(q, &a);
                for (auto &iv : a.reads) if (overlap(iv.first, iv.second, dst, dst + numel)) clash = true;
                if (k == i && q.copy_from >= 0 && overlap(q.in0, q.in0 + (int64_t)q.ic * q.ih * q.iw, dst, dst + numel)) clash = true; /* (reads a copy, but keep it simple) */
            }
            if (clash) break;
            /* earlier inputs of the same concat (the slivers that survive it) may read the stream too -- with the planner's buffer
             * rotation the "first" input often IS this tensor (SURVEY C.4).  They run after the conv, when the forwarded copy is
             * already in place and nothing has modified it: read that copy instead, so that the original store can die */
            for (size_t k = i + 1; k < j; k++) {
                Op &q = ops[k];
                if (q.kind != OP_CONCAT || q.mode != EXEC_PARALLEL || q.xlat || q.ic != q.oc) continue;
                const int64_t qn = (int64_t)q.n, qdst = q.out + q.coff;
                if (q.in0 < src || q.in0 + qn > src + numel) continue;
                const int64_t nin = q.in0 + (dst - src);
                if (overlap(nin, nin + qn, qdst, qdst + qn)) continue;
                q.in0 = nin; q.note += " (reads the forwarded copy)";
            }
            o.fwd_out = dst; o.fwd_stream = stream;
            o.whi = std::max(o.whi, dst + numel);
            o.note += " +fwd";
            if (numel == n) { c.kind = OP_NOP; c.note = "written by the producing conv (concat forwarding)"; }
            else { c.in0 += numel; c.coff += (int)numel; c.wlo += numel; c.n -= (uint64_t)numel; c.note += " (head written by the producing conv)"; }
            break;
        }
    }
}

static void elide_dead_stores(Program *p, const IvSet &observed, const IvSet &host_written) {
    IvSet live_in; /* live at the start of a run */
    Access a;
    for (int iter = 0; iter < 8; iter++) {
        IvSet live = observed;
        for (auto &iv : live_in.v) live.add(iv.first, iv.second);
        for (size_t k = p->ops.size(); k-- > 0;) {
            Op &o = p->ops[k];
            if (o.fused_layers == 0 && o.fwd_out >= 0 && o.kind == OP_CONV_I8_NCHW && o.store_y &&
                !live.hits(o.out, o.out + (int64_t)o.oc * o.oh * o.ow)) { o.store_y = false; o.note += " -Y"; } /* only the forwarded copy is read */
            if (o.fused_layers > 0 && (o.kind == OP_CONV_I8_NCHW || o.kind == OP_CONV_I8_NHWC)) {
                const int64_t numel = (int64_t)o.oc * o.oh * o.ow;
                if (getenv("MARS_LIVE_DEBUG") && iter == 0) { /* how many output planes of every stream are live after the op */
                    const int64_t P = (int64_t)o.oh * o.ow;
                    auto cnt = [&](int64_t base) { int n = 0; if (base < 0) return -1; for (int c = 0; c < o.oc; c++) n += live.hits(base + c * P, base + (c + 1) * P) ? 1 : 0; return n; };
                    fprintf(stderr, "live op %zu layer %d oc %d: Y %d%s S %d Z %d%s\n", k, o.layer, o.oc, cnt(o.out), o.store_y ? "" : "(off)", cnt(o.out_s), cnt(o.out_z), o.store_z ? "" : "(off)");
                }
                /* later stages of the chain overwrite equal ranges, so test each against what is live AFTER the op */
                if (o.store_y && !live.hits(o.out, o.out + numel)) { o.store_y = false; o.note += " -Y"; }
                if (o.out_s >= 0 && !live.hits(o.out_s, o.out_s + numel)) { o.out_s = -1; o.note += " -S"; }
                if (o.out_z >= 0 && o.store_z && (o.nhwc_consumer >= 0 || o.fwd_out >= 0) && !live.hits(o.out_z, o.out_z + numel)) { o.store_z = false; o.note += " -Z"; }
            }
            op_access(o, &a);
            for (auto &iv : a.kills) live.sub(iv.first, iv.second);
            for (auto &iv : a.reads) live.add(iv.first, iv.second);
        }
        for (auto &iv : host_written.v) live.sub(iv.first, iv.second); /* the host rewrites the inputs before every run */
        if (live == live_in) break;
        live_in = live;
    }
}

mars_error_t compile_program(const mars_header_t &h, const mars_runtime_tensor_t *tensors,
                             const mars_runtime_layer_t *layers, const std::vector<size_t> &toff,
                             size_t weights_size, size_t arena_size, int opt_level, int depthwise_mode,
                             Program *out, int f32_mode, const HeadSet *heads) {
    out->ops.clear();
    out->const_pool.clear();
    out->scratch_bytes = 0;
    out->linked_bytes = 0;
    out->max_extent = 0;
    Ctx c{h, tensors, toff, (int64_t)weights_size, (int64_t)arena_size, out};
    for (uint32_t i = 0; i < h.num_layers; i++) {
        const mars_layer_t &L = layers[i].desc;
        mars_error_t e = MARS_OK;
        switch ((int)L.type) {
            case MARS_LAYER_CONV2D: e = compile_conv(c, (int)i, L, 0); break;
            case MARS_LAYER_DEPTHWISE_CONV2D:
                if (depthwise_mode) e = compile_conv(c, (int)i, L, 1); /* else no-op, reference :1168-1170 */
                break;
            case MARS_LAYER_MAXPOOL: case MARS_LAYER_UPSAMPLE: e = compile_spatial(c, (int)i, L); break;
            case MARS_LAYER_RELU: case MARS_LAYER_RELU6: case MARS_LAYER_LEAKY_RELU:
            case MARS_LAYER_SIGMOID: case MARS_LAYER_ADD: case MARS_LAYER_MUL:
                e = compile_eltwise(c, (int)i, L); break;
            case MARS_LAYER_CONCAT: e = compile_concat(c, (int)i, L); break;
            case MARS_LAYER_BATCHNORM: e = compile_batchnorm(c, (int)i, L); break;
            case MARS_LAYER_AVGPOOL: case MARS_LAYER_SILU: case MARS_LAYER_RESHAPE:
            case MARS_LAYER_TRANSPOSE: case MARS_LAYER_SOFTMAX:
                break; /* no-ops in the reference (:1175-1213) */
            default: /* GLOBAL_AVGPOOL(4), FC(16), unknown: reference :1218-1220 */
                out->ops.push_back(fail_op((int)i, MARS_ERR_INVALID_LAYER, "unknown layer type"));
                break;
        }
        if (e != MARS_OK) return e;
    }
    if (heads && !heads->empty()) {
        mars_error_t e = insert_heads(c, *heads);
        if (e != MARS_OK) return e;
    }
    if (opt_level >= 1) select_tensor_core_convs(out, f32_mode);
    if (opt_level >= 2) fuse_silu(out, (int64_t)weights_size);
    if (opt_level >= 2) link_nhwc_copies(out);
    if (opt_level >= 3) {
        IvSet observed, host_written;
        for (uint32_t i = 0; i < h.num_outputs && i < 4; i++) { /* callers may read a whole output work buffer (alloc_size) */
            uint32_t ti = h.output_tensor_ids[i];
            if (ti < h.num_tensors) observed.add((int64_t)toff[ti], (int64_t)toff[ti] + (int64_t)tensors[ti].alloc_size);
        }
        for (uint32_t i = 0; i < h.num_inputs && i < 4; i++) {
            uint32_t ti = h.input_tensor_ids[i];
            if (ti >= h.num_tensors) continue;
            const mars_tensor_t &d = tensors[ti].desc;
            int64_t es = (d.dtype == MARS_DTYPE_FLOAT32 || d.dtype == MARS_DTYPE_INT32) ? 4 : (d.dtype == MARS_DTYPE_INT16 ? 2 : 1);
            host_written.add((int64_t)toff[ti], (int64_t)toff[ti] + (int64_t)numel_of(d) * es);
        }
        elide_dead_stores(out, observed, host_written); /* first: which streams of a conv are stored at all */
        forward_concat_inputs(out);
        elide_dead_stores(out, observed, host_written); /* again: the original of a forwarded stream is usually dead now */
    }
    /* tables are addressed in 256-byte units; keep the pool non-empty so the upload is uniform */
    if (out->const_pool.empty()) out->const_pool.resize(256, 0);
    return MARS_OK;
}

static const char *kind_name(int k) {
    static const char *n[] = {"nop", "conv_i8_nchw", "conv_i8_nhwc", "conv_f32_nchw", "dw_i8", "byte_relu",
                              "sigmoid_i8", "sigmoid_f32", "mul_i8", "add_i8", "mul_f32", "add_f32", "relu_i8",
                              "relu_f32", "bn_i8", "bn_f32", "maxpool", "concat", "concat_periodic", "upsample", "lut_i8",
                              "yolo_head", "gfl_head"};
    return (k >= 0 && k < OP_KIND_COUNT) ? n[k] : "?";
}
static const char *mode_name(int m) {
    switch (m) {
        case EXEC_PARALLEL: return "parallel";
        case EXEC_OC_PASSES: return "oc-passes";
        case EXEC_OC_PASSES_SCRATCH: return "oc-passes+scratch";
        case EXEC_PIXEL_SERIAL: return "pixel-serial";
        case EXEC_SERIAL: return "serial";
        default: return m >= 1000 ? "FAIL" : "?";
    }
}

std::string describe_program(const Program &p) {
    std::string s;
    char line[512];
    for (size_t i = 0; i < p.ops.size(); i++) {
        const Op &o = p.ops[i];
        char rq[16] = ""; /* int8 tensor-core convs of a compiled model: the epilogue's requantisation variant */
        if (o.rq >= 0) snprintf(rq, sizeof rq, " rq=%d", o.rq);
        snprintf(line, sizeof line,
                 "op %3zu layer %3d %-16s %-18s impl=%d%s in=%lld out=%lld ic=%d ih=%d iw=%d oc=%d oh=%d ow=%d k=%dx%d s=%d,%d p=%d,%d n=%llu fused=%d%s %s\n",
                 i, o.layer, kind_name(o.kind), mode_name(o.mode), o.impl, rq, (long long)o.in0, (long long)o.out, o.ic,
                 o.ih, o.iw, o.oc, o.oh, o.ow, o.kh, o.kw, o.sh, o.sw, o.pt, o.pl, (unsigned long long)o.n,
                 o.fused_layers, o.xlat ? " xlat" : "", o.note.c_str());
        s += line;
    }
    return s;
}

} // namespace marsb200
