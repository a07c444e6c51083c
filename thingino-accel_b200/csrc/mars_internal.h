/*
 * mars_internal.h -- private types of libmars_b200.so.
 *
 * Data layout in HBM (DESIGN.md §3):
 *   d_weights : the model's weight blob, one copy per GPU, shared by every image;
 *   d_slots   : `capacity` image slots, each = the reference's work buffers
 *               [buf0 | buf1 | (buf2)] exactly as the planner of reference
 *               src/mars/mars_runtime.c:248-337 lays them out behind the weights.
 * Every tensor is addressed by its byte offset in the reference's arena
 * ("arena offset"): offsets below weights_size resolve into d_weights, the rest
 * into the image's slot.  A layer compiles into one or more `Op`s over arena offsets.
 */
#ifndef MARS_INTERNAL_H
#define MARS_INTERNAL_H

#include <stddef.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/mars_b200.h"

namespace marsb200 {

enum OpKind : int {
    OP_NOP = 0,
    OP_CONV_I8_NCHW,   /* reference src/mars/mxu_conv.c:630-670 */
    OP_CONV_I8_NHWC,   /* reference src/mars/mxu_conv.c:713-757 */
    OP_CONV_F32_NCHW,  /* reference src/mars/mxu_conv.c:673-710 */
    OP_DW_I8,          /* restated depthwise (parity unpinned) */
    OP_BYTE_RELU,      /* reference src/mars/mars_runtime.c:700-707 */
    OP_SIGMOID_I8,     /* reference src/mars/mars_runtime.c:752-768 (as a 256-entry table) */
    OP_SIGMOID_F32,    /* :742-749 */
    OP_MUL_I8, OP_ADD_I8,   /* :818-835, :885-902 */
    OP_MUL_F32, OP_ADD_F32, /* :807-815, :874-882 */
    OP_RELU_I8,        /* :1072-1085 (relu / relu6 / leaky as a 256-entry table) */
    OP_RELU_F32,       /* :1066-1071 */
    OP_BN_I8, OP_BN_F32, /* :1092-1158 */
    OP_MAXPOOL,        /* :908-960 */
    OP_CONCAT,         /* :963-1000, one op per input, in order */
    OP_CONCAT_PERIODIC,/* in-place concat input with constant shift (SURVEY C.4b) */
    OP_UPSAMPLE,       /* :1003-1044 */
    OP_LUT_I8,         /* fused chain of int8 unary layers as one table */
    OP_YOLO_HEAD,      /* anchor-grid decode of one YOLO head conv output (mars_b200_set_yolo_heads), right after the conv */
    OP_GFL_HEAD,       /* GFL decode of one NanoDet head conv output (mars_b200_set_gfl_heads), right after the conv */
    OP_KIND_COUNT
};

enum ExecMode : int {
    EXEC_PARALLEL = 0,  /* one thread (or tile) per output element, any order */
    EXEC_OC_PASSES,     /* NCHW conv whose output aliases its input: one launch per output channel */
    EXEC_OC_PASSES_SCRATCH, /* same, each pass staged through a scratch plane */
    EXEC_PIXEL_SERIAL,  /* NHWC conv in place: thread per pixel, output channels in order */
    EXEC_SERIAL         /* literal reference loop order on one thread per image */
};

enum ConvImpl : int {
    CONV_DIRECT = 0,    /* exact direct kernel (any shape) */
    CONV_TC_NCHW,       /* tcgen05 implicit GEMM (conv_tc.cu): NCHW / OIHW layers and, despite the name, NHWC / OHWI ones */
    CONV_TC_F32         /* tcgen05 kind::tf32 implicit GEMM for float32 layers (conv_tf32.cu) */
};

/* epilogue applied to an int8 value produced by an op (fused following layers) */
struct Epilogue {
    int lut_off;        /* >=0: offset of a 256-byte table in the const pool applied to the int8 result */
    int64_t extra_out[2]; /* additional arena offsets the *pre-table* stages are also written to, -1 = none */
    int extra_lut[2];     /* table applied for each extra output (-1 = identity) */
};

struct Op {
    int kind = OP_NOP;
    int mode = EXEC_PARALLEL;
    int impl = CONV_DIRECT;
    int layer = -1;        /* originating layer index */
    int fused_layers = 0;  /* how many following layers were folded into this op */
    bool xlat = false;     /* some operand straddles the weights/slot boundary: per-access translation */
    int64_t in0 = -1, in1 = -1, in2 = -1, out = -1, w = -1, bias = -1; /* arena offsets */
    int ic = 0, ih = 0, iw = 0, oc = 0, oh = 0, ow = 0;
    int kh = 1, kw = 1, sh = 1, sw = 1, pt = 0, pl = 0;
    int coff = 0;          /* concat channel offset / periodic shift */
    int in_ctot = 0;       /* concat: channels of this input */
    float f0 = 0, f1 = 0, f2 = 0; /* scales: conv combined scale; eltwise sa, sb, inv/so */
    uint64_t n = 0;        /* element count for flat ops */
    int lut = -1;          /* const-pool offset of a 256-byte table (sigmoid/relu/fused) */
    int post_relu = 0;     /* conv: byte-ReLU folded into the epilogue */
    int post_lut = -1;     /* conv: fused following unary chain */
    /* conv with the following SIGMOID and MUL layers folded into its epilogue: y = conv output
     * byte, S = lut_s[y] stored at out_s, Z = lut_z[y] stored at out_z; store_y=false when a
     * later stage of the same chain overwrites Y's bytes anyway */
    bool store_y = true, store_z = true;
    int64_t out_s = -1, out_z = -1;
    int lut_s = -1, lut_z = -1;
    /* producer -> consumer link (SURVEY C.6): a kxk tensor-core conv reads a channel-innermost, zero-padded copy of
     * its input; when that input is exactly one output stream of an earlier tensor-core conv, the producer's
     * epilogue writes the copy itself (nhwc_consumer / nhwc_stream: 0 = Z, 1 = S, 2 = Y) and the consumer skips its
     * own layout pre-pass (copy_from = producer op, copy_off = byte offset of its region in the per-image link area) */
    int copy_from = -1, nhwc_consumer = -1, nhwc_stream = -1;
    int64_t copy_off = 0;
    /* concat forwarding (opt level 3): the op's stream fwd_stream (0 = Z, 1 = S, 2 = Y) is ALSO written at arena offset fwd_out --
     * its place in the output of the concat that would copy it there later (program.cpp forward_concat_inputs) */
    int64_t fwd_out = -1;
    int fwd_stream = -1;
    /* write/read extents for hazard analysis and bounds checks */
    int64_t wlo = 0, whi = 0;
    /* OP_YOLO_HEAD / OP_GFL_HEAD: the head tensor is [in0, in0 + n) with grid oh x ow, `lut` = const-pool offset of its 256-float
     * sigmoid table (OP_GFL_HEAD: followed by the 256-float table E[d] = expf(-(d * scale))), f0 = confidence threshold,
     * sh = stride (8 << head_level).  OP_GFL_HEAD: f2 = cell centre offset (0.5 or 0), iw x ih = network input size */
    int head_level = -1, head_nc = 0, head_reg_max = 0;
    bool head_nhwc = false;
    int rq = -1; /* int8 tensor-core conv: requantisation variant of its planned epilogue (tc_rq), set when the model compiles */
    std::string note;
};

/* one detection head conv (YOLOv5 Detect or NanoDet GFL) as the layer table describes it */
struct HeadTensor {
    uint32_t id = 0;   /* tensor id (mars_tensor_t.id) of the head conv's output */
    int tensor = -1;   /* its tensor table index */
    int layer = -1;    /* the CONV2D layer that writes it */
    int channels = 0, nc = 0, gh = 0, gw = 0, stride = 0;
    bool nhwc = false;
    float scale = 0.0f;
};

/* the detection heads a model decodes inside its program: one kind or none (each setter replaces what is set) */
enum HeadKind : int { HEADS_NONE = 0, HEADS_YOLO, HEADS_GFL };
struct HeadSet {
    int kind = HEADS_NONE;
    std::vector<HeadTensor> heads; /* in level order */
    float conf = 0.25f;
    int reg_max = 0, centre = 0;   /* HEADS_GFL (centre: MARS_B200_GFL_CENTRE_*) */
    bool empty() const { return heads.empty(); }
};

/* the three YOLOv5 Detect levels of reference examples/yolo_detect.cpp:176-181: stride and (w, h) of each of the level's anchors */
struct HeadAnchors { float wh[6]; };
struct YoloLevel {
    int stride;
    HeadAnchors anchors;
};
static const YoloLevel YOLO_LEVELS[3] = {
    {8, {{10, 13, 16, 30, 33, 23}}}, {16, {{30, 61, 62, 45, 59, 119}}}, {32, {{116, 90, 156, 198, 373, 326}}}};

struct Program {
    std::vector<Op> ops;
    std::vector<uint8_t> const_pool; /* 256-byte tables, uploaded once */
    size_t scratch_bytes = 0;        /* per-image scratch for EXEC_OC_PASSES_SCRATCH */
    size_t linked_bytes = 0;         /* per-image bytes of producer-written conv input copies */
    size_t max_extent = 0;           /* highest arena offset (exclusive) any op reads or writes: an image slot must reach that far */
};

/* device-side view of the arena; passed by value to kernels */
struct ArenaView {
    const uint8_t *wbase; /* d_weights */
    uint8_t *sbase;       /* slot 0 of the launch */
    uint64_t W;           /* weights_size: arena offsets >= W live in the slot */
    uint64_t slot_stride;
    const uint8_t *cpool; /* const pool */
    uint8_t *scratch;     /* per-image scratch base */
    uint64_t scratch_stride;
};

struct Model; /* defined in runtime.cu */

/* ---- host-side helpers shared between translation units ---- */
size_t tensor_byte_size(const mars_tensor_t *t);
int find_tensor(const mars_header_t &h, const mars_runtime_tensor_t *tensors, uint32_t id);
void set_last_error(const char *fmt, ...);
/* once per CUDA device: true the first time it is called with this mask on the current device (function attributes and
 * SM counts are per device; the API supports several devices in one process) */
bool first_time_on_device(unsigned long long *mask);
/* sig[v + 128] = 1 / (1 + expf(-(v * scale))) for v = -128..127: the host libm's expf, one rounding per operation */
void build_sigmoid_table(float scale, float sig[256]);

/* compile the layer table into ops (program.cpp) */
mars_error_t compile_program(const mars_header_t &h, const mars_runtime_tensor_t *tensors,
                             const mars_runtime_layer_t *layers, const std::vector<size_t> &toff,
                             size_t weights_size, size_t arena_size, int opt_level, int depthwise_mode,
                             Program *out, int f32_mode = 0, const HeadSet *heads = nullptr);
std::string describe_program(const Program &p);
/* the outputs of the three CONV2D layers of a YOLOv5 Detect block in stride order 8 / 16 / 32 (host only); 0 when there are none */
int find_yolo_heads(const mars_header_t &h, const mars_runtime_tensor_t *tensors, const mars_runtime_layer_t *layers, uint32_t *ids, int cap);
/* checks n head tensor ids for mars_b200_set_yolo_heads: MARS_ERR_INVALID_TENSOR (with mars_b200_last_error) or MARS_OK + *out */
mars_error_t resolve_yolo_heads(const mars_header_t &h, const mars_runtime_tensor_t *tensors, const mars_runtime_layer_t *layers,
                                const std::vector<size_t> &toff, size_t weights_size, const uint32_t *ids, int n, std::vector<HeadTensor> *out);
/* the last 1x1 CONV2D per stride 8 / 16 / 32 (/ 64) with nc + 4 (reg_max + 1) channels, no activation and no compute reader, in
 * stride order (host only); returns 3 or 4, or 0 when the strides found are not 8, 16, 32 (, 64) */
int find_gfl_heads(const mars_header_t &h, const mars_runtime_tensor_t *tensors, const mars_runtime_layer_t *layers, int nc, int reg_max,
                   uint32_t *ids, int cap);
/* the parameters of mars_b200_set_gfl_heads: MARS_ERR_INVALID_TENSOR (with mars_b200_last_error) or MARS_OK */
mars_error_t check_gfl_params(int nc, int reg_max, int centre, float conf);
/* checks n GFL head tensor ids and the parameters for mars_b200_set_gfl_heads, like resolve_yolo_heads */
mars_error_t resolve_gfl_heads(const mars_header_t &h, const mars_runtime_tensor_t *tensors, const mars_runtime_layer_t *layers,
                               const std::vector<size_t> &toff, size_t weights_size, const uint32_t *ids, int n, int nc, int reg_max,
                               int centre, float conf, std::vector<HeadTensor> *out);
/* E[d] = expf(-(d * scale)) for d = 0..255: the host libm's expf, one rounding per operation (the GFL softmax) */
void build_gfl_exp_table(float scale, float e[256]);

} // namespace marsb200

#endif
