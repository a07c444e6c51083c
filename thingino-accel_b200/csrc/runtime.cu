/*
 * runtime.cu -- libmars_b200.so: the mars C runtime API over an HBM arena.
 *
 * Host side (stays C-callable, mirrors reference src/mars/mars_runtime.c):
 *   mars_load_memory/file : parse the .mars tables, run the reference's work-buffer
 *                           planner (:248-337) to get every tensor's ARENA OFFSET, upload
 *                           the weight blob once, compile the layer table into device ops;
 *   mars_run              : H2D of the input work buffers, replay the ops on one image
 *                           slot, D2H of the output work buffers (synchronous, like the
 *                           reference's :439-459);
 *   mars_b200_*           : the same ops over a batch of image slots resident in HBM,
 *                           plus YOLO decode + NMS on the device.
 * There is no CPU execution path: without a CUDA device every entry point fails with
 * MARS_ERR_NNA_INIT_FAILED.
 */
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <map>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/mxu_ops.h"
#include "../../include/mars_math.h"
#include "../../include/nna.h"
#include "../../include/nna_memory.h"
#include "conv_tc.h"
#include "conv_tf32.h"
#include "kernels_exact.cuh"
#include "kernels_fast.cuh"
#include "mars_internal.h"
#include "postproc.cuh"
#include "preproc.cuh"
#include "nna_layout.cuh"
#include "track.cuh"
#include "zones.cuh"

namespace marsb200 {

/* ---- diagnostics ------------------------------------------------------------ */
static thread_local char g_err[768];
void set_last_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    if (getenv("MARS_VERBOSE")) fprintf(stderr, "mars_b200: %s\n", g_err);
}

#define CU_OK(call, ret)                                                                       \
    do {                                                                                       \
        cudaError_t e__ = (call);                                                              \
        if (e__ != cudaSuccess) {                                                              \
            set_last_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return ret;                                                                        \
        }                                                                                      \
    } while (0)

/* an owned device array of T; moves, never copies, and frees itself */
template <typename T = uint8_t> struct DevBuf {
    T *p = nullptr;
    DevBuf() = default;
    explicit DevBuf(size_t n) { alloc(n); }
    ~DevBuf() { cudaFree(p); }
    DevBuf(DevBuf &&o) noexcept : p(o.p) { o.p = nullptr; }
    DevBuf &operator=(DevBuf &&o) noexcept {
        if (this != &o) { cudaFree(p); p = o.p; o.p = nullptr; }
        return *this;
    }
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    void reset() { cudaFree(p); p = nullptr; }
    /* replaces the array by n (at least one) fresh elements; false, empty and the reason in the last error when that fails */
    bool alloc(size_t n) {
        reset();
        const cudaError_t e = cudaMalloc(&p, (n ? n : 1) * sizeof(T));
        if (e == cudaSuccess) return true;
        p = nullptr;
        set_last_error("cudaMalloc of %zu bytes failed: %s", (n ? n : 1) * sizeof(T), cudaGetErrorString(e));
        return false;
    }
};

bool first_time_on_device(unsigned long long *mask) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev > 63) return true;
    if ((*mask >> dev) & 1ull) return false;
    *mask |= 1ull << dev;
    return true;
}

/* ---- process-wide device state (reference: g_nna_dev, src/device.c:105-131) -- */
static int g_strict = -1; /* -1: MARS_STRICT from the environment; 1: a failed tensor-core plan is an error, not a silent drop to the direct kernels */
static bool strict_mode() {
    if (g_strict < 0) { const char *e = getenv("MARS_STRICT"); g_strict = (e && atoi(e) != 0) ? 1 : 0; }
    return g_strict != 0;
}
static int g_device = -1;
static bool g_ready = false;
static size_t g_arena_bytes = 0;
struct Model;
static Model *g_last_model = nullptr;

static int pick_device() {
    if (g_device >= 0) return g_device;
    const char *e = getenv("MARS_DEVICE");
    if (e && *e) return atoi(e);
    e = getenv("LOCAL_RANK"); /* one process per GPU under torchrun */
    if (e && *e) {
        int n = 0;
        if (cudaGetDeviceCount(&n) == cudaSuccess && n > 0) return atoi(e) % n;
    }
    return 0;
}

static int device_up() {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        set_last_error("no CUDA device: %s (this library has no CPU fallback)", cudaGetErrorString(e));
        return NNA_ERROR_DEVICE;
    }
    int d = pick_device();
    if (d >= n) {
        set_last_error("device ordinal %d out of range (%d visible)", d, n);
        return NNA_ERROR_DEVICE;
    }
    e = cudaSetDevice(d);
    if (e != cudaSuccess) {
        set_last_error("cudaSetDevice(%d): %s", d, cudaGetErrorString(e));
        return NNA_ERROR_DEVICE;
    }
    g_device = d;
    g_ready = true;
    return NNA_SUCCESS;
}

/* ---- helpers shared with program.cpp ---------------------------------------- */
/* reference src/mars/mars_runtime.c:80-124: byte size by dtype AND format tag */
size_t tensor_byte_size(const mars_tensor_t *t) {
    size_t es;
    switch (t->dtype) {
        case MARS_DTYPE_FLOAT32: case MARS_DTYPE_INT32: es = 4; break;
        case MARS_DTYPE_INT16: es = 2; break;
        default: es = 1;
    }
    if (t->format == MARS_FORMAT_NDHWC32 && t->ndims >= 4) {
        int c32 = (t->shape[1] + 31) / 32;
        return (size_t)(t->shape[0] * c32 * t->shape[2] * t->shape[3] * 32) * es;
    }
    if (t->format == MARS_FORMAT_NMHWSOIB2 && t->ndims >= 4) {
        int no = (t->shape[0] + 31) / 32, mi = (t->shape[1] + 31) / 32;
        return (size_t)(no * mi * t->shape[2] * t->shape[3] * 1024);
    }
    size_t numel = 1;
    for (uint32_t i = 0; i < t->ndims && i < MARS_MAX_DIMS; i++) numel *= (size_t)t->shape[i];
    if (t->dtype == MARS_DTYPE_UINT4) return (numel + 1) / 2;
    return numel * es;
}

/* reference src/mars/mars_runtime.c:713-721: first table entry with a matching id */
int find_tensor(const mars_header_t &h, const mars_runtime_tensor_t *tensors, uint32_t id) {
    if (id == 0xFFFFFFFFu) return -1;
    for (uint32_t i = 0; i < h.num_tensors; i++)
        if (tensors[i].desc.id == id) return (int)i;
    return -1;
}

/* ---- the private model object ------------------------------------------------ */
static const uint32_t MODEL_TAG = 0x4232304Du; /* "M02B" */

/* CAP records and one count per image slot */
template <typename R, int CAP = MARS_MAX_DETS> struct RecordSet {
    DevBuf<R> rec;
    DevBuf<int32_t> cnt;
    bool alloc(int slots) { return rec.alloc((size_t)slots * CAP) && cnt.alloc((size_t)slots); }
    R *at(int slot) const { return rec.p + (size_t)slot * CAP; }
};

/* the per-slot device state besides the slots themselves, (re)allocated together by set_capacity */
struct SlotRecords {
    RecordSet<mars_det_t> raw, det;      /* the output0 path: parsed candidates, kept detections */
    RecordSet<mars_box_t> box_raw, box;  /* the heads path: decoded candidates, kept corner boxes */
    RecordSet<mars_box_t> fbox;          /* frame records of the region merge (mars_b200_merge_rois_resident) */
    RecordSet<mars_b200_track_box_t, MARS_B200_MAX_TRACKS> trk; /* tracked boxes (mars_b200_track_resident) */
    DevBuf<mars_b200_zone_frame_t> zone; /* one zone record per slot, beside its tracked boxes (k_zones) */
    DevBuf<unsigned> nms_mask;           /* NMS_SCRATCH_WORDS per slot: suppression bit matrices */
    DevBuf<int2> frame;                  /* original frame size per slot (0 = none), for the letterbox inverse */
};

struct Model {
    mars_model_t pub; /* must stay first: applications hold &pub */
    uint32_t tag = MODEL_TAG;
    int device = 0;
    size_t arena_size = 0, weights_size = 0, buffer_size = 0, slot_bytes = 0, slot_stride = 0;
    int num_buffers = 0;
    std::vector<size_t> toff;
    uint8_t *h_arena = nullptr;  /* pinned host mirror of [weights | buf0 | buf1 | (buf2)] */
    DevBuf<> weights;
    DevBuf<> slots;
    int capacity = 0;
    DevBuf<> scratch;
    size_t scratch_stride = 0;
    DevBuf<> cpool;
    DevBuf<> tc_scratch;         /* padded / phase-split conv inputs, one region per image slot */
    size_t tc_scratch_stride = 0;
    DevBuf<> linked;             /* producer-written conv input copies (Program::linked_bytes per image), pads stay zero */
    size_t linked_stride = 0;
    Program prog;
    int opt_level = 3, depthwise_mode = 0;
    int f32_mode = 2; /* float32 convolutions: 0 = exact-order fp32 (bit-exact control), 1 = tf32, 2 = tf32x3 (conv_tf32.cu) */
    cudaStream_t stream = nullptr, h2d_stream = nullptr, d2h_stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    float last_ms = 0.0f;
    uint64_t launches = 0;
    /* asynchronous batches (mars_b200_submit_batch / wait_batch): one in flight per half of the slot pool */
    struct Pending { bool active = false; int n = 0, maxd = 0; int32_t *counts = nullptr; } pending[2];
    /* letterbox pre-processing (preproc.cuh): tap lists per (in, out) size of one axis -- camera sizes repeat, and the
     * downscale taps cost O(in x out) on the host -- the float rows of one launch, and staging for frames and descriptor
     * tables: one set per pool of the frames submit, one for the synchronous and device-frame calls (PRE_SYNC) */
    std::map<std::pair<int, int>, ResizeTaps> pre_taps;
    DevBuf<float> preH;
    size_t preH_cap = 0;
    struct PreStage {
        DevBuf<> frames, tab;    /* device frames, device table */
        uint8_t *h_tab = nullptr; /* pinned table */
        size_t frames_cap = 0, tab_cap = 0, h_cap = 0;
        cudaEvent_t ev = nullptr; /* the last upload from h_tab */
    } pre_stage[3];
    /* captured steps (mars_b200_step_resident): one CUDA graph per (first, n, threshold, with_detect) seen twice */
    struct StepGraph { int first, n, with_detect; uint32_t thresh_bits; int seen; cudaGraphExec_t exec; uint64_t launches; };
    std::vector<StepGraph> graphs;
    bool graphs_broken = false;
    SlotRecords rec; /* device-resident detections, boxes and frame sizes */
    /* detection heads (mars_b200_set_yolo_heads / mars_b200_set_gfl_heads) */
    HeadSet heads;
    DevBuf<DecodeTables> tab;
    float tab_scale = 0.0f;
    bool tab_valid = false;
    /* per-op profile (CUDA events around every op when enabled) */
    int profile = 0;
    std::vector<cudaEvent_t> prof_ev;
    std::vector<double> prof_ms;
    std::vector<uint64_t> prof_calls;
    bool prof_pending = false;
    /* tensor-core conv plans (conv_tc.cu) */
    std::vector<TcPlan> tc;
    bool compiled = false;
    uint64_t weights_hash = 0; /* FNV-1a of the host weight blob the compiled plans were built from */
    /* multi-object tracking (mars_b200_set_tracking, track.cuh): MARS_B200_MAX_TRACKS track slots and the counters per stream, the
     * parameters, and the device staging of mars_b200_track_boxes (in: stream table, counts, boxes; out: counts, records) */
    int track_streams = 0;
    mars_b200_track_params_t track_params = MARS_B200_TRACK_PARAMS_DEFAULT;
    DevBuf<TrackSlot> tracks;
    DevBuf<TrackMeta> track_meta;
    DevBuf<> track_in, track_out;
    size_t track_in_cap = 0, track_out_cap = 0;
    /* zones and counting lines (mars_b200_set_zones, zones.cuh): per tracker stream its geometry, the analytics state of its
     * tracks and its line totals, allocated by the first set_zones; which streams have geometry, and how many */
    DevBuf<ZoneGeom> zone_geom;
    DevBuf<ZoneTrack> zone_state;
    DevBuf<ZoneMeta> zone_meta;
    std::vector<uint8_t> zone_on;
    int zone_streams = 0;
};

static Model *as_model(mars_model_t *p) {
    if (!p) return nullptr;
    Model *m = reinterpret_cast<Model *>(p);
    return m->tag == MODEL_TAG ? m : nullptr;
}

static inline uint8_t *dev_addr(const Model *m, size_t off, int slot) {
    return off < m->weights_size ? m->weights.p + off : m->slots.p + (size_t)slot * m->slot_stride + (off - m->weights_size);
}

static uint64_t fnv1a(const uint8_t *p, size_t n) {
    uint64_t h = 1469598103934665603ull;
    for (size_t i = 0; i < n; i++) { h ^= p[i]; h *= 1099511628211ull; }
    return h;
}

static void release_graphs(Model *m) {
    for (auto &g : m->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    m->graphs.clear();
}

static void model_release(Model *m) {
    if (!m) return;
    cudaSetDevice(m->device);
    if (m->stream) cudaStreamSynchronize(m->stream);
    release_graphs(m);
    tc_release(m->tc);
    for (auto e : m->prof_ev) cudaEventDestroy(e);
    if (m->h_arena) cudaFreeHost(m->h_arena);
    if (m->ev0) cudaEventDestroy(m->ev0);
    if (m->ev1) cudaEventDestroy(m->ev1);
    for (int i = 0; i < 2; i++) {
        if (m->ev_in[i]) cudaEventDestroy(m->ev_in[i]);
        if (m->ev_done[i]) cudaEventDestroy(m->ev_done[i]);
        if (m->ev_out[i]) cudaEventDestroy(m->ev_out[i]);
    }
    for (auto &st : m->pre_stage) {
        if (st.ev) cudaEventSynchronize(st.ev);
        if (st.ev) cudaEventDestroy(st.ev);
        if (st.h_tab) cudaFreeHost(st.h_tab);
    }
    if (m->stream) cudaStreamDestroy(m->stream);
    if (m->h2d_stream) cudaStreamDestroy(m->h2d_stream);
    if (m->d2h_stream) cudaStreamDestroy(m->d2h_stream);
    free(m->pub.tensors);
    free(m->pub.layers);
    if (g_last_model == m) g_last_model = nullptr;
    m->tag = 0;
    delete m; /* frees the device buffers */
}

/* (re)allocate `capacity` image slots; the slots both capacities share keep their contents and frame sizes.  The new set is
 * complete before it replaces the old one: on failure the model keeps its slots */
static mars_error_t set_capacity(Model *m, int capacity) {
    if (capacity < 1) capacity = 1;
    if (capacity == m->capacity) return MARS_OK;
    const size_t c = (size_t)capacity, keep = (size_t)std::min(capacity, m->capacity);
    CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED);
    DevBuf<> slots, scratch;
    SlotRecords r;
    if (!slots.alloc(c * m->slot_stride) || (m->scratch_stride && !scratch.alloc(c * m->scratch_stride)) || !r.raw.alloc(capacity) ||
        !r.det.alloc(capacity) || !r.box_raw.alloc(capacity) || !r.box.alloc(capacity) || !r.fbox.alloc(capacity) ||
        !r.trk.alloc(capacity) || !r.zone.alloc(c) || !r.nms_mask.alloc(c * NMS_SCRATCH_WORDS) || !r.frame.alloc(c))
        return MARS_ERR_ALLOC_FAILED;
    CU_OK(cudaMemsetAsync(slots.p, 0, c * m->slot_stride, m->stream), MARS_ERR_ALLOC_FAILED);
    CU_OK(cudaMemsetAsync(r.frame.p, 0, c * sizeof(int2), m->stream), MARS_ERR_ALLOC_FAILED);
    CU_OK(cudaMemsetAsync(r.zone.p, 0, c * sizeof(mars_b200_zone_frame_t), m->stream), MARS_ERR_ALLOC_FAILED);
    for (int32_t *cnt : {r.raw.cnt.p, r.det.cnt.p, r.box_raw.cnt.p, r.box.cnt.p, r.fbox.cnt.p, r.trk.cnt.p})
        CU_OK(cudaMemsetAsync(cnt, 0, c * sizeof(int32_t), m->stream), MARS_ERR_ALLOC_FAILED);
    if (m->slots.p) {
        CU_OK(cudaMemcpyAsync(slots.p, m->slots.p, keep * m->slot_stride, cudaMemcpyDeviceToDevice, m->stream), MARS_ERR_ALLOC_FAILED);
        CU_OK(cudaMemcpyAsync(r.frame.p, m->rec.frame.p, keep * sizeof(int2), cudaMemcpyDeviceToDevice, m->stream), MARS_ERR_ALLOC_FAILED);
    }
    CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED);
    m->slots = std::move(slots);
    m->scratch = std::move(scratch);
    m->rec = std::move(r);
    m->capacity = capacity;
    m->pub.ddr_paddr = m->slots.p;
    for (uint32_t i = 0; i < m->pub.header.num_tensors; i++) m->pub.tensors[i].paddr = dev_addr(m, m->toff[i], 0);
    /* tensor maps embed slot addresses and the slot count */
    tc_release(m->tc);
    m->tc_scratch.reset();
    m->tc_scratch_stride = 0;
    m->linked.reset();
    m->linked_stride = 0;
    m->compiled = false;
    return MARS_OK;
}

static mars_error_t compile_model(Model *m) {
    if (m->compiled) return MARS_OK;
    release_graphs(m); /* kernel parameters (slot addresses, tensor maps, tables) are about to change */
    Program p;
    mars_error_t e = compile_program(m->pub.header, m->pub.tensors, m->pub.layers, m->toff, m->weights_size,
                                     m->arena_size, m->opt_level, m->depthwise_mode, &p, m->f32_mode, &m->heads);
    if (e != MARS_OK) return e;
    m->prog = std::move(p);
    if (!m->cpool.alloc(m->prog.const_pool.size())) return MARS_ERR_ALLOC_FAILED;
    CU_OK(cudaMemcpy(m->cpool.p, m->prog.const_pool.data(), m->prog.const_pool.size(), cudaMemcpyHostToDevice),
          MARS_ERR_ALLOC_FAILED);
    if (m->prog.scratch_bytes > m->scratch_stride) {
        m->scratch_stride = (m->prog.scratch_bytes + 255) & ~(size_t)255;
        if (!m->scratch.alloc((size_t)m->capacity * m->scratch_stride)) return MARS_ERR_ALLOC_FAILED;
    }
    tc_release(m->tc);
    m->tc.assign(m->prog.ops.size(), TcPlan());
    size_t need = 0;
    for (const Op &o : m->prog.ops) {
        if (o.impl == CONV_TC_NCHW) need = std::max(need, tc_scratch_need(o));
        if (o.impl == CONV_TC_F32) need = std::max(need, tf32_scratch_need(o, m->f32_mode));
    }
    need = (need + 1023) & ~(size_t)1023;
    if (need > m->tc_scratch_stride || (need && !m->tc_scratch.p)) {
        m->tc_scratch_stride = need;
        if (!m->tc_scratch.alloc((size_t)m->capacity * need)) return MARS_ERR_ALLOC_FAILED;
    }
    /* the link area is private to one compiled program: pads must be zero, so (re)allocate it zeroed every time */
    m->linked.reset();
    m->linked_stride = (m->prog.linked_bytes + 1023) & ~(size_t)1023;
    if (m->linked_stride) {
        if (!m->linked.alloc((size_t)m->capacity * m->linked_stride)) return MARS_ERR_ALLOC_FAILED;
        CU_OK(cudaMemset(m->linked.p, 0, (size_t)m->capacity * m->linked_stride), MARS_ERR_ALLOC_FAILED);
    }
    ArenaGeom g{m->weights.p, m->slots.p, m->weights_size, m->slot_stride, m->capacity, m->h_arena, m->prog.const_pool.data()};
    for (size_t i = 0; i < m->prog.ops.size(); i++) {
        Op &o = m->prog.ops[i];
        if (o.impl == CONV_TC_F32) { /* float32 layer on the tf32 tensor path; a failed plan simply stays on the exact kernel */
            if (!tf32_plan(o, g, m->f32_mode, m->tc_scratch.p, m->tc_scratch_stride, &m->tc[i])) {
                if (strict_mode()) {
                    char why[600];
                    snprintf(why, sizeof why, "%s", g_err);
                    set_last_error("strict mode: tf32 plan failed for layer %d (%s)", o.layer, why);
                    tc_release(m->tc);
                    return MARS_ERR_LAYER_FAILED;
                }
                o.impl = CONV_DIRECT;
            }
            continue;
        }
        if (o.impl != CONV_TC_NCHW) continue;
        const Op *consumer = o.nhwc_consumer >= 0 ? &m->prog.ops[o.nhwc_consumer] : nullptr;
        if (!tc_plan(o, g, m->tc_scratch.p, m->tc_scratch_stride, m->linked.p, m->linked_stride, consumer, &m->tc[i])) {
            /* a fused op cannot simply fall back (its followers were folded): recompile exact -- unless the caller asked
             * to be told (mars_b200_set_strict / MARS_STRICT=1): the direct kernels are ~100x slower */
            if (strict_mode()) {
                char why[600];
                snprintf(why, sizeof why, "%s", g_err);
                set_last_error("strict mode: tensor-core plan failed for layer %d (%s)", o.layer, why);
                tc_release(m->tc);
                return MARS_ERR_LAYER_FAILED;
            }
            fprintf(stderr, "mars_b200: tensor-core plan failed for layer %d (%s); using the direct CUDA kernels\n", o.layer, g_err);
            tc_release(m->tc);
            m->opt_level = 0;
            return compile_model(m);
        }
        o.rq = tc_rq(m->tc[i]);
    }
    m->prof_ms.assign(m->prog.ops.size(), 0.0);
    m->prof_calls.assign(m->prog.ops.size(), 0);
    m->weights_hash = fnv1a(m->h_arena, m->weights_size);
    /* tables, the zeroed link area and the repacked weights are complete before a (non-blocking) stream uses them */
    CU_OK(cudaDeviceSynchronize(), MARS_ERR_LAYER_FAILED);
    m->compiled = true;
    return MARS_OK;
}

/* ---- op launch ---------------------------------------------------------------- */
static KOp to_kop(const Op &o) {
    KOp k;
    k.kind = o.kind; k.mode = o.mode;
    k.in0 = o.in0; k.in1 = o.in1; k.in2 = o.in2; k.out = o.out; k.w = o.w; k.bias = o.bias;
    k.ic = o.ic; k.ih = o.ih; k.iw = o.iw; k.oc = o.oc; k.oh = o.oh; k.ow = o.ow;
    k.kh = o.kh; k.kw = o.kw; k.sh = o.sh; k.sw = o.sw; k.pt = o.pt; k.pl = o.pl;
    k.coff = o.coff;
    k.f0 = o.f0; k.f1 = o.f1; k.f2 = o.f2;
    k.n = o.n;
    k.lut = o.lut; k.post_relu = o.post_relu; k.post_lut = o.post_lut;
    k.pass_oc = 0; k.use_scratch = 0;
    k.out_s = o.fused_layers > 0 ? o.out_s : -1;
    k.out_z = (o.fused_layers > 0 && o.store_z) ? o.out_z : -1;
    k.lut_s = o.lut_s; k.lut_z = o.lut_z; k.store_y = o.store_y ? 1 : 0;
    /* int8 mul / add: |a * sa| <= 128 |sa| etc.; with everything finite and the scaled result below 2^30 neither the x86
     * overflow rule nor NaN handling of the reference's float -> int conversion can trigger */
    k.fast_bin = 0;
    if (o.kind == OP_MUL_I8 || o.kind == OP_ADD_I8) {
        const double a = 128.0 * fabs((double)o.f0), b = 128.0 * fabs((double)o.f1), inv = fabs((double)o.f2);
        const double top = (o.kind == OP_MUL_I8 ? a * b : a + b) * inv + 1.0;
        k.fast_bin = (std::isfinite(o.f0) && std::isfinite(o.f1) && std::isfinite(o.f2) && top < 1073741824.0 && a < 1e30 && b < 1e30) ? 1 : 0;
    }
    return k;
}

static inline unsigned blocks_for(uint64_t n, unsigned per) { return (unsigned)((n + per - 1) / per); }

static mars_error_t launch_op(Model *m, size_t op_index, int first, int n, bool full_pass) {
    const Op &o = m->prog.ops[op_index];
    if (o.mode >= 1000) {
        set_last_error("layer %d: %s", o.layer, o.note.c_str());
        return (mars_error_t)(-(o.mode - 1000));
    }
    if (o.kind == OP_NOP || n <= 0) return MARS_OK;
    if (o.kind == OP_YOLO_HEAD) {
        const int C = o.oc, P = o.oh * o.ow;
        k_head_decode<<<n, 256, 0, m->stream>>>(reinterpret_cast<const int8_t *>(dev_addr(m, (size_t)o.in0, first)), m->slot_stride, o.oh, o.ow,
                                                o.head_nc, o.head_nhwc ? 5 + o.head_nc : (5 + o.head_nc) * P, o.head_nhwc ? 1 : P,
                                                o.head_nhwc ? C : 1, reinterpret_cast<const float *>(m->cpool.p + o.lut), (float)o.sh,
                                                YOLO_LEVELS[o.head_level].anchors, o.f0, o.head_level > 0, m->rec.box_raw.at(first),
                                                m->rec.box_raw.cnt.p + first, MARS_MAX_DETS, HEAD_MAX_CAND);
        m->launches++;
        CU_OK(cudaGetLastError(), MARS_ERR_LAYER_FAILED);
        return MARS_OK;
    }
    if (o.kind == OP_GFL_HEAD) {
        k_gfl_decode<<<n, 256, 0, m->stream>>>(reinterpret_cast<const int8_t *>(dev_addr(m, (size_t)o.in0, first)), m->slot_stride, o.oh, o.ow,
                                               o.head_nc, o.head_reg_max, o.head_nhwc ? 1 : o.oh * o.ow, o.head_nhwc ? o.oc : 1,
                                               reinterpret_cast<const float *>(m->cpool.p + o.lut), (float)o.sh, o.f2, (float)o.iw, (float)o.ih,
                                               o.f0, o.head_level > 0, m->rec.box_raw.at(first), m->rec.box_raw.cnt.p + first,
                                               MARS_MAX_DETS, HEAD_MAX_CAND);
        m->launches++;
        CU_OK(cudaGetLastError(), MARS_ERR_LAYER_FAILED);
        return MARS_OK;
    }
    ArenaView v;
    v.wbase = m->weights.p;
    v.sbase = m->slots.p + (size_t)first * m->slot_stride;
    v.W = m->weights_size;
    v.slot_stride = m->slot_stride;
    v.cpool = m->cpool.p;
    v.scratch = m->scratch.p ? m->scratch.p + (size_t)first * m->scratch_stride : nullptr;
    v.scratch_stride = m->scratch_stride;
    KOp k = to_kop(o);
    cudaStream_t s = m->stream;
    const bool xl = o.xlat;
    const int is_conv = o.kind == OP_CONV_I8_NCHW || o.kind == OP_CONV_I8_NHWC || o.kind == OP_CONV_F32_NCHW || o.kind == OP_DW_I8;
    if (o.mode == EXEC_SERIAL) {
        if (xl) k_serial<true><<<n, 32, 0, s>>>(v, k); else k_serial<false><<<n, 32, 0, s>>>(v, k);
        m->launches++;
    } else if (is_conv) {
        const uint64_t P = (uint64_t)o.oh * o.ow;
        const int es = o.kind == OP_CONV_F32_NCHW ? 4 : 1;
        if (o.impl == CONV_TC_F32 && m->tc[op_index].f32) {
            if (!tf32_launch(m->tc[op_index], m->slots.p, first, n, s, &m->launches)) return MARS_ERR_LAYER_FAILED;
        } else if (o.impl == CONV_TC_NCHW && m->tc[op_index].i8) {
            if (!tc_launch(m->tc[op_index], m->slots.p, first, n, full_pass, s, &m->launches)) return MARS_ERR_LAYER_FAILED;
        } else if (o.mode == EXEC_PARALLEL) {
            if (o.kind == OP_CONV_I8_NCHW && !xl && fast_conv_nchw_ok(k)) {
                launch_fast_conv_nchw(v, k, n, s);
            } else if (o.kind == OP_DW_I8 && !xl && m->opt_level >= 1 && dw_nchw4_ok(v, k)) {
                k_dw_nchw4<<<dim3(blocks_for((uint64_t)o.oc * o.oh * (o.ow >> 2), 256), n), 256, 0, s>>>(v, k);
            } else {
                dim3 g(blocks_for(P * o.oc, 256), n);
                if (xl) k_conv_point<true><<<g, 256, 0, s>>>(v, k); else k_conv_point<false><<<g, 256, 0, s>>>(v, k);
            }
            m->launches++;
        } else if (o.mode == EXEC_OC_PASSES || o.mode == EXEC_OC_PASSES_SCRATCH) {
            dim3 g(blocks_for(P, 256), n);
            for (int oc = 0; oc < o.oc; oc++) {
                k.pass_oc = oc;
                k.use_scratch = o.mode == EXEC_OC_PASSES_SCRATCH;
                if (xl) k_conv_point<true><<<g, 256, 0, s>>>(v, k); else k_conv_point<false><<<g, 256, 0, s>>>(v, k);
                m->launches++;
                if (k.use_scratch) {
                    dim3 gc(blocks_for(P * es, 256), n);
                    k_pass_commit<<<gc, 256, 0, s>>>(v, k, es);
                    m->launches++;
                }
            }
        } else if (o.mode == EXEC_PIXEL_SERIAL && o.kind == OP_CONV_I8_NCHW && m->opt_level >= 1 && inplace_reg_ok(v, k)) {
            launch_inplace_reg(v, k, n, s);
            m->launches++;
        } else if (o.mode == EXEC_PIXEL_SERIAL && o.kind == OP_CONV_I8_NCHW && o.fused_layers > 0) {
            set_last_error("layer %d: fused in-place conv needs the register kernel", o.layer); /* the planner fuses only what inplace_reg_ok accepts */
            return MARS_ERR_LAYER_FAILED;
        } else if (o.mode == EXEC_PIXEL_SERIAL && o.kind == OP_CONV_I8_NCHW) {
            dim3 g(blocks_for(P, 128), n);
            const size_t smem = (size_t)o.ic * 128 + (size_t)o.oc * o.ic;
            static unsigned long long attr_set = 0;
            if (first_time_on_device(&attr_set)) cudaFuncSetAttribute(k_conv1x1_nchw_inplace, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            k_conv1x1_nchw_inplace<<<g, 128, smem, s>>>(v, k);
            m->launches++;
        } else if (o.mode == EXEC_PIXEL_SERIAL) {
            dim3 g(blocks_for(P, 128), n);
            if (xl) k_conv_nhwc_pixel_serial<true><<<g, 128, 0, s>>>(v, k); else k_conv_nhwc_pixel_serial<false><<<g, 128, 0, s>>>(v, k);
            m->launches++;
        }
    } else if (o.kind == OP_MAXPOOL || o.kind == OP_UPSAMPLE || o.kind == OP_CONCAT || o.kind == OP_CONCAT_PERIODIC) {
        uint64_t total = (o.kind == OP_CONCAT || o.kind == OP_CONCAT_PERIODIC) ? o.n : (uint64_t)o.oh * o.ow * o.ic;
        if (o.kind == OP_CONCAT_PERIODIC) {
            /* chunks of `coff` bytes depend on the previous chunk only through position j mod coff,
             * whose source bytes [0, coff) are never written: order-free (SURVEY C.4b) */
        }
        if (!xl && m->opt_level >= 1 && fast_spatial_ok(v, k)) {
            launch_fast_spatial(v, k, n, s);
        } else {
            dim3 g(blocks_for(total, 256), n);
            if (xl) k_spatial<true><<<g, 256, 0, s>>>(v, k); else k_spatial<false><<<g, 256, 0, s>>>(v, k);
        }
        m->launches++;
    } else {
        if (!xl && m->opt_level >= 1 && fast_flat_ok(v, k)) {
            launch_fast_flat(v, k, n, s);
        } else {
            dim3 g(blocks_for(o.n, 256), n);
            if (xl) k_flat<true><<<g, 256, 0, s>>>(v, k); else k_flat<false><<<g, 256, 0, s>>>(v, k);
        }
        m->launches++;
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_last_error("layer %d launch failed: %s", o.layer, cudaGetErrorString(e));
        return MARS_ERR_LAYER_FAILED;
    }
    return MARS_OK;
}

/* all ops (or the ops of one layer) over slots [first, first+n) on m->stream */
static mars_error_t enqueue_ops(Model *m, int first, int n, int only_layer) {
    mars_error_t e = compile_model(m);
    if (e != MARS_OK) return e;
    const size_t nops = m->prog.ops.size();
    if (m->profile && m->prof_ev.size() < nops + 1) {
        while (m->prof_ev.size() < nops + 1) {
            cudaEvent_t ev;
            CU_OK(cudaEventCreate(&ev), MARS_ERR_ALLOC_FAILED);
            m->prof_ev.push_back(ev);
        }
    }
    const bool prof = m->profile && only_layer < 0;
    for (size_t i = 0; i < nops; i++) {
        if (only_layer >= 0 && m->prog.ops[i].layer != only_layer) continue;
        if (prof) cudaEventRecord(m->prof_ev[i], m->stream);
        e = launch_op(m, i, first, n, only_layer < 0);
        if (e != MARS_OK) return e;
    }
    if (prof) {
        cudaEventRecord(m->prof_ev[nops], m->stream);
        m->prof_pending = true;
    }
    return MARS_OK;
}

/* after the stream was synchronised: fold the per-op event intervals of the last full pass */
static void profile_collect(Model *m) {
    if (!m->prof_pending) return;
    m->prof_pending = false;
    const size_t nops = m->prog.ops.size();
    for (size_t i = 0; i < nops; i++) {
        float ms = 0.0f;
        if (cudaEventElapsedTime(&ms, m->prof_ev[i], m->prof_ev[i + 1]) == cudaSuccess) {
            m->prof_ms[i] += ms;
            m->prof_calls[i]++;
        }
    }
}

/* the start of every model entry point: *m = the model behind the handle, made the current device */
static mars_error_t enter(mars_model_t *model, Model **m) {
    *m = as_model(model);
    if (!*m) return MARS_ERR_INVALID_FILE;
    CU_OK(cudaSetDevice((*m)->device), MARS_ERR_NNA_INIT_FAILED);
    return MARS_OK;
}
/* ... of an entry point that works on slots [first, first+n) */
static mars_error_t enter(mars_model_t *model, Model **m, int first, int n) {
    mars_error_t e = enter(model, m);
    if (e == MARS_OK && (first < 0 || n < 0 || first + n > (*m)->capacity)) {
        set_last_error("slots [%d,%d) outside the batch capacity %d (mars_b200_set_batch)", first, first + n, (*m)->capacity);
        e = MARS_ERR_INVALID_TENSOR;
    }
    return e;
}

static mars_error_t need_heads(Model *m, const char *what) {
    if (!m->heads.empty()) return MARS_OK;
    set_last_error("%s: no detection heads configured (mars_b200_set_yolo_heads / mars_b200_set_gfl_heads)", what);
    return MARS_ERR_INVALID_TENSOR;
}

/* a setting the compiled program depends on is about to change: wait for the work that uses it; the next call recompiles (and
 * drops the captured graphs) */
static void invalidate_program(Model *m) {
    cudaSetDevice(m->device);
    cudaStreamSynchronize(m->stream);
    m->compiled = false;
}

/* a synchronous call: enqueue() on the compute stream between ev0 and ev1, wait for it, and keep its device time as last_ms.
 * The stream is idle afterwards, so a pending per-op profile pass is complete and folded in. */
template <typename F> static mars_error_t timed_call(Model *m, const char *what, F enqueue) {
    cudaEventRecord(m->ev0, m->stream);
    mars_error_t e = enqueue();
    cudaEventRecord(m->ev1, m->stream);
    const cudaError_t ce = cudaStreamSynchronize(m->stream);
    if (e == MARS_OK && ce != cudaSuccess) {
        set_last_error("%s: %s", what, cudaGetErrorString(ce));
        e = MARS_ERR_LAYER_FAILED;
    }
    if (e == MARS_OK) { cudaEventElapsedTime(&m->last_ms, m->ev0, m->ev1); profile_collect(m); }
    return e;
}

/* ---- decode + NMS on the device ----------------------------------------------- */
/* reference src/mars/mars_yolo_test.c:84,92 -- host libm expf, one rounding per operation.  obj is the sigmoid table: :84 takes
 * expf(-v * scale) and the table expf(-(v * scale)); negation commutes with the rounded product, so expf sees the same bits */
static void build_decode_tables(float scale, DecodeTables *t) {
    build_sigmoid_table(scale, t->obj);
    for (int v = -128; v < 128; v++) {
        volatile float s = (float)v * scale;
        volatile float e2 = expf(-s);
        volatile float den2 = 1.0f + e2;
        t->den[v + 128] = den2;
    }
    volatile float e3 = expf(1e9f);
    volatile float d3 = 1.0f + e3;
    t->den[256] = d3;
}

static mars_error_t ensure_tables(Model *m, float scale) {
    if (m->tab_valid && memcmp(&m->tab_scale, &scale, 4) == 0) return MARS_OK;
    DecodeTables t;
    build_decode_tables(scale, &t);
    if (!m->tab.p && !m->tab.alloc(1)) return MARS_ERR_ALLOC_FAILED;
    CU_OK(cudaMemcpyAsync(m->tab.p, &t, sizeof t, cudaMemcpyHostToDevice, m->stream), MARS_ERR_LAYER_FAILED);
    CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED); /* t is a stack object */
    m->tab_scale = scale;
    m->tab_valid = true;
    return MARS_OK;
}

static mars_error_t enqueue_detect(Model *m, int first, int n, float thresh) {
    if (m->pub.header.num_outputs < 1) return MARS_ERR_INVALID_TENSOR;
    uint32_t oi = m->pub.header.output_tensor_ids[0];
    if (oi >= m->pub.header.num_tensors) return MARS_ERR_INVALID_TENSOR;
    const mars_tensor_t &d = m->pub.tensors[oi].desc;
    if (d.ndims < 3 || d.shape[2] != 85 || d.shape[1] <= 0 || m->toff[oi] < m->weights_size) {
        set_last_error("detect: output 0 is not an int8 [1,N,85] head (reference src/mars/mars_yolo_test.c:187)");
        return MARS_ERR_INVALID_TENSOR;
    }
    mars_error_t e = ensure_tables(m, d.scale);
    if (e != MARS_OK) return e;
    const int8_t *data = reinterpret_cast<const int8_t *>(dev_addr(m, m->toff[oi], first));
    k_parse_output<<<n, 256, 0, m->stream>>>(data, m->slot_stride, d.shape[1], d.scale, m->tab.p, m->rec.raw.at(first),
                                             m->rec.raw.cnt.p + first, 1000, MARS_MAX_DETS);
    CU_OK(launch_nms_center(m->rec.raw.at(first), m->rec.raw.cnt.p + first, m->rec.det.at(first),
                            m->rec.det.cnt.p + first, MARS_MAX_DETS, thresh, n, m->rec.nms_mask.p + (size_t)first * NMS_SCRATCH_WORDS, m->stream),
          MARS_ERR_LAYER_FAILED);
    m->launches += 3; /* parse, NMS sort, NMS suppression */
    CU_OK(cudaGetLastError(), MARS_ERR_LAYER_FAILED);
    return MARS_OK;
}

/* corner NMS + letterbox inverse over the candidates the program's OP_YOLO_HEAD / OP_GFL_HEAD ops left for slots [first, first+n) */
static mars_error_t enqueue_heads_nms(Model *m, int first, int n, float thresh) {
    const mars_tensor_t &in = m->pub.tensors[m->pub.header.input_tensor_ids[0]].desc; /* checked by the heads setters */
    const bool nhwc = in.format == MARS_FORMAT_NHWC;
    const int net_h = nhwc ? in.shape[1] : in.shape[2], net_w = nhwc ? in.shape[2] : in.shape[3];
    k_nms_corner_batch<<<n, NMSB_THREADS, 0, m->stream>>>(m->rec.box_raw.at(first), m->rec.box_raw.cnt.p + first,
                                                         m->rec.box.at(first), m->rec.box.cnt.p + first, MARS_MAX_DETS, thresh,
                                                         m->rec.nms_mask.p + (size_t)first * NMS_SCRATCH_WORDS, m->rec.frame.p + first, net_w, net_h);
    m->launches++;
    CU_OK(cudaGetLastError(), MARS_ERR_LAYER_FAILED);
    return MARS_OK;
}

static inline double now_us() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3;
}

/* a device buffer of at least `need` elements; growing waits for the compute stream, whose launches may still read the old one */
template <typename T> static bool pre_grow(Model *m, DevBuf<T> &b, size_t *cap, size_t need) {
    if (need <= *cap) return true;
    cudaStreamSynchronize(m->stream);
    *cap = 0;
    if (!b.alloc(need)) return false;
    *cap = need;
    return true;
}

/* kept records of slots [first, first+n) of a record set -> dets[n][maxd], counts[n] on stream s */
template <typename R, int CAP>
static mars_error_t copy_dets(const RecordSet<R, CAP> &rs, int first, int n, void *dets, int32_t *counts, int maxd, cudaStream_t s) {
    if (maxd > std::min(1000, CAP)) maxd = std::min(1000, CAP);
    if (maxd < 0) maxd = 0;
    CU_OK(cudaMemcpyAsync(counts, rs.cnt.p + first, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, s), MARS_ERR_LAYER_FAILED);
    if (maxd > 0)
        CU_OK(cudaMemcpy2DAsync(dets, (size_t)maxd * sizeof(R), rs.at(first), (size_t)CAP * sizeof(R), (size_t)maxd * sizeof(R),
                                (size_t)n, cudaMemcpyDeviceToHost, s), MARS_ERR_LAYER_FAILED);
    return MARS_OK;
}

template <typename R, int CAP>
static mars_error_t download_records(mars_model_t *model, RecordSet<R, CAP> SlotRecords::*set, int first, int n, R *dets, int32_t *counts,
                                     int maxd) {
    Model *m;
    mars_error_t e = dets && counts ? enter(model, &m, first, n) : MARS_ERR_INVALID_FILE;
    if (e == MARS_OK) e = copy_dets(m->rec.*set, first, n, dets, counts, maxd, m->stream);
    if (e != MARS_OK) return e;
    CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED);
    for (int i = 0; i < n; i++) if (counts[i] > maxd) counts[i] = maxd;
    return MARS_OK;
}

/* ---- multi-object tracking (track.cuh) ----------------------------------------------------------------------------------- */
static mars_error_t need_tracking(Model *m, const char *what) {
    if (m->track_streams > 0) return MARS_OK;
    set_last_error("%s: tracking is not set (mars_b200_set_tracking)", what);
    return MARS_ERR_INVALID_TENSOR;
}

/* tracking is set and the n entries of a call name streams of it, each at most once */
static mars_error_t check_streams(Model *m, const char *what, int n, const int32_t *streams) {
    mars_error_t e = need_tracking(m, what);
    if (e != MARS_OK) return e;
    if (n > 0 && !streams) { set_last_error("%s: no stream table", what); return MARS_ERR_INVALID_FILE; }
    std::vector<uint8_t> seen((size_t)m->track_streams, 0);
    for (int i = 0; i < n; i++) {
        const int s = streams[i];
        if (s < 0 || s >= m->track_streams) {
            set_last_error("%s: entry %d: stream %d outside [0, %d) (mars_b200_set_tracking)", what, i, s, m->track_streams);
            return MARS_ERR_INVALID_TENSOR;
        }
        if (seen[s]++) { set_last_error("%s: entry %d: stream %d named twice in one call", what, i, s); return MARS_ERR_INVALID_TENSOR; }
    }
    return MARS_OK;
}

/* the tracker on the compute stream: entry i = the detections at boxes + i * box_stride (counts[i]) as the next frame of stream
 * streams[i] (a device table), tracked boxes to out + i * out_stride and out_counts[i].  The zone analytics follow while any
 * stream has geometry, or always when with_zones; their records go to zones[i] (null: none) */
static mars_error_t enqueue_track(Model *m, const mars_box_t *boxes, const int32_t *counts, int box_stride, const int32_t *streams, int n,
                                  mars_b200_track_box_t *out, int32_t *out_counts, int out_stride, mars_b200_zone_frame_t *zones = nullptr,
                                  bool with_zones = false) {
    if (n <= 0) return MARS_OK;
    k_track<<<n, TRK_THREADS, 0, m->stream>>>(boxes, counts, box_stride, streams, m->tracks.p, m->track_meta.p, m->track_params, out,
                                             out_counts, out_stride);
    m->launches++;
    CU_OK(cudaGetLastError(), MARS_ERR_LAYER_FAILED);
    if (m->zone_streams > 0 || with_zones) {
        k_zones<<<n, ZN_THREADS, 0, m->stream>>>(streams, m->tracks.p, m->track_meta.p, out, out_counts, out_stride, m->zone_geom.p,
                                                m->zone_state.p, m->zone_meta.p, zones);
        m->launches++;
        CU_OK(cudaGetLastError(), MARS_ERR_LAYER_FAILED);
    }
    return MARS_OK;
}
} // namespace marsb200

using namespace marsb200;

/* ================================================================================ */
/* the reference API (include/mars_runtime.h)                                        */
/* ================================================================================ */
extern "C" {

/* reference src/mars/mars_runtime.c:58-76 */
const char *mars_get_error_string(mars_error_t err) {
    static const char *s[] = {"OK", "Invalid magic number", "Version mismatch", "Memory allocation failed",
                              "Invalid file format", "NNA initialization failed", "Layer execution failed",
                              "Invalid tensor", "Invalid layer"};
    int i = -(int)err;
    return (i >= 0 && i < 9) ? s[i] : "Unknown error";
}

/* The header, tensor and layer tables of a .mars blob, without touching a device.  MARS_ERR_INVALID_MAGIC,
 * MARS_ERR_VERSION_MISMATCH (*h holds the header), or MARS_ERR_INVALID_FILE when the blob is shorter than its header, its tables
 * or its weights: the reference would read past the buffer there. */
static mars_error_t parse_tables(const void *data, size_t size, mars_header_t *h, std::vector<mars_runtime_tensor_t> *tensors,
                                 std::vector<mars_runtime_layer_t> *layers) {
    if (!data || size < sizeof(mars_header_t)) return MARS_ERR_INVALID_FILE;
    memcpy(h, data, sizeof *h);
    if (h->magic != MARS_MAGIC) return MARS_ERR_INVALID_MAGIC;
    if (h->version_major != MARS_VERSION_MAJOR) return MARS_ERR_VERSION_MISMATCH;
    const size_t tables = sizeof *h + (size_t)h->num_tensors * sizeof(mars_tensor_t) + (size_t)h->num_layers * sizeof(mars_layer_t);
    if (size < tables || h->weights_offset > size || h->weights_size > size - h->weights_offset) {
        set_last_error("file truncated: %zu bytes, tables need %zu, weights [%llu,+%llu)", size, tables,
                       (unsigned long long)h->weights_offset, (unsigned long long)h->weights_size);
        return MARS_ERR_INVALID_FILE;
    }
    tensors->assign(h->num_tensors ? h->num_tensors : 1, mars_runtime_tensor_t());
    layers->assign(h->num_layers ? h->num_layers : 1, mars_runtime_layer_t());
    memset(tensors->data(), 0, tensors->size() * sizeof(mars_runtime_tensor_t));
    memset(layers->data(), 0, layers->size() * sizeof(mars_runtime_layer_t));
    const uint8_t *p = (const uint8_t *)data + sizeof *h;
    for (uint32_t i = 0; i < h->num_tensors; i++, p += sizeof(mars_tensor_t)) memcpy(&(*tensors)[i].desc, p, sizeof(mars_tensor_t));
    for (uint32_t i = 0; i < h->num_layers; i++, p += sizeof(mars_layer_t)) memcpy(&(*layers)[i].desc, p, sizeof(mars_layer_t));
    return MARS_OK;
}

/* The work-buffer planner of reference src/mars/mars_runtime.c:248-337 (SURVEY Appendix C.1) behind weights of
 * h.weights_size <= arena bytes, producing arena offsets: weight tensors point into the blob (:321-326), runtime tensors go
 * round-robin into *num_buffers work buffers of *buffer_size bytes (:316-334).  False when the buffers do not fit the arena. */
static bool plan_work_buffers(const mars_header_t &h, mars_runtime_tensor_t *tensors, size_t arena, size_t *num_buffers,
                              size_t *buffer_size, std::vector<size_t> *toff) {
    const size_t W = (size_t)h.weights_size, remaining = arena - W;
    size_t maxsz = 0;
    for (uint32_t i = 0; i < h.num_tensors; i++)
        if (tensors[i].desc.data_size == 0) maxsz = std::max(maxsz, (tensor_byte_size(&tensors[i].desc) + 63) & ~(size_t)63);
    size_t nb = 3, bs = maxsz;
    if (bs * nb > remaining) nb = 2;
    if (bs * nb > remaining) {
        bs = (remaining / 2) & ~(size_t)63;
        if (bs < 65536) return false;
    }
    toff->assign(h.num_tensors ? h.num_tensors : 1, 0);
    for (uint32_t i = 0, k = 0; i < h.num_tensors; i++) {
        mars_runtime_tensor_t &t = tensors[i];
        if (t.desc.data_size > 0) {
            (*toff)[i] = (size_t)t.desc.data_offset;
            t.alloc_size = (size_t)t.desc.data_size;
        } else {
            (*toff)[i] = W + (size_t)(k % nb) * bs;
            t.alloc_size = bs;
            k++;
        }
    }
    *num_buffers = nb;
    *buffer_size = bs;
    return true;
}

/* s -> dst, cut to cap - 1 bytes and NUL-terminated; returns the length of s */
static size_t copy_out(const std::string &s, char *dst, size_t cap) {
    if (dst && cap) {
        const size_t n = std::min(cap - 1, s.size());
        memcpy(dst, s.data(), n);
        dst[n] = 0;
    }
    return s.size();
}

/* The planner's decisions for a .mars blob without touching a device: parses the tables, lays the tensors out as mars_load_memory
 * does, compiles the layer table at `opt_level` and writes the op list (one line per op: kind, mode, kernel choice, fused /
 * linked / forwarded / elided streams) to dst.  Returns the length of the description (0 on error).  Host logic only -- the CPU
 * test suite checks fusion, concat trimming and forwarding through it. */
size_t mars_b200_plan_describe(const void *data, size_t size, size_t arena_bytes, int opt_level, char *dst, size_t cap) {
    mars_header_t h;
    std::vector<mars_runtime_tensor_t> tensors;
    std::vector<mars_runtime_layer_t> layers;
    if (parse_tables(data, size, &h, &tensors, &layers) != MARS_OK) return 0;
    const size_t arena = arena_bytes ? arena_bytes : (size_t)8 << 20;
    size_t nb, bs;
    std::vector<size_t> toff;
    if (h.weights_size > arena || !plan_work_buffers(h, tensors.data(), arena, &nb, &bs, &toff)) return 0;
    Program prog;
    if (compile_program(h, tensors.data(), layers.data(), toff, (size_t)h.weights_size, arena, opt_level, 0, &prog,
                        2 /* the library's default float32 mode: tf32x3 */) != MARS_OK)
        return 0;
    return copy_out(describe_program(prog), dst, cap);
}

/* The outputs of the three CONV2D layers of a YOLOv5 Detect block, stride 8 / 16 / 32, without touching a device */
int mars_b200_find_yolo_heads(const void *data, size_t size, uint32_t *tensor_ids, int cap) {
    mars_header_t h;
    std::vector<mars_runtime_tensor_t> tensors;
    std::vector<mars_runtime_layer_t> layers;
    if (parse_tables(data, size, &h, &tensors, &layers) != MARS_OK) return 0;
    return find_yolo_heads(h, tensors.data(), layers.data(), tensor_ids, cap);
}

/* The NanoDet GFL head convs, stride 8 / 16 / 32 (/ 64), without touching a device */
int mars_b200_find_gfl_heads(const void *data, size_t size, int nc, int reg_max, uint32_t *tensor_ids, int cap) {
    mars_header_t h;
    std::vector<mars_runtime_tensor_t> tensors;
    std::vector<mars_runtime_layer_t> layers;
    if (parse_tables(data, size, &h, &tensors, &layers) != MARS_OK) return 0;
    return find_gfl_heads(h, tensors.data(), layers.data(), nc, reg_max, tensor_ids, cap);
}

/* reference src/mars/mars_runtime.c:126-349 */
mars_error_t mars_load_memory(const void *data, size_t size, mars_model_t **out_model) {
    if (!out_model) return MARS_ERR_INVALID_FILE;
    mars_header_t h;
    std::vector<mars_runtime_tensor_t> tensors;
    std::vector<mars_runtime_layer_t> layers;
    const mars_error_t pe = parse_tables(data, size, &h, &tensors, &layers);
    if (pe == MARS_ERR_INVALID_MAGIC) fprintf(stderr, "Mars: Invalid magic 0x%08x (expected 0x%08x)\n", h.magic, MARS_MAGIC);
    if (pe == MARS_ERR_VERSION_MISMATCH)
        fprintf(stderr, "Mars: Version mismatch %d.%d (expected %d.x)\n", h.version_major, h.version_minor, MARS_VERSION_MAJOR);
    if (pe != MARS_OK) return pe;
    if (!g_ready && device_up() != NNA_SUCCESS) return MARS_ERR_NNA_INIT_FAILED;
    CU_OK(cudaSetDevice(g_device), MARS_ERR_NNA_INIT_FAILED);

    Model *m = new (std::nothrow) Model();
    if (!m) return MARS_ERR_ALLOC_FAILED;
    memset(&m->pub, 0, sizeof m->pub);
    m->device = g_device;
    { const char *e = getenv("MARS_F32_MODE"); if (e && *e) m->f32_mode = std::max(0, std::min(2, atoi(e))); }
    m->pub.header = h;
    m->pub.tensors = (mars_runtime_tensor_t *)calloc(tensors.size(), sizeof(mars_runtime_tensor_t));
    m->pub.layers = (mars_runtime_layer_t *)calloc(layers.size(), sizeof(mars_runtime_layer_t));
    if (!m->pub.tensors || !m->pub.layers) { model_release(m); return MARS_ERR_ALLOC_FAILED; }
    memcpy(m->pub.tensors, tensors.data(), tensors.size() * sizeof(mars_runtime_tensor_t));
    memcpy(m->pub.layers, layers.data(), layers.size() * sizeof(mars_runtime_layer_t));

    /* arena size: the reference's literal 8 MiB (:209) unless the application asked for more */
    size_t arena = g_arena_bytes;
    if (!arena) {
        const char *e = getenv("MARS_ARENA_BYTES");
        if (e && *e) arena = (size_t)strtoull(e, nullptr, 0);
    }
    if (!arena) arena = (size_t)8 << 20;
    m->arena_size = arena;
    m->weights_size = (size_t)h.weights_size;
    if (m->weights_size > arena) {
        fprintf(stderr, "Mars: Weights too large (%zu > %zu)\n", m->weights_size, arena);
        model_release(m);
        return MARS_ERR_ALLOC_FAILED;
    }
    size_t nb, bs;
    if (!plan_work_buffers(h, m->pub.tensors, arena, &nb, &bs, &m->toff)) {
        fprintf(stderr, "Mars: Not enough DDR for work buffers (set MARS_ARENA_BYTES / mars_b200_set_arena_bytes)\n");
        model_release(m);
        return MARS_ERR_ALLOC_FAILED;
    }
    m->num_buffers = (int)nb;
    m->buffer_size = bs;
    m->slot_bytes = nb * bs;
    m->slot_stride = (m->slot_bytes + 1023) & ~(size_t)1023;
    if (m->slot_stride == 0) m->slot_stride = 1024;

    if (cudaHostAlloc((void **)&m->h_arena, arena + 4096, cudaHostAllocDefault) != cudaSuccess) {
        set_last_error("pinned host mirror of %zu bytes: %s", arena, cudaGetErrorString(cudaGetLastError()));
        model_release(m);
        return MARS_ERR_ALLOC_FAILED;
    }
    memset(m->h_arena, 0, arena + 4096);
    memcpy(m->h_arena, (const uint8_t *)data + h.weights_offset, m->weights_size);
    /* 64 KiB of zeroed slack behind the weights keeps stray device reads mapped */
    if (!m->weights.alloc(m->weights_size + 65536) ||
        cudaMemset(m->weights.p, 0, m->weights_size + 65536) != cudaSuccess ||
        cudaMemcpy(m->weights.p, m->h_arena, m->weights_size, cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&m->h2d_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&m->d2h_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&m->ev0) != cudaSuccess || cudaEventCreate(&m->ev1) != cudaSuccess) {
        set_last_error("device setup: %s", cudaGetErrorString(cudaGetLastError()));
        model_release(m);
        return MARS_ERR_ALLOC_FAILED;
    }
    for (int i = 0; i < 2; i++) {
        cudaEventCreateWithFlags(&m->ev_in[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&m->ev_done[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&m->ev_out[i], cudaEventDisableTiming);
    }
    for (auto &st : m->pre_stage) cudaEventCreateWithFlags(&st.ev, cudaEventDisableTiming);

    for (uint32_t i = 0; i < h.num_tensors; i++) {
        m->pub.tensors[i].vaddr = m->toff[i] <= arena ? m->h_arena + m->toff[i] : nullptr;
        m->pub.tensors[i].is_external = false;
    }
    m->pub.ddr_base = m->h_arena;
    m->pub.ddr_size = arena;
    m->pub.oram_base = nullptr;
    m->pub.oram_paddr = nullptr;
    m->pub.oram_size = 0;
    m->pub.weights = m->h_arena;
    m->pub.weights_size = m->weights_size;

    /* An image slot must reach as far as any layer reads or writes.  In the reference an access behind the last work buffer
     * lands in unused arena (extents taken from another tensor or dtype, the reduced-buffer case); here it would land in the
     * next image's slot, so the slot is sized to the furthest access of a dry compile (it stays private and zero-initialised). */
    {
        Program dry;
        mars_error_t de = compile_program(m->pub.header, m->pub.tensors, m->pub.layers, m->toff, m->weights_size, m->arena_size, 0,
                                          m->depthwise_mode, &dry);
        if (de != MARS_OK) { model_release(m); return de; }
        if (dry.max_extent > m->weights_size + m->slot_bytes) {
            m->slot_bytes = dry.max_extent - m->weights_size;
            m->slot_stride = (m->slot_bytes + 1023) & ~(size_t)1023;
        }
    }
    mars_error_t e = set_capacity(m, 1);
    if (e == MARS_OK) e = compile_model(m);
    if (e != MARS_OK) { model_release(m); return e; }
    g_last_model = m;
    *out_model = &m->pub;
    return MARS_OK;
}

/* reference src/mars/mars_runtime.c:351-386 */
mars_error_t mars_load_file(const char *path, mars_model_t **model) {
    if (!path || !model) return MARS_ERR_INVALID_FILE;
    FILE *f = fopen(path, "rb");
    if (!f) {
        fprintf(stderr, "Mars: Cannot open %s\n", path);
        return MARS_ERR_INVALID_FILE;
    }
    fseek(f, 0, SEEK_END);
    long sz = ftell(f);
    fseek(f, 0, SEEK_SET);
    if (sz <= 0) { fclose(f); return MARS_ERR_INVALID_FILE; }
    void *buf = malloc((size_t)sz);
    if (!buf) { fclose(f); return MARS_ERR_ALLOC_FAILED; }
    size_t got = fread(buf, 1, (size_t)sz, f);
    fclose(f);
    if (got != (size_t)sz) { free(buf); return MARS_ERR_INVALID_FILE; }
    mars_error_t e = mars_load_memory(buf, (size_t)sz, model);
    free(buf); /* the model owns a copy of the weights inside the arena (:384) */
    return e;
}

void mars_free(mars_model_t *model) { model_release(as_model(model)); }

/* reference src/mars/mars_runtime.c:395-411: the header ids are used as table indices */
mars_runtime_tensor_t *mars_get_input(mars_model_t *model, int index) {
    if (!model || index < 0 || (uint32_t)index >= model->header.num_inputs) return nullptr;
    uint32_t id = model->header.input_tensor_ids[index];
    return id < model->header.num_tensors ? &model->tensors[id] : nullptr;
}
mars_runtime_tensor_t *mars_get_output(mars_model_t *model, int index) {
    if (!model || index < 0 || (uint32_t)index >= model->header.num_outputs) return nullptr;
    uint32_t id = model->header.output_tensor_ids[index];
    return id < model->header.num_tensors ? &model->tensors[id] : nullptr;
}
int mars_get_num_inputs(mars_model_t *model) { return model ? (int)model->header.num_inputs : 0; }
int mars_get_num_outputs(mars_model_t *model) { return model ? (int)model->header.num_outputs : 0; }

/* reference src/mars/mars_runtime.c:421-434 */
void mars_print_summary(mars_model_t *model) {
    if (!model) return;
    Model *m = as_model(model);
    printf("Mars Model Summary:\n");
    printf("  Layers: %u\n", model->header.num_layers);
    printf("  Tensors: %u\n", model->header.num_tensors);
    printf("  Inputs: %u\n", model->header.num_inputs);
    printf("  Outputs: %u\n", model->header.num_outputs);
    printf("  Weights: %zu bytes\n", model->weights_size);
    printf("  DDR: %zu bytes @ %p\n", model->ddr_size, model->ddr_base);
    if (m) printf("  B200: device %d, %d work buffers x %zu bytes, %d image slot(s), %zu device ops\n", m->device,
                  m->num_buffers, m->buffer_size, m->capacity, m->prog.ops.size());
}

/* the host mirror's work buffers <-> slot 0 on the compute stream: those holding the model's inputs (or outputs), each once,
 * or with MARS_MIRROR=full the whole slot */
static mars_error_t mirror_work_buffers(Model *m, bool outputs) {
    static int full_mirror = -1;
    if (full_mirror < 0) { const char *e = getenv("MARS_MIRROR"); full_mirror = (e && !strcmp(e, "full")) ? 1 : 0; }
    const mars_header_t &h = m->pub.header;
    const cudaMemcpyKind kind = outputs ? cudaMemcpyDeviceToHost : cudaMemcpyHostToDevice;
    uint8_t *host = m->h_arena + m->weights_size, *dev = m->slots.p;
    if (full_mirror) {
        CU_OK(cudaMemcpyAsync(outputs ? host : dev, outputs ? dev : host, m->slot_bytes, kind, m->stream), MARS_ERR_LAYER_FAILED);
        return MARS_OK;
    }
    bool done[3] = {false, false, false};
    for (uint32_t i = 0; i < (outputs ? h.num_outputs : h.num_inputs) && i < 4; i++) {
        const uint32_t ti = outputs ? h.output_tensor_ids[i] : h.input_tensor_ids[i];
        if (ti >= h.num_tensors || m->toff[ti] < m->weights_size) continue;
        const size_t b = (m->toff[ti] - m->weights_size) / m->buffer_size, off = b * m->buffer_size;
        if (b < 3 && !done[b]) {
            done[b] = true;
            CU_OK(cudaMemcpyAsync(outputs ? host + off : dev + off, outputs ? dev + off : host + off, m->buffer_size, kind, m->stream),
                  MARS_ERR_LAYER_FAILED);
        }
    }
    return MARS_OK;
}

/* reference src/mars/mars_runtime.c:439-459: synchronous, one image */
mars_error_t mars_run(mars_model_t *model) {
    Model *m;
    mars_error_t e = enter(model, &m);
    if (e != MARS_OK) return e;
    double t0 = now_us();
    e = mirror_work_buffers(m, false);
    if (e != MARS_OK) return e;
    e = enqueue_ops(m, 0, 1, -1);
    if (e != MARS_OK) { cudaStreamSynchronize(m->stream); return e; }
    e = mirror_work_buffers(m, true);
    if (e != MARS_OK) return e;
    cudaError_t ce = cudaStreamSynchronize(m->stream);
    if (ce != cudaSuccess) {
        set_last_error("mars_run: %s", cudaGetErrorString(ce));
        return MARS_ERR_LAYER_FAILED;
    }
    for (uint32_t i = 0; i < model->header.num_layers; i++) model->layers[i].is_executed = true;
    model->inference_count++;
    model->total_inference_us += (uint64_t)(now_us() - t0); /* the reference declares but never fills this */
    return MARS_OK;
}

/* ================================================================================ */
/* additive B200 entry points (include/mars_b200.h)                                  */
/* ================================================================================ */
const char *mars_b200_version(void) { return "mars-b200 0.1 (sm_100a)"; }
int mars_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return (int)MARS_ERR_NNA_INIT_FAILED;
    return n;
}
int mars_b200_set_device(int ordinal) {
    g_device = ordinal;
    g_ready = false;
    return device_up() == NNA_SUCCESS ? 0 : (int)MARS_ERR_NNA_INIT_FAILED;
}
void mars_b200_set_arena_bytes(size_t bytes) { g_arena_bytes = bytes; }
const char *mars_b200_last_error(void) { return g_err; }

mars_error_t mars_b200_arena_upload(mars_model_t *model, int slot) {
    Model *m;
    mars_error_t e = enter(model, &m, slot, 1);
    if (e != MARS_OK) return e;
    /* the host mirror of the weights is writable (model->weights, tensor->vaddr, as in the reference): the tensor-core plans
     * hold a repacked copy and requantisation bounds derived from the blob, so an edit invalidates the compiled program */
    if (m->compiled && fnv1a(m->h_arena, m->weights_size) != m->weights_hash) invalidate_program(m);
    CU_OK(cudaMemcpyAsync(m->weights.p, m->h_arena, m->weights_size, cudaMemcpyHostToDevice, m->stream), MARS_ERR_LAYER_FAILED);
    size_t nbytes = std::min(m->slot_bytes, m->arena_size - m->weights_size);
    CU_OK(cudaMemcpyAsync(m->slots.p + (size_t)slot * m->slot_stride, m->h_arena + m->weights_size, nbytes,
                          cudaMemcpyHostToDevice, m->stream), MARS_ERR_LAYER_FAILED);
    CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED);
    return compile_model(m);
}

mars_error_t mars_b200_arena_download(mars_model_t *model, int slot, void *host_dst, size_t bytes) {
    Model *m;
    mars_error_t e = enter(model, &m, slot, 1);
    if (e != MARS_OK) return e;
    uint8_t *dst = host_dst ? (uint8_t *)host_dst : m->h_arena;
    if (!host_dst || bytes > m->weights_size + m->slot_bytes) bytes = std::min(m->arena_size, m->weights_size + m->slot_bytes);
    size_t wb = std::min(bytes, m->weights_size);
    CU_OK(cudaMemcpyAsync(dst, m->weights.p, wb, cudaMemcpyDeviceToHost, m->stream), MARS_ERR_LAYER_FAILED);
    if (bytes > wb)
        CU_OK(cudaMemcpyAsync(dst + wb, m->slots.p + (size_t)slot * m->slot_stride, bytes - wb, cudaMemcpyDeviceToHost,
                              m->stream), MARS_ERR_LAYER_FAILED);
    CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED);
    return MARS_OK;
}

mars_error_t mars_b200_arena_clear(mars_model_t *model) {
    Model *m;
    mars_error_t e = enter(model, &m);
    if (e != MARS_OK) return e;
    CU_OK(cudaMemsetAsync(m->slots.p, 0, (size_t)m->capacity * m->slot_stride, m->stream), MARS_ERR_LAYER_FAILED);
    CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED);
    memset(m->h_arena + m->weights_size, 0, m->arena_size - m->weights_size);
    return MARS_OK;
}

mars_error_t mars_b200_run_layer(mars_model_t *model, uint32_t layer) {
    Model *m;
    mars_error_t e = enter(model, &m);
    if (e != MARS_OK) return e;
    if (layer >= model->header.num_layers) return MARS_ERR_INVALID_LAYER;
    e = enqueue_ops(m, 0, 1, (int)layer);
    cudaError_t ce = cudaStreamSynchronize(m->stream);
    if (e == MARS_OK && ce != cudaSuccess) {
        set_last_error("run_layer %u: %s", layer, cudaGetErrorString(ce));
        e = MARS_ERR_LAYER_FAILED;
    }
    return e;
}

size_t mars_b200_describe(mars_model_t *model, char *dst, size_t cap) {
    Model *m = as_model(model);
    if (!m) return 0;
    if (compile_model(m) != MARS_OK) return 0;
    return copy_out(describe_program(m->prog), dst, cap);
}

void mars_b200_set_opt_level(mars_model_t *model, int level) {
    Model *m = as_model(model);
    if (!m || m->opt_level == level) return;
    invalidate_program(m);
    m->opt_level = level;
}
void mars_b200_set_strict(int on) { g_strict = on ? 1 : 0; }

/* make `hs` the model's detection heads; recompiles (and drops the captured graphs) only when something changed */
static mars_error_t replace_heads(Model *m, HeadSet hs) {
    const HeadSet &o = m->heads;
    bool same = hs.kind == o.kind && hs.heads.size() == o.heads.size() &&
                (hs.empty() || (memcmp(&hs.conf, &o.conf, 4) == 0 && hs.reg_max == o.reg_max && hs.centre == o.centre));
    for (size_t k = 0; same && k < hs.heads.size(); k++) same = hs.heads[k].id == o.heads[k].id && hs.heads[k].nc == o.heads[k].nc;
    if (same) return MARS_OK;
    invalidate_program(m);
    m->heads = std::move(hs);
    return MARS_OK;
}

mars_error_t mars_b200_set_yolo_heads(mars_model_t *model, const uint32_t *tensor_ids, int n, float conf_thresh) {
    Model *m = as_model(model);
    if (!m) return MARS_ERR_INVALID_FILE;
    HeadSet hs;
    if (n != 0) {
        uint32_t found[3];
        if (!tensor_ids) {
            n = find_yolo_heads(m->pub.header, m->pub.tensors, m->pub.layers, found, 3);
            if (n == 0) { set_last_error("set_yolo_heads: the model has no YOLOv5 Detect head convolutions"); return MARS_ERR_INVALID_TENSOR; }
            tensor_ids = found;
        }
        mars_error_t e = resolve_yolo_heads(m->pub.header, m->pub.tensors, m->pub.layers, m->toff, m->weights_size, tensor_ids, n, &hs.heads);
        if (e != MARS_OK) return e;
        hs.kind = HEADS_YOLO;
        hs.conf = conf_thresh;
    }
    return replace_heads(m, std::move(hs));
}

mars_error_t mars_b200_set_gfl_heads(mars_model_t *model, const uint32_t *tensor_ids, int n, int nc, int reg_max, int centre, float conf_thresh) {
    Model *m = as_model(model);
    if (!m) return MARS_ERR_INVALID_FILE;
    HeadSet hs;
    if (n != 0) {
        mars_error_t e = check_gfl_params(nc, reg_max, centre, conf_thresh);
        if (e != MARS_OK) return e;
        uint32_t found[4];
        if (!tensor_ids) {
            n = find_gfl_heads(m->pub.header, m->pub.tensors, m->pub.layers, nc, reg_max, found, 4);
            if (n == 0) {
                set_last_error("set_gfl_heads: the model has no GFL head convolutions with %d + 4 * (%d + 1) channels at strides 8, 16, 32", nc, reg_max);
                return MARS_ERR_INVALID_TENSOR;
            }
            tensor_ids = found;
        }
        e = resolve_gfl_heads(m->pub.header, m->pub.tensors, m->pub.layers, m->toff, m->weights_size, tensor_ids, n, nc, reg_max, centre,
                              conf_thresh, &hs.heads);
        if (e != MARS_OK) return e;
        hs.kind = HEADS_GFL;
        hs.conf = conf_thresh;
        hs.reg_max = reg_max;
        hs.centre = centre;
    }
    return replace_heads(m, std::move(hs));
}

mars_error_t mars_b200_set_frame_size(mars_model_t *model, int first, int n, int w, int h) {
    Model *m;
    mars_error_t e = enter(model, &m, first, n);
    if (e != MARS_OK) return e;
    if (w < 0 || h < 0 || (w == 0) != (h == 0)) {
        set_last_error("set_frame_size: %d x %d is not a frame size (0 x 0 clears it)", w, h);
        return MARS_ERR_INVALID_TENSOR;
    }
    std::vector<int2> fr((size_t)n, make_int2(w, h));
    if (n > 0) CU_OK(cudaMemcpyAsync(m->rec.frame.p + first, fr.data(), (size_t)n * sizeof(int2), cudaMemcpyHostToDevice, m->stream), MARS_ERR_LAYER_FAILED);
    CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED);
    return MARS_OK;
}
void mars_b200_set_f32_mode(mars_model_t *model, int mode) {
    Model *m = as_model(model);
    if (!m || m->f32_mode == mode) return;
    invalidate_program(m);
    m->f32_mode = mode < 0 ? 0 : (mode > 2 ? 2 : mode);
}
void mars_b200_set_depthwise_mode(mars_model_t *model, int mode) {
    Model *m = as_model(model);
    if (!m || m->depthwise_mode == mode) return;
    invalidate_program(m);
    m->depthwise_mode = mode;
}

mars_error_t mars_b200_set_batch(mars_model_t *model, int capacity) {
    Model *m;
    mars_error_t e = enter(model, &m);
    if (e == MARS_OK) e = set_capacity(m, capacity);
    if (e == MARS_OK) e = compile_model(m);
    return e;
}
int mars_b200_get_batch(mars_model_t *model) {
    Model *m = as_model(model);
    return m ? m->capacity : 0;
}

static size_t io_bytes(mars_model_t *model, int output) {
    mars_runtime_tensor_t *t = output ? mars_get_output(model, 0) : mars_get_input(model, 0);
    if (!t) return 0;
    size_t n = 1;
    for (uint32_t i = 0; i < t->desc.ndims && i < MARS_MAX_DIMS; i++) n *= (size_t)(t->desc.shape[i] < 0 ? 0 : t->desc.shape[i]);
    size_t es = (t->desc.dtype == MARS_DTYPE_FLOAT32 || t->desc.dtype == MARS_DTYPE_INT32) ? 4 : (t->desc.dtype == MARS_DTYPE_INT16 ? 2 : 1);
    return n * es;
}
size_t mars_b200_input_bytes(mars_model_t *model) { return io_bytes(model, 0); }
size_t mars_b200_output_bytes(mars_model_t *model) { return io_bytes(model, 1); }

static mars_error_t copy_io(Model *m, int first, int n, void *host, size_t stride, int output, cudaStream_t s) {
    mars_model_t *model = &m->pub;
    uint32_t ti = output ? model->header.output_tensor_ids[0] : model->header.input_tensor_ids[0];
    if ((output ? model->header.num_outputs : model->header.num_inputs) < 1 || ti >= model->header.num_tensors ||
        m->toff[ti] < m->weights_size)
        return MARS_ERR_INVALID_TENSOR;
    size_t bytes = io_bytes(model, output);
    if (bytes > m->buffer_size) bytes = m->buffer_size;
    if (n == 0 || bytes == 0) return MARS_OK;
    if (stride < bytes) stride = bytes;
    uint8_t *dev = dev_addr(m, m->toff[ti], first);
    if (output)
        CU_OK(cudaMemcpy2DAsync(host, stride, dev, m->slot_stride, bytes, (size_t)n, cudaMemcpyDeviceToHost, s), MARS_ERR_LAYER_FAILED);
    else
        CU_OK(cudaMemcpy2DAsync(dev, m->slot_stride, host, stride, bytes, (size_t)n, cudaMemcpyHostToDevice, s), MARS_ERR_LAYER_FAILED);
    return MARS_OK;
}

mars_error_t mars_b200_upload_inputs(mars_model_t *model, int first, int n, const void *host, size_t stride) {
    Model *m;
    mars_error_t e = host ? enter(model, &m, first, n) : MARS_ERR_INVALID_FILE;
    if (e == MARS_OK) e = copy_io(m, first, n, const_cast<void *>(host), stride, 0, m->stream);
    if (e != MARS_OK) return e;
    CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED);
    return MARS_OK;
}
mars_error_t mars_b200_download_outputs(mars_model_t *model, int first, int n, void *host, size_t stride) {
    Model *m;
    mars_error_t e = host ? enter(model, &m, first, n) : MARS_ERR_INVALID_FILE;
    if (e == MARS_OK) e = copy_io(m, first, n, host, stride, 1, m->stream);
    if (e != MARS_OK) return e;
    CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED);
    return MARS_OK;
}

/* ---- letterbox pre-processing of ragged batches (preproc.cuh) ------------------------------------------------------ */
enum { PRE_SYNC = 2 }; /* pre_stage index of the synchronous and device-frame calls; 0 and 1 are the pools */
enum PreSource { PRE_HOST_SYNC, PRE_DEVICE, PRE_HOST_POOL };

/* the letterbox target: input tensor 0 of the slots, a 4-d int8 tensor (reference src/mars/mars_yolo_test.c:157-159) */
static mars_error_t pre_target(Model *m, const char *what, uint32_t *ti, int *tw, int *th, int *nhwc) {
    if (m->pub.header.num_inputs < 1) return MARS_ERR_INVALID_TENSOR;
    *ti = m->pub.header.input_tensor_ids[0];
    if (*ti >= m->pub.header.num_tensors || m->toff[*ti] < m->weights_size) return MARS_ERR_INVALID_TENSOR;
    const mars_tensor_t &d = m->pub.tensors[*ti].desc;
    if (d.dtype != MARS_DTYPE_INT8 || d.ndims < 4) {
        set_last_error("%s: input 0 must be a 4-d int8 tensor (reference src/mars/mars_yolo_test.c:157-159)", what);
        return MARS_ERR_INVALID_TENSOR;
    }
    *nhwc = d.format == MARS_FORMAT_NHWC;
    *th = *nhwc ? d.shape[1] : d.shape[2];
    *tw = *nhwc ? d.shape[2] : d.shape[3];
    if (*th <= 0 || *tw <= 0 || (size_t)*tw * *th * 3 > m->buffer_size) return MARS_ERR_INVALID_TENSOR;
    return MARS_OK;
}

/* One frame of a call, whichever public struct it arrived in: an RGB8 frame (p0) or the luma (p0) and chroma (p1) planes of
 * an NV12 frame, with their row pitches (0 in the public struct = tight rows, resolved here), the size, the format and the
 * NV12 colour variant.  Validation, staging and the letterbox launches see only this. */
struct FrameSrc {
    const uint8_t *p0, *p1;
    size_t pitch0, pitch1;
    int w, h, fmt, colour;
};
/* the public frame tables -> *s; null when there is no table */
static const std::vector<FrameSrc> *rgb_sources(int n, const mars_b200_frame_t *frames, std::vector<FrameSrc> *s) {
    if (!frames) return nullptr;
    s->resize(n > 0 ? n : 0);
    for (int f = 0; f < n; f++) {
        const mars_b200_frame_t &a = frames[f];
        (*s)[f] = FrameSrc{a.rgb, nullptr, a.row_stride ? a.row_stride : (size_t)a.w * 3, 0, a.w, a.h, PRE_RGB8, 0};
    }
    return s;
}
static const std::vector<FrameSrc> *nv12_sources(int n, const mars_b200_nv12_frame_t *frames, std::vector<FrameSrc> *s) {
    if (!frames) return nullptr;
    s->resize(n > 0 ? n : 0);
    for (int f = 0; f < n; f++) {
        const mars_b200_nv12_frame_t &a = frames[f];
        (*s)[f] = FrameSrc{a.y, a.uv, a.y_stride ? a.y_stride : (size_t)a.w, a.uv_stride ? a.uv_stride : (size_t)2 * ((a.w + 1) / 2),
                           a.w, a.h, PRE_NV12, a.colour};
    }
    return s;
}

/* every frame of a call is checked before any device work, so that a rejected call writes no slot */
static mars_error_t pre_check_frames(Model *m, const char *what, const std::vector<FrameSrc> *table, int tw, int th, bool device,
                                     std::vector<LetterboxGeom> *g) {
    if (!table) { set_last_error("%s: no frame table", what); return MARS_ERR_INVALID_FILE; }
    const std::vector<FrameSrc> &frames = *table;
    const int n = (int)frames.size();
    g->resize(n);
    for (int f = 0; f < n; f++) {
        const FrameSrc &fr = frames[f];
        const bool nv12 = fr.fmt == PRE_NV12;
        const char *plane[2] = {nv12 ? "y" : "rgb", "uv"};
        const uint8_t *ptr[2] = {fr.p0, fr.p1};
        const int planes = nv12 ? 2 : 1;
        for (int p = 0; p < planes; p++)
            if (!ptr[p]) { set_last_error("%s: frame %d: %s is NULL", what, f, plane[p]); return MARS_ERR_INVALID_FILE; }
        if (fr.w <= 0 || fr.h <= 0) { set_last_error("%s: frame %d: %d x %d is not a frame size", what, f, fr.w, fr.h); return MARS_ERR_INVALID_TENSOR; }
        const size_t row0 = (size_t)fr.w * (nv12 ? 1 : 3), row1 = (size_t)2 * ((fr.w + 1) / 2);
        if (fr.pitch0 < row0) {
            set_last_error("%s: frame %d: %s %zu < %s = %zu", what, f, nv12 ? "y_stride" : "row_stride", fr.pitch0, nv12 ? "w" : "w * 3", row0);
            return MARS_ERR_INVALID_TENSOR;
        }
        if (nv12 && fr.pitch1 < row1) {
            set_last_error("%s: frame %d: uv_stride %zu < 2 * ceil(w / 2) = %zu", what, f, fr.pitch1, row1);
            return MARS_ERR_INVALID_TENSOR;
        }
        if (nv12 && (fr.colour < 0 || fr.colour >= PRE_YUV_VARIANTS)) {
            set_last_error("%s: frame %d: colour %d is not a MARS_B200_YUV_* variant", what, f, fr.colour);
            return MARS_ERR_INVALID_TENSOR;
        }
        const LetterboxGeom q = letterbox_geom(fr.w, fr.h, tw, th);
        if (q.nw <= 0 || q.nh <= 0 || q.nw > tw || q.nh > th) {
            set_last_error("%s: frame %d: cannot letterbox %dx%d into %dx%d", what, f, fr.w, fr.h, tw, th);
            return MARS_ERR_INVALID_TENSOR;
        }
        for (int p = 0; device && p < planes; p++) {
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, ptr[p]) != cudaSuccess ||
                (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) || at.device != m->device) {
                cudaGetLastError();
                set_last_error("%s: frame %d: %s is not device memory of device %d", what, f, plane[p], m->device);
                return MARS_ERR_INVALID_FILE;
            }
        }
        (*g)[f] = q;
    }
    return MARS_OK;
}

/* the region table of a call (mars_b200_roi_t) */
struct RoiList {
    int n;
    const mars_b200_roi_t *p;
};

/* Every region of a call is checked before any device work: frame in [0, n_frames) and not decreasing (the regions of a frame
 * are contiguous: that fixes the concatenation order of the merge), x, y >= 0, w, h > 0, inside its frame (when there is a frame
 * table), a letterbox at least one pixel wide and tall (when g is given: *g receives each region's geometry), and region r in
 * slot first + r within the batch capacity. */
static mars_error_t pre_check_rois(Model *m, const char *what, int first, int n_frames, const std::vector<FrameSrc> *frames, const RoiList &rois,
                                   int tw, int th, std::vector<LetterboxGeom> *g) {
    if (rois.n < 0 || (rois.n > 0 && !rois.p)) { set_last_error("%s: no region table for %d regions", what, rois.n); return MARS_ERR_INVALID_FILE; }
    if (first < 0 || first + rois.n > m->capacity) {
        const int r = first < 0 ? 0 : m->capacity - first;
        set_last_error("%s: region %d: slot %d outside the batch capacity %d (mars_b200_set_batch)", what, r, first + r, m->capacity);
        return MARS_ERR_INVALID_TENSOR;
    }
    if (g) g->resize(rois.n);
    for (int r = 0; r < rois.n; r++) {
        const mars_b200_roi_t &q = rois.p[r];
        if (q.frame < 0 || q.frame >= n_frames) {
            set_last_error("%s: region %d: frame %d outside [0, %d)", what, r, q.frame, n_frames);
            return MARS_ERR_INVALID_TENSOR;
        }
        if (r > 0 && q.frame < rois.p[r - 1].frame) {
            set_last_error("%s: region %d: frame %d after frame %d (the regions of a frame must be contiguous, frames ascending)", what, r,
                           q.frame, rois.p[r - 1].frame);
            return MARS_ERR_INVALID_TENSOR;
        }
        if (q.x < 0 || q.y < 0 || q.w <= 0 || q.h <= 0) {
            set_last_error("%s: region %d: %d x %d at (%d, %d) is not a region", what, r, q.w, q.h, q.x, q.y);
            return MARS_ERR_INVALID_TENSOR;
        }
        if (frames) {
            const FrameSrc &a = (*frames)[q.frame];
            if ((long long)q.x + q.w > a.w || (long long)q.y + q.h > a.h) {
                set_last_error("%s: region %d: %d x %d at (%d, %d) reaches past frame %d (%d x %d)", what, r, q.w, q.h, q.x, q.y, q.frame, a.w, a.h);
                return MARS_ERR_INVALID_TENSOR;
            }
        }
        if (g) {
            const LetterboxGeom lg = letterbox_geom(q.w, q.h, tw, th);
            if (lg.nw <= 0 || lg.nh <= 0 || lg.nw > tw || lg.nh > th) {
                set_last_error("%s: region %d: cannot letterbox %dx%d into %dx%d", what, r, q.w, q.h, tw, th);
                return MARS_ERR_INVALID_TENSOR;
            }
            (*g)[r] = lg;
        }
    }
    return MARS_OK;
}

/* the merge table of k_merge_rois for validated regions: the first region of each frame (n_frames + 1 entries), then (x, y) of
 * each region */
static void merge_table(int n_frames, const RoiList &rois, std::vector<int> *tab) {
    tab->assign((size_t)n_frames + 1 + 2 * (size_t)rois.n, 0);
    for (int f = 0, r = 0; f <= n_frames; f++) {
        while (r < rois.n && rois.p[r].frame < f) r++;
        (*tab)[f] = r;
    }
    for (int r = 0; r < rois.n; r++) {
        (*tab)[n_frames + 1 + 2 * r] = rois.p[r].x;
        (*tab)[n_frames + 2 + 2 * r] = rois.p[r].y;
    }
}

static const ResizeTaps &cached_taps(Model *m, int in, int out) {
    const auto key = std::make_pair(in, out);
    auto it = m->pre_taps.find(key);
    if (it != m->pre_taps.end()) return it->second;
    ResizeTaps &t = m->pre_taps[key];
    build_resize_taps(in, out, &t);
    return t;
}

/* host frames [f0, f1) of a table -> their staging offsets, tight rows (pre_frame_bytes): one copy per RGB8 frame, one per NV12
 * plane.  RGB8 frames of one size with tight rows that sit equally spaced in host memory (mars_b200_preprocess_batch) go in
 * one copy. */
static cudaError_t pre_stage_frames(const PreTable &t, const FrameSrc *frames, int f0, int f1, uint8_t *d_stage, cudaStream_t s) {
    for (int f = f0; f < f1;) {
        const FrameSrc &a = frames[f];
        if (a.fmt == PRE_NV12) {
            const size_t row1 = (size_t)2 * ((a.w + 1) / 2);
            cudaError_t ce = cudaMemcpy2DAsync(d_stage + t.stage[f], (size_t)a.w, a.p0, a.pitch0, (size_t)a.w, (size_t)a.h, cudaMemcpyHostToDevice, s);
            if (ce == cudaSuccess)
                ce = cudaMemcpy2DAsync(d_stage + t.stage[f] + (size_t)a.w * a.h, row1, a.p1, a.pitch1, row1, (size_t)((a.h + 1) / 2),
                                       cudaMemcpyHostToDevice, s);
            if (ce != cudaSuccess) return ce;
            f++;
            continue;
        }
        const size_t row = (size_t)a.w * 3, pitch = a.pitch0, bytes = row * a.h;
        int e = f + 1;
        ptrdiff_t gap = 0;
        if (pitch == row && e < f1) {
            gap = frames[e].p0 - a.p0;
            while (e < f1 && gap >= (ptrdiff_t)bytes && frames[e].fmt == PRE_RGB8 && frames[e].w == a.w && frames[e].h == a.h &&
                   frames[e].pitch0 == row && frames[e].p0 - a.p0 == gap * (e - f) && t.stage[e] == t.stage[f] + bytes * (e - f))
                e++;
        }
        const cudaError_t ce = e > f + 1 ? cudaMemcpy2DAsync(d_stage + t.stage[f], bytes, a.p0, (size_t)gap, bytes, (size_t)(e - f), cudaMemcpyHostToDevice, s)
                                         : cudaMemcpy2DAsync(d_stage + t.stage[f], row, a.p0, pitch, row, (size_t)a.h, cudaMemcpyHostToDevice, s);
        if (ce != cudaSuccess) return ce;
        f = e;
    }
    return cudaSuccess;
}

/* the blob of t -> the stage's device table on stream s.  The pinned copy is rewritten only once the last upload from it has
 * completed; growing the device table waits for the compute stream (pre_grow). */
static mars_error_t pre_upload(Model *m, Model::PreStage &st, const PreTable &t, cudaStream_t s) {
    const size_t tab = t.bytes();
    if (!pre_grow(m, st.tab, &st.tab_cap, tab)) {
        set_last_error("preprocess: out of device memory for a %zu-byte table", tab);
        return MARS_ERR_ALLOC_FAILED;
    }
    CU_OK(cudaEventSynchronize(st.ev), MARS_ERR_LAYER_FAILED);
    if (tab > st.h_cap) {
        if (st.h_tab) cudaFreeHost(st.h_tab);
        st.h_tab = nullptr; st.h_cap = 0;
        CU_OK(cudaHostAlloc((void **)&st.h_tab, tab, cudaHostAllocDefault), MARS_ERR_ALLOC_FAILED);
        st.h_cap = tab;
    }
    t.pack(st.h_tab);
    CU_OK(cudaMemcpyAsync(st.tab.p, st.h_tab, tab, cudaMemcpyHostToDevice, s), MARS_ERR_LAYER_FAILED);
    CU_OK(cudaEventRecord(st.ev, s), MARS_ERR_LAYER_FAILED);
    return MARS_OK;
}

/* Letterboxes validated frames into input tensor ti of slots first, first+1, ... and records each slot's source size for the
 * letterbox inverse; the launches go on the compute stream.  Without rois slot first + f gets frame f (geometry g[f]); with
 * rois slot first + r gets region r (geometry g[r]) of frame rois[r].frame -- each frame staged once, whatever its number of
 * regions.  tail: an int table carried in the same upload (the region merge table, or the stream table of the tracker), whose
 * device address goes to *tail_dev.
 *   PRE_HOST_SYNC : host frames staged on the compute stream, launch by launch without regions (the caller synchronises);
 *   PRE_DEVICE    : device frames read in place;
 *   PRE_HOST_POOL : host frames and the table copied on the copy stream, then ev_in, which the compute stream waits for. */
static mars_error_t enqueue_letterbox(Model *m, Model::PreStage &st, int first, const std::vector<FrameSrc> &frames,
                                      const std::vector<LetterboxGeom> &g, uint32_t ti, int nhwc, PreSource how, cudaEvent_t ev_in,
                                      const RoiList *rois = nullptr, const std::vector<int> *tail = nullptr, const int **tail_dev = nullptr) {
    const int n = (int)g.size(), nfr = (int)frames.size();
    if (n == 0) return MARS_OK;
    if (m->pre_taps.size() > 64) m->pre_taps.clear();
    auto frame_of = [rois](int e) { return rois ? rois->p[e].frame : e; };
    std::vector<int> fmt(n);
    for (int e = 0; e < n; e++) fmt[e] = frames[frame_of(e)].fmt;
    PreTable t;
    pre_table_build(g.data(), fmt.data(), n, [m](int in, int out) -> const ResizeTaps & { return cached_taps(m, in, out); }, &t);
    std::vector<size_t> fbytes(nfr);
    for (int f = 0; f < nfr; f++) fbytes[f] = pre_frame_bytes(frames[f].fmt, frames[f].w, frames[f].h);
    const bool per_launch = how == PRE_HOST_SYNC && !rois;
    pre_table_stage(&t, fbytes.data(), nfr, per_launch);
    if (tail) t.merge = *tail;
    if ((how != PRE_DEVICE && !pre_grow(m, st.frames, &st.frames_cap, t.stage_bytes)) || !pre_grow(m, m->preH, &m->preH_cap, t.h_floats)) {
        set_last_error("preprocess: out of device memory for %d frames", n);
        return MARS_ERR_ALLOC_FAILED;
    }
    for (int e = 0; e < n; e++) {
        PreFrame &d = t.fr[e];
        const int f = frame_of(e);
        const FrameSrc &a = frames[f];
        const bool nv12 = a.fmt == PRE_NV12;
        d.colour = a.colour;
        if (rois) { d.ox = rois->p[e].x; d.oy = rois->p[e].y; }
        if (how == PRE_DEVICE) {
            d.src = a.p0; d.uv = a.p1;
            d.row_stride = a.pitch0; d.uv_stride = a.pitch1;
        } else { /* the tight staging layout of pre_stage_frames */
            d.src = st.frames.p + t.stage[f];
            d.row_stride = (size_t)a.w * (nv12 ? 1 : 3);
            d.uv = nv12 ? d.src + (size_t)a.w * a.h : nullptr;
            d.uv_stride = nv12 ? (size_t)2 * ((a.w + 1) / 2) : 0;
        }
    }
    cudaStream_t cs = how == PRE_HOST_POOL ? m->h2d_stream : m->stream;
    mars_error_t e = pre_upload(m, st, t, cs);
    if (e != MARS_OK) return e;
    if (tail_dev) *tail_dev = reinterpret_cast<const int *>(st.tab.p + t.merge_offset());
    if (how == PRE_HOST_POOL || (how == PRE_HOST_SYNC && !per_launch)) {
        CU_OK(pre_stage_frames(t, frames.data(), 0, nfr, st.frames.p, cs), MARS_ERR_LAYER_FAILED);
        if (how == PRE_HOST_POOL) {
            cudaEventRecord(ev_in, cs);
            cudaStreamWaitEvent(m->stream, ev_in, 0);
        }
    }
    int8_t *dst = reinterpret_cast<int8_t *>(dev_addr(m, m->toff[ti], first));
    for (size_t k = 0; k + 1 < t.first.size(); k++) {
        if (per_launch) CU_OK(pre_stage_frames(t, frames.data(), t.first[k], t.first[k + 1], st.frames.p, m->stream), MARS_ERR_LAYER_FAILED);
        CU_OK(launch_letterbox(t, (int)k, st.tab.p, m->preH.p, dst, m->slot_stride, nhwc, m->rec.frame.p + first, m->stream), MARS_ERR_LAYER_FAILED);
        m->launches += 2;
    }
    return MARS_OK;
}

/* the checks of a letterbox call after its slot range: the target, the frames and (with rois) the regions; *g receives the
 * geometry of each slot's source, frame or region */
static mars_error_t pre_validate(Model *m, const char *what, int first, const std::vector<FrameSrc> *frames, const RoiList *rois, bool device,
                                 uint32_t *ti, int *nhwc, std::vector<LetterboxGeom> *g) {
    int tw, th;
    mars_error_t e = pre_target(m, what, ti, &tw, &th, nhwc);
    if (e == MARS_OK) e = pre_check_frames(m, what, frames, tw, th, device, g);
    if (e == MARS_OK && rois) e = pre_check_rois(m, what, first, (int)frames->size(), frames, *rois, tw, th, g);
    return e;
}

/* The letterbox calls on the compute stream: host frames staged and letterboxed as one timed call (synchronous), or device
 * frames read in place (enqueued only).  rois: slot first + r gets region r of the n frames (the regions check their own slot
 * range). */
static mars_error_t preprocess(mars_model_t *model, const char *what, int first, int n, const std::vector<FrameSrc> *frames, PreSource how,
                               const RoiList *rois = nullptr) {
    Model *m;
    mars_error_t e = rois ? enter(model, &m) : enter(model, &m, first, n);
    if (e != MARS_OK) return e;
    uint32_t ti;
    int nhwc;
    std::vector<LetterboxGeom> g;
    e = pre_validate(m, what, first, frames, rois, how == PRE_DEVICE, &ti, &nhwc, &g);
    if (e != MARS_OK) return e;
    auto enqueue = [&] { return enqueue_letterbox(m, m->pre_stage[PRE_SYNC], first, *frames, g, ti, nhwc, how, nullptr, rois); };
    return how == PRE_DEVICE ? enqueue() : timed_call(m, what, enqueue);
}

/* Pre-processing in front of mars_run, as the reference's caller does it on the CPU (src/mars/mars_yolo_test.c:40-77 and
 * :157-165): n RGB8 frames of w x h pixels (host memory, frame_stride bytes apart, >= w*h*3) are letterboxed into input
 * tensor 0 of slots [first, first+n) -- stbir_resize_uint8 semantics, gray border -17, px - 128, NCHW or NHWC as the
 * tensor's format field says.  Synchronous like mars_b200_upload_inputs.  A table of identical frames on the ragged path. */
mars_error_t mars_b200_preprocess_batch(mars_model_t *model, int first, int n, const uint8_t *frames, size_t frame_stride, int w, int h) {
    Model *m = as_model(model);
    if (!m || !frames) return MARS_ERR_INVALID_FILE;
    if (w <= 0 || h <= 0) { set_last_error("preprocess: %d x %d is not a frame size", w, h); return MARS_ERR_INVALID_TENSOR; }
    const size_t frame_bytes = (size_t)(w > 0 ? w : 0) * (h > 0 ? h : 0) * 3;
    if (frame_stride < frame_bytes) frame_stride = frame_bytes;
    std::vector<FrameSrc> fr((size_t)(n > 0 ? n : 0));
    for (int f = 0; f < n; f++) fr[f] = FrameSrc{frames + (size_t)f * frame_stride, nullptr, (size_t)w * 3, 0, w, h, PRE_RGB8, 0};
    return preprocess(model, "preprocess", first, n, &fr, PRE_HOST_SYNC);
}

mars_error_t mars_b200_preprocess_frames(mars_model_t *model, int first, int n, const mars_b200_frame_t *frames) {
    std::vector<FrameSrc> s;
    return preprocess(model, "preprocess_frames", first, n, rgb_sources(n, frames, &s), PRE_HOST_SYNC);
}
mars_error_t mars_b200_preprocess_frames_nv12(mars_model_t *model, int first, int n, const mars_b200_nv12_frame_t *frames) {
    std::vector<FrameSrc> s;
    return preprocess(model, "preprocess_frames_nv12", first, n, nv12_sources(n, frames, &s), PRE_HOST_SYNC);
}

mars_error_t mars_b200_preprocess_frames_device(mars_model_t *model, int first, int n, const mars_b200_frame_t *frames) {
    std::vector<FrameSrc> s;
    return preprocess(model, "preprocess_frames_device", first, n, rgb_sources(n, frames, &s), PRE_DEVICE);
}
mars_error_t mars_b200_preprocess_frames_nv12_device(mars_model_t *model, int first, int n, const mars_b200_nv12_frame_t *frames) {
    std::vector<FrameSrc> s;
    return preprocess(model, "preprocess_frames_nv12_device", first, n, nv12_sources(n, frames, &s), PRE_DEVICE);
}

/* regions of frames (mars_b200_tile_rois) -> one slot each */
mars_error_t mars_b200_preprocess_rois(mars_model_t *model, int first, int n_frames, const mars_b200_frame_t *frames, int n_rois,
                                       const mars_b200_roi_t *rois) {
    std::vector<FrameSrc> s;
    const RoiList rl{n_rois, rois};
    return preprocess(model, "preprocess_rois", first, n_frames, rgb_sources(n_frames, frames, &s), PRE_HOST_SYNC, &rl);
}
mars_error_t mars_b200_preprocess_rois_nv12_device(mars_model_t *model, int first, int n_frames, const mars_b200_nv12_frame_t *frames,
                                                   int n_rois, const mars_b200_roi_t *rois) {
    std::vector<FrameSrc> s;
    const RoiList rl{n_rois, rois};
    return preprocess(model, "preprocess_rois_nv12_device", first, n_frames, nv12_sources(n_frames, frames, &s), PRE_DEVICE, &rl);
}

/* the region merge of frames [0, n_frames) of a call whose regions occupy slots [first, first + n_rois): tab = the merge table
 * on the device; the kept boxes of the step's corner NMS in, frame records first + f out */
static mars_error_t enqueue_merge(Model *m, int first, int n_frames, const int *tab, float thresh) {
    if (n_frames <= 0) return MARS_OK;
    k_merge_rois<<<n_frames, NMSB_THREADS, 0, m->stream>>>(m->rec.box.at(first), m->rec.box.cnt.p + first, MARS_MAX_DETS, tab,
                                                          n_frames, m->rec.fbox.at(first), m->rec.fbox.cnt.p + first, thresh,
                                                          m->rec.nms_mask.p + (size_t)first * NMS_SCRATCH_WORDS);
    m->launches++;
    CU_OK(cudaGetLastError(), MARS_ERR_LAYER_FAILED);
    return MARS_OK;
}

/* The merge reads the step's kept boxes and uses the suppression scratch rows of frame records [first, first + n_frames), free
 * once the step's own NMS has run (stream order).  Enqueued on the compute stream. */
mars_error_t mars_b200_merge_rois_resident(mars_model_t *model, int first, int n_frames, int n_rois, const mars_b200_roi_t *rois, float merge_thresh) {
    Model *m;
    mars_error_t e = enter(model, &m, first, n_frames);
    if (e != MARS_OK) return e;
    const RoiList rl{n_rois, rois};
    e = pre_check_rois(m, "merge_rois_resident", first, n_frames, nullptr, rl, 0, 0, nullptr);
    if (e != MARS_OK || n_frames == 0) return e;
    PreTable t;
    merge_table(n_frames, rl, &t.merge);
    Model::PreStage &st = m->pre_stage[PRE_SYNC];
    e = pre_upload(m, st, t, m->stream);
    if (e != MARS_OK) return e;
    return enqueue_merge(m, first, n_frames, reinterpret_cast<const int *>(st.tab.p), merge_thresh);
}

mars_error_t mars_b200_run_resident(mars_model_t *model, int first, int n) {
    Model *m;
    mars_error_t e = enter(model, &m, first, n);
    if (e != MARS_OK) return e;
    return timed_call(m, "run_resident", [&] { return enqueue_ops(m, first, n, -1); });
}

mars_error_t mars_b200_detect_resident(mars_model_t *model, int first, int n, float nms_thresh) {
    Model *m;
    mars_error_t e = enter(model, &m, first, n);
    if (e != MARS_OK) return e;
    return timed_call(m, "detect_resident", [&] { return enqueue_detect(m, first, n, nms_thresh); });
}

/* The ~110 launches of a step replayed as one CUDA graph: the second time a (first, n, threshold) combination is seen the
 * launch sequence is captured from the compute stream, afterwards it is replayed -- the kernels and their parameters are
 * the same, only the host-side launch work and the inter-kernel launch latency go.  MARS_GRAPH=0 disables it; profiling
 * (per-op events) and anything that cannot be captured fall back to plain launches. */
static bool graphs_enabled() {
    static const bool on = !(getenv("MARS_GRAPH") && atoi(getenv("MARS_GRAPH")) == 0);
    return on;
}

/* what follows the layers of a step; also the graph cache key */
enum StepFlavour : int { STEP_LAYERS = 0, STEP_DETECT = 1 /* parse_output of output0 + centre NMS */, STEP_HEADS = 2 /* corner NMS of the heads */ };

static mars_error_t enqueue_step(Model *m, int first, int n, float nms_thresh, int with_detect) {
    mars_error_t e = enqueue_ops(m, first, n, -1);
    if (e == MARS_OK && with_detect == STEP_DETECT) e = enqueue_detect(m, first, n, nms_thresh);
    if (e == MARS_OK && with_detect == STEP_HEADS) e = enqueue_heads_nms(m, first, n, nms_thresh);
    return e;
}

static mars_error_t enqueue_step_graphed(Model *m, int first, int n, float nms_thresh, int with_detect) {
    if (!graphs_enabled() || m->graphs_broken || m->profile || n <= 0) return enqueue_step(m, first, n, nms_thresh, with_detect);
    uint32_t tb;
    memcpy(&tb, &nms_thresh, 4);
    Model::StepGraph *g = nullptr;
    for (auto &c : m->graphs)
        if (c.first == first && c.n == n && c.with_detect == with_detect && c.thresh_bits == tb) g = &c;
    if (!g) {
        if (m->graphs.size() >= 16) release_graphs(m);
        m->graphs.push_back(Model::StepGraph{first, n, with_detect, tb, 0, nullptr, 0});
        g = &m->graphs.back();
    }
    if (g->exec) {
        if (cudaGraphLaunch(g->exec, m->stream) != cudaSuccess) { m->graphs_broken = true; return MARS_ERR_LAYER_FAILED; }
        m->launches += g->launches;
        return MARS_OK;
    }
    if (++g->seen < 2) return enqueue_step(m, first, n, nms_thresh, with_detect); /* first time: plain (also does the lazy one-time setup) */
    const uint64_t before = m->launches;
    cudaGraph_t graph = nullptr;
    if (cudaStreamBeginCapture(m->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
        m->graphs_broken = true;
        cudaGetLastError();
        return enqueue_step(m, first, n, nms_thresh, with_detect);
    }
    mars_error_t e = enqueue_step(m, first, n, nms_thresh, with_detect);
    const cudaError_t ce = cudaStreamEndCapture(m->stream, &graph);
    if (e != MARS_OK || ce != cudaSuccess || !graph || cudaGraphInstantiate(&g->exec, graph, 0) != cudaSuccess) {
        if (graph) cudaGraphDestroy(graph);
        g->exec = nullptr;
        m->graphs_broken = true;
        cudaGetLastError();
        m->launches = before;
        return e != MARS_OK ? e : enqueue_step(m, first, n, nms_thresh, with_detect);
    }
    cudaGraphDestroy(graph);
    g->launches = m->launches - before;
    if (cudaGraphLaunch(g->exec, m->stream) != cudaSuccess) { m->graphs_broken = true; return MARS_ERR_LAYER_FAILED; }
    return MARS_OK;
}

/* the step of slots [first, first+n), as one timed call (timed) or enqueued only */
static mars_error_t step_resident(mars_model_t *model, const char *what, int first, int n, float nms_thresh, int flavour, bool timed) {
    Model *m;
    mars_error_t e = enter(model, &m, first, n);
    if (e == MARS_OK && flavour == STEP_HEADS) e = need_heads(m, what);
    if (e == MARS_OK) e = compile_model(m);
    if (e != MARS_OK) return e;
    auto enqueue = [&] { return enqueue_step_graphed(m, first, n, nms_thresh, flavour); };
    return timed ? timed_call(m, what, enqueue) : enqueue();
}

/* run + detect as one timed region (the bench's resident step) */
mars_error_t mars_b200_step_resident(mars_model_t *model, int first, int n, float nms_thresh, int with_detect) {
    return step_resident(model, "step_resident", first, n, nms_thresh, with_detect ? STEP_DETECT : STEP_LAYERS, true);
}

/* the same step, enqueued only: the call returns as soon as the launches (one CUDA-graph replay from the second time on) are on the
 * model's compute stream; the caller orders its own work behind them there (mars_b200_compute_stream) and synchronises itself */
mars_error_t mars_b200_enqueue_step_resident(mars_model_t *model, int first, int n, float nms_thresh, int with_detect) {
    return step_resident(model, "enqueue_step_resident", first, n, nms_thresh, with_detect ? STEP_DETECT : STEP_LAYERS, false);
}

/* all layers (with the head decodes the program holds), corner NMS and the letterbox inverse as one timed region */
mars_error_t mars_b200_step_heads_resident(mars_model_t *model, int first, int n, float nms_thresh) {
    return step_resident(model, "step_heads_resident", first, n, nms_thresh, STEP_HEADS, true);
}
mars_error_t mars_b200_enqueue_step_heads_resident(mars_model_t *model, int first, int n, float nms_thresh) {
    return step_resident(model, "enqueue_step_heads_resident", first, n, nms_thresh, STEP_HEADS, false);
}

mars_error_t mars_b200_detect_heads_resident(mars_model_t *model, int first, int n, float nms_thresh) {
    Model *m;
    mars_error_t e = enter(model, &m, first, n);
    if (e == MARS_OK) e = need_heads(m, "detect_heads_resident");
    if (e == MARS_OK) e = compile_model(m);
    if (e != MARS_OK) return e;
    return timed_call(m, "detect_heads_resident", [&] { return enqueue_heads_nms(m, first, n, nms_thresh); });
}

mars_error_t mars_b200_download_detections(mars_model_t *model, int first, int n, mars_det_t *dets, int32_t *counts, int maxd) {
    return download_records(model, &SlotRecords::det, first, n, dets, counts, maxd);
}
mars_error_t mars_b200_download_boxes(mars_model_t *model, int first, int n, mars_box_t *boxes, int32_t *counts, int maxd) {
    return download_records(model, &SlotRecords::box, first, n, boxes, counts, maxd);
}
mars_error_t mars_b200_download_frame_boxes(mars_model_t *model, int first, int n, mars_box_t *boxes, int32_t *counts, int maxd) {
    return download_records(model, &SlotRecords::fbox, first, n, boxes, counts, maxd);
}

mars_error_t mars_b200_set_tracking(mars_model_t *model, int n_streams, const mars_b200_track_params_t *p) {
    Model *m;
    mars_error_t e = enter(model, &m);
    if (e != MARS_OK) return e;
    const mars_b200_track_params_t q = p ? *p : mars_b200_track_params_t MARS_B200_TRACK_PARAMS_DEFAULT;
    if (n_streams < 0 || n_streams > (1 << 20)) {
        set_last_error("set_tracking: %d streams (0 .. %d)", n_streams, 1 << 20);
        return MARS_ERR_INVALID_TENSOR;
    }
    const float th[6] = {q.high_thresh, q.low_thresh, q.new_thresh, q.sim_high, q.sim_low, q.sim_unconfirmed};
    bool ok = q.low_thresh >= 0.0f && q.low_thresh <= q.high_thresh && q.max_lost >= 0 && (q.class_aware == 0 || q.class_aware == 1);
    for (int i = 0; i < 6; i++) ok = ok && std::isfinite(th[i]) && (i < 3 || (th[i] >= 0.0f && th[i] < 1.0f));
    if (!ok) {
        set_last_error("set_tracking: parameters (high %g, low %g, new %g, gates %g %g %g, max_lost %d, class_aware %d) need finite "
                       "values, 0 <= low <= high, gates in [0, 1), max_lost >= 0, class_aware 0 or 1",
                       q.high_thresh, q.low_thresh, q.new_thresh, q.sim_high, q.sim_low, q.sim_unconfirmed, q.max_lost, q.class_aware);
        return MARS_ERR_INVALID_TENSOR;
    }
    CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED); /* the old tables may still be in use */
    DevBuf<TrackSlot> tracks;
    DevBuf<TrackMeta> meta;
    if (n_streams > 0) {
        if (!tracks.alloc((size_t)n_streams * MARS_B200_MAX_TRACKS) || !meta.alloc((size_t)n_streams)) return MARS_ERR_ALLOC_FAILED;
        CU_OK(cudaMemsetAsync(meta.p, 0, (size_t)n_streams * sizeof(TrackMeta), m->stream), MARS_ERR_ALLOC_FAILED);
        CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED);
    }
    m->tracks = std::move(tracks);
    m->track_meta = std::move(meta);
    m->track_streams = n_streams;
    m->track_params = q;
    m->zone_geom.reset();
    m->zone_state.reset();
    m->zone_meta.reset();
    m->zone_on.assign((size_t)n_streams, 0);
    m->zone_streams = 0;
    return MARS_OK;
}

mars_error_t mars_b200_reset_tracks(mars_model_t *model, int first_stream, int n) {
    Model *m;
    mars_error_t e = enter(model, &m);
    if (e == MARS_OK) e = need_tracking(m, "reset_tracks");
    if (e != MARS_OK) return e;
    if (first_stream < 0 || n < 0 || (long long)first_stream + n > m->track_streams) {
        set_last_error("reset_tracks: streams [%d, %lld) outside [0, %d)", first_stream, (long long)first_stream + n, m->track_streams);
        return MARS_ERR_INVALID_TENSOR;
    }
    if (n > 0) CU_OK(cudaMemsetAsync(m->track_meta.p + first_stream, 0, (size_t)n * sizeof(TrackMeta), m->stream), MARS_ERR_LAYER_FAILED);
    /* the track IDs start over, so the analytics state of these streams would name other tracks: it goes too, the geometry stays */
    if (n > 0 && m->zone_meta.p)
        CU_OK(cudaMemsetAsync(m->zone_meta.p + first_stream, 0, (size_t)n * sizeof(ZoneMeta), m->stream), MARS_ERR_LAYER_FAILED);
    return MARS_OK;
}

/* the stream table goes through the synchronous calls' pinned staging, as mars_b200_merge_rois_resident's merge table does */
mars_error_t mars_b200_track_resident(mars_model_t *model, int first, int n, const int32_t *streams) {
    Model *m;
    mars_error_t e = enter(model, &m, first, n);
    if (e == MARS_OK) e = check_streams(m, "track_resident", n, streams);
    if (e == MARS_OK) e = need_heads(m, "track_resident");
    if (e != MARS_OK || n == 0) return e;
    PreTable t;
    t.merge.assign(streams, streams + n);
    Model::PreStage &st = m->pre_stage[PRE_SYNC];
    e = pre_upload(m, st, t, m->stream);
    if (e != MARS_OK) return e;
    return enqueue_track(m, m->rec.box.at(first), m->rec.box.cnt.p + first, MARS_MAX_DETS, reinterpret_cast<const int32_t *>(st.tab.p), n,
                         m->rec.trk.at(first), m->rec.trk.cnt.p + first, MARS_B200_MAX_TRACKS, m->rec.zone.p + first);
}

mars_error_t mars_b200_download_tracks(mars_model_t *model, int first, int n, mars_b200_track_box_t *out, int32_t *counts, int maxd) {
    Model *m = as_model(model);
    if (m && need_tracking(m, "download_tracks") != MARS_OK) return MARS_ERR_INVALID_TENSOR;
    return download_records(model, &SlotRecords::trk, first, n, out, counts, maxd);
}

/* the checks of mars_b200_set_zones; the message names the zone or line and the field */
static bool zones_valid(const mars_b200_zone_t *zones, int n_zones, const mars_b200_line_t *lines, int n_lines) {
    auto anchor_ok = [](int a) { return a == MARS_B200_ANCHOR_BOTTOM || a == MARS_B200_ANCHOR_CENTRE; };
    for (int k = 0; k < n_zones; k++) {
        const mars_b200_zone_t &z = zones[k];
        if (z.n_verts < 3 || z.n_verts > MARS_B200_MAX_ZONE_VERTS) {
            set_last_error("set_zones: zone %d: n_verts %d (3 .. %d)", k, z.n_verts, MARS_B200_MAX_ZONE_VERTS);
            return false;
        }
        for (int i = 0; i < z.n_verts; i++)
            if (!std::isfinite(z.x[i]) || !std::isfinite(z.y[i])) {
                set_last_error("set_zones: zone %d: vertex %d (%g, %g) is not finite", k, i, z.x[i], z.y[i]);
                return false;
            }
        if (z.class_id < -1) { set_last_error("set_zones: zone %d: class_id %d (-1: any, or >= 0)", k, z.class_id); return false; }
        if (!anchor_ok(z.anchor)) { set_last_error("set_zones: zone %d: anchor %d (0 bottom, 1 centre)", k, z.anchor); return false; }
        if (z.min_dwell < 0) { set_last_error("set_zones: zone %d: min_dwell %d (>= 0)", k, z.min_dwell); return false; }
    }
    for (int k = 0; k < n_lines; k++) {
        const mars_b200_line_t &l = lines[k];
        if (!std::isfinite(l.x0) || !std::isfinite(l.y0) || !std::isfinite(l.x1) || !std::isfinite(l.y1)) {
            set_last_error("set_zones: line %d: ends (%g, %g) (%g, %g) are not finite", k, l.x0, l.y0, l.x1, l.y1);
            return false;
        }
        if (l.x0 == l.x1 && l.y0 == l.y1) { set_last_error("set_zones: line %d: ends coincide at (%g, %g)", k, l.x0, l.y0); return false; }
        if (l.class_id < -1) { set_last_error("set_zones: line %d: class_id %d (-1: any, or >= 0)", k, l.class_id); return false; }
        if (!anchor_ok(l.anchor)) { set_last_error("set_zones: line %d: anchor %d (0 bottom, 1 centre)", k, l.anchor); return false; }
    }
    return true;
}

mars_error_t mars_b200_set_zones(mars_model_t *model, int stream, const mars_b200_zone_t *zones, int n_zones, const mars_b200_line_t *lines,
                                 int n_lines) {
    Model *m;
    mars_error_t e = enter(model, &m);
    if (e == MARS_OK) e = need_tracking(m, "set_zones");
    if (e != MARS_OK) return e;
    if (stream < 0 || stream >= m->track_streams) {
        set_last_error("set_zones: stream %d outside [0, %d) (mars_b200_set_tracking)", stream, m->track_streams);
        return MARS_ERR_INVALID_TENSOR;
    }
    if (n_zones < 0 || n_zones > MARS_B200_MAX_ZONES || n_lines < 0 || n_lines > MARS_B200_MAX_LINES || (n_zones > 0 && !zones) ||
        (n_lines > 0 && !lines)) {
        set_last_error("set_zones: %d zones (0 .. %d) and %d lines (0 .. %d), each table present when its count is positive", n_zones,
                       MARS_B200_MAX_ZONES, n_lines, MARS_B200_MAX_LINES);
        return MARS_ERR_INVALID_TENSOR;
    }
    if (!zones_valid(zones, n_zones, lines, n_lines)) return MARS_ERR_INVALID_TENSOR;
    CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED); /* tracker calls in flight read the geometry and the state */
    if (!m->zone_geom.p) {
        const size_t ns = (size_t)m->track_streams;
        DevBuf<ZoneGeom> geom;
        DevBuf<ZoneTrack> state;
        DevBuf<ZoneMeta> meta;
        if (!geom.alloc(ns) || !state.alloc(ns * MARS_B200_MAX_TRACKS) || !meta.alloc(ns)) return MARS_ERR_ALLOC_FAILED;
        CU_OK(cudaMemsetAsync(geom.p, 0, ns * sizeof(ZoneGeom), m->stream), MARS_ERR_ALLOC_FAILED);
        CU_OK(cudaMemsetAsync(meta.p, 0, ns * sizeof(ZoneMeta), m->stream), MARS_ERR_ALLOC_FAILED);
        CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_ALLOC_FAILED);
        m->zone_geom = std::move(geom);
        m->zone_state = std::move(state);
        m->zone_meta = std::move(meta);
    }
    ZoneGeom g;
    memset(&g, 0, sizeof g);
    g.n_zones = n_zones;
    g.n_lines = n_lines;
    if (n_zones) memcpy(g.zone, zones, (size_t)n_zones * sizeof(mars_b200_zone_t));
    if (n_lines) memcpy(g.line, lines, (size_t)n_lines * sizeof(mars_b200_line_t));
    /* on the compute stream, so that the tracker calls that follow see the new geometry and the cleared state; g is a stack
     * object, so the call waits for the copy */
    CU_OK(cudaMemcpyAsync(m->zone_geom.p + stream, &g, sizeof g, cudaMemcpyHostToDevice, m->stream), MARS_ERR_LAYER_FAILED);
    CU_OK(cudaMemsetAsync(m->zone_meta.p + stream, 0, sizeof(ZoneMeta), m->stream), MARS_ERR_LAYER_FAILED);
    CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED);
    const uint8_t on = n_zones > 0 || n_lines > 0;
    m->zone_streams += (int)on - (int)m->zone_on[stream];
    m->zone_on[stream] = on;
    return MARS_OK;
}

mars_error_t mars_b200_download_zones(mars_model_t *model, int first, int n, mars_b200_zone_frame_t *out) {
    Model *m;
    mars_error_t e = out || n == 0 ? enter(model, &m, first, n) : MARS_ERR_INVALID_FILE;
    if (e == MARS_OK) e = need_tracking(m, "download_zones");
    if (e != MARS_OK || n == 0) return e;
    CU_OK(cudaMemcpyAsync(out, m->rec.zone.p + first, (size_t)n * sizeof(mars_b200_zone_frame_t), cudaMemcpyDeviceToHost, m->stream),
          MARS_ERR_LAYER_FAILED);
    CU_OK(cudaStreamSynchronize(m->stream), MARS_ERR_LAYER_FAILED);
    return MARS_OK;
}

mars_error_t mars_b200_track_boxes(mars_model_t *model, int n, const int32_t *streams, const mars_box_t *boxes, const int32_t *counts,
                                   int box_stride, mars_b200_track_box_t *out, int32_t *out_counts, int maxd) {
    return mars_b200_track_boxes_zones(model, n, streams, boxes, counts, box_stride, out, out_counts, maxd, nullptr);
}

mars_error_t mars_b200_track_boxes_zones(mars_model_t *model, int n, const int32_t *streams, const mars_box_t *boxes, const int32_t *counts,
                                         int box_stride, mars_b200_track_box_t *out, int32_t *out_counts, int maxd,
                                         mars_b200_zone_frame_t *zone_out) {
    Model *m;
    mars_error_t e = enter(model, &m);
    if (e == MARS_OK) e = check_streams(m, "track_boxes", n, streams);
    if (e != MARS_OK) return e;
    if (n < 0 || (n > 0 && (!counts || !out || !out_counts))) { set_last_error("track_boxes: no count or output table"); return MARS_ERR_INVALID_FILE; }
    int maxc = 1;
    for (int i = 0; i < n; i++) {
        if (counts[i] < 0 || counts[i] > TRK_MAX_DETS || counts[i] > box_stride || (counts[i] > 0 && !boxes)) {
            set_last_error("track_boxes: entry %d: %d boxes (0 .. min(box_stride %d, %d))", i, counts[i], box_stride, TRK_MAX_DETS);
            return MARS_ERR_INVALID_TENSOR;
        }
        maxc = std::max(maxc, (int)counts[i]);
    }
    if (n == 0) return MARS_OK;
    maxd = std::max(0, std::min(maxd, MARS_B200_MAX_TRACKS));
    /* in: [streams | counts | boxes n x maxc], out: [counts | records n x MARS_B200_MAX_TRACKS | (zone records n)], each part
     * 256-byte aligned */
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t ints = up((size_t)n * sizeof(int32_t)), in_bytes = 2 * ints + (size_t)n * maxc * sizeof(mars_box_t);
    const size_t rec_bytes = (size_t)n * MARS_B200_MAX_TRACKS * sizeof(mars_b200_track_box_t);
    const size_t out_bytes = ints + rec_bytes + (zone_out ? (size_t)n * sizeof(mars_b200_zone_frame_t) : 0);
    if (!pre_grow(m, m->track_in, &m->track_in_cap, in_bytes) || !pre_grow(m, m->track_out, &m->track_out_cap, out_bytes)) return MARS_ERR_ALLOC_FAILED;
    std::vector<uint8_t> blob(in_bytes, 0);
    memcpy(blob.data(), streams, (size_t)n * sizeof(int32_t));
    memcpy(blob.data() + ints, counts, (size_t)n * sizeof(int32_t));
    for (int i = 0; i < n; i++)
        memcpy(blob.data() + 2 * ints + (size_t)i * maxc * sizeof(mars_box_t), boxes + (size_t)i * box_stride, (size_t)counts[i] * sizeof(mars_box_t));
    const int32_t *d_streams = reinterpret_cast<const int32_t *>(m->track_in.p), *d_counts = reinterpret_cast<const int32_t *>(m->track_in.p + ints);
    const mars_box_t *d_boxes = reinterpret_cast<const mars_box_t *>(m->track_in.p + 2 * ints);
    int32_t *d_out_counts = reinterpret_cast<int32_t *>(m->track_out.p);
    mars_b200_track_box_t *d_out = reinterpret_cast<mars_b200_track_box_t *>(m->track_out.p + ints);
    mars_b200_zone_frame_t *d_zones = zone_out ? reinterpret_cast<mars_b200_zone_frame_t *>(m->track_out.p + ints + rec_bytes) : nullptr;
    e = timed_call(m, "track_boxes", [&]() -> mars_error_t {
        CU_OK(cudaMemcpyAsync(m->track_in.p, blob.data(), in_bytes, cudaMemcpyHostToDevice, m->stream), MARS_ERR_LAYER_FAILED);
        mars_error_t r = enqueue_track(m, d_boxes, d_counts, maxc, d_streams, n, d_out, d_out_counts, MARS_B200_MAX_TRACKS, d_zones,
                                       zone_out != nullptr);
        if (r != MARS_OK) return r;
        if (zone_out)
            CU_OK(cudaMemcpyAsync(zone_out, d_zones, (size_t)n * sizeof(mars_b200_zone_frame_t), cudaMemcpyDeviceToHost, m->stream),
                  MARS_ERR_LAYER_FAILED);
        CU_OK(cudaMemcpyAsync(out_counts, d_out_counts, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, m->stream), MARS_ERR_LAYER_FAILED);
        if (maxd > 0)
            CU_OK(cudaMemcpy2DAsync(out, (size_t)maxd * sizeof(mars_b200_track_box_t), d_out, MARS_B200_MAX_TRACKS * sizeof(mars_b200_track_box_t),
                                    (size_t)maxd * sizeof(mars_b200_track_box_t), (size_t)n, cudaMemcpyDeviceToHost, m->stream),
                  MARS_ERR_LAYER_FAILED);
        return MARS_OK;
    });
    if (e == MARS_OK)
        for (int i = 0; i < n; i++) out_counts[i] = std::min(out_counts[i], maxd);
    return e;
}

/* end to end from host buffers, double-buffered over the two halves of the slot pool:
 * H2D of chunk c+1 and D2H of chunk c-1 overlap the kernels of chunk c */
static mars_error_t batch_pipeline(Model *m, int n, const void *inputs, size_t in_stride, void *outputs, size_t out_stride,
                                   mars_det_t *dets, int32_t *counts, int maxd, float thresh) {
    if (n <= 0) return MARS_OK;
    const size_t in_bytes = io_bytes(&m->pub, 0);
    if (in_stride < in_bytes) in_stride = in_bytes;
    const size_t out_bytes = io_bytes(&m->pub, 1);
    if (out_stride < out_bytes) out_stride = out_bytes;
    if (maxd > 1000) maxd = 1000;
    const int chunk = m->capacity >= 2 ? m->capacity / 2 : 1;
    const int halves = m->capacity >= 2 ? 2 : 1;
    mars_error_t e = MARS_OK;
    cudaEventRecord(m->ev0, m->stream);
    int c = 0;
    for (int done = 0; done < n && e == MARS_OK; done += chunk, c++) {
        const int h = c % halves, first = h * chunk, cnt = std::min(chunk, n - done);
        /* the half is free once its previous results were copied out */
        if (c >= halves) cudaStreamWaitEvent(m->h2d_stream, m->ev_out[h], 0);
        e = copy_io(m, first, cnt, (uint8_t *)const_cast<void *>(inputs) + (size_t)done * in_stride, in_stride, 0, m->h2d_stream);
        if (e != MARS_OK) break;
        cudaEventRecord(m->ev_in[h], m->h2d_stream);
        cudaStreamWaitEvent(m->stream, m->ev_in[h], 0);
        e = enqueue_ops(m, first, cnt, -1);
        if (e == MARS_OK && dets) e = enqueue_detect(m, first, cnt, thresh);
        if (e != MARS_OK) break;
        cudaEventRecord(m->ev_done[h], m->stream);
        cudaStreamWaitEvent(m->d2h_stream, m->ev_done[h], 0);
        if (dets) e = copy_dets(m->rec.det, first, cnt, dets + (size_t)done * maxd, counts + done, maxd, m->d2h_stream);
        if (e == MARS_OK && outputs) e = copy_io(m, first, cnt, (uint8_t *)outputs + (size_t)done * out_stride, out_stride, 1, m->d2h_stream);
        cudaEventRecord(m->ev_out[h], m->d2h_stream);
    }
    cudaEventRecord(m->ev1, m->stream);
    cudaError_t c1 = cudaStreamSynchronize(m->h2d_stream), c2 = cudaStreamSynchronize(m->stream), c3 = cudaStreamSynchronize(m->d2h_stream);
    if (e == MARS_OK && (c1 != cudaSuccess || c2 != cudaSuccess || c3 != cudaSuccess)) {
        set_last_error("batch pipeline: %s", cudaGetErrorString(c1 != cudaSuccess ? c1 : (c2 != cudaSuccess ? c2 : c3)));
        e = MARS_ERR_LAYER_FAILED;
    }
    if (e == MARS_OK) {
        cudaEventElapsedTime(&m->last_ms, m->ev0, m->ev1);
        if (dets) for (int i = 0; i < n; i++) if (counts[i] > maxd) counts[i] = maxd;
    }
    return e;
}

mars_error_t mars_b200_detect_batch(mars_model_t *model, int n, const void *inputs, size_t in_stride, mars_det_t *dets,
                                    int32_t *counts, int maxd, float nms_thresh) {
    Model *m;
    mars_error_t e = inputs && dets && counts ? enter(model, &m) : MARS_ERR_INVALID_FILE;
    return e == MARS_OK ? batch_pipeline(m, n, inputs, in_stride, nullptr, 0, dets, counts, maxd, nms_thresh) : e;
}

mars_error_t mars_b200_run_batch(mars_model_t *model, int n, const void *inputs, size_t in_stride, void *outputs, size_t out_stride) {
    Model *m;
    mars_error_t e = inputs && outputs ? enter(model, &m) : MARS_ERR_INVALID_FILE;
    return e == MARS_OK ? batch_pipeline(m, n, inputs, in_stride, outputs, out_stride, nullptr, nullptr, 0, 0.0f) : e;
}

/* where the images of a pooled submit come from: host input tensors 0, `stride` bytes apart, or (from_frames) host frames
 * letterboxed into the slots -- one frame per slot, or with rois one region of them per slot (frames is null when the caller
 * passed no table) */
struct SubmitIn {
    const void *tensors;
    size_t stride;
    bool from_frames;
    const std::vector<FrameSrc> *frames;
    const RoiList *rois;
};
/* what a pooled submit reads back, which also picks the step: the kept detections of output0 (decode + centre NMS), the kept
 * corner boxes of the heads, the frame records of the region merge (rois), the tracked boxes of the heads' boxes (frames only:
 * the stream table travels in the letterbox upload), or the raw output tensor 0 (the layers alone) */
struct SubmitOut {
    enum Kind { DETS, BOXES, FRAME_BOXES, TRACKS, TENSOR } kind;
    void *dst; /* records [records][maxd], or output tensors `stride` bytes apart */
    int32_t *counts;
    int maxd;
    size_t stride;
    const int32_t *streams = nullptr; /* TRACKS: the tracker stream of each image */
    mars_b200_zone_frame_t *zones = nullptr; /* TRACKS: the zone record of each image (null: not read back) */
};

/* Asynchronous form of mars_b200_detect_batch: the slot pool is split into two halves ("pools" 0 and 1); a batch of up to
 * capacity/2 images is queued on one half -- H2D on the copy stream, layers + decode + NMS on the compute stream, D2H of the
 * detection records on the read-back stream -- and the call returns.  While it runs the caller submits the next batch to the
 * other half, so the host->device copy of batch k+1 and the read-back of batch k-1 overlap the kernels of batch k.
 * Inputs and outputs must stay valid (and should be pinned, e.g. nna_malloc) until mars_b200_wait_batch(pool) returns.
 * With frames the letterbox launches go on the compute stream in front of the (graphed) step; with rois the boxes of the
 * n = rois->n regions are merged per frame after the step (k_merge_rois, merge_thresh) and read back as frames->size() frame
 * records. */
static mars_error_t submit_batch(mars_model_t *model, const char *what, int pool, int n, const SubmitIn &in, SubmitOut out,
                                 float nms_thresh, float merge_thresh = 0.0f) {
    const bool records = out.kind != SubmitOut::TENSOR;
    const int flavour = out.kind == SubmitOut::DETS ? STEP_DETECT : records ? STEP_HEADS : STEP_LAYERS;
    Model *m = as_model(model);
    if (m && flavour == STEP_HEADS && need_heads(m, what) != MARS_OK) return MARS_ERR_INVALID_TENSOR;
    if (m && in.from_frames && !in.frames) { set_last_error("%s: no frame table", what); return MARS_ERR_INVALID_FILE; }
    if (!(in.from_frames || in.tensors) || !out.dst || (records && !out.counts) || pool < 0 || pool > 1) return MARS_ERR_INVALID_FILE;
    mars_error_t e = enter(model, &m);
    if (e != MARS_OK) return e;
    const int half = m->capacity / 2;
    if (half < 1 || n < 0 || n > half) {
        set_last_error("%s: %d %s do not fit half of the slot pool (capacity %d; mars_b200_set_batch)", what, n, in.rois ? "regions" : "images",
                       m->capacity);
        return MARS_ERR_INVALID_TENSOR;
    }
    const int nrec = in.rois ? (int)in.frames->size() : n; /* records read back */
    if (in.rois && nrec > half) {
        set_last_error("%s: %d frames do not fit half of the slot pool (capacity %d; mars_b200_set_batch)", what, nrec, m->capacity);
        return MARS_ERR_INVALID_TENSOR;
    }
    if (m->pending[pool].active) {
        set_last_error("%s: pool %d still has a batch in flight (mars_b200_wait_batch first)", what, pool);
        return MARS_ERR_LAYER_FAILED;
    }
    if (out.kind == SubmitOut::TRACKS) {
        e = in.from_frames ? check_streams(m, what, n, out.streams) : MARS_ERR_INVALID_FILE;
        if (e != MARS_OK) return e;
        if (out.maxd > MARS_B200_MAX_TRACKS) out.maxd = MARS_B200_MAX_TRACKS;
    }
    if (out.maxd > 1000) out.maxd = 1000;
    if (out.maxd < 0) out.maxd = 0;
    const size_t in_stride = std::max(in.stride, io_bytes(&m->pub, 0)), out_stride = std::max(out.stride, io_bytes(&m->pub, 1));
    const int first = pool * half;
    uint32_t ti = 0;
    int nhwc = 0;
    std::vector<LetterboxGeom> g;
    if (in.from_frames) {
        e = pre_validate(m, what, first, in.frames, in.rois, false, &ti, &nhwc, &g);
        if (e != MARS_OK) return e;
    }
    e = compile_model(m); /* also drops captured graphs of an older program (set_opt_level, set_depthwise_mode) */
    if (e != MARS_OK) return e;
    if (n > 0) {
        /* the half is free: its previous batch was waited for (read-back complete) before this call -- its staging too */
        std::vector<int> tail;
        if (in.rois) merge_table(nrec, *in.rois, &tail);
        if (out.kind == SubmitOut::TRACKS) tail.assign(out.streams, out.streams + n);
        const int *tail_dev = nullptr;
        if (in.from_frames) {
            e = enqueue_letterbox(m, m->pre_stage[pool], first, *in.frames, g, ti, nhwc, PRE_HOST_POOL, m->ev_in[pool], in.rois, &tail,
                                  &tail_dev);
            if (e != MARS_OK) return e;
        } else {
            e = copy_io(m, first, n, const_cast<void *>(in.tensors), in_stride, 0, m->h2d_stream);
            if (e != MARS_OK) return e;
            cudaEventRecord(m->ev_in[pool], m->h2d_stream);
            cudaStreamWaitEvent(m->stream, m->ev_in[pool], 0);
        }
        e = enqueue_step_graphed(m, first, n, nms_thresh, flavour);
        if (e == MARS_OK && in.rois) e = enqueue_merge(m, first, nrec, tail_dev, merge_thresh);
        if (e == MARS_OK && out.kind == SubmitOut::TRACKS)
            e = enqueue_track(m, m->rec.box.at(first), m->rec.box.cnt.p + first, MARS_MAX_DETS, tail_dev, n, m->rec.trk.at(first),
                              m->rec.trk.cnt.p + first, MARS_B200_MAX_TRACKS, m->rec.zone.p + first, out.zones != nullptr);
        if (e != MARS_OK) { cudaStreamSynchronize(m->stream); return e; }
        cudaEventRecord(m->ev_done[pool], m->stream);
        cudaStreamWaitEvent(m->d2h_stream, m->ev_done[pool], 0);
        switch (out.kind) {
            case SubmitOut::DETS: e = copy_dets(m->rec.det, first, nrec, out.dst, out.counts, out.maxd, m->d2h_stream); break;
            case SubmitOut::BOXES: e = copy_dets(m->rec.box, first, nrec, out.dst, out.counts, out.maxd, m->d2h_stream); break;
            case SubmitOut::FRAME_BOXES: e = copy_dets(m->rec.fbox, first, nrec, out.dst, out.counts, out.maxd, m->d2h_stream); break;
            case SubmitOut::TRACKS:
                e = copy_dets(m->rec.trk, first, nrec, out.dst, out.counts, out.maxd, m->d2h_stream);
                if (e == MARS_OK && out.zones)
                    CU_OK(cudaMemcpyAsync(out.zones, m->rec.zone.p + first, (size_t)n * sizeof(mars_b200_zone_frame_t), cudaMemcpyDeviceToHost,
                                          m->d2h_stream), MARS_ERR_LAYER_FAILED);
                break;
            case SubmitOut::TENSOR: e = copy_io(m, first, n, out.dst, out_stride, 1, m->d2h_stream); break;
        }
        if (e != MARS_OK) return e;
    } else {
        for (int i = 0; i < nrec; i++) out.counts[i] = 0; /* frames without regions */
    }
    cudaEventRecord(m->ev_out[pool], m->d2h_stream);
    Model::Pending &pd = m->pending[pool];
    pd.active = true;
    pd.n = records ? nrec : 0; pd.maxd = out.maxd; pd.counts = out.counts;
    return MARS_OK;
}
mars_error_t mars_b200_submit_batch(mars_model_t *model, int pool, int n, const void *inputs, size_t in_stride, mars_det_t *dets,
                                    int32_t *counts, int maxd, float nms_thresh) {
    return submit_batch(model, "submit_batch", pool, n, SubmitIn{inputs, in_stride, false, nullptr, nullptr},
                        SubmitOut{SubmitOut::DETS, dets, counts, maxd, 0}, nms_thresh);
}
/* mars_b200_submit_batch with the YOLO heads decode (mars_b200_set_yolo_heads): boxes[n][maxd] corner boxes, frame coordinates for
 * slots with a frame size */
mars_error_t mars_b200_submit_heads_batch(mars_model_t *model, int pool, int n, const void *inputs, size_t in_stride, mars_box_t *boxes,
                                          int32_t *counts, int maxd, float nms_thresh) {
    return submit_batch(model, "submit_heads_batch", pool, n, SubmitIn{inputs, in_stride, false, nullptr, nullptr},
                        SubmitOut{SubmitOut::BOXES, boxes, counts, maxd, 0}, nms_thresh);
}

/* mars_b200_submit_heads_batch from RGB8 or NV12 frames of any sizes and row pitches (host memory): H2D of each frame (each
 * NV12 plane) on the copy stream, the letterbox launches on the compute stream in front of the (graphed) step, frame
 * coordinates for every slot */
mars_error_t mars_b200_submit_frames_heads_batch(mars_model_t *model, int pool, int n, const mars_b200_frame_t *frames, mars_box_t *boxes,
                                                 int32_t *counts, int maxd, float nms_thresh) {
    std::vector<FrameSrc> s;
    return submit_batch(model, "submit_frames_heads_batch", pool, n, SubmitIn{nullptr, 0, true, rgb_sources(n, frames, &s), nullptr},
                        SubmitOut{SubmitOut::BOXES, boxes, counts, maxd, 0}, nms_thresh);
}
mars_error_t mars_b200_submit_frames_nv12_heads_batch(mars_model_t *model, int pool, int n, const mars_b200_nv12_frame_t *frames,
                                                      mars_box_t *boxes, int32_t *counts, int maxd, float nms_thresh) {
    std::vector<FrameSrc> s;
    return submit_batch(model, "submit_frames_nv12_heads_batch", pool, n, SubmitIn{nullptr, 0, true, nv12_sources(n, frames, &s), nullptr},
                        SubmitOut{SubmitOut::BOXES, boxes, counts, maxd, 0}, nms_thresh);
}

/* the tiled flow of mars_b200_submit_frames_heads_batch: regions of the frames letterboxed into the pool's slots, their boxes
 * merged per frame (k_merge_rois) and read back per frame */
mars_error_t mars_b200_submit_rois_heads_batch(mars_model_t *model, int pool, int n_frames, const mars_b200_frame_t *frames, int n_rois,
                                               const mars_b200_roi_t *rois, mars_box_t *boxes, int32_t *counts, int maxd, float nms_thresh,
                                               float merge_thresh) {
    std::vector<FrameSrc> s;
    const RoiList rl{n_rois, rois};
    return submit_batch(model, "submit_rois_heads_batch", pool, n_rois, SubmitIn{nullptr, 0, true, rgb_sources(n_frames, frames, &s), &rl},
                        SubmitOut{SubmitOut::FRAME_BOXES, boxes, counts, maxd, 0}, nms_thresh, merge_thresh);
}
mars_error_t mars_b200_submit_rois_nv12_heads_batch(mars_model_t *model, int pool, int n_frames, const mars_b200_nv12_frame_t *frames,
                                                    int n_rois, const mars_b200_roi_t *rois, mars_box_t *boxes, int32_t *counts, int maxd,
                                                    float nms_thresh, float merge_thresh) {
    std::vector<FrameSrc> s;
    const RoiList rl{n_rois, rois};
    return submit_batch(model, "submit_rois_nv12_heads_batch", pool, n_rois,
                        SubmitIn{nullptr, 0, true, nv12_sources(n_frames, frames, &s), &rl},
                        SubmitOut{SubmitOut::FRAME_BOXES, boxes, counts, maxd, 0}, nms_thresh, merge_thresh);
}

/* mars_b200_submit_frames[_nv12]_heads_batch, then the tracker on the pool's slots; the tracked boxes are read back */
mars_error_t mars_b200_submit_frames_track_batch(mars_model_t *model, int pool, int n, const mars_b200_frame_t *frames, const int32_t *streams,
                                                 mars_b200_track_box_t *out, int32_t *counts, int maxd, float nms_thresh) {
    std::vector<FrameSrc> s;
    return submit_batch(model, "submit_frames_track_batch", pool, n, SubmitIn{nullptr, 0, true, rgb_sources(n, frames, &s), nullptr},
                        SubmitOut{SubmitOut::TRACKS, out, counts, maxd, 0, streams}, nms_thresh);
}
mars_error_t mars_b200_submit_frames_nv12_track_batch(mars_model_t *model, int pool, int n, const mars_b200_nv12_frame_t *frames,
                                                      const int32_t *streams, mars_b200_track_box_t *out, int32_t *counts, int maxd,
                                                      float nms_thresh) {
    std::vector<FrameSrc> s;
    return submit_batch(model, "submit_frames_nv12_track_batch", pool, n, SubmitIn{nullptr, 0, true, nv12_sources(n, frames, &s), nullptr},
                        SubmitOut{SubmitOut::TRACKS, out, counts, maxd, 0, streams}, nms_thresh);
}
/* the track submits with the zone record of every frame read back too */
mars_error_t mars_b200_submit_frames_zones_batch(mars_model_t *model, int pool, int n, const mars_b200_frame_t *frames, const int32_t *streams,
                                                 mars_b200_track_box_t *out, int32_t *counts, int maxd, mars_b200_zone_frame_t *zones,
                                                 float nms_thresh) {
    std::vector<FrameSrc> s;
    if (!zones) {
        set_last_error("submit_frames_zones_batch: no zone record table (zones is NULL; mars_b200_submit_frames_track_batch reads back no zone records)");
        return MARS_ERR_INVALID_FILE;
    }
    return submit_batch(model, "submit_frames_zones_batch", pool, n, SubmitIn{nullptr, 0, true, rgb_sources(n, frames, &s), nullptr},
                        SubmitOut{SubmitOut::TRACKS, out, counts, maxd, 0, streams, zones}, nms_thresh);
}
mars_error_t mars_b200_submit_frames_nv12_zones_batch(mars_model_t *model, int pool, int n, const mars_b200_nv12_frame_t *frames,
                                                      const int32_t *streams, mars_b200_track_box_t *out, int32_t *counts, int maxd,
                                                      mars_b200_zone_frame_t *zones, float nms_thresh) {
    std::vector<FrameSrc> s;
    if (!zones) {
        set_last_error("submit_frames_nv12_zones_batch: no zone record table (zones is NULL; mars_b200_submit_frames_nv12_track_batch reads back no zone records)");
        return MARS_ERR_INVALID_FILE;
    }
    return submit_batch(model, "submit_frames_nv12_zones_batch", pool, n, SubmitIn{nullptr, 0, true, nv12_sources(n, frames, &s), nullptr},
                        SubmitOut{SubmitOut::TRACKS, out, counts, maxd, 0, streams, zones}, nms_thresh);
}

/* mars_b200_submit_batch without the YOLO post-process: the raw output tensor 0 of every image is read back instead
 * (models whose output is not a [1, N, 85] head: NanoDet-style heads, float32 models).  Same pools, same wait. */
mars_error_t mars_b200_submit_run_batch(mars_model_t *model, int pool, int n, const void *inputs, size_t in_stride, void *outputs, size_t out_stride) {
    return submit_batch(model, "submit_run_batch", pool, n, SubmitIn{inputs, in_stride, false, nullptr, nullptr},
                        SubmitOut{SubmitOut::TENSOR, outputs, nullptr, 0, out_stride}, 0.0f);
}

mars_error_t mars_b200_wait_batch(mars_model_t *model, int pool) {
    if (pool < 0 || pool > 1) return MARS_ERR_INVALID_FILE;
    Model *m;
    mars_error_t e = enter(model, &m);
    if (e != MARS_OK || !m->pending[pool].active) return e;
    cudaError_t ce = cudaEventSynchronize(m->ev_out[pool]);
    Model::Pending &pd = m->pending[pool];
    pd.active = false;
    if (ce != cudaSuccess) {
        set_last_error("wait_batch: %s", cudaGetErrorString(ce));
        return MARS_ERR_LAYER_FAILED;
    }
    for (int i = 0; i < pd.n; i++) if (pd.counts[i] > pd.maxd) pd.counts[i] = pd.maxd;
    return MARS_OK;
}

/* the CUDA stream (cudaStream_t) every kernel of this model is launched on: work a caller enqueues there -- e.g. an NCCL
 * gather of the resident detection records -- is ordered after the batch that produced them and before the next one */
void *mars_b200_compute_stream(mars_model_t *model) {
    Model *m = as_model(model);
    return m ? (void *)m->stream : nullptr;
}
uint64_t mars_b200_launch_count(mars_model_t *model) {
    Model *m = as_model(model);
    return m ? m->launches : 0;
}
/* device addresses of the resident detection records (for a device-side gather):
 * dets = mars_det_t[capacity][1024], counts = int32[capacity] */
void mars_b200_detections_device(mars_model_t *model, void **dets, void **counts, int *stride_dets) {
    Model *m = as_model(model);
    if (dets) *dets = m ? m->rec.det.rec.p : nullptr;
    if (counts) *counts = m ? m->rec.det.cnt.p : nullptr;
    if (stride_dets) *stride_dets = MARS_MAX_DETS;
}
float mars_b200_last_gpu_ms(mars_model_t *model) {
    Model *m = as_model(model);
    return m ? m->last_ms : 0.0f;
}

/* per-op profile: enable, run, read back "op kind layer ms calls bytes macs" lines */
void mars_b200_set_profile(mars_model_t *model, int on) {
    Model *m = as_model(model);
    if (!m) return;
    m->profile = on;
    if (on) {
        std::fill(m->prof_ms.begin(), m->prof_ms.end(), 0.0);
        std::fill(m->prof_calls.begin(), m->prof_calls.end(), 0);
    }
}
int mars_b200_num_ops(mars_model_t *model) {
    Model *m = as_model(model);
    if (!m || compile_model(m) != MARS_OK) return 0;
    return (int)m->prog.ops.size();
}
/* info[0]=kind [1]=layer [2]=impl [3]=mode [4]=ic [5]=oc [6]=oh [7]=ow [8]=kh [9]=kw [10]=fused_layers [11]=ih [12]=iw;
 * ms = accumulated CUDA-event milliseconds, calls = timed launches of this op */
int mars_b200_op_info(mars_model_t *model, int op, int32_t *info, double *ms, uint64_t *calls, uint64_t *flat_n) {
    Model *m = as_model(model);
    if (!m || op < 0 || (size_t)op >= m->prog.ops.size()) return -1;
    const Op &o = m->prog.ops[op];
    if (info) {
        info[0] = o.kind; info[1] = o.layer; info[2] = o.impl; info[3] = o.mode; info[4] = o.ic; info[5] = o.oc;
        info[6] = o.oh; info[7] = o.ow; info[8] = o.kh; info[9] = o.kw; info[10] = o.fused_layers; info[11] = o.ih; info[12] = o.iw;
    }
    if (ms) *ms = (size_t)op < m->prof_ms.size() ? m->prof_ms[op] : 0.0;
    if (calls) *calls = (size_t)op < m->prof_calls.size() ? m->prof_calls[op] : 0;
    if (flat_n) *flat_n = o.n;
    return 0;
}

/* geometry of the arena, for tests: out[0]=weights_size [1]=buffer_size [2]=num_buffers [3]=slot_stride [4]=arena_size */
void mars_b200_geometry(mars_model_t *model, size_t *out5) {
    Model *m = as_model(model);
    if (!m || !out5) return;
    out5[0] = m->weights_size; out5[1] = m->buffer_size; out5[2] = (size_t)m->num_buffers; out5[3] = m->slot_stride; out5[4] = m->arena_size;
}
size_t mars_b200_tensor_offset(mars_model_t *model, uint32_t index) {
    Model *m = as_model(model);
    if (!m || index >= model->header.num_tensors) return (size_t)-1;
    return m->toff[index];
}

/* ---- several GPUs behind one C call (SURVEY 8e; north_star: "work is partitioned across the GPUs of one box by sharding the
 * image batch, with no inter-GPU traffic on the hot path") --------------------------------------------------------------
 * A group holds one replica of the model per device.  mars_b200_group_detect_batch shards the n images into contiguous
 * blocks of ceil(n / G), runs every block on its GPU from its own host thread (H2D, all layers, decode, NMS, D2H, pipelined
 * in chunks exactly like mars_b200_detect_batch) and returns when all are done; the detection records land directly in the
 * caller's arrays, which is the "gather" of a single-process caller (bench.py, one process per GPU, gathers over NCCL). */
struct mars_b200_group {
    std::vector<mars_model_t *> models;
    std::vector<int> devices;
};

mars_error_t mars_b200_group_load(const void *data, size_t size, const int *devices, int n_devices, int per_gpu_batch, mars_b200_group_t **out) {
    if (!data || !out || n_devices < 1 || per_gpu_batch < 1) return MARS_ERR_INVALID_FILE;
    int visible = 0;
    if (cudaGetDeviceCount(&visible) != cudaSuccess || visible < 1) {
        set_last_error("no CUDA device (this library has no CPU fallback)");
        return MARS_ERR_NNA_INIT_FAILED;
    }
    mars_b200_group *g = new (std::nothrow) mars_b200_group();
    if (!g) return MARS_ERR_ALLOC_FAILED;
    const int saved = g_device;
    mars_error_t e = MARS_OK;
    for (int i = 0; i < n_devices && e == MARS_OK; i++) {
        const int d = devices ? devices[i] : i;
        if (d < 0 || d >= visible) { set_last_error("group: device ordinal %d out of range (%d visible)", d, visible); e = MARS_ERR_NNA_INIT_FAILED; break; }
        if (mars_b200_set_device(d) != 0) { e = MARS_ERR_NNA_INIT_FAILED; break; }
        mars_model_t *m = nullptr;
        e = mars_load_memory(data, size, &m);
        if (e == MARS_OK) e = mars_b200_set_batch(m, per_gpu_batch);
        if (e != MARS_OK) { if (m) mars_free(m); break; }
        g->models.push_back(m);
        g->devices.push_back(d);
    }
    if (saved >= 0) mars_b200_set_device(saved);
    if (e != MARS_OK) {
        for (auto *m : g->models) mars_free(m);
        delete g;
        return e;
    }
    *out = g;
    return MARS_OK;
}

void mars_b200_group_free(mars_b200_group_t *g) {
    if (!g) return;
    for (auto *m : g->models) mars_free(m);
    delete g;
}

int mars_b200_group_size(mars_b200_group_t *g) { return g ? (int)g->models.size() : 0; }
mars_model_t *mars_b200_group_model(mars_b200_group_t *g, int i) { return (g && i >= 0 && (size_t)i < g->models.size()) ? g->models[i] : nullptr; }

mars_error_t mars_b200_group_detect_batch(mars_b200_group_t *g, int n, const void *inputs, size_t in_stride, mars_det_t *dets, int32_t *counts,
                                          int maxd, float nms_thresh) {
    if (!g || g->models.empty() || !inputs || !dets || !counts || n < 0) return MARS_ERR_INVALID_FILE;
    const int G = (int)g->models.size();
    const size_t in_bytes = mars_b200_input_bytes(g->models[0]);
    if (in_stride < in_bytes) in_stride = in_bytes;
    if (maxd > 1000) maxd = 1000;
    if (maxd < 0) maxd = 0;
    const int per = (n + G - 1) / G;
    std::vector<mars_error_t> err((size_t)G, MARS_OK);
    std::vector<std::string> why((size_t)G);
    std::vector<std::thread> th;
    for (int r = 0; r < G; r++) {
        const int first = std::min(r * per, n), cnt = std::max(0, std::min(per, n - first));
        if (cnt == 0) continue;
        th.emplace_back([=, &err, &why]() {
            err[r] = mars_b200_detect_batch(g->models[r], cnt, (const uint8_t *)inputs + (size_t)first * in_stride, in_stride,
                                            dets + (size_t)first * maxd, counts + first, maxd, nms_thresh);
            if (err[r] != MARS_OK) why[r] = g_err; /* the diagnostic is thread-local: carry it to the caller's thread */
        });
    }
    for (auto &t : th) t.join();
    for (int r = 0; r < G; r++)
        if (err[r] != MARS_OK) { set_last_error("group: GPU %d: %s", g->devices[r], why[r].c_str()); return err[r]; }
    return MARS_OK;
}

} /* extern "C" */

#include "seam.inc"
