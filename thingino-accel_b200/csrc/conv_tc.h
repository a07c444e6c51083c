/*
 * conv_tc.h -- host interface of the tcgen05 int8 implicit-GEMM convolution (conv_tc.cu).
 * A TcPlan holds what is fixed per (layer, arena): the TMA tensor maps over the NCHW
 * activation planes of every image slot and over the repacked weights, the tile shape and
 * the fused-epilogue description.
 */
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "mars_internal.h"

namespace marsb200 {

struct ArenaGeom {
    uint8_t *d_weights;
    uint8_t *d_slots;
    size_t W, slot_stride;
    int capacity;
    const uint8_t *h_weights; /* host copy of the weight blob (requantisation bounds are computed from the real weights) */
    const uint8_t *h_cpool;   /* host copy of the const pool (256-byte tables) */
};

struct TcPlanImpl;  /* conv_tc.cu */
struct F32PlanImpl; /* conv_tf32.cu */
/* the tensor-core plan of one op, owned: int8 (tc_plan) or float32 (tf32_plan); neither = no plan */
struct TcPlan {
    TcPlanImpl *i8 = nullptr;
    F32PlanImpl *f32 = nullptr;
};

/* ---- shared by the int8 (conv_tc.cu) and float32 (conv_tf32.cu) planners ---- */
/* M tile (output pixels = TMEM lanes of an accumulator), most kernel taps, most output channels */
constexpr int TC_BM = 128, TC_MAX_TAPS = 36, TC_MAX_CO = 1024;
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
/* the driver's cuTensorMapEncodeTiled (looked up once through the runtime), or null */
EncodeTiledFn encode_tiled();
/* byte-typed 3-d map: dims (d0 bytes, d1 rows, d2 images / taps), strides s1, s2, box {b0, b1, 1} */
bool make_map3(CUtensorMap *m, void *base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t s1, uint64_t s2, uint32_t b0, uint32_t b1,
               CUtensorMapSwizzle sw);
/* 4-d map over channel-innermost activations: dims (C, W, H, images), box {bc channels, bw, bh, 1} traversed with stride es in W
 * and H (the box covers bw / es x bh / es pixels); coordinates outside the tensor read as zeros */
bool make_map4(CUtensorMap *m, void *base, uint64_t C, uint64_t W, uint64_t H, uint64_t N, uint64_t img_stride, uint32_t bc, uint32_t bw,
               uint32_t bh, uint32_t es, CUtensorMapSwizzle sw);
inline int round_up(int x, int a) { return (x + a - 1) / a * a; }
/* N tile for `oc` output channels: all of them (padded to 16) up to 256, else 256 or 128 columns (the last tile may be ragged) */
int tc_n_tile(int oc);
/* how many N tiles the kernel would use for `oc` output channels */
int tc_n_tiles(int oc);
/* bytes of K per pipeline step for `kbytes` bytes of K per tap: 128, 64 or 32 */
int tc_bk(int kbytes);
/* K-major operands with `bk`-byte rows: UMMA layout type (2 = SW128, 4 = SW64, 6 = SW32) and the matching TMA swizzle */
uint32_t tc_umma_layout(int bk);
CUtensorMapSwizzle tc_swizzle(int bk);
/* multiprocessors of the current device (148 when the query fails) */
int tc_sm_count();

/* The channel-innermost input copy of a kxk conv in which a kernel tap is a flat row shift: mode 1 (stride 1) pads every row with
 * kw-1 zero columns (pitch Wp), mode 2 (stride 2) splits the image into its 2x2 phases, planes of `plane` pixels with pitch Wp.
 * npix = pixel rows of the copy.  Written by a layout pre-pass (copy_src_pixel, tc_common.cuh gives each row's source pixel) or
 * by the producing conv's epilogue. */
struct PixelCopy {
    int mode = 0; /* 0: the op's shape has no such copy */
    int Wp = 0, plane = 0, npix = 0, pt = 0, pl = 0;
    /* row offset of tap (kh, kw) from the row of the output pixel */
    int tap_shift(int kh, int kw) const { return mode == 1 ? (kh - pt) * Wp + kw : ((kh & 1) * 2 + (kw & 1)) * plane + (kh / 2) * Wp + kw / 2; }
};
PixelCopy pixel_copy(const Op &o);

/* can this op run on the tensor-core kernel at all (shape / hazard rules)? */
bool tc_supported(const Op &o);
/* does the kernel read its activations from a private copy (pre-pass) rather than the arena? */
bool tc_uses_copy(const Op &o);
/* is that copy the padded / phase-split channel-innermost layout a producing conv's epilogue can write directly? */
bool tc_linkable(const Op &o);
/* per-image bytes of the padded / phase-split input copy the op needs (0 = reads the arena) */
size_t tc_scratch_need(const Op &o);
/* build the plan: tensor maps, repacked weights, epilogue description */
/* linked / linked_stride: the per-image area of producer-written copies (Op::copy_off, Program::linked_bytes);
 * consumer: the op whose input copy this op's epilogue writes (Op::nhwc_consumer), or null */
bool tc_plan(const Op &o, const ArenaGeom &g, uint8_t *scratch, size_t scratch_stride, uint8_t *linked, size_t linked_stride,
             const Op *consumer, TcPlan *plan);
/* pre-pass (if any) + conv kernel for image slots [first, first+n) */
/* use_linked: read the producer-written copy (full passes) instead of running the layout pre-pass on the arena tensor */
bool tc_launch(const TcPlan &plan, uint8_t *slots_base, int first, int n, bool use_linked, cudaStream_t s, uint64_t *launches);
/* the requantisation variant (0..3, see select_requant) of an int8 plan, or -1 when the op has none */
int tc_rq(const TcPlan &plan);
void tc_release(std::vector<TcPlan> &plans);

} // namespace marsb200
