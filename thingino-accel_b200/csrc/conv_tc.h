/*
 * conv_tc.h -- host interface of the tcgen05 int8 implicit-GEMM convolution (conv_tc.cu).
 * A TcPlan holds what is fixed per (layer, arena): the TMA tensor maps over the NCHW
 * activation planes of every image slot and over the repacked weights, the tile shape and
 * the fused-epilogue description.
 */
#pragma once
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

struct TcPlan {
    bool valid = false;
    void *impl = nullptr; /* TcPlanImpl* (conv_tc.cu) or F32PlanImpl* (conv_tf32.cu, f32 == true), owned */
    bool f32 = false;
};

/* can this op run on the tensor-core kernel at all (shape / hazard rules)? */
bool tc_supported(const Op &o);
/* how many N tiles the kernel would use for `oc` output channels */
int tc_n_tiles(int oc);
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
void tc_release(std::vector<TcPlan> &plans);

} // namespace marsb200
