/*
 * conv_tf32.h -- host interface of the tcgen05 kind::tf32 convolution for float32 models (conv_tf32.cu).
 * mode: 1 = tf32 (operands rounded to tf32), 2 = tf32x3 (hi/lo operand split, three MMAs per k-step: fp32-grade products).
 */
#pragma once
#include "conv_tc.h"

namespace marsb200 {

bool tf32_supported(const Op &o, int mode);
/* per-image bytes of the channel-innermost fp32 input copy (two copies in mode 2) */
size_t tf32_scratch_need(const Op &o, int mode);
bool tf32_plan(const Op &o, const ArenaGeom &g, int mode, uint8_t *scratch, size_t scratch_stride, TcPlan *plan);
bool tf32_launch(const TcPlan &plan, uint8_t *slots_base, int first, int n, cudaStream_t s, uint64_t *launches);
/* frees a plan tf32_plan built (null: nothing) */
void tf32_release(F32PlanImpl *t);

} // namespace marsb200
