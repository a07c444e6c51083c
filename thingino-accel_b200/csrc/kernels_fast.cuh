/*
 * kernels_fast.cuh -- vectorised variants of the memory-bound layer kernels.
 *
 * Each is bit-identical to its point function in kernels_exact.cuh (same fp32 operation
 * sequence, same tables) and is only selected for hazard-free ops (EXEC_PARALLEL, operands not
 * straddling the weights/slot boundary) whose operands are 16-byte aligned; everything else
 * stays on the exact kernels.  16 bytes per thread per access, 256-byte tables staged in
 * shared memory, grid = (chunks, images).
 */
#pragma once
#include "kernels_exact.cuh"

namespace marsb200 {

__device__ __forceinline__ uint32_t lut4(const uint8_t *lut, uint32_t w) {
    return (uint32_t)lut[(uint8_t)((w & 0xFF) ^ 0x80)] | ((uint32_t)lut[(uint8_t)(((w >> 8) & 0xFF) ^ 0x80)] << 8) |
           ((uint32_t)lut[(uint8_t)(((w >> 16) & 0xFF) ^ 0x80)] << 16) | ((uint32_t)lut[(uint8_t)((w >> 24) ^ 0x80)] << 24);
}

/* out[i] = table[in[i]] (sigmoid / relu / fused unary chains), table index = value + 128 */
__global__ void __launch_bounds__(256) k_lut16(ArenaView v, KOp o) {
    __shared__ uint8_t lut[256];
    lut[threadIdx.x] = v.cpool[o.lut + threadIdx.x];
    __syncthreads();
    const Img im = make_img(v, blockIdx.y);
    const uint8_t *in = im.s_minus_W + o.in0;
    uint8_t *out = im.s_minus_W + o.out;
    const int64_t nv = (int64_t)(o.n >> 4);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x) {
        uint4 a = reinterpret_cast<const uint4 *>(in)[i];
        a.x = lut4(lut, a.x); a.y = lut4(lut, a.y); a.z = lut4(lut, a.z); a.w = lut4(lut, a.w);
        reinterpret_cast<uint4 *>(out)[i] = a;
    }
    if (blockIdx.x == 0 && threadIdx.x < (int)(o.n & 15)) {
        const int64_t i = (nv << 4) + threadIdx.x;
        out[i] = lut[(uint8_t)(in[i] ^ 0x80)];
    }
}

/* the same four elements without the int -> float conversions (the XU pipe, 16 lanes per SM, bounded the kernel at three
 * conversions per element): (float)(int8) = as_float(0x4B400000 + sign-extended byte) - 1.5 * 2^23, exact; the final truncation is
 * one saturating cvt.rzi.s8 -- equal to the reference's (int32) cast + clamp whenever the value is finite and below 2^31, which the
 * host checks from the scales (KOp::fast_bin) */
__device__ __forceinline__ uint32_t bin4_fast(uint32_t a, uint32_t b, int is_mul, float sa, float sb, float inv) {
    uint32_t r[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const uint32_t sel = (uint32_t)k | ((uint32_t)(k | 8) << 4) | ((uint32_t)(k | 8) << 8) | ((uint32_t)(k | 8) << 12); /* byte k, then its sign three times */
        uint32_t xa, xb; /* prmt in its default mode: selector values 8..15 replicate the sign bit of byte (value & 7) */
        asm("prmt.b32 %0, %1, %2, %3;" : "=r"(xa) : "r"(a), "r"(0u), "r"(sel));
        asm("prmt.b32 %0, %1, %2, %3;" : "=r"(xb) : "r"(b), "r"(0u), "r"(sel));
        const float fa = __fadd_rn(__int_as_float((int)(xa + 0x4B400000u)), -12582912.0f);
        const float fb = __fadd_rn(__int_as_float((int)(xb + 0x4B400000u)), -12582912.0f);
        const float va = __fmul_rn(fa, sa), vb = __fmul_rn(fb, sb);
        const float y = is_mul ? __fmul_rn(va, vb) : __fadd_rn(va, vb);
        const float u = __fadd_rn(__fmul_rn(y, inv), 0.5f);
        int q;
        asm("cvt.rzi.s8.f32 %0, %1;" : "=r"(q) : "f"(u));
        r[k] = (uint32_t)q;
    }
    return __byte_perm(__byte_perm(r[0], r[1], 0x0040), __byte_perm(r[2], r[3], 0x0040), 0x5410);
}

__device__ __forceinline__ uint32_t bin4(uint32_t a, uint32_t b, int is_mul, float sa, float sb, float inv) {
    uint32_t r = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const float va = __fmul_rn((float)(int8_t)(a >> (8 * k)), sa), vb = __fmul_rn((float)(int8_t)(b >> (8 * k)), sb);
        const float y = is_mul ? __fmul_rn(va, vb) : __fadd_rn(va, vb);
        r |= (uint32_t)(uint8_t)requant_mul_inv(y, inv) << (8 * k);
    }
    return r;
}

/* int8 mul / add (reference src/mars/mars_runtime.c:818-835, :885-902) */
__global__ void __launch_bounds__(256) k_bin16(ArenaView v, KOp o) {
    const Img im = make_img(v, blockIdx.y);
    const uint8_t *a = im.s_minus_W + o.in0, *b = im.s_minus_W + o.in1;
    uint8_t *out = im.s_minus_W + o.out;
    const int is_mul = o.kind == OP_MUL_I8;
    const int64_t nv = (int64_t)(o.n >> 4);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x) {
        const uint4 x = reinterpret_cast<const uint4 *>(a)[i], y = reinterpret_cast<const uint4 *>(b)[i];
        uint4 r;
        if (o.fast_bin) {
            r.x = bin4_fast(x.x, y.x, is_mul, o.f0, o.f1, o.f2); r.y = bin4_fast(x.y, y.y, is_mul, o.f0, o.f1, o.f2);
            r.z = bin4_fast(x.z, y.z, is_mul, o.f0, o.f1, o.f2); r.w = bin4_fast(x.w, y.w, is_mul, o.f0, o.f1, o.f2);
        } else {
            r.x = bin4(x.x, y.x, is_mul, o.f0, o.f1, o.f2); r.y = bin4(x.y, y.y, is_mul, o.f0, o.f1, o.f2);
            r.z = bin4(x.z, y.z, is_mul, o.f0, o.f1, o.f2); r.w = bin4(x.w, y.w, is_mul, o.f0, o.f1, o.f2);
        }
        reinterpret_cast<uint4 *>(out)[i] = r;
    }
    if (blockIdx.x == 0 && threadIdx.x < (int)(o.n & 15)) {
        const int64_t i = (nv << 4) + threadIdx.x;
        const float va = __fmul_rn((float)(int8_t)a[i], o.f0), vb = __fmul_rn((float)(int8_t)b[i], o.f1);
        out[i] = (uint8_t)requant_mul_inv(is_mul ? __fmul_rn(va, vb) : __fadd_rn(va, vb), o.f2);
    }
}

/* Restated depthwise convolution (parity unpinned: the reference's DEPTHWISE_CONV2D is a no-op, src/mars/mars_runtime.c:1168-1170;
 * convention of mars-compiler/src/main.rs:877-881), NCHW, four adjacent output pixels of one channel per thread: the input window of
 * a kernel row is shared by the four (L1), every tap weight is loaded once for all of them, one 4-byte store.  Same arithmetic as dw_i8_point (int32 wrap-around accumulation in tap order, requant_conv);
 * selected for hazard-free layers with ow % 4 == 0 and kernels up to 7 wide. */
__global__ void __launch_bounds__(256) k_dw_nchw4(ArenaView v, KOp o) {
    const Img im = make_img(v, blockIdx.y);
    const int ow4 = o.ow >> 2;
    const int64_t total = (int64_t)o.oc * o.oh * ow4;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int x4 = (int)(t % ow4), oh = (int)((t / ow4) % o.oh), c = (int)(t / ((int64_t)ow4 * o.oh));
    const int8_t *in = reinterpret_cast<const int8_t *>(im.s_minus_W + o.in0) + (int64_t)c * o.ih * o.iw;
    const int8_t *w = reinterpret_cast<const int8_t *>(im.w + o.w) + (int64_t)c * o.kh * o.kw;
    const uint32_t b = (uint32_t)bias_i32<false>(im, o, c);
    uint32_t acc[4] = {b, b, b, b};
    const int iw0 = x4 * 4 * o.sw - o.pl; /* input column of output 0, tap 0 */
    for (int y = 0; y < o.kh; y++) {
        const int ih = oh * o.sh - o.pt + y;
        if (ih < 0 || ih >= o.ih) continue;
        const int8_t *row = in + (int64_t)ih * o.iw;
        for (int x = 0; x < o.kw; x++) {
            const int wv = (int)w[y * o.kw + x];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int iw = iw0 + j * o.sw + x;
                if (iw >= 0 && iw < o.iw) acc[j] += (uint32_t)((int)row[iw] * wv); /* taps outside the plane are skipped, like dw_i8_point */
            }
        }
    }
    uint32_t r = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        int8_t q = requant_conv((int32_t)acc[j], o.f0);
        if (o.post_relu && q < 0) q = 0;
        if (o.post_lut >= 0) q = (int8_t)v.cpool[o.post_lut + (int)q + 128];
        r |= (uint32_t)(uint8_t)q << (8 * j);
    }
    *reinterpret_cast<uint32_t *>(wr_ptr(im, o.out) + ((int64_t)c * o.oh + oh) * o.ow + x4 * 4) = r;
}
static inline bool dw_nchw4_ok(const ArenaView &v, const KOp &o) {
    return o.kind == OP_DW_I8 && o.coff == 0 && o.mode == EXEC_PARALLEL && o.ow > 0 && o.ow % 4 == 0 && o.sw >= 1 && o.kw >= 1 && o.in0 >= (int64_t)v.W && o.out >= (int64_t)v.W && ((o.out - (int64_t)v.W) & 3) == 0 && o.w >= 0 &&
           o.w + (int64_t)o.oc * o.kh * o.kw <= (int64_t)v.W && (o.bias < 0 || o.bias + 4 * (int64_t)o.oc <= (int64_t)v.W);
}

/* concat input whose channel count equals the output's (every concat of the shipped YOLO files,
 * SURVEY C.4): out[t + coff] = in[t], a shifted flat copy.  VEC = bytes per access. */
template <int VEC>
__global__ void __launch_bounds__(256) k_shift_copy(ArenaView v, KOp o, int periodic) {
    const Img im = make_img(v, blockIdx.y);
    uint8_t *out = im.s_minus_W + o.out + o.coff;
    const uint8_t *in = periodic ? (const uint8_t *)(im.s_minus_W + o.out) : (const uint8_t *)(im.s_minus_W + o.in0);
    const int64_t nv = (int64_t)o.n / VEC;
    const int64_t per = o.coff / VEC; /* periodic: source index wraps every coff bytes (SURVEY C.4b) */
    const bool small = nv < (int64_t)0x7FFFFFFF; /* 32-bit remainder: the 64-bit one (a ~100-instruction sequence) bounded the periodic fill */
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t si = periodic ? (small ? (int64_t)((uint32_t)i % (uint32_t)per) : i % per) : i;
        if (VEC == 16) reinterpret_cast<uint4 *>(out)[i] = reinterpret_cast<const uint4 *>(in)[si];
        else if (VEC == 4) reinterpret_cast<uint32_t *>(out)[i] = reinterpret_cast<const uint32_t *>(in)[si];
        else out[i] = in[si];
    }
    if (blockIdx.x == 0 && threadIdx.x < (int)((int64_t)o.n % VEC)) {
        const int64_t i = nv * VEC + threadIdx.x;
        out[i] = periodic ? in[i % o.coff] : in[i];
    }
}

/* In-place NCHW 1x1 conv (see k_conv1x1_nchw_inplace in kernels_exact.cuh for why one thread per pixel walking the output
 * channels in order is exact) with the pixel's channel vector in REGISTERS: CI4 packed words per thread, weights and
 * biases in shared memory read as 16-byte broadcasts, dp4a accumulation (exact int32, order-free).  The feedback
 * "pass oc reads planes ic < oc in their output form" becomes a byte insert into word oc/4, a compile-time register
 * index because the loop over output-channel groups is fully unrolled.  blockDim.x = 128 pixels;
 * smem = (Co * CI4 + Co) * 4 bytes. */
template <int CI4>
__global__ void __launch_bounds__(128) k_conv1x1_inplace_reg(ArenaView v, KOp o) {
    extern __shared__ uint32_t smem_w[];
    const Img im = make_img(v, blockIdx.y);
    uint32_t *ws = smem_w;                                        /* [oc][CI4] */
    int32_t *bs = reinterpret_cast<int32_t *>(smem_w + o.oc * CI4); /* [oc] */
    const int64_t P = (int64_t)o.oh * o.ow;
    const int64_t p = (int64_t)blockIdx.x * 128 + threadIdx.x;
    const uint8_t *in = im.s_minus_W + o.in0;
    const uint32_t *w = reinterpret_cast<const uint32_t *>(im.w + o.w); /* weights lie in the blob, 4-byte aligned (checked on the host) */
    for (int i = threadIdx.x; i < o.oc * CI4; i += 128) ws[i] = w[i];
    for (int i = threadIdx.x; i < o.oc; i += 128) bs[i] = bias_i32<false>(im, o, i);
    uint32_t x[CI4];
    if (p < P) {
#pragma unroll
        for (int k = 0; k < CI4; k++) {
            const uint8_t *q = in + (int64_t)(4 * k) * P + p;
            x[k] = (uint32_t)q[0] | ((uint32_t)q[P] << 8) | ((uint32_t)q[2 * P] << 16) | ((uint32_t)q[3 * P] << 24);
        }
    }
    __syncthreads();
    if (p >= P) return;
    uint8_t *out = wr_ptr(im, o.out) + p;
    /* fused followers (planner: fuse_silu): S and Z are tables of the output byte (reference src/mars/mars_runtime.c:724-838) */
    uint8_t *out_s = o.out_s >= 0 ? wr_ptr(im, o.out_s) + p : nullptr, *out_z = o.out_z >= 0 ? wr_ptr(im, o.out_z) + p : nullptr;
    const uint8_t *ts = o.lut_s >= 0 ? v.cpool + o.lut_s + 128 : nullptr, *tz = o.lut_z >= 0 ? v.cpool + o.lut_z + 128 : nullptr;
    const bool store_y = o.store_y != 0;
    const float cs = o.f0;
#pragma unroll
    for (int g = 0; g < CI4; g++) { /* output channels 4g .. 4g+3 feed back into word g */
        if (4 * g >= o.oc) break;
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const int oc = 4 * g + r;
            if (oc < o.oc) {
                int acc = bs[oc];
                const uint4 *wr = reinterpret_cast<const uint4 *>(ws + oc * CI4);
#pragma unroll
                for (int k4 = 0; k4 < CI4 / 4; k4++) {
                    const uint4 w4 = wr[k4];
                    acc = __dp4a((int)x[4 * k4], (int)w4.x, acc); acc = __dp4a((int)x[4 * k4 + 1], (int)w4.y, acc);
                    acc = __dp4a((int)x[4 * k4 + 2], (int)w4.z, acc); acc = __dp4a((int)x[4 * k4 + 3], (int)w4.w, acc);
                }
                const int8_t y = requant_conv(acc, cs);
                if (store_y) out[(int64_t)oc * P] = (uint8_t)y;
                if (out_s) out_s[(int64_t)oc * P] = __ldg(ts + y);
                if (out_z) out_z[(int64_t)oc * P] = __ldg(tz + y);
                x[g] = (x[g] & ~(0xFFu << (8 * r))) | ((uint32_t)(uint8_t)y << (8 * r));
            }
        }
    }
    for (int oc = 4 * CI4; oc < o.oc; oc++) { /* more outputs than inputs: no feedback beyond plane ic-1 */
        int acc = bs[oc];
        const uint4 *wr = reinterpret_cast<const uint4 *>(ws + oc * CI4);
#pragma unroll
        for (int k4 = 0; k4 < CI4 / 4; k4++) {
            const uint4 w4 = wr[k4];
            acc = __dp4a((int)x[4 * k4], (int)w4.x, acc); acc = __dp4a((int)x[4 * k4 + 1], (int)w4.y, acc);
            acc = __dp4a((int)x[4 * k4 + 2], (int)w4.z, acc); acc = __dp4a((int)x[4 * k4 + 3], (int)w4.w, acc);
        }
        const int8_t y = requant_conv(acc, cs);
        if (store_y) out[(int64_t)oc * P] = (uint8_t)y;
        if (out_s) out_s[(int64_t)oc * P] = __ldg(ts + y);
        if (out_z) out_z[(int64_t)oc * P] = __ldg(tz + y);
    }
}

static inline bool inplace_reg_ok(const ArenaView &v, const KOp &o) {
    return (o.ic == 32 || o.ic == 64 || o.ic == 128) && o.w >= 0 && (o.w & 3) == 0 &&
           o.w + (int64_t)o.oc * o.ic <= (int64_t)v.W && (size_t)o.oc * (o.ic / 4 + 1) * 4 <= 160 * 1024;
}
static inline void launch_inplace_reg(const ArenaView &v, const KOp &o, int n_img, cudaStream_t s) {
    const unsigned P = (unsigned)o.oh * o.ow;
    dim3 g((P + 127) / 128, n_img);
    const size_t smem = (size_t)o.oc * (o.ic / 4 + 1) * 4;
    static unsigned long long attr = 0; /* function attributes are per device */
    if (first_time_on_device(&attr)) {
        cudaFuncSetAttribute(k_conv1x1_inplace_reg<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
        cudaFuncSetAttribute(k_conv1x1_inplace_reg<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
        cudaFuncSetAttribute(k_conv1x1_inplace_reg<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
    }
    if (o.ic == 32) k_conv1x1_inplace_reg<8><<<g, 128, smem, s>>>(v, o);
    else if (o.ic == 64) k_conv1x1_inplace_reg<16><<<g, 128, smem, s>>>(v, o);
    else k_conv1x1_inplace_reg<32><<<g, 128, smem, s>>>(v, o);
}

static inline unsigned fast_grid(uint64_t items, unsigned per_block = 256) {
    uint64_t b = (items + per_block - 1) / per_block;
    return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(b, 148 * 16));
}

/* ---- selection + launch ---------------------------------------------------------- */
/* shifted flat copy whose source and destination are only 4-byte aligned relative to each other: 16-byte stores on the
 * destination's alignment, four 4-byte loads each; head and tail words one by one.  n4 = words to copy. */
__global__ void __launch_bounds__(256) k_shift_copy_d16(ArenaView v, KOp o) {
    const Img im = make_img(v, blockIdx.y);
    uint32_t *out = reinterpret_cast<uint32_t *>(im.s_minus_W + o.out + o.coff);
    const uint32_t *in = reinterpret_cast<const uint32_t *>(im.s_minus_W + o.in0);
    const int64_t n4 = (int64_t)o.n >> 2;
    const int head = (int)((16 - (reinterpret_cast<uintptr_t>(out) & 15)) & 15) >> 2; /* words before the first aligned 16 bytes */
    const int64_t nv = n4 > head ? (n4 - head) >> 2 : 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t *sp = in + head + 4 * i;
        reinterpret_cast<uint4 *>(out + head)[i] = make_uint4(sp[0], sp[1], sp[2], sp[3]);
    }
    if (blockIdx.x == 0) {
        if ((int)threadIdx.x < head && threadIdx.x < n4) out[threadIdx.x] = in[threadIdx.x];
        const int64_t done = head + 4 * nv;
        if (done + threadIdx.x < n4) out[done + threadIdx.x] = in[done + threadIdx.x];
        const int64_t b = (n4 << 2) + threadIdx.x; /* tail bytes */
        if (b < (int64_t)o.n) reinterpret_cast<uint8_t *>(out)[b] = reinterpret_cast<const uint8_t *>(in)[b];
    }
}

/* in-place concat input = periodic replication (SURVEY C.4b): A[out + j] = A[out + (j mod s)] for s <= j < n + s, with the
 * first s bytes (never written here) as the pattern.  Written as a fill: the pattern is expanded in shared memory to
 * L = lcm(s, 16) bytes, so every 16-byte aligned destination vector is one aligned 16-byte read of it; write-only traffic.
 * grid = (chunks, images), smem = L bytes. */
__global__ void __launch_bounds__(256) k_fill_periodic(ArenaView v, KOp o, int L) {
    extern __shared__ __align__(16) uint8_t fp_pat[];
    const Img im = make_img(v, blockIdx.y);
    uint8_t *base = im.s_minus_W + o.out; /* pattern at [0, s), destination [s, s + n) */
    const int s = o.coff;
    for (int k = threadIdx.x; k < L; k += blockDim.x) fp_pat[k] = base[k % s];
    __syncthreads();
    const int64_t lo = s, hi = (int64_t)s + (int64_t)o.n;
    /* 16-byte vectors relative to `base` rounded down: base itself is 16-byte aligned? not necessarily -> align on the address */
    const uintptr_t b0 = reinterpret_cast<uintptr_t>(base);
    const int64_t a_lo = (int64_t)(((b0 + lo + 15) & ~(uintptr_t)15) - b0), a_hi = (int64_t)(((b0 + hi) & ~(uintptr_t)15) - b0);
    if (a_lo < a_hi) {
        const int64_t nv = (a_hi - a_lo) >> 4;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x) {
            const int64_t j = a_lo + (i << 4); /* offset from base; the pattern phase of byte j is j mod s */
            const int ph = (int)(j % L);
            uint4 w;
            if ((ph & 15) == 0) w = *reinterpret_cast<const uint4 *>(fp_pat + ph);
            else { /* base not 16-byte aligned relative to the period: assemble bytewise (rare) */
                uint8_t t[16];
                for (int b = 0; b < 16; b++) t[b] = fp_pat[(ph + b) % L];
                w = *reinterpret_cast<const uint4 *>(t);
            }
            *reinterpret_cast<uint4 *>(base + j) = w;
        }
    }
    if (blockIdx.x == 0) { /* ragged ends */
        const int64_t e_lo = a_lo < a_hi ? a_lo : hi, s_hi = a_lo < a_hi ? a_hi : hi;
        for (int64_t j = lo + threadIdx.x; j < e_lo; j += blockDim.x) base[j] = fp_pat[j % L];
        for (int64_t j = s_hi + threadIdx.x; j < hi; j += blockDim.x) base[j] = fp_pat[j % L];
    }
}

static inline bool aligned16(int64_t x) { return (x & 15) == 0; }

static inline bool fast_flat_ok(const ArenaView &v, const KOp &o) {
    const int64_t W = (int64_t)v.W;
    if (o.mode != EXEC_PARALLEL || o.n < 64 || o.in0 < W || o.out < W) return false;
    switch (o.kind) {
        case OP_SIGMOID_I8: case OP_RELU_I8: case OP_LUT_I8:
            return o.lut >= 0 && aligned16(o.in0 - W) && aligned16(o.out - W);
        case OP_MUL_I8: case OP_ADD_I8:
            return o.in1 >= W && aligned16(o.in0 - W) && aligned16(o.in1 - W) && aligned16(o.out - W);
        default: return false;
    }
}
static inline void launch_fast_flat(const ArenaView &v, const KOp &o, int n_img, cudaStream_t s) {
    dim3 g(fast_grid(o.n >> 4), n_img);
    if (o.kind == OP_MUL_I8 || o.kind == OP_ADD_I8) k_bin16<<<g, 256, 0, s>>>(v, o);
    else k_lut16<<<g, 256, 0, s>>>(v, o);
}

/* maxpool / upsample over 4 channels per thread (reference src/mars/mars_runtime.c:934-956, :1027-1040; NHWC indexing of
 * shape[1..3] whatever the tag, SURVEY C.4): signed per-byte max with __vmaxs4, window clipped at the bottom/right edge,
 * pads ignored, exactly like the point functions. */
__global__ void __launch_bounds__(256) k_spatial_vec4(ArenaView v, KOp o) {
    const Img im = make_img(v, blockIdx.y);
    const uint32_t *in = reinterpret_cast<const uint32_t *>(im.s_minus_W + o.in0);
    uint32_t *out = reinterpret_cast<uint32_t *>(im.s_minus_W + o.out);
    const int c4 = o.ic >> 2;
    const int64_t total = (int64_t)o.oh * o.ow * c4;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(t % c4);
        const int64_t p = t / c4;
        const int oh = (int)(p / o.ow), ow = (int)(p - (int64_t)oh * o.ow);
        uint32_t r;
        if (o.kind == OP_MAXPOOL) {
            r = 0x80808080u; /* four times -128 */
            const int ih0 = oh * o.sh, iw0 = ow * o.sw;
            const int ky = min(o.kh, o.ih - ih0), kx = min(o.kw, o.iw - iw0);
            for (int y = 0; y < ky; y++) {
                const uint32_t *row = in + ((int64_t)(ih0 + y) * o.iw + iw0) * c4 + c;
                for (int x = 0; x < kx; x++) r = __vmaxs4(r, row[(int64_t)x * c4]);
            }
        } else {
            int ih = oh / o.sh; if (ih >= o.ih) ih = o.ih - 1;
            int iw = ow / o.sw; if (iw >= o.iw) iw = o.iw - 1;
            r = in[((int64_t)ih * o.iw + iw) * c4 + c];
        }
        out[t] = r;
    }
}

/* stride-1 maxpool, separable: a block stages a strip of input rows in shared memory, takes the horizontal window
 * maximum (kw loads per word instead of kh*kw), then the vertical one.  Rows are iw*ic bytes = RW words; windows are
 * clipped at the right / bottom edge and pads are ignored, exactly like maxpool_point.  grid = (strips, images),
 * smem = 2 * (TH + kh - 1) * RW words. */
__global__ void __launch_bounds__(256) k_maxpool_sep(ArenaView v, KOp o, int TH) {
    extern __shared__ uint32_t mp_smem[];
    const Img im = make_img(v, blockIdx.y);
    const uint32_t *in = reinterpret_cast<const uint32_t *>(im.s_minus_W + o.in0);
    uint32_t *out = reinterpret_cast<uint32_t *>(im.s_minus_W + o.out);
    const int c4 = o.ic >> 2, RW = o.iw * c4, OW = o.ow * c4;
    const int r0 = blockIdx.x * TH, nout = min(TH, o.oh - r0), nin = min(nout + o.kh - 1, o.ih - r0);
    uint32_t *raw = mp_smem, *hm = mp_smem + (TH + o.kh - 1) * RW;
    for (int t = threadIdx.x; t < nin * RW; t += blockDim.x) raw[t] = in[(int64_t)r0 * RW + t];
    __syncthreads();
    for (int t = threadIdx.x; t < nin * OW; t += blockDim.x) { /* horizontal: output column x covers input columns x .. x+kw-1 */
        const int y = t / OW, xw = t - y * OW, x = xw / c4;
        const int kx = min(o.kw, o.iw - x);
        uint32_t r = 0x80808080u;
        const uint32_t *p = raw + y * RW + xw;
        for (int k = 0; k < kx; k++) r = __vmaxs4(r, p[k * c4]);
        hm[y * OW + xw] = r;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < nout * OW; t += blockDim.x) { /* vertical: output row y covers input rows y .. y+kh-1 */
        const int y = t / OW, xw = t - y * OW;
        const int ky = min(o.kh, nin - y);
        uint32_t r = 0x80808080u;
        for (int k = 0; k < ky; k++) r = __vmaxs4(r, hm[(y + k) * OW + xw]);
        out[(int64_t)(r0 + y) * OW + xw] = r;
    }
}

/* 5x5 stride-1 maxpool (the SPPF pools): one thread per output column word walks down the rows with the horizontal maxima
 * of the current and the next four rows in registers -- no shared memory, no barriers, long-lived threads whose loads for
 * the following rows are in flight while the current row is reduced.  Same clipping as k_maxpool_sep (right / bottom edge,
 * pads ignored; -128 is the identity).  grid = (column blocks, row chunks, images).
 * The maxima are taken on sign-extended 16-bit pairs: __vmaxs4 is emulated on sm_100a (the first version of this kernel was
 * ALU bound at 113 instructions per output word, ncu: alu 75 %), VIMNMX3.S16 is one instruction for three operands. */
struct S16x4 { uint32_t lo, hi; }; /* bytes 0,1 and 2,3 of a word as two s16x2 words */
__device__ __forceinline__ S16x4 s16x4_from_s8x4(uint32_t w) { return {__byte_perm(w, 0u, 0x9180u), __byte_perm(w, 0u, 0xB3A2u)}; }
__device__ __forceinline__ S16x4 s16x4_max3(S16x4 a, S16x4 b, S16x4 c) { return {__vimax3_s16x2(a.lo, b.lo, c.lo), __vimax3_s16x2(a.hi, b.hi, c.hi)}; }
__device__ __forceinline__ uint32_t s8x4_from_s16x4(S16x4 a) { return __byte_perm(a.lo, a.hi, 0x6420u); }
__global__ void __launch_bounds__(128) k_maxpool5_col(ArenaView v, KOp o, int rows_per_block) {
    const Img im = make_img(v, blockIdx.z);
    const int c4 = o.ic >> 2, RW = o.iw * c4, OW = o.ow * c4;
    const int xw = blockIdx.x * 128 + threadIdx.x;
    if (xw >= OW) return;
    const int x = xw / c4, kx = min(5, o.iw - x);
    const int y0 = blockIdx.y * rows_per_block, y1 = min(y0 + rows_per_block, o.oh);
    const uint32_t *in = reinterpret_cast<const uint32_t *>(im.s_minus_W + o.in0) + (x * c4 + (xw - x * c4));
    uint32_t *out = reinterpret_cast<uint32_t *>(im.s_minus_W + o.out) + xw + (int64_t)y0 * OW;
    const uint32_t NEG = 0x80808080u;
    /* word offsets of the window's columns; columns past the right edge re-read column 0 (max is idempotent) */
    const int o1 = kx > 1 ? c4 : 0, o2 = kx > 2 ? 2 * c4 : 0, o3 = kx > 3 ? 3 * c4 : 0, o4 = kx > 4 ? 4 * c4 : 0;
    const uint32_t *p = in + (int64_t)y0 * RW;
    int r = y0;
    const uint32_t *const p_last = in + (int64_t)(o.ih - 1) * RW;
    auto hmax = [&]() -> S16x4 { /* horizontal window maximum of input row r (then advances); rows past the bottom edge do not exist */
        /* no branch: a row past the edge re-reads the last row and is replaced by the identity afterwards, so the loads of the
         * unrolled rows are independent and all in flight together (the branchy version was latency bound: one row per round trip) */
        const bool ok = r < o.ih;
        const uint32_t *q = ok ? p : p_last;
        const uint32_t w0 = q[0], w1 = q[o1], w2 = q[o2], w3 = q[o3], w4 = q[o4];
        const S16x4 a = s16x4_from_s8x4(ok ? w0 : NEG), b = s16x4_from_s8x4(w1), c = s16x4_from_s8x4(w2), d = s16x4_from_s8x4(w3), e = s16x4_from_s8x4(w4);
        S16x4 m = s16x4_max3(s16x4_max3(a, b, c), d, e);
        if (!ok) m = s16x4_from_s8x4(NEG);
        r++; p += RW;
        return m;
    };
    S16x4 h0 = hmax(), h1 = hmax(), h2 = hmax(), h3 = hmax();
#pragma unroll 4
    for (int y = y0; y < y1; y++) {
        const S16x4 h4 = hmax();
        *out = s8x4_from_s16x4(s16x4_max3(s16x4_max3(h0, h1, h2), h3, h4));
        out += OW;
        h0 = h1; h1 = h2; h2 = h3; h3 = h4;
    }
}

/* nearest upsample (reference src/mars/mars_runtime.c:1027-1040: ih = min(oh / sh, ih - 1), same for columns): one block
 * per (output row, image); a thread produces consecutive output words (fully coalesced stores), reading the input row
 * through L1.  Divisions by multiplication. */
#define UPS_ROWS 8
__global__ void __launch_bounds__(256) k_upsample_rep(ArenaView v, KOp o) {
    const Img im = make_img(v, blockIdx.y);
    const int c4 = o.ic >> 2, orw = o.ow * c4;
    const unsigned m_c4 = 0xFFFFFFFFu / (unsigned)c4 + 1u, m_sw = 0xFFFFFFFFu / (unsigned)o.sw + 1u; /* floor(a / d) = umulhi(a, m) */
    /* UPS_ROWS output rows per block: the rows of the small planes are a few hundred bytes, one block per row was all launch overhead */
    for (int row = blockIdx.x * UPS_ROWS; row < min((int)(blockIdx.x + 1) * UPS_ROWS, o.oh); row++) {
        const uint32_t *in = reinterpret_cast<const uint32_t *>(im.s_minus_W + o.in0) + (int64_t)min(row / o.sh, o.ih - 1) * o.iw * c4;
        uint32_t *out = reinterpret_cast<uint32_t *>(im.s_minus_W + o.out) + (int64_t)row * orw;
        for (int w = threadIdx.x; w < orw; w += blockDim.x) {
            const int xo = (int)__umulhi((unsigned)w, m_c4), c = w - xo * c4;
            const int xi = min(o.sw == 1 ? xo : (int)__umulhi((unsigned)xo, m_sw), o.iw - 1);
            out[w] = in[xi * c4 + c];
        }
    }
}

/* concat input with fewer channels than the output (a real channel concat: NHWC-convention models, reference
 * src/mars/mars_runtime.c:963-1000): pixel p copies its ic bytes to out[p * oc + coff]; 16 bytes per thread, consecutive
 * threads walk the channel chunks of a pixel and then the next pixel (coalesced on both sides) */
__global__ void __launch_bounds__(256) k_concat_strided16(ArenaView v, KOp o) {
    const Img im = make_img(v, blockIdx.y);
    const uint4 *in = reinterpret_cast<const uint4 *>(im.s_minus_W + o.in0);
    uint8_t *out = im.s_minus_W + o.out + o.coff;
    const int cpp = o.ic >> 4; /* 16-byte chunks per pixel */
    const unsigned m_cpp = 0xFFFFFFFFu / (unsigned)cpp + 1u;
    const int64_t total = (int64_t)(o.n >> 4);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned px = cpp == 1 ? (unsigned)i : __umulhi((unsigned)i, m_cpp), c = (unsigned)i - px * (unsigned)cpp;
        *reinterpret_cast<uint4 *>(out + (int64_t)px * o.oc + 16 * c) = in[i];
    }
}

static inline bool fast_spatial_ok(const ArenaView &v, const KOp &o) {
    if (o.mode != EXEC_PARALLEL || o.out < (int64_t)v.W) return false;
    if (o.kind == OP_CONCAT && o.ic != o.oc) /* strided: 16-byte chunks on both sides, 32-bit chunk index */
        return o.in0 >= (int64_t)v.W && o.ic > 0 && o.ic % 16 == 0 && o.oc % 16 == 0 && o.coff % 16 == 0 && o.n >= 64 && o.n < (1ull << 35) &&
               (o.n >> 4) < 0x7FFFFFFFull && ((o.in0 - (int64_t)v.W) & 15) == 0 && ((o.out - (int64_t)v.W) & 15) == 0;
    if (o.kind == OP_CONCAT) return o.in0 >= (int64_t)v.W && o.ic == o.oc && o.n >= 64;
    if (o.kind == OP_CONCAT_PERIODIC) return o.coff > 0 && o.n >= 64;
    if (o.kind == OP_MAXPOOL || o.kind == OP_UPSAMPLE)
        return o.in0 >= (int64_t)v.W && o.ic > 0 && o.ic % 4 == 0 && ((o.in0 - (int64_t)v.W) & 3) == 0 && ((o.out - (int64_t)v.W) & 3) == 0 &&
               o.ih > 0 && o.iw > 0 && o.sh > 0 && o.sw > 0;
    return false;
}
/* the one-load-many-stores kernel needs input and output ranges that do not touch (the planner only sends hazard-free ops here,
 * but the check is cheap) */
static inline bool upsample_ranges_overlap(const KOp &o) {
    const int64_t ib = (int64_t)o.ih * o.iw * o.ic, ob = (int64_t)o.oh * o.ow * o.ic;
    return o.in0 < o.out + ob && o.out < o.in0 + ib;
}
/* nearest upsample whose output is covered by whole input pixels (oh <= ih * sh, ow <= iw * sw, so that y / sh and x / sw never
 * clamp): a thread owns one INPUT word and stores it to its (up to) sh x sw output positions -- one load, sh * sw stores and one
 * index split per input word instead of two divisions per output word (ncu on k_upsample_rep: alu 64 %, xu 28 %, 47
 * instructions per output warp-word).  Only the input rows / columns the output reads are visited. */
__global__ void __launch_bounds__(256) k_upsample_exact(ArenaView v, KOp o) {
    const Img im = make_img(v, blockIdx.z);
    const int c4 = o.ic >> 2, irw = o.iw * c4, orw = o.ow * c4;
    const int w = blockIdx.x * 256 + threadIdx.x, yi = blockIdx.y;
    const int xi = w / c4, c = w - xi * c4;
    if (xi * o.sw >= o.ow) return; /* (also: w beyond the input row) */
    const uint32_t val = (reinterpret_cast<const uint32_t *>(im.s_minus_W + o.in0))[(int64_t)yi * irw + w];
    uint32_t *out = reinterpret_cast<uint32_t *>(im.s_minus_W + o.out) + (int64_t)yi * o.sh * orw + xi * o.sw * c4 + c;
    const int ny = min(o.sh, o.oh - yi * o.sh), nx = min(o.sw, o.ow - xi * o.sw);
    for (int dy = 0; dy < ny; dy++, out += orw)
        for (int dx = 0; dx < nx; dx++) out[dx * c4] = val;
}

static inline void launch_fast_spatial(const ArenaView &v, const KOp &o, int n_img, cudaStream_t s) {
    if (o.kind == OP_MAXPOOL && o.sh == 1 && o.sw == 1 && o.kh == 5 && o.kw == 5 && o.oh <= o.ih && o.ow <= o.iw && n_img <= 65535) {
        const int OW = o.ow * (o.ic >> 2), rows = 64;
        k_maxpool5_col<<<dim3((OW + 127) / 128, (o.oh + rows - 1) / rows, n_img), 128, 0, s>>>(v, o, rows);
        return;
    }
    if (o.kind == OP_MAXPOOL && o.sh == 1 && o.sw == 1 && o.kh >= 1 && o.kw >= 1 && o.oh <= o.ih && o.ow <= o.iw) {
        const int RW = o.iw * (o.ic >> 2);
        int TH = 32;
        while (TH > 1 && (size_t)2 * (TH + o.kh - 1) * RW * 4 > 96 * 1024) TH >>= 1;
        if ((size_t)2 * (TH + o.kh - 1) * RW * 4 <= 96 * 1024) {
            static unsigned long long attr = 0;
            if (first_time_on_device(&attr)) cudaFuncSetAttribute(k_maxpool_sep, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
            dim3 g((o.oh + TH - 1) / TH, n_img);
            k_maxpool_sep<<<g, 256, (size_t)2 * (TH + o.kh - 1) * RW * 4, s>>>(v, o, TH);
            return;
        }
    }
    if (o.kind == OP_UPSAMPLE && o.sh >= 1 && o.sw >= 1 && o.sw <= 4 && o.sh <= 4 && o.oh <= o.ih * o.sh && o.ow <= o.iw * o.sw && o.oh <= 65535 * o.sh &&
        n_img <= 65535 && !upsample_ranges_overlap(o)) {
        const int rows_in = (o.oh + o.sh - 1) / o.sh, cols_in = (o.ow + o.sw - 1) / o.sw; /* the input rows / pixels the output reads */
        k_upsample_exact<<<dim3((cols_in * (o.ic >> 2) + 255) / 256, rows_in, n_img), 256, 0, s>>>(v, o);
        return;
    }
    if (o.kind == OP_UPSAMPLE && o.oh <= 65535 && (long long)o.ow * (o.ic >> 2) < 65536) {
        k_upsample_rep<<<dim3((o.oh + UPS_ROWS - 1) / UPS_ROWS, n_img), 256, 0, s>>>(v, o);
        return;
    }
    if (o.kind == OP_MAXPOOL || o.kind == OP_UPSAMPLE) {
        /* one output word per thread: the loads of a thread are dependent, so parallelism comes from the number of warps */
        dim3 g((unsigned)(((uint64_t)o.oh * o.ow * (o.ic >> 2) + 255) / 256), n_img);
        k_spatial_vec4<<<g, 256, 0, s>>>(v, o);
        return;
    }
    if (o.kind == OP_CONCAT && o.ic != o.oc) {
        k_concat_strided16<<<dim3(fast_grid(o.n >> 4), n_img), 256, 0, s>>>(v, o);
        return;
    }
    const int periodic = o.kind == OP_CONCAT_PERIODIC;
    if (periodic && o.coff > 0 && o.n >= 4096) {
        int g = o.coff, b = 16;
        while (b) { int t = g % b; g = b; b = t; } /* gcd(coff, 16) */
        const long long L = (long long)o.coff / g * 16;
        if (L <= 16384) {
            k_fill_periodic<<<dim3(fast_grid(o.n >> 4), n_img), 256, L, s>>>(v, o, (int)L);
            return;
        }
    }
    const int64_t dst = o.out + o.coff, src = periodic ? o.out : o.in0;
    /* slot bases are 1 KiB aligned and W-relative offsets keep their low bits: alignment of the
     * arena offsets minus W is what counts, and v.W is subtracted from both alike */
    const int64_t rel_d = dst - (int64_t)v.W, rel_s = src - (int64_t)v.W;
    int vec = 1;
    if (((rel_d | rel_s) & 15) == 0 && (!periodic || (o.coff & 15) == 0)) vec = 16;
    else if (((rel_d | rel_s) & 3) == 0 && (!periodic || (o.coff & 3) == 0)) vec = 4;
    dim3 g(fast_grid(o.n / vec), n_img);
    if (vec == 16) k_shift_copy<16><<<g, 256, 0, s>>>(v, o, periodic);
    else if (vec == 4 && !periodic && o.n >= 1024) k_shift_copy_d16<<<dim3(fast_grid(o.n / 16), n_img), 256, 0, s>>>(v, o);
    else if (vec == 4) k_shift_copy<4><<<g, 256, 0, s>>>(v, o, periodic);
    else k_shift_copy<1><<<g, 256, 0, s>>>(v, o, periodic);
}

static inline bool fast_conv_nchw_ok(const KOp &) { return false; }
static inline void launch_fast_conv_nchw(const ArenaView &, const KOp &, int, cudaStream_t) {}

} // namespace marsb200
