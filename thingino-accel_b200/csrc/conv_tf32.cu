/*
 * conv_tf32.cu -- float32 convolution as an implicit GEMM on tcgen05 (kind::tf32, fp32 accumulators in TMEM), sm_100a.
 *
 * Replaces the reference's conv2d_float32_mxu (src/mars/mxu_conv.c:673-710: fp32 NCHW x OIHW, `sum = bias; sum += in * w` in
 * ic -> kh -> kw order, no activation) for hazard-free layers of float32 models.  This is the TOLERANCE path of the north
 * star (<= 1e-3 relative on the logits); the exact-order FFMA-free kernel (kernels_exact.cuh, conv_f32_nchw_point) stays the
 * bit-exact control and is what mars_b200_set_f32_mode(model, 0) selects.
 *
 *   GEMM view   D[M = 128 pixels][N = out channels] = A[M][K] * B[N][K],  K = taps x in channels, both operands K-major.
 *   A operand   a channel-innermost fp32 copy of the input written by a pre-pass (k_f32_to_kmajor): rows padded with k-1
 *               zero columns for stride 1, a 2x2 phase split for stride 2, so that a kernel tap is a flat row shift (the
 *               layouts of conv_tc.cu's int8 copies with 4-byte elements), channels padded to a multiple of 8.
 *   precision   kind::tf32 uses 10 mantissa bits of each fp32 operand.  Mode 1 (tf32): the pre-pass and the weight repack round
 *               to nearest tf32 first (unbiased, ~5e-4 relative per product).  Mode 2 (tf32x3, default): every operand is
 *               split exactly, x = hi + lo with hi = x rounded to tf32 (stored with its 13 low bits zero, so the tensor core
 *               sees exactly hi whether it truncates or rounds -- measured: passing the raw x as `hi` left 2e-4 of error)
 *               and lo = x - hi, and three MMAs per k-step accumulate hi*hi + lo*hi + hi*lo -- ~2^-21 relative per product,
 *               fp32 accumulation, so the result differs from the reference's sequential fp32 sum by summation order only.
 *   epilogue    + fp32 bias, one coalesced 128-byte store per channel and warp into the NCHW output plane.
 *   roles       warps 0..7 epilogue (two per TMEM lane quadrant), warp 8 = TMEM allocator + MMA issuer, warp 9 = TMA producer;
 *               persistent CTAs, one per SM, walking (image, M tile, N tile) units.
 */
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "conv_tf32.h"
#include "tc_common.cuh"

namespace marsb200 {

namespace {

constexpr int F_EPI = 8;

struct F32Params {
    int Co, Ho, Wo, Wp, mflat, plane;
    int n_tile, n_tiles, m_tiles, ntaps, ksteps, stages, acc_bufs, tmem_cols, x3;
    uint32_t idesc, layout, bk; /* bk: bytes of K per pipeline step (128 / 64 / 32) */
    uint32_t a_tile_bytes, b_tile_bytes, stage_bytes;
    int a_shift[TC_MAX_TAPS];
    int lo_rows;             /* row offset of the `lo` copy inside the A tensor map (tf32x3) */
    const float *bias;
    uint8_t *out_base;       /* slot 0 of the launch */
    unsigned long long slot_stride;
    long long out_off;
    unsigned wp_magic;
    int img0, n_img;
};

__global__ void __launch_bounds__((F_EPI + 2) * 32, 1)
k_conv_tf32(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const F32Params p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_full[8], bar_empty[8], bar_tfull[4], bar_tempty[4];
    __shared__ uint32_t tmem_base_slot;
    __shared__ float s_bias[TC_MAX_CO];
    __shared__ int s_shift[TC_MAX_TAPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int tiles_per_img = p.m_tiles * p.n_tiles;
    const int nsteps = p.ntaps * p.ksteps;
    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; s++) { mbar_init(smem_u32(&bar_full[s]), 1); mbar_init(smem_u32(&bar_empty[s]), 1); }
        for (int b = 0; b < p.acc_bufs; b++) { mbar_init(smem_u32(&bar_tfull[b]), 1); mbar_init(smem_u32(&bar_tempty[b]), F_EPI); }
        mbar_fence_init();
    }
    if (warp == F_EPI) tmem_alloc(smem_u32(&tmem_base_slot), (uint32_t)p.tmem_cols);
    for (int i = threadIdx.x; i < TC_MAX_CO; i += blockDim.x) s_bias[i] = (p.bias && i < p.Co) ? p.bias[i] : 0.0f;
    if (threadIdx.x < TC_MAX_TAPS) s_shift[threadIdx.x] = p.a_shift[threadIdx.x];
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_d = tmem_base_slot;

    if (warp < F_EPI) {
        /* ===== epilogue: thread = output pixel (TMEM lane), 16 channels per TMEM load ===== */
        const int quad = warp & 3, part = warp >> 2, parts = F_EPI >> 2;
        const int r = quad * 32 + lane;
        const int n_units = p.n_tile >> 4;
        const long long plane = p.plane;
        const uint32_t acc_lane = tmem_d + ((uint32_t)(quad * 32) << 16);
        int ab = 0, aph = 0;
        for (TileIter ti(blockIdx.x, gridDim.x, tiles_per_img); ti.img < p.n_img; ti.next()) {
            mbar_wait_relaxed(smem_u32(&bar_tfull[ab]), aph);
            tcgen05_fence_after();
            const int mt = p.n_tiles == 1 ? ti.rem : ti.rem / p.n_tiles, n0 = (ti.rem - mt * p.n_tiles) * p.n_tile;
            const int q = mt * TC_BM + r;
            const int oh = (int)__umulhi((unsigned)q, p.wp_magic), ow = q - oh * p.Wp;
            const bool valid = q < p.mflat && ow < p.Wo;
            float *o = reinterpret_cast<float *>(p.out_base + (unsigned long long)ti.img * p.slot_stride + p.out_off) + ((long long)n0 * plane + (long long)oh * p.Wo + ow);
            for (int u = part; u < n_units; u += parts) {
                uint32_t v[16];
                tmem_ld16_issue(acc_lane + (uint32_t)(ab * p.n_tile + u * 16), v);
                tmem_ld_wait(v);
                if (u + parts >= n_units) { /* last read of this accumulator by this warp */
                    tcgen05_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(smem_u32(&bar_tempty[ab]));
                }
                const int c0 = n0 + u * 16;
                if (valid) {
#pragma unroll
                    for (int j = 0; j < 16; j++)
                        if (c0 + j < p.Co) o[(long long)(u * 16 + j) * plane] = __fadd_rn(__uint_as_float(v[j]), s_bias[c0 + j]);
                }
            }
            if (part >= n_units) { /* narrow N tile: this warp only releases */
                __syncwarp();
                if (lane == 0) mbar_arrive(smem_u32(&bar_tempty[ab]));
            }
            if (++ab == p.acc_bufs) { ab = 0; aph ^= 1; }
        }
    } else if (warp == F_EPI) {
        if (lane == 0) { /* ===== MMA issuer ===== */
            const uint32_t hi_k = ((8u * p.bk) >> 4) | (1u << 14) | (p.layout << 29); /* SBO = 8 rows, version 1, swizzle */
            const uint32_t a_lo0 = (smem_base >> 4) | (1u << 16);
            const uint32_t st16 = p.stage_bytes >> 4, at16 = p.a_tile_bytes >> 4, bt16 = p.b_tile_bytes >> 4;
            const int nj = (int)(p.bk >> 5); /* K = 8 tf32 = 32 bytes per MMA */
            int s = 0, ph = 0, buf = 0, aph = 1;
            for (TileIter ti(blockIdx.x, gridDim.x, tiles_per_img); ti.img < p.n_img; ti.next()) {
                mbar_wait(smem_u32(&bar_tempty[buf]), aph);
                tcgen05_fence_after();
                const uint32_t acc = tmem_d + (uint32_t)(buf * p.n_tile);
                for (int i = 0; i < nsteps; i++) {
                    mbar_wait(smem_u32(&bar_full[s]), ph);
                    tcgen05_fence_after();
                    /* stage: [A hi | A lo | B hi | B lo] (x3) or [A | B] */
                    const uint32_t a_hi_d = a_lo0 + s * st16, a_lo_d = a_hi_d + at16;
                    const uint32_t b_hi_d = a_hi_d + (p.x3 ? 2u : 1u) * at16, b_lo_d = b_hi_d + bt16;
                    for (int j = 0; j < nj; j++) {
                        umma_tf32(acc, a_hi_d + 2u * j, hi_k, b_hi_d + 2u * j, hi_k, p.idesc, (uint32_t)((i | j) != 0));
                        if (p.x3) {
                            umma_tf32(acc, a_lo_d + 2u * j, hi_k, b_hi_d + 2u * j, hi_k, p.idesc, 1u);
                            umma_tf32(acc, a_hi_d + 2u * j, hi_k, b_lo_d + 2u * j, hi_k, p.idesc, 1u);
                        }
                    }
                    umma_commit(smem_u32(&bar_empty[s]));
                    if (++s == p.stages) { s = 0; ph ^= 1; }
                }
                umma_commit(smem_u32(&bar_tfull[buf]));
                if (++buf == p.acc_bufs) { buf = 0; aph ^= 1; }
            }
        }
    } else if (lane == 0) { /* ===== TMA producer ===== */
        const uint32_t tx = (p.x3 ? 2u : 1u) * (p.a_tile_bytes + (uint32_t)p.n_tile * p.bk);
        int s = 0, ph = 1;
        for (TileIter ti(blockIdx.x, gridDim.x, tiles_per_img); ti.img < p.n_img; ti.next()) {
            const int mt = p.n_tiles == 1 ? ti.rem : ti.rem / p.n_tiles, n0 = (ti.rem - mt * p.n_tiles) * p.n_tile;
            const int q0 = mt * TC_BM, zc = p.img0 + ti.img;
            for (int tap = 0; tap < p.ntaps; tap++) {
                const int qa = q0 + s_shift[tap];
                for (int kb = 0; kb < p.ksteps; kb++) {
                    mbar_wait(smem_u32(&bar_empty[s]), ph);
                    const uint32_t full = smem_u32(&bar_full[s]), dst = smem_base + s * p.stage_bytes;
                    mbar_expect_tx(full, tx);
                    tma_load_3d(dst, &mapA, full, kb * (int)p.bk, qa, zc);
                    if (p.x3) {
                        tma_load_3d(dst + p.a_tile_bytes, &mapA, full, kb * (int)p.bk, qa + p.lo_rows, zc);
                        tma_load_3d(dst + 2 * p.a_tile_bytes, &mapB, full, kb * (int)p.bk, n0, 2 * tap);
                        tma_load_3d(dst + 2 * p.a_tile_bytes + p.b_tile_bytes, &mapB, full, kb * (int)p.bk, n0, 2 * tap + 1);
                    } else tma_load_3d(dst + p.a_tile_bytes, &mapB, full, kb * (int)p.bk, n0, tap);
                    if (++s == p.stages) { s = 0; ph ^= 1; }
                }
            }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == F_EPI) {
        tcgen05_fence_after();
        tmem_dealloc(tmem_d, (uint32_t)p.tmem_cols);
    }
}

__device__ __forceinline__ float tf32_round(float x) { /* round to nearest, ties away (cvt.rna); the result has 13 zero low bits */
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

/* pre-pass: arena NCHW fp32 -> channel-innermost fp32 copy (source pixel: copy_src_pixel): dst[pix][c] for
 * pix < npix, c < Cp (channels >= C are zero); split != 0: a second copy behind the first (and `guard` zero rows) holds lo = x - hi;
 * split == 0: the values are rounded to tf32.  32 pixels x 32 channels per block through shared memory. */
__global__ void __launch_bounds__(256) k_f32_to_kmajor(const uint8_t *src_base, unsigned long long src_stride, uint8_t *dst_base, unsigned long long dst_stride,
                                                      int C, int Cp, int H, int W, int Wp, int plane, int npix, int stride2, int pt, int pl, int split, int guard) {
    __shared__ float tile[32][33];
    const float *src = reinterpret_cast<const float *>(src_base + (unsigned long long)blockIdx.z * src_stride);
    float *dst = reinterpret_cast<float *>(dst_base + (unsigned long long)blockIdx.z * dst_stride);
    const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    {
        const int pix = p0 + tx;
        int ih = -1, iw = -1;
        if (pix < npix) copy_src_pixel(pix, stride2, Wp, plane, pt, pl, ih, iw);
        const bool inb = ih >= 0 && ih < H && iw >= 0 && iw < W;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int c = c0 + ty + 8 * k;
            tile[ty + 8 * k][tx] = (inb && c < C) ? src[((long long)c * H + ih) * W + iw] : 0.0f;
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int pix = p0 + ty + 8 * k, c = c0 + tx;
        if (pix < npix + guard && c < Cp) { /* rows npix .. npix+guard-1: zeros (taps of the last tiles run past the copy; with two
                                             * copies in one tensor map the TMA's out-of-bounds zero fill only protects the second) */
            const float x = tile[tx][ty + 8 * k];
            if (split) {
                const float hi = tf32_round(x); /* stored with its 13 low bits zero: whatever the tensor core does with them, it sees hi */
                dst[(long long)pix * Cp + c] = hi;
                if (pix < npix) dst[((long long)npix + guard + pix) * Cp + c] = __fsub_rn(x, hi); /* exact; |lo| <= 2^-11 |x| */
            } else if (pix < npix) dst[(long long)pix * Cp + c] = tf32_round(x);
        }
    }
}

/* OIHW fp32 -> [tap][2][Co_pad][Cip] (split: hi = w, lo = w - trunc(w)) or [tap][Co_pad][Cip] (rounded), zero padded */
__global__ void k_repack_f32(const float *w, float *dst, int Co, int Co_pad, int Ci, int Cip, int ntaps, int split) {
    const long long per = (long long)Co_pad * Cip, total = (long long)ntaps * per;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int ci = (int)(i % Cip);
        const long long r = i / Cip;
        const int co = (int)(r % Co_pad), tap = (int)(r / Co_pad);
        const float x = (co < Co && ci < Ci) ? w[((long long)co * Ci + ci) * ntaps + tap] : 0.0f;
        if (split) {
            const float hi = tf32_round(x);
            dst[(2ll * tap) * per + (long long)co * Cip + ci] = hi;
            dst[(2ll * tap + 1) * per + (long long)co * Cip + ci] = __fsub_rn(x, hi);
        } else dst[(long long)tap * per + (long long)co * Cip + ci] = tf32_round(x);
    }
}

struct F32Geom {
    bool ok = false;
    PixelCopy copy;
    int ntaps = 0, Cp = 0, guard = 0;
    size_t scratch_bytes = 0;
};
F32Geom f32_geometry(const Op &o, int mode) {
    F32Geom g;
    if (mode <= 0 || o.kind != OP_CONV_F32_NCHW || o.mode != EXEC_PARALLEL || o.xlat) return g;
    if (o.oc < 1 || o.sh != o.sw || o.sh < 1 || o.sh > 2 || o.kh < 1 || o.kh != o.kw) return g;
    if (o.oh <= 0 || o.ow <= 0 || o.ih <= 0 || o.iw <= 0 || o.ic <= 0 || round_up(o.oc, 16) > TC_MAX_CO) return g;
    if (o.pt < 0 || o.pl < 0 || o.pl >= o.kw || o.pt >= o.kh) return g;
    if ((long long)o.oh * o.ow * o.oc * o.ic * o.kh * o.kw < (1ll << 22)) return g; /* tiny layers stay on the exact kernel */
    g.ntaps = o.kh * o.kw;
    if (g.ntaps > TC_MAX_TAPS) return g;
    g.Cp = round_up(o.ic, 8);
    g.copy = pixel_copy(o);
    const PixelCopy &c = g.copy;
    if (!c.mode) return g;
    if ((unsigned long long)(o.oh * (long long)c.Wp + 2 * c.Wp) * (unsigned)c.Wp >= (1ull << 32)) return g;
    /* zero rows between the hi and the lo copy: the deepest tap of the last M tile */
    g.guard = mode >= 2 ? TC_BM + (c.mode == 1 ? (o.kh - 1) * c.Wp + o.kw - 1 : ((o.kh - 1) / 2) * c.Wp + (o.kw - 1) / 2) + 8 : 0;
    g.scratch_bytes = (size_t)(mode >= 2 ? 2 * c.npix + g.guard : c.npix) * g.Cp * 4;
    g.ok = true;
    return g;
}

} // namespace

struct F32PlanImpl {
    CUtensorMap mapA, mapB;
    F32Params p;
    PixelCopy copy;
    int C = 0, Cp = 0, H = 0, W = 0, split = 0, guard = 0, sms = 148;
    const uint8_t *src_slot0 = nullptr;
    uint8_t *scratch = nullptr;
    size_t scratch_stride = 0, slot_stride = 0, smem = 0;
    float *d_wr = nullptr;
};

bool tf32_supported(const Op &o, int mode) { return f32_geometry(o, mode).ok; }
size_t tf32_scratch_need(const Op &o, int mode) { const F32Geom g = f32_geometry(o, mode); return g.ok ? g.scratch_bytes : 0; }

bool tf32_plan(const Op &o, const ArenaGeom &ag, int mode, uint8_t *scratch, size_t scratch_stride, TcPlan *plan) {
    const F32Geom g = f32_geometry(o, mode);
    if (!g.ok || !encode_tiled()) return false;
    if (o.in0 < (int64_t)ag.W || o.out < (int64_t)ag.W || o.w >= (int64_t)ag.W || o.w % 4 || g.scratch_bytes > scratch_stride) return false;
    if (o.bias >= 0 && (o.bias % 4 || o.bias + 4 * (int64_t)o.oc > (int64_t)ag.W)) return false;
    F32PlanImpl *t = new F32PlanImpl();
    F32Params &p = t->p;
    memset(&p, 0, sizeof p);
    const int x3 = mode >= 2 ? 1 : 0;
    p.x3 = x3;
    const PixelCopy &c = g.copy;
    p.Co = o.oc; p.Ho = o.oh; p.Wo = o.ow; p.Wp = c.Wp; p.mflat = o.oh * c.Wp; p.plane = o.oh * o.ow;
    const int co_pad = round_up(o.oc, 16);
    p.n_tile = tc_n_tile(o.oc);
    p.n_tiles = tc_n_tiles(o.oc);
    const int kbytes = g.Cp * 4; /* K extent of one tap in bytes */
    p.bk = tc_bk(kbytes);
    p.ksteps = kbytes / (int)p.bk;
    p.ntaps = g.ntaps;
    p.layout = tc_umma_layout(p.bk);
    p.a_tile_bytes = (uint32_t)(TC_BM * p.bk);
    p.b_tile_bytes = (uint32_t)round_up(p.n_tile * (int)p.bk, 1024);
    p.stage_bytes = (x3 ? 2u : 1u) * (p.a_tile_bytes + p.b_tile_bytes);
    p.stages = std::max(2, std::min(8, (200 * 1024) / (int)p.stage_bytes));
    t->smem = 1024 + (size_t)p.stages * p.stage_bytes;
    p.acc_bufs = std::max(1, std::min(4, 512 / p.n_tile));
    if (p.acc_bufs < 2) p.acc_bufs = 2; /* n_tile <= 256: two buffers always fit the 512 columns */
    p.tmem_cols = 512;
    /* cute/arch/mma_sm100_desc.hpp InstrDescriptor: c = F32 (1), a = b = TF32 (2), both K-major, N >> 3, M >> 4 */
    p.idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.n_tile >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
    for (int kh = 0; kh < o.kh; kh++)
        for (int kw = 0; kw < o.kw; kw++) p.a_shift[kh * o.kw + kw] = c.tap_shift(kh, kw);
    p.lo_rows = c.npix + g.guard;
    p.bias = o.bias >= 0 ? reinterpret_cast<const float *>(ag.d_weights + o.bias) : nullptr;
    p.slot_stride = ag.slot_stride;
    p.out_off = o.out - (int64_t)ag.W;
    p.m_tiles = (p.mflat + TC_BM - 1) / TC_BM;
    p.wp_magic = (unsigned)((1ull << 32) / (unsigned)c.Wp) + 1u;
    if ((long long)p.m_tiles * p.n_tiles * ag.capacity >= (1ll << 31)) { delete t; return false; }
    t->copy = c; t->C = o.ic; t->Cp = g.Cp; t->H = o.ih; t->W = o.iw; t->split = x3; t->guard = g.guard;
    t->src_slot0 = ag.d_slots + (o.in0 - (int64_t)ag.W);
    t->scratch = scratch; t->scratch_stride = scratch_stride; t->slot_stride = ag.slot_stride;
    const size_t wr_floats = (size_t)g.ntaps * (x3 ? 2 : 1) * co_pad * g.Cp;
    if (cudaMalloc(&t->d_wr, wr_floats * 4) != cudaSuccess) { delete t; return false; }
    k_repack_f32<<<256, 256>>>(reinterpret_cast<const float *>(ag.d_weights + o.w), t->d_wr, o.oc, co_pad, o.ic, g.Cp, g.ntaps, x3);
    bool ok = cudaDeviceSynchronize() == cudaSuccess;
    const CUtensorMapSwizzle ksw = tc_swizzle(p.bk);
    ok = ok && make_map3(&t->mapA, scratch, (uint64_t)kbytes, (uint64_t)(x3 ? 2 * c.npix + g.guard : c.npix), (uint64_t)ag.capacity, (uint64_t)kbytes, scratch_stride,
                         p.bk, TC_BM, ksw);
    ok = ok && make_map3(&t->mapB, t->d_wr, (uint64_t)kbytes, (uint64_t)co_pad, (uint64_t)g.ntaps * (x3 ? 2 : 1), (uint64_t)kbytes,
                         (uint64_t)co_pad * kbytes, p.bk, (uint32_t)p.n_tile, ksw);
    t->sms = tc_sm_count();
    ok = ok && cudaFuncSetAttribute((const void *)k_conv_tf32, cudaFuncAttributeMaxDynamicSharedMemorySize, 210 * 1024) == cudaSuccess;
    if (!ok) { cudaFree(t->d_wr); delete t; return false; }
    if (getenv("MARS_TC_VERBOSE"))
        fprintf(stderr, "tf32_plan layer %d: %dx%d k%d s%d ci %d co %d | n_tile %d stages %d bk %u x3 %d smem %zu\n", o.layer, o.oh, o.ow, o.kh, o.sh, o.ic,
                o.oc, p.n_tile, p.stages, p.bk, x3, t->smem);
    plan->f32 = t;
    return true;
}

bool tf32_launch(const TcPlan &plan, uint8_t *slots_base, int first, int n, cudaStream_t s, uint64_t *launches) {
    F32PlanImpl *t = plan.f32;
    if (!t) return false;
    const uint8_t *src = t->src_slot0 + (size_t)first * t->slot_stride;
    uint8_t *scr = t->scratch + (size_t)first * t->scratch_stride;
    dim3 g((t->copy.npix + t->guard + 31) / 32, (t->Cp + 31) / 32, n);
    k_f32_to_kmajor<<<g, 256, 0, s>>>(src, t->slot_stride, scr, t->scratch_stride, t->C, t->Cp, t->H, t->W, t->copy.Wp, t->copy.plane, t->copy.npix,
                                      t->copy.mode == 2, t->copy.pt, t->copy.pl, t->split, t->guard);
    (*launches)++;
    F32Params p = t->p;
    p.out_base = slots_base + (size_t)first * t->slot_stride;
    p.img0 = first;
    p.n_img = n;
    const long long total = (long long)p.m_tiles * p.n_tiles * n;
    const unsigned grid = (unsigned)std::min<long long>(total, (long long)t->sms);
    k_conv_tf32<<<grid, (F_EPI + 2) * 32, t->smem, s>>>(t->mapA, t->mapB, p);
    (*launches)++;
    return cudaGetLastError() == cudaSuccess;
}

void tf32_release(F32PlanImpl *t) {
    if (t) { cudaFree(t->d_wr); delete t; }
}

} // namespace marsb200
