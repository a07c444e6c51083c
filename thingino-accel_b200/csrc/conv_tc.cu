/*
 * conv_tc.cu -- int8 convolution as an implicit GEMM on tcgen05 (sm_100a), persistent and warp-specialised.
 *
 * Replaces the reference's conv2d_int8_mxu (src/mars/mxu_conv.c:630-670; MIPS variant :144-408 built on the
 * 64-byte S4MACSSB dot product) for hazard-free NCHW/OIHW layers, together with the SIGMOID and MUL layers the
 * planner folded into it (src/mars/mars_runtime.c:724-838).  DESIGN.md section 5.1 is the long form.
 *
 *   GEMM view   D[M = 128 pixels][N = out channels] = A[M][K] * B[N][K],  K = taps x in channels.
 *   A operand   1x1 convs: the NCHW activation planes themselves -- one K-row = 128 consecutive pixels of one
 *               input channel (MN-major A, legal for kind::i8), loaded by TMA straight from the arena (128B swizzle).
 *               kxk convs: a kernel tap (kh,kw) is a FLAT pixel shift.  TMA faults ("illegal instruction", measured
 *               on B200) when the innermost box coordinate is not 16-byte aligned, so 1-pixel shifts cannot be
 *               applied to NCHW planes; A comes from a channel-innermost (NHWC) copy instead -- rows padded with k-1
 *               zero columns for stride 1, a 2x2 phase split for stride 2 -- and is K-major like B.  The copy is
 *               written by the PRODUCING conv's epilogue when there is one (Op::copy_from), by the k_to_nhwc
 *               pre-pass otherwise; it is also what lets fused outputs overwrite the layer's own input buffer, as
 *               the reference's work-buffer aliasing demands.  Stride 1 with resident weights: one load of the
 *               unit's rows plus halo serves all taps as row-shifted operands ("halo" mode).
 *               6x6 stride-2 stem (Ci <= 4): 3x3 over the space-to-depth image; 16-byte pixels read through a no-swizzle
 *               descriptor as overlapping 32-byte K rows ("s2d" mode).  Other small-Ci shapes: producer warps build
 *               the K rows in shared memory ("gather" mode).
 *   B operand   weights repacked once at load to [tap][Co][Ci] (K-major); resident in shared memory when small.
 *   D           int32 in TMEM (128 lanes = pixels, N columns per M tile, ring of accumulator groups).
 *   epilogue    + int32 bias (wrap-around), requantisation with the x86 float->int rule (SURVEY A.1), one lookup
 *               in a 512-entry word table holding the clamped int8 and its fused followers, NCHW byte stores and
 *               the optional channel-innermost side output.
 *   roles       warps 0..EPI-1 epilogue (two or four per TMEM lane quadrant), warp EPI = TMEM allocator + MMA
 *               issuer (one lane), warp EPI+1 = TMA producer (one lane) or EPI+1..EPI+4 = gather producers.
 *               CTA b walks work units b, b+grid, ... ; two CTAs per SM unless the N tile needs all of TMEM.
 */
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "conv_tc.h"
#include "conv_tf32.h"
#include "tc_common.cuh"

namespace marsb200 {

/* tuning aids (MARS_TC_DEBUG: 2 = epilogue only drains TMEM, 3 = 2 + no per-step TMA loads, 4 = 2 + no MMAs, 6 = prologue and
 * teardown only, 7 / 9 = epilogue warps only hand the accumulators back): compiled in with -DMARS_TC_TUNING, otherwise the tests
 * on them vanish from the kernels (they sat in the epilogue's inner loop) */
#ifdef MARS_TC_TUNING
#define TC_DBG(p) ((p).dbg)
#else
#define TC_DBG(p) 0
#endif
/* warp roles: warps 0..EPI-1 epilogue (EPI = 8, or 16 when one CTA owns the SM; quadrant = warp & 3), warp EPI = TMEM
 * allocator + MMA issuer (one elected lane), warp EPI+1 = TMA producer (lane 0) -- gather mode: warps EPI+1..EPI+4 */

struct TcParams {
    int Co, Ho, Wo, Wp;      /* Wp = row pitch of the flat pixel index */
    int mflat, plane;        /* Ho * Wp, Ho * Wo */
    int n_tile, n_tiles, m_tiles, bk, ksteps_per_tap, ntaps, stages;
    int tmem_cols;
    uint32_t idesc;
    uint32_t b_layout;       /* UMMA LayoutType of the K-major operands: 2 = SW128, 4 = SW64, 6 = SW32 */
    int a_kmajor;            /* 0: A = NCHW planes (MN-major, SW128); 1: A = channel-innermost rows (K-major, swizzle = bk) */
    uint32_t a_stage_bytes, b_stage_bytes, tx_bytes, a_tx_bytes; /* a_tx_bytes: bytes the A loads of one pipeline step deliver */
    int a_shift[TC_MAX_TAPS];
    const int32_t *bias;     /* device pointer or null */
    float cs;
    int q_m, q_s;            /* RQ 3 (integer requantisation): multiplier m = cs * 2^(32 + q_s), shift */
    long long q_c;           /* RQ 3: rounding addend c; the kernel forms c64[ch] = bias[ch] * m + c */
    uint32_t cm_off;         /* RQ 3: offset of the int64 per-channel addends in dynamic shared memory */
    /* TST (plane stores through shared memory): staging area [team][2][NST][16 channels][128 pixels] in dynamic shared memory,
     * copied out by the team's threads, 16 pixels of one channel each */
    uint32_t stg_off;
    const uint32_t *lutw;    /* 256-entry word table: index = r + 128, byte k = value of output stream k, byte 3 = side-output stream */
    uint32_t tab_off, tab_rep; /* offset of the replicated table ([256][tab_rep] words) in dynamic shared memory; copies (8, 16 or 32) */
    uint8_t *out_base;       /* slot 0 of the launch */
    unsigned long long slot_stride;
    long long out_off[3];    /* slot-relative byte offset of output stream k (NCHW), -1 = not stored */
    /* optional channel-innermost side output: the padded / phase-split copy the consuming kxk conv reads (SURVEY C.6) */
    int nhwc_sel;            /* -1 = none, else the table byte to write */
    int nhwc_mode, nhwc_Wp, nhwc_plane, nhwc_pt, nhwc_pl, nhwc_C;
    uint8_t *nhwc_base;
    unsigned long long nhwc_stride;
    unsigned wp_magic;       /* floor(2^32 / Wp) + 1 */
    int a_row_bytes;         /* bytes of one A row in a halo stage: bk, or 16 in s2d mode */
    int toep;                /* s2d mode: A rows are 16-byte pixels read as overlapping 32-byte K rows (no swizzle) */
    int halo, halo_min, halo_rb, halo_nb; /* kxk stride 1 / s2d: one A load per (tile, k block) covers all taps: rows q0+halo_min .., halo_nb boxes of halo_rb rows */
    int halo_wide;           /* s2d: the halo region travels as 256-byte rows (16 pixels): halo_rb counts those rows, halo_min is a multiple of 16 */
    int acc_bufs;            /* TMEM accumulator ring depth */
    int grp, m_groups;       /* M tiles (128 rows each) per pipeline step and accumulator hand-over; groups per image */
    uint32_t a_tile_bytes;   /* bytes of one M tile's A block per k-step (a_stage_bytes = grp of them, or the halo region) */
    int dbg;                 /* tuning aid (MARS_TC_DEBUG): 2 = epilogue only drains TMEM, 3 = 2 + no per-step TMA loads, 4 = 2 + no MMAs */
    int b_resident;          /* all weight blocks of the (single) N tile stay in shared memory for the whole launch */
    int img0, n_img;         /* first image (TMA coordinate of the slot dimension), images of this launch */
    /* gather mode: A rows are built from a private NCHW copy of the input (small Ci, e.g. the 6x6 stride-2 stem) */
    const uint8_t *g_src;
    unsigned long long g_stride;
    int gC, gH, gW, gS, gpt, gpl, gKH, gKW, gKt;
    int tw_shift, tiles_x;   /* M tile = (1 << tw_shift) x (128 >> tw_shift) output pixels */
    int gPH, gPWW, gdx;      /* patch rows per channel, 4-byte words per patch row, byte column of tap x = 0 */
    int g_align2;
    /* rect mode (channel-innermost activations read straight from the arena, conv2d_int8_nhwc_mxu): an M tile is tw x th output
     * pixels, a tap (kh, kw) is ONE 4-d TMA box {bk channels, tw pixels, th rows, 1 image} at input pixel (s*x0 + kw - pl,
     * s*y0 + kh - pt) with traversal stride s; pixels outside the image arrive as zeros (the reference skips those taps) */
    int rect, tw, th, rs, rpt, rpl;
    unsigned tw_magic;       /* floor(2^32 / tw) + 1 */
    int onhwc_vec;           /* OUT 2: 16-byte stores are legal (Co % 16 == 0, 16-byte aligned tensors) */
};

/* ---- requantisation ------------------------------------------------------------
 * reference src/mars/mxu_conv.c:663-666: r = (int32)(sc + (sc >= 0 ? 0.5f : -0.5f)), sc = (float)acc * cs, clamped to
 * int8, with the x86 cvttss2si rule (NaN and |v| >= 2^31 become INT_MIN, hence -128).  Both variants return the clamped
 * value r in [-128, 127]; the fused followers (sigmoid, SiLU product, byte-ReLU) are one lookup r -> word afterwards.
 *
 * FAST (chosen per layer on the host when max|acc| < 2^22 and |cs| < 512, so |sc| < 2^31 and nothing overflows): the
 * int -> float conversion is an integer add of 0x4B400000 (folded into the bias word) and one float subtract,
 *   (float)acc = as_float(acc + 0x4B400000) - 1.5 * 2^23          exact for |acc| < 2^22,
 * done for two channels at a time with the packed FADD2 / FMUL2 of sm_100 (same IEEE rounding per half).  The final
 * truncation + clamp is one F2I.S8.TRUNC (float -> int conversions saturate in PTX).  Measured (tools/epi_bench.cu,
 * profiles/r02a_epi_bench.txt): 9.3 cycles per warp-element per scheduler against 11.9 for the round-1 sequence, which
 * avoided the conversion with five integer-pipe instructions; the integer pipe (16 lanes per scheduler) is what limits
 * the epilogue.  The +-0.5 add stays a scalar FADD: ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 (one
 * rounding), which is not the reference's arithmetic. */
/* RQ = 0: general (I2F, x86 overflow rule); 1: FAST, sign-exact, F2I; 2: FAST, round-half-up without conversion instructions;
 * 3: the integer form (requant_int).  select_requant picks one per layer.
 *
 * RQ 2 is chosen when the integer form does not fit (scales <= 0 or >= 0.49, or the rare positive scale whose thresholds no
 * integer triple reproduces), max |acc + bias| < 2^22, |cs| < 512 and no accumulator value in range lands on a negative tie.
 * Most builder scales fit the integer form, so RQ 2 is now the exception.  ncu on the F2I variant showed the XU pipe
 * (conversions, 16 lanes per SM) 87 % busy: one F2I per output element is what limited the epilogue.  floor(fl(sc + 0.5f)) needs none: a round-down add of 1.5 * 2^23 leaves
 * floor(h) in the low mantissa bits, and one VIADDMNMX.RELU (DPX) subtracts the exponent pattern and clamps to [0, 255]
 * = r + 128.  Round-half-up differs from the reference's round-half-away only when sc is a NEGATIVE exact tie -(n + 0.5)
 * (or -pred(0.5), where fl(sc - 0.5f) rounds to -1): the host enumerates those few floats per layer and selects RQ 2 only
 * when no accumulator value in the layer's range maps onto one of them (halfup_requant_ok). */
template <int RQ>
__device__ __forceinline__ void requant_pair(int32_t t0, int32_t t1, float cs, int &r0, int &r1) {
    float s0, s1;
    if (RQ != 0) {
        unsigned long long a, b, c2;
        asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "r"(t0), "r"(t1));
        asm("add.rn.f32x2 %0, %1, %2;" : "=l"(b) : "l"(a), "l"(0xCB400000CB400000ull)); /* - 12582912.0f, twice */
        asm("mov.b64 %0, {%1, %1};" : "=l"(c2) : "f"(cs));
        asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(a) : "l"(b), "l"(c2));
        asm("mov.b64 {%0, %1}, %2;" : "=f"(s0), "=f"(s1) : "l"(a));
    } else {
        s0 = __fmul_rn(__int2float_rn(t0), cs);
        s1 = __fmul_rn(__int2float_rn(t1), cs);
    }
    if (RQ == 2) { /* returns r + 128 in [0, 255] */
        const int i0 = __float_as_int(__fadd_rd(__fadd_rn(s0, 0.5f), 12582912.0f)), i1 = __float_as_int(__fadd_rd(__fadd_rn(s1, 0.5f), 12582912.0f));
        r0 = __viaddmin_s32_relu(i0, -(0x4B400000 - 128), 255);
        r1 = __viaddmin_s32_relu(i1, -(0x4B400000 - 128), 255);
        return;
    }
    const float h0 = __fadd_rn(s0, copysignf(0.5f, s0)), h1 = __fadd_rn(s1, copysignf(0.5f, s1)); /* +-0: both signs truncate to 0 */
    asm("cvt.rzi.s8.f32 %0, %1;" : "=r"(r0) : "f"(h0)); /* truncate + clamp to [-128, 127]; NaN -> 0 */
    asm("cvt.rzi.s8.f32 %0, %1;" : "=r"(r1) : "f"(h1));
    if (RQ == 0) { /* x86: +overflow and NaN -> INT_MIN -> -128 */
        if (!(h0 < 2147483648.0f)) r0 = -128;
        if (!(h1 < 2147483648.0f)) r1 = -128;
    }
}

/* ---- requantisation, integer form (RQ 3) ----------------------------------------
 * The reference's r(t) = clamp((int32)(fl(t * cs) + copysign(0.5f, .))) (src/mars/mxu_conv.c:663-666) is a monotone step function
 * of the integer t = acc + bias with 255 steps.  So is g(t) = clamp(floor((t * m + c) / 2^(32 + s))) for integers m, c, s, and two
 * monotone step functions are equal exactly when their 255 thresholds are: the host finds the reference's thresholds by bisection
 * over the layer's accumulator range and looks for a c that reproduces all of them (int_requant_fit; m = cs * 2^(32 + s) exactly,
 * s as large as keeps m below 2^31).  When one exists -- almost always: it fails for scales with short mantissas, whose exact ties
 * the float arithmetic rounds away from zero on both sides -- the epilogue needs one IMAD.HI, one shift and one clamp per element
 * instead of the magic-number int -> float conversion, two packed float operations, two float adds and the clamp; the bias is
 * folded into the 64-bit addend (c64[ch] = bias[ch] * m + c), and there is no accumulator-range restriction (RQ 1 / 2 need
 * |t| < 2^22).  Returns r + 128 in [0, 255] like RQ 2. */
__device__ __forceinline__ int requant_int(uint32_t acc, int c_lo, int c_hi, int m, int sh) {
    const long long c = (long long)(((unsigned long long)(uint32_t)c_hi << 32) | (uint32_t)c_lo);
    const long long x = (long long)(int32_t)acc * (long long)m + c;
    return __viaddmin_s32_relu((int)(x >> 32) >> sh, 128, 255);
}

/* the 16 table words (or plain bytes) of one unit: 16 accumulator columns (output channels) of this thread's pixel.
 * cm: shared address of the unit's per-channel constants -- int32 bias (+ the int->float magic when RQ 1 / 2), or the int64
 * addends of RQ 3; cs: the conv scale, for RQ 3 the bits of the multiplier m; qs: the shift s of RQ 3.
 * TAB = the op has fused followers: r indexes this lane's copy of the 256-entry word table (byte k = value of output
 * stream k, byte 3 = the side-output stream); the table is replicated per lane ([256][32] words), so the data-dependent
 * lookups of a warp never meet in a bank (the shared 512-entry table of round 1 cost ~3 wavefronts per lookup). */
template <int RQ, bool TAB>
__device__ __forceinline__ void unit_words(const uint32_t (&v)[16], uint32_t cm, uint32_t tab_lane, uint32_t tab_stride, float cs, int qs, uint32_t (&w)[16]) {
    constexpr bool R128 = RQ >= 2; /* the requantisation returns r + 128 */
    if (RQ == 3) {
        const int m = __float_as_int(cs);
#pragma unroll
        for (int j2 = 0; j2 < 8; j2++) {
            const int4 c4 = lds_v4(cm + (uint32_t)j2 * 16u);
            const int r0 = requant_int(v[2 * j2], c4.x, c4.y, m, qs), r1 = requant_int(v[2 * j2 + 1], c4.z, c4.w, m, qs);
            w[2 * j2] = TAB ? lds_u32(tab_lane + (uint32_t)r0 * tab_stride) : (uint32_t)r0 ^ 0x80u;
            w[2 * j2 + 1] = TAB ? lds_u32(tab_lane + (uint32_t)r1 * tab_stride) : (uint32_t)r1 ^ 0x80u;
        }
    } else {
#pragma unroll
        for (int j4 = 0; j4 < 4; j4++) {
            const int4 c4 = lds_v4(cm + (uint32_t)j4 * 16u);
            const int cc[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
            for (int k = 0; k < 4; k += 2) {
                int r0, r1;
                requant_pair<RQ>((int32_t)(v[j4 * 4 + k] + (uint32_t)cc[k]), (int32_t)(v[j4 * 4 + k + 1] + (uint32_t)cc[k + 1]), cs, r0, r1);
                w[j4 * 4 + k] = TAB ? lds_u32(tab_lane + (uint32_t)r0 * tab_stride) : (R128 ? (uint32_t)r0 ^ 0x80u : (uint32_t)r0);
                w[j4 * 4 + k + 1] = TAB ? lds_u32(tab_lane + (uint32_t)r1 * tab_stride) : (R128 ? (uint32_t)r1 ^ 0x80u : (uint32_t)r1);
            }
        }
    }
}
/* one channel pair (j, j+1) of a ragged unit */
template <int RQ, bool TAB>
__device__ __forceinline__ void pair_words(uint32_t v0, uint32_t v1, uint32_t cm, int j, uint32_t tab_lane, uint32_t tab_stride, float cs, int qs,
                                           uint32_t &w0, uint32_t &w1) {
    constexpr bool R128 = RQ >= 2;
    int r0, r1;
    if (RQ == 3) {
        const int4 c4 = lds_v4(cm + 8u * (uint32_t)j);
        r0 = requant_int(v0, c4.x, c4.y, __float_as_int(cs), qs); r1 = requant_int(v1, c4.z, c4.w, __float_as_int(cs), qs);
    } else requant_pair<RQ>((int32_t)(v0 + lds_u32(cm + 4u * j)), (int32_t)(v1 + lds_u32(cm + 4u * j + 4u)), cs, r0, r1);
    w0 = TAB ? lds_u32(tab_lane + (uint32_t)r0 * tab_stride) : (R128 ? (uint32_t)r0 ^ 0x80u : (uint32_t)r0);
    w1 = TAB ? lds_u32(tab_lane + (uint32_t)r1 * tab_stride) : (R128 ? (uint32_t)r1 ^ 0x80u : (uint32_t)r1);
}

/* ---- epilogue of one unit: 16 accumulator columns (output channels) of this thread's pixel -----------------
 * NST = number of NCHW output streams stored (table bytes 0..NST-1), NHWC = also pack the side byte of every 16 channels
 * into one 16-byte store of the consumer's channel-innermost copy.  o0..o2 point at channel c0 of this pixel; nch = how
 * many of the 16 channels exist (16 = all, <= 0 = none / pixel outside the image). */
template <int RQ, bool TAB, int NST, bool NHWC, int PAIR>
__device__ __forceinline__ void epilogue_unit(const uint32_t (&v)[16], uint32_t cm, uint32_t tab_lane, uint32_t tab_stride, float cs, int qs,
                                              uint8_t *o0, uint8_t *o1, uint8_t *o2, long long plane, int nch, uint8_t *nh, uint32_t (&keep)[4]) {
    if (nch <= 0) return; /* cm: shared address of the unit's per-channel constants; tab_lane: shared address of entry r = 0 of this lane's table */
    if (nch >= 16) {
        uint32_t w[16], pk[4];
        unit_words<RQ, TAB>(v, cm, tab_lane, tab_stride, cs, qs, w);
#pragma unroll
        for (int j4 = 0; j4 < 4; j4++) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                if (NST > 0) { *o0 = (uint8_t)w[4 * j4 + k]; o0 += plane; }
                if (NST > 1) { *o1 = (uint8_t)(w[4 * j4 + k] >> 8); o1 += plane; }
                if (NST > 2) { *o2 = (uint8_t)(w[4 * j4 + k] >> 16); o2 += plane; }
            }
            if (NHWC) { /* the side-output stream sits in the top byte of the table word (plain conv: the value itself) */
                const uint32_t sel = TAB ? 0x0073u : 0x0040u;
                pk[j4] = __byte_perm(__byte_perm(w[4 * j4], w[4 * j4 + 1], sel), __byte_perm(w[4 * j4 + 2], w[4 * j4 + 3], sel), 0x5410);
            }
        }
        /* side output: units (2k, 2k+1) of a pixel are handled back to back by this thread (the work split is in pairs) and go
         * out as ONE 32-byte store (STG.256): half as many partially written 128-byte lines on their way to L2 as two 16-byte
         * stores -- the L1 -> L2 request path is what saturates in the layers with a side output (profiles/r02i).  PAIR 1 = first
         * unit of a pair: the packed bytes wait in `keep`; PAIR 2 = second unit: store both */
        if (NHWC) {
            if (PAIR == 1) { keep[0] = pk[0]; keep[1] = pk[1]; keep[2] = pk[2]; keep[3] = pk[3]; }
            else if (PAIR == 2)
                asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(nh - 16), "r"(keep[0]), "r"(keep[1]), "r"(keep[2]), "r"(keep[3]),
                             "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]) : "memory");
            else *reinterpret_cast<uint4 *>(nh) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
    } else { /* ragged last unit (e.g. 255 head channels); a side-output consumer always has Ci = Co, a multiple of 32 */
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
            if (j < nch) {
                uint32_t w0, w1;
                pair_words<RQ, TAB>(v[j], v[j + 1], cm, j, tab_lane, tab_stride, cs, qs, w0, w1);
                if (NST > 0) o0[(long long)j * plane] = (uint8_t)w0;
                if (NST > 1) o1[(long long)j * plane] = (uint8_t)(w0 >> 8);
                if (NST > 2) o2[(long long)j * plane] = (uint8_t)(w0 >> 16);
                if (j + 1 < nch) {
                    if (NST > 0) o0[(long long)(j + 1) * plane] = (uint8_t)w1;
                    if (NST > 1) o1[(long long)(j + 1) * plane] = (uint8_t)(w1 >> 8);
                    if (NST > 2) o2[(long long)(j + 1) * plane] = (uint8_t)(w1 >> 16);
                }
            }
        }
    }
}

/* TST: the NCHW streams of the unit go into the team's staging block [stream][16 channels][128 pixels] (this thread's pixel =
 * byte r of every row; immediate offsets, no pointer arithmetic); the team's threads copy the block out afterwards.  The side output
 * (NHWC) is stored directly as before. */
template <int RQ, bool TAB, int NST, bool NHWC>
__device__ __forceinline__ void epilogue_unit_staged(const uint32_t (&v)[16], uint32_t cm, uint32_t tab_lane, uint32_t tab_stride, float cs, int qs,
                                                     uint32_t stg_r, bool side_ok, uint8_t *nh) {
    uint32_t w[16], pk[4];
    unit_words<RQ, TAB>(v, cm, tab_lane, tab_stride, cs, qs, w);
#pragma unroll
    for (int j = 0; j < 16; j++) {
        if (NST > 0) sts_u8(stg_r + (uint32_t)j * 128u, w[j]);
        if (NST > 1) sts_u8(stg_r + 2048u + (uint32_t)j * 128u, w[j] >> 8);
        if (NST > 2) sts_u8(stg_r + 4096u + (uint32_t)j * 128u, w[j] >> 16);
    }
    if (NHWC) {
        const uint32_t sel = TAB ? 0x0073u : 0x0040u;
#pragma unroll
        for (int j4 = 0; j4 < 4; j4++)
            pk[j4] = __byte_perm(__byte_perm(w[4 * j4], w[4 * j4 + 1], sel), __byte_perm(w[4 * j4 + 2], w[4 * j4 + 3], sel), 0x5410);
        if (side_ok) *reinterpret_cast<uint4 *>(nh) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
}

/* OUT 2: the same 16 channels written channel-innermost -- one 16-byte store per stream (bytes of stream k = byte k of the
 * table words); `vec` = the tensor allows 16-byte stores (Co % 16 == 0), otherwise (e.g. 255 head channels) bytes.
 * o0..o2 point at channel c0 of this pixel in each stream's NHWC tensor. */
template <int RQ, bool TAB, int NST>
__device__ __forceinline__ void epilogue_unit_nhwc(const uint32_t (&v)[16], uint32_t cm, uint32_t tab_lane, uint32_t tab_stride, float cs, int qs,
                                                   uint8_t *o0, uint8_t *o1, uint8_t *o2, int nch, bool vec) {
    if (nch <= 0) return;
    uint32_t w[16], pk[3][4];
    unit_words<RQ, TAB>(v, cm, tab_lane, tab_stride, cs, qs, w);
#pragma unroll
    for (int j4 = 0; j4 < 4; j4++) {
        pk[0][j4] = __byte_perm(__byte_perm(w[4 * j4], w[4 * j4 + 1], 0x0040), __byte_perm(w[4 * j4 + 2], w[4 * j4 + 3], 0x0040), 0x5410);
        if (NST > 1) pk[1][j4] = __byte_perm(__byte_perm(w[4 * j4], w[4 * j4 + 1], 0x0051), __byte_perm(w[4 * j4 + 2], w[4 * j4 + 3], 0x0051), 0x5410);
        if (NST > 2) pk[2][j4] = __byte_perm(__byte_perm(w[4 * j4], w[4 * j4 + 1], 0x0062), __byte_perm(w[4 * j4 + 2], w[4 * j4 + 3], 0x0062), 0x5410);
    }
    if (vec && nch >= 16) {
        *reinterpret_cast<uint4 *>(o0) = make_uint4(pk[0][0], pk[0][1], pk[0][2], pk[0][3]);
        if (NST > 1) *reinterpret_cast<uint4 *>(o1) = make_uint4(pk[1][0], pk[1][1], pk[1][2], pk[1][3]);
        if (NST > 2) *reinterpret_cast<uint4 *>(o2) = make_uint4(pk[2][0], pk[2][1], pk[2][2], pk[2][3]);
    } else {
#pragma unroll
        for (int j = 0; j < 16; j++) {
            if (j < nch) {
                o0[j] = (uint8_t)(pk[0][j >> 2] >> (8 * (j & 3)));
                if (NST > 1) o1[j] = (uint8_t)(pk[1][j >> 2] >> (8 * (j & 3)));
                if (NST > 2) o2[j] = (uint8_t)(pk[2][j >> 2] >> (8 * (j & 3)));
            }
        }
    }
}

/* ---- the kernel ----------------------------------------------------------------
 * Persistent: CTA b walks tiles b, b + gridDim.x, ... of the launch's (image, M tile, N tile) space; barriers, TMEM
 * and tables are set up once.  The accumulator is double buffered in TMEM, so the epilogue of tile t overlaps the
 * loads and MMAs of tile t+1.  Epilogue warps never synchronise with each other: thread = output pixel (TMEM lane),
 * registers = 16 output channels; per channel the 32 lanes of a warp store 32 consecutive pixels of one NCHW plane.
 * OUT: 0 = NCHW planes, 1 = NCHW planes + the consumer's channel-innermost side copy, 2 = channel-innermost (NHWC) output
 * tensors, 16 bytes per thread and unit.
 * GATHER (small Ci, e.g. the 6x6 stride-2 stem): M tiles are tw x th output pixels; four producer warps stage the
 * input patch of the tile in shared memory (next tile's patch is in flight in registers meanwhile) and build the
 * 128-byte K rows of the A operand from it, in the 128B-swizzled K-major layout TMA would have produced. */
template <int RQ, bool GATHER, bool TAB, int NST, int OUT, int EPI, bool TST = false>
__global__ void __launch_bounds__((EPI + (GATHER ? 5 : 2)) * 32, EPI == 8 ? 2 : 1)
k_conv_tc(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const TcParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_full[8], bar_empty[8], bar_tmem_full[8], bar_tmem_empty[8], bar_b;
    __shared__ uint32_t tmem_base_slot;
    __shared__ __align__(16) int32_t s_cm[TC_MAX_CO];   /* bias (+ the int->float magic when FAST) */
    __shared__ __align__(16) int s_koff[GATHER ? 128 : 4]; /* gather: patch-relative byte offset of tap k */
    __shared__ int s_shift[TC_MAX_TAPS];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t a_base = smem_base, b_base = smem_base + p.stages * p.a_stage_bytes;
    const int nsteps = p.ntaps * p.ksteps_per_tap;
    const int tiles_per_img = p.m_groups * p.n_tiles; /* scheduling unit = a group of p.grp M tiles x one N tile */
    /* gather-mode shared regions behind the weight tile */
    uint8_t *g_patch = smem_al + (size_t)p.stages * p.a_stage_bytes + p.b_stage_bytes; /* gather: B is one resident block */
    int *g_poff = reinterpret_cast<int *>(g_patch + 3 * 4096); /* three patch buffers, then per patch word: offset inside the input */
    int *g_pyx = g_poff + 1024;                            /* per patch word: patch row << 16 | byte column */

    if (threadIdx.x == 0) {
        /* one MMA-issuing lane per M tile of a group: each commits (arrives) on its own */
        for (int s = 0; s < p.stages; s++) { mbar_init(smem_u32(&bar_full[s]), GATHER ? 4 : 1); mbar_init(smem_u32(&bar_empty[s]), p.grp); }
        for (int b = 0; b < p.acc_bufs; b++) { mbar_init(smem_u32(&bar_tmem_full[b]), p.grp); mbar_init(smem_u32(&bar_tmem_empty[b]), EPI); }
        mbar_init(smem_u32(&bar_b), 1);
        mbar_fence_init();
    }
    constexpr int WARP_MMA = EPI, WARP_PROD = EPI + 1; /* then: TMA producer (lane 0) or four gather producer warps */
    if (warp == WARP_MMA) { /* TMEM allocation is a warp-wide operation; this warp also frees it */
        tmem_alloc(smem_u32(&tmem_base_slot), (uint32_t)p.tmem_cols);
    }
    if (RQ == 3) { /* int64 addends c64[ch] = bias[ch] * m + c in dynamic shared memory (p.cm_off), all N tiles */
        long long *cm64 = reinterpret_cast<long long *>(smem_al + p.cm_off);
        for (int i = threadIdx.x; i < p.n_tiles * p.n_tile; i += blockDim.x)
            cm64[i] = (long long)((p.bias && i < p.Co) ? p.bias[i] : 0) * (long long)p.q_m + p.q_c;
    } else {
        for (int i = threadIdx.x; i < TC_MAX_CO; i += blockDim.x)
            s_cm[i] = (int32_t)((uint32_t)((p.bias && i < p.Co) ? p.bias[i] : 0) + (RQ != 0 ? 0x4B400000u : 0u));
    }
    if (TAB) { /* [256][rep] words: lane l reads copy l % rep; with rep = 32 (bank = lane) the data-dependent lookups never conflict */
        uint32_t *tab = reinterpret_cast<uint32_t *>(smem_al + p.tab_off);
        const int sh = p.tab_rep == 32 ? 5 : (p.tab_rep == 16 ? 4 : 3);
        for (int i = threadIdx.x; i < (256 << sh); i += blockDim.x) tab[i] = __ldg(p.lutw + (i >> sh));
    }
    /* per tap: flat pixel shift (TMA coordinate); halo mode: start of the tap's rows inside the stage, in 16-byte units */
    if (threadIdx.x < TC_MAX_TAPS) s_shift[threadIdx.x] = p.halo ? ((p.a_shift[threadIdx.x] - p.halo_min) * p.a_row_bytes) >> 4 : p.a_shift[threadIdx.x];
    if (GATHER) {
        const int PP = p.gPWW * 4;
        for (int k = threadIdx.x; k < 128; k += blockDim.x) {
            const int ci = k / (p.gKH * p.gKW), r = k - ci * p.gKH * p.gKW, y = r / p.gKW, x = r - y * p.gKW;
            const int off = k < p.gKt ? (ci * p.gPH + y) * PP + x + p.gdx : 0;
            if (!p.g_align2) s_koff[k] = off;
            else if ((k & 1) == 0) s_koff[k >> 1] = off; /* one entry per byte pair (k, k+1) */
        }
        for (int i = threadIdx.x; i < p.gC * p.gPH * p.gPWW; i += blockDim.x) {
            const int ci = i / (p.gPH * p.gPWW), r = i - ci * p.gPH * p.gPWW, py = r / p.gPWW, wi = r - py * p.gPWW;
            g_poff[i] = (ci * p.gH + py) * p.gW + 4 * wi;
            g_pyx[i] = (py << 16) | (4 * wi);
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_d = tmem_base_slot;
    if (TC_DBG(p) == 6) goto teardown; /* tuning aid: prologue + teardown only */

    if (warp < EPI) {
        /* ===== epilogue: TMEM -> registers -> requantised byte -> (word table) -> stores =====
         * Work items of an accumulator group are (M tile g, 16-column unit u) pairs, g-major; the EPI / 4 warps of a TMEM
         * lane quadrant take contiguous blocks of them, so the per-M-tile values (pixel coordinates, output pointers) are
         * recomputed as rarely as possible.  The TMEM load of item k+1 is issued before item k is processed, so the load
         * latency (and, at a group boundary, the wait for the next accumulator when it is already there) hides behind
         * the arithmetic and the stores of the current item. */
        const int quad = warp & 3, part = warp >> 2, parts = EPI >> 2;
        const int r = quad * 32 + lane; /* accumulator row = pixel of the tile */
        const int n_units = p.n_tile >> 4;
        const long long plane = p.plane;
        const float cs = RQ == 3 ? __int_as_float(p.q_m) : p.cs; /* RQ 3: the multiplier travels in the scale's place */
        const int qs = p.q_s;
        const uint32_t acc_lane = tmem_d + ((uint32_t)(quad * 32) << 16);
        const uint32_t sa_cm = RQ == 3 ? smem_base + p.cm_off : smem_u32(s_cm);
        constexpr uint32_t CMB = RQ == 3 ? 8u : 4u; /* bytes per channel constant */
        const uint32_t tab_stride = 4u * p.tab_rep; /* bytes between consecutive table entries */
        const uint32_t tab_lane = smem_base + p.tab_off + (RQ >= 2 ? 0u : 128u * tab_stride) + 4u * ((uint32_t)lane & (p.tab_rep - 1u)); /* this lane's copy: entry r = 0 (RQ 2 / 3: entry r = -128, the requantisation returns r + 128) */
        const uint32_t sa_full = smem_u32(&bar_tmem_full[0]), sa_empty = smem_u32(&bar_tmem_empty[0]);
        const bool flat = !GATHER && !p.rect && p.Wp == p.Wo && OUT != 1; /* no pad columns: the tile row index IS the pixel index */
        uint8_t *const obase = p.out_base + r; /* + image * slot_stride + pixel + channel * plane + stream offset */
        const int G = p.grp, gcols = p.grp * p.n_tile;
        /* OUT 1: items are handed out in pairs of units (the side output is stored per pair) */
        const int total_items = G * n_units, ipp = OUT == 1 ? 2 * ((total_items / 2 + parts - 1) / parts) : (total_items + parts - 1) / parts;
        const int i_lo = part * ipp, i_hi = min(total_items, i_lo + ipp);
        if (i_lo >= i_hi || TC_DBG(p) == 7 || TC_DBG(p) == 9) { /* narrow group: nothing to read for this warp, it only releases the accumulators */
            int ab = 0, aph = 0; /* accumulator ring position and phase */
            for (TileIter ti(blockIdx.x, gridDim.x, tiles_per_img); ti.img < p.n_img; ti.next()) {
                mbar_wait_relaxed(sa_full + 8u * ab, aph);
                __syncwarp();
                if (lane == 0) mbar_arrive(sa_empty + 8u * ab);
                if (++ab == p.acc_bufs) { ab = 0; aph ^= 1; }
            }
        } else {
            /* this warp's block of items, as (M tile, unit range) runs: [g_first, u_first) ... [g_last, u_last] */
            const int g_first = i_lo / n_units, u_first = i_lo - g_first * n_units;
            const int g_last = (i_hi - 1) / n_units, u_last_end = i_hi - g_last * n_units; /* units [0, u_last_end) of the last M tile */
            int ab = 0, aph = 0;
            uint32_t va[16], vb[16];
            /* TST: the four warps of a part (one per TMEM lane quadrant) form a team that fills one staging block per unit and,
             * behind a barrier, copies it out; consecutive units alternate between two blocks, so the writes of the next unit
             * cannot meet the copy-out of this one */
            const uint32_t stg_team = smem_base + p.stg_off + (uint32_t)part * (2u * NST * 2048u) + (uint32_t)r;
            uint32_t cnt = 0;
            for (TileIter ti(blockIdx.x, gridDim.x, tiles_per_img); ti.img < p.n_img; ti.next()) {
                mbar_wait_relaxed(sa_full + 8u * ab, aph);
                tcgen05_fence_after();
                const int mg = p.n_tiles == 1 ? ti.rem : ti.rem / p.n_tiles;
                const int n0 = (ti.rem - mg * p.n_tiles) * p.n_tile;
                const uint32_t acc_grp = acc_lane + (uint32_t)(ab * gcols);
                uint8_t *const img_base = obase + ((unsigned long long)ti.img * p.slot_stride + (long long)n0 * plane);
                const uint32_t cm0 = sa_cm + CMB * (uint32_t)n0;
                for (int g = g_first; g <= g_last; g++) {
                    const int u_lo = g == g_first ? u_first : 0, u_hi = g == g_last ? u_last_end : n_units;
                    /* per-M-tile values: pixel of this lane, validity, output pointers */
                    const int mt = mg * G + g;
                    int oh = 0, ow = 0, pix;
                    bool valid;
                    if (flat) {
                        pix = mt * TC_BM; /* + r, folded into obase */
                        valid = pix + r < p.mflat;
                    } else {
                        if (GATHER) {
                            const int ty = mt / p.tiles_x, tx = mt - ty * p.tiles_x;
                            oh = ty * (TC_BM >> p.tw_shift) + (r >> p.tw_shift);
                            ow = (tx << p.tw_shift) + (r & ((1 << p.tw_shift) - 1));
                            valid = oh < p.Ho && ow < p.Wo;
                        } else if (p.rect) { /* tw x th output pixels, row-major inside the tile */
                            const int ty = mt / p.tiles_x, tx = mt - ty * p.tiles_x;
                            const int ry = (int)__umulhi((unsigned)r, p.tw_magic), rx = r - ry * p.tw;
                            oh = ty * p.th + ry; ow = tx * p.tw + rx;
                            valid = ry < p.th && oh < p.Ho && ow < p.Wo;
                        } else {
                            const int q = mt * TC_BM + r;
                            oh = (int)__umulhi((unsigned)q, p.wp_magic); ow = q - oh * p.Wp; /* q / Wp, exact for q * Wp < 2^32 (checked on the host) */
                            valid = q < p.mflat && ow < p.Wo;
                        }
                        pix = oh * p.Wo + ow - r;
                    }
                    const int co_left = valid ? p.Co - n0 : 0; /* channels of this N tile that exist for this pixel (<= 0: nothing to store) */
                    /* channel n0 + 16 u_lo of this pixel: NCHW planes, or (OUT 2) the pixel's channel vector */
                    uint8_t *pix_base = OUT == 2 ? p.out_base + ((unsigned long long)ti.img * p.slot_stride + (long long)(pix + r) * p.Co + n0 + u_lo * 16)
                                                 : img_base + pix + (long long)(u_lo * 16) * plane;
                    uint8_t *nh = nullptr;
                    if (OUT == 1) {
                        long long dp;
                        if (p.nhwc_mode == 2) {
                            const int yy = oh + p.nhwc_pt, xx = ow + p.nhwc_pl;
                            dp = (long long)(((yy & 1) << 1) | (xx & 1)) * p.nhwc_plane + (long long)(yy >> 1) * p.nhwc_Wp + (xx >> 1);
                        } else dp = (long long)oh * p.nhwc_Wp + ow + p.nhwc_pl;
                        nh = p.nhwc_base + (unsigned long long)ti.img * p.nhwc_stride + dp * p.nhwc_C + n0;
                    }
                    const long long plane16 = OUT == 2 ? 16 : plane * 16;
                    const uint32_t acc_g = acc_grp + (uint32_t)(g * p.n_tile);
                    const bool last_g = g == g_last;
                    /* TST copy-out: thread r of the team owns the 16-pixel chunk (r & 7) of channel (r >> 3) of every unit (the
                     * chunk starts on a 16-pixel boundary of its row: Wo and Wp are multiples of 16) */
                    const int cq = mt * TC_BM + (r & 7) * 16, cy = (int)__umulhi((unsigned)cq, p.wp_magic), cx = cq - cy * p.Wp;
                    const bool c_ok = cx < p.Wo && cy < p.Ho;
                    const long long c_off = (long long)(unsigned long long)ti.img * (long long)p.slot_stride + (long long)cy * p.Wo + cx;
                    auto staged = [&](const uint32_t (&v)[16], int uu) {
                        const uint32_t sb = stg_team + (cnt & 1u) * (NST * 2048u);
                        epilogue_unit_staged<RQ, TAB, NST, OUT == 1>(v, cm0 + 16u * CMB * (uint32_t)uu, tab_lane, tab_stride, cs, qs, sb, valid, nh + uu * 16);
                        asm volatile("bar.sync %0, 128;" ::"r"(1 + part) : "memory");
                        const int c = n0 + uu * 16 + (r >> 3);
                        const uint32_t src = sb - (uint32_t)r + (uint32_t)(r >> 3) * 128u + (uint32_t)(r & 7) * 16u;
                        if (c_ok && c < p.Co) {
                            uint8_t *dst = p.out_base + (c_off + (long long)c * plane);
                            const int4 d0 = lds_v4(src);
                            *reinterpret_cast<int4 *>(dst + p.out_off[0]) = d0;
                            if (NST > 1) { const int4 d1 = lds_v4(src + 2048u); *reinterpret_cast<int4 *>(dst + p.out_off[1]) = d1; }
                            if (NST > 2) { const int4 d2 = lds_v4(src + 4096u); *reinterpret_cast<int4 *>(dst + p.out_off[2]) = d2; }
                        }
                        cnt++;
                    };
                    /* units u_lo .. u_hi-1 of this M tile, the TMEM load of the next one in flight while one is processed */
                    int u = u_lo;
                    uint32_t keep[4] = {0u, 0u, 0u, 0u}; /* OUT 1: the first unit's side bytes of a pair (runs start at even units and have even length) */
                    tmem_ld16_issue(acc_g + (uint32_t)(u * 16), va);
                    for (;;) {
                        tmem_ld_wait(va);
                        if (u + 1 < u_hi) tmem_ld16_issue(acc_g + (uint32_t)((u + 1) * 16), vb);
                        else if (last_g) { /* last read of this accumulator group by this warp: hand it back */
                            tcgen05_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(sa_empty + 8u * ab);
                        }
                        if (TC_DBG(p) >= 2) { if (va[0] == 0x12345678u && va[7] == 0x9abcdef0u) pix_base[p.out_off[0]] = 1; }
                        else if (TST) staged(va, u);
                        else if (OUT == 2) epilogue_unit_nhwc<RQ, TAB, NST>(va, cm0 + 16u * CMB * (uint32_t)u, tab_lane, tab_stride, cs, qs, pix_base + p.out_off[0], pix_base + p.out_off[1],
                                                                            pix_base + p.out_off[2], co_left - u * 16, p.onhwc_vec != 0);
                        else epilogue_unit<RQ, TAB, NST, OUT == 1, OUT == 1 ? 1 : 0>(va, cm0 + 16u * CMB * (uint32_t)u, tab_lane, tab_stride, cs, qs, pix_base + p.out_off[0], pix_base + p.out_off[1],
                                                                   pix_base + p.out_off[2], plane, co_left - u * 16, nh + u * 16, keep);
                        pix_base += plane16;
                        if (++u >= u_hi) break;
                        tmem_ld_wait(vb);
                        if (u + 1 < u_hi) tmem_ld16_issue(acc_g + (uint32_t)((u + 1) * 16), va);
                        else if (last_g) {
                            tcgen05_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(sa_empty + 8u * ab);
                        }
                        if (TC_DBG(p) >= 2) { if (vb[0] == 0x12345678u && vb[7] == 0x9abcdef0u) pix_base[p.out_off[0]] = 1; }
                        else if (TST) staged(vb, u);
                        else if (OUT == 2) epilogue_unit_nhwc<RQ, TAB, NST>(vb, cm0 + 16u * CMB * (uint32_t)u, tab_lane, tab_stride, cs, qs, pix_base + p.out_off[0], pix_base + p.out_off[1],
                                                                            pix_base + p.out_off[2], co_left - u * 16, p.onhwc_vec != 0);
                        else epilogue_unit<RQ, TAB, NST, OUT == 1, OUT == 1 ? 2 : 0>(vb, cm0 + 16u * CMB * (uint32_t)u, tab_lane, tab_stride, cs, qs, pix_base + p.out_off[0], pix_base + p.out_off[1],
                                                                   pix_base + p.out_off[2], plane, co_left - u * 16, nh + u * 16, keep);
                        pix_base += plane16;
                        if (++u >= u_hi) break;
                    }
                }
                if (++ab == p.acc_bufs) { ab = 0; aph ^= 1; }
            }
        }
    } else if (warp == WARP_MMA) {
        if (lane < p.grp) { /* ===== MMA issuers: lane g issues the MMAs of M tile g of every group =====
            * Issuing one small MMA costs a thread ~300 cycles (measured: 9 taps x K=32, N=32 are issue-bound, not
            * tensor-bound), so the M tiles of a group -- independent accumulators -- are issued by different lanes of this
            * warp, each committing (arriving) on its own.  All MMAs of one accumulator stay on one lane, i.e. in order.
            * Everything loop-invariant (descriptor halves, barrier addresses, strides in 16-byte descriptor units) is
            * computed up front and the descriptors are advanced by additions. */
            const uint32_t k_sbo16 = (8u * (uint32_t)p.bk) >> 4;
            /* descriptor high word: SBO >> 4 at [32,46), version 1 at [46,48), layout type at [61,64) */
            const uint32_t hi_k = k_sbo16 | (1u << 14) | (p.b_layout << 29);
            /* s2d mode: canonical no-swizzle K-major layout with SBO = 128 (8 rows of 16 bytes) and LBO = 16: element (r, k) at
             * byte 16 r + k, i.e. a 32-byte K row is the pixel's 16 channels followed by the NEXT pixel's (SURVEY 8a row 6) */
            const uint32_t hi_a = p.toep ? ((128u >> 4) | (1u << 14)) : (p.a_kmajor ? hi_k : ((1024u >> 4) | (1u << 14) | (2u << 29)));
            /* low word: start address >> 4 at [0,14), LBO >> 4 at [16,30) (16 bytes for the K-major operands) */
            const uint32_t a_lo0 = (a_base >> 4) | (p.a_kmajor ? (1u << 16) : 0u), a_st16 = p.a_stage_bytes >> 4;
            const uint32_t b_lo0 = (b_base >> 4) | (1u << 16), b_st16 = p.b_stage_bytes >> 4;
            /* per MMA (K = 32): K-major operands advance 32 bytes inside the swizzle atom; the MN-major A (NCHW planes,
             * 128B swizzle) advances 32 K-rows of 128 bytes = 4 atoms of 8 rows */
            const uint32_t a_j16 = p.a_kmajor ? 2u : 256u;
            const int nj = p.bk >> 5, stages = p.stages, acc_bufs = p.acc_bufs, n_tile = p.n_tile, n_img = p.n_img, G = p.grp;
            const uint32_t a_tile16 = p.a_tile_bytes >> 4, g_rows16 = (uint32_t)(TC_BM * p.a_row_bytes) >> 4;
            const int ntaps = p.ntaps, ksteps = p.ksteps_per_tap;
            const uint32_t idesc = p.idesc;
            const bool b_res = GATHER || p.b_resident, halo = p.halo != 0;
            const uint32_t sa_full = smem_u32(&bar_full[0]), sa_empty = smem_u32(&bar_empty[0]);
            const uint32_t sa_tfull = smem_u32(&bar_tmem_full[0]), sa_tempty = smem_u32(&bar_tmem_empty[0]);
            if (b_res) mbar_wait(smem_u32(&bar_b), 0);
            int s = 0, ph = 0, buf = 0, aph = 1; /* waits on the accumulator-empty barriers start with the opposite parity */
            for (TileIter ti(blockIdx.x, gridDim.x, tiles_per_img); ti.img < n_img; ti.next()) {
                mbar_wait(sa_tempty + 8u * buf, aph); /* epilogue drained this accumulator */
                tcgen05_fence_after();
                const uint32_t acc = tmem_d + (uint32_t)(buf * G * n_tile);
                if (halo) {
                    /* a tap = the same rows shifted: the operand simply starts (shift) rows further down.  The swizzle is a
                     * function of the absolute shared-memory address (measured: a start address that is not a multiple of
                     * the 8-row atom needs NO descriptor base offset), so TMA's layout is read back as is */
                    for (int kb = 0; kb < ksteps; kb++) {
                        mbar_wait(sa_full + 8u * s, ph);
                        tcgen05_fence_after();
                        const uint32_t a_st = a_lo0 + s * a_st16;
                        { /* M tile g of the group starts 128 rows further down the same stage */
                            const int g = lane;
                            uint32_t b_lo = b_lo0 + kb * b_st16;
                            for (int tap = 0; tap < ntaps; tap++, b_lo += ksteps * b_st16) {
                                const uint32_t a_lo = a_st + g * g_rows16 + (uint32_t)s_shift[tap]; /* halo mode: row shift in 16-byte units */
                                for (int j = 0; j < nj; j++)
                                    umma_i8(acc + (uint32_t)(g * n_tile), a_lo + 2u * j, hi_a, b_lo + 2u * j, hi_k, idesc, (uint32_t)((kb | tap | j) != 0));
                            }
                        }
                        umma_commit(sa_empty + 8u * s);
                        if (++s == stages) { s = 0; ph ^= 1; }
                    }
                } else {
                    for (int i = 0; i < nsteps; i++) {
                        mbar_wait(sa_full + 8u * s, ph);
                        tcgen05_fence_after();
                        const uint32_t a_st = a_lo0 + s * a_st16 + lane * a_tile16, b_lo = b_lo0 + (b_res ? i : s) * b_st16;
                        if (TC_DBG(p) != 4 && TC_DBG(p) != 9)
                            for (int j = 0; j < nj; j++)
                                umma_i8(acc + (uint32_t)(lane * n_tile), a_st + a_j16 * j, hi_a, b_lo + 2u * j, hi_k, idesc, (uint32_t)((i | j) != 0));
                        umma_commit(sa_empty + 8u * s); /* frees the stage when these MMAs retire */
                        if (++s == stages) { s = 0; ph ^= 1; }
                    }
                }
                umma_commit(sa_tfull + 8u * buf);
                if (++buf == acc_bufs) { buf = 0; aph ^= 1; }
            }
        }
    } else if (!GATHER) {
        if (warp == WARP_PROD && lane == 0) { /* ===== TMA producer (same care for the per-step instruction count) ===== */
            const int bk = p.bk, ntaps = p.ntaps, ksteps = p.ksteps_per_tap, stages = p.stages, n_img = p.n_img, n_tiles = p.n_tiles;
            const uint32_t a_stb = p.a_stage_bytes, b_stb = p.b_stage_bytes, a_tb = p.a_tile_bytes;
            const int G = p.grp;
            const bool b_res = p.b_resident != 0, a_km = p.a_kmajor != 0;
            const uint32_t sa_full = smem_u32(&bar_full[0]), sa_empty = smem_u32(&bar_empty[0]);
            if (b_res) { /* the whole repacked weight matrix of this N tile set stays in shared memory */
                mbar_expect_tx(smem_u32(&bar_b), (uint32_t)(nsteps * p.n_tile * bk));
                for (int tap = 0, i = 0; tap < ntaps; tap++)
                    for (int kb = 0; kb < ksteps; kb++, i++)
                        tma_load_3d(b_base + i * b_stb, &mapB, smem_u32(&bar_b), kb * bk, 0, tap);
            }
            int s = 0, ph = 1; /* waits on the empty barriers start with the opposite parity */
            if (p.halo) {
                const int nb = p.halo_nb, rb = p.halo_rb;
                /* wide mode: the same bytes as 256-byte rows of 16 pixels (TMA's cost is per row: measured ~2 cycles per 16-byte row) */
                const int wide = p.halo_wide ? 16 : 1;
                const uint32_t tx = (uint32_t)(nb * rb * p.a_row_bytes * wide), box_b = (uint32_t)(rb * p.a_row_bytes * wide);
                for (TileIter ti(blockIdx.x, gridDim.x, tiles_per_img); ti.img < n_img; ti.next()) {
                    const int q0 = ti.rem * G * TC_BM, zc = p.img0 + ti.img; /* n_tiles == 1 with resident weights; q0 and halo_min are multiples of 16 in wide mode */
                    const int qr = (q0 + p.halo_min) / wide;
                    for (int kb = 0; kb < ksteps; kb++) {
                        mbar_wait(sa_empty + 8u * s, ph);
                        const uint32_t full = sa_full + 8u * s, dst = a_base + s * a_stb;
                        if (TC_DBG(p) == 3 || TC_DBG(p) == 9) { mbar_arrive(full); if (++s == stages) { s = 0; ph ^= 1; } continue; }
                        mbar_expect_tx(full, tx);
                        for (int b = 0; b < nb; b++) tma_load_3d(dst + b * box_b, &mapA, full, kb * bk, qr + b * rb, zc);
                        if (++s == stages) { s = 0; ph ^= 1; }
                    }
                }
            } else {
                const uint32_t tx = p.a_tx_bytes + (b_res ? 0u : (uint32_t)(p.n_tile * bk));
                const bool rect = p.rect != 0;
                for (TileIter ti(blockIdx.x, gridDim.x, tiles_per_img); ti.img < n_img; ti.next()) {
                    const int mg = n_tiles == 1 ? ti.rem : ti.rem / n_tiles, n0 = (ti.rem - mg * n_tiles) * p.n_tile;
                    const int q0 = mg * G * TC_BM, zc = p.img0 + ti.img;
                    for (int tap = 0; tap < ntaps; tap++) {
                        const int sh = s_shift[tap], qa = q0 + sh; /* rect mode: sh = kh << 16 | kw */
                        for (int kb = 0; kb < ksteps; kb++) {
                            mbar_wait(sa_empty + 8u * s, ph);
                            const uint32_t full = sa_full + 8u * s;
                            if (TC_DBG(p) == 3 || TC_DBG(p) == 9) { mbar_arrive(full); if (++s == stages) { s = 0; ph ^= 1; } continue; }
                            mbar_expect_tx(full, tx);
                            for (int g = 0; g < G; g++) { /* rows beyond the tensor (last, partial group) are zero-filled */
                                if (rect) {
                                    const int mt = mg * G + g, ty = mt / p.tiles_x, tx0 = mt - ty * p.tiles_x;
                                    tma_load_4d(a_base + s * a_stb + g * a_tb, &mapA, full, kb * bk, tx0 * p.tw * p.rs + (sh & 0xFFFF) - p.rpl,
                                                ty * p.th * p.rs + (sh >> 16) - p.rpt, zc);
                                } else if (a_km) tma_load_3d(a_base + s * a_stb + g * a_tb, &mapA, full, kb * bk, qa + g * TC_BM, zc);
                                else tma_load_3d(a_base + s * a_stb + g * a_tb, &mapA, full, q0 + g * TC_BM, kb * bk, zc);
                            }
                            if (!b_res) tma_load_3d(b_base + s * b_stb, &mapB, full, kb * bk, n0, tap);
                            if (++s == stages) { s = 0; ph ^= 1; }
                        }
                    }
                }
            }
        }
    } else {
        /* ===== gather producer: 128 threads, one A row (output pixel) each ===== */
        if (warp == WARP_PROD && lane == 0) { /* the whole weight matrix once */
            mbar_expect_tx(smem_u32(&bar_b), (uint32_t)(p.n_tile * 128));
            tma_load_3d(b_base, &mapB, smem_u32(&bar_b), 0, 0, 0);
        }
        const int pr = (warp - WARP_PROD) * 32 + lane;
        const int PP = p.gPWW * 4, nwords = p.gC * p.gPH * p.gPWW;
        const int th = TC_BM >> p.tw_shift;
        const int tb = ((pr >> p.tw_shift) * p.gS) * PP + (pr & ((1 << p.tw_shift) - 1)) * p.gS; /* this pixel's origin in the patch */
        const int nchunks = (p.gKt + 15) >> 4;
        /* the input patch of a tile travels global -> shared with cp.async (zero fill outside the image), three
         * patch buffers deep: while the rows of tile t are built, the patches of tiles t+1 and t+2 are in flight */
        const uint32_t patch_sa = smem_u32(g_patch);
        auto issue = [&](int img, int mt, int buf) { /* n_tiles == 1 in gather mode: tile inside the image = M tile */
            const int ty = mt / p.tiles_x, tx = mt - ty * p.tiles_x;
            const int y0 = ty * th * p.gS - p.gpt, xs = (tx << p.tw_shift) * p.gS - p.gpl - p.gdx;
            const uint8_t *src = p.g_src + (unsigned long long)img * p.g_stride + ((long long)y0 * p.gW + xs);
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int wi = pr + 128 * i;
                if (wi < nwords) {
                    const int yx = g_pyx[wi], y = y0 + (yx >> 16), x = xs + (yx & 0xFFFF);
                    const bool ok = (unsigned)y < (unsigned)p.gH && (unsigned)x < (unsigned)p.gW;
                    const uint8_t *a = ok ? src + g_poff[wi] : p.g_src;
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(patch_sa + (uint32_t)(buf * 4096 + wi * 4)), "l"(a), "r"(ok ? 4 : 0) : "memory");
                }
            }
        };
        int s = 0, ph = 1, g = 0, gi = 0, t = 0;
        const int G = p.grp;
        TileIter ti(blockIdx.x, gridDim.x, tiles_per_img), tii = ti; /* consume / issue positions */
        for (int k = 0; k < 2; k++) {
            if (tii.img < p.n_img) { issue(tii.img, tii.rem * G + gi, k); if (++gi == G) { gi = 0; tii.next(); } }
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
        for (; ti.img < p.n_img; t++) {
            asm volatile("bar.sync 2, 128;" ::: "memory"); /* everyone has built the rows of tile t-1: its patch buffer is free */
            if (tii.img < p.n_img) { issue(tii.img, tii.rem * G + gi, (t + 2) % 3); if (++gi == G) { gi = 0; tii.next(); } }
            asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group 2;" ::: "memory"); /* this thread's part of tile t's patch has landed ... */
            asm volatile("bar.sync 2, 128;" ::: "memory");        /* ... and everybody else's */
            const int gcur = g;
            if (++g == G) { g = 0; ti.next(); }
            if (gcur == 0) mbar_wait_relaxed(smem_u32(&bar_empty[s]), ph); /* the stage holds the whole group */
            uint8_t *row = smem_al + (size_t)s * p.a_stage_bytes + (size_t)gcur * p.a_tile_bytes + pr * 128;
            const uint8_t *pb = g_patch + (t % 3) * 4096 + tb;
            /* K columns >= Kt meet zero weights (k_repack_rows pads B with zeros), so whatever bytes sit there are
             * harmless: table entries beyond Kt point at offset 0 and 16-byte chunks beyond Kt are not written at all */
            if (p.g_align2) { /* taps come in aligned byte pairs (even stride, even kernel width): 2-byte loads */
#pragma unroll
                for (int c = 0; c < 8; c++) {
                    if (c < nchunks) {
                        const int4 pa = reinterpret_cast<const int4 *>(s_koff)[c * 2], pc = reinterpret_cast<const int4 *>(s_koff)[c * 2 + 1];
                        uint4 wv;
                        wv.x = (uint32_t)*reinterpret_cast<const uint16_t *>(pb + pa.x) | ((uint32_t)*reinterpret_cast<const uint16_t *>(pb + pa.y) << 16);
                        wv.y = (uint32_t)*reinterpret_cast<const uint16_t *>(pb + pa.z) | ((uint32_t)*reinterpret_cast<const uint16_t *>(pb + pa.w) << 16);
                        wv.z = (uint32_t)*reinterpret_cast<const uint16_t *>(pb + pc.x) | ((uint32_t)*reinterpret_cast<const uint16_t *>(pb + pc.y) << 16);
                        wv.w = (uint32_t)*reinterpret_cast<const uint16_t *>(pb + pc.z) | ((uint32_t)*reinterpret_cast<const uint16_t *>(pb + pc.w) << 16);
                        *reinterpret_cast<uint4 *>(row + ((c ^ (pr & 7)) << 4)) = wv;
                    }
                }
            } else {
#pragma unroll
                for (int c = 0; c < 8; c++) {
                    if (c < nchunks) {
                        uint32_t wds[4];
#pragma unroll
                        for (int g = 0; g < 4; g++) {
                            const int4 o4 = reinterpret_cast<const int4 *>(s_koff)[c * 4 + g];
                            wds[g] = (uint32_t)pb[o4.x] | ((uint32_t)pb[o4.y] << 8) | ((uint32_t)pb[o4.z] << 16) | ((uint32_t)pb[o4.w] << 24);
                        }
                        *reinterpret_cast<uint4 *>(row + ((c ^ (pr & 7)) << 4)) = make_uint4(wds[0], wds[1], wds[2], wds[3]);
                    }
                }
            }
            if (gcur == G - 1) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); /* generic-proxy writes -> visible to the MMA's async proxy */
                __syncwarp();
                if (lane == 0) mbar_arrive(smem_u32(&bar_full[s]));
                if (++s == p.stages) { s = 0; ph ^= 1; }
            }
        }
    }
teardown:
    tcgen05_fence_before();
    __syncthreads();
    if (warp == WARP_MMA) {
        tcgen05_fence_after();
        tmem_dealloc(tmem_d, (uint32_t)p.tmem_cols);
    }
}

/* ---- pre-pass: arena NCHW -> channel-innermost copy with zero padding --------------- */
/* dst[pix][c] for pix < npix (source pixel: copy_src_pixel).
 * 32 pixels x 32 channels per block through shared memory: coalesced reads along pixels,
 * coalesced writes along channels. */
__global__ void __launch_bounds__(256) k_to_nhwc(const uint8_t *src_base, unsigned long long src_stride, uint8_t *dst_base,
                                                 unsigned long long dst_stride, int C, int Cp, int H, int W, int Wp, int plane, int npix,
                                                 int stride2, int pt, int pl) { /* Cp >= C: bytes per pixel of the copy */
    __shared__ uint8_t tile[32][33];
    const uint8_t *src = src_base + (unsigned long long)blockIdx.z * src_stride;
    uint8_t *dst = dst_base + (unsigned long long)blockIdx.z * dst_stride;
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
            tile[ty + 8 * k][tx] = (inb && c < C) ? src[((long long)c * H + ih) * W + iw] : (uint8_t)0;
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int pix = p0 + ty + 8 * k, c = c0 + tx;
        if (pix < npix && c < Cp) dst[(long long)pix * Cp + c] = tile[tx][ty + 8 * k]; /* channels C..Cp-1: zeros (padded K) */
    }
}
/* ---- s2d mode (6x6 stride-2 pad-2 conv with <= 4 input channels = 3x3 stride-1 pad-1 conv over the 2x2 space-to-depth
 * image): P[(y+1)*Wp + (x+1)][16] = the 2x2 input block (2y+py, 2x+px) of every channel, byte c' = ci*4 + py*2 + px,
 * zero border and zero beyond 4*C bytes.  One thread per P pixel. */
__global__ void __launch_bounds__(256) k_s2d16(const uint8_t *__restrict__ src_base, unsigned long long src_stride, uint8_t *__restrict__ dst_base,
                                               unsigned long long dst_stride, int C, int H, int W, int Wp, int npix, int src_nhwc) {
    const uint8_t *src = src_base + (unsigned long long)blockIdx.y * src_stride;
    uint4 *dst = reinterpret_cast<uint4 *>(dst_base + (unsigned long long)blockIdx.y * dst_stride);
    /* four pixels per thread, 256 apart: all their loads are issued before the first store (the kernel is pure latency) */
    constexpr int PPT = 4;
    const int base = blockIdx.x * (256 * PPT) + threadIdx.x;
    const unsigned wp_magic = 0xFFFFFFFFu / (unsigned)Wp + 1u; /* floor(a / Wp) = umulhi(a, magic), a < 2^31 / Wp (host-checked mflat bound) */
    uint32_t w[PPT][4];
#pragma unroll
    for (int k = 0; k < PPT; k++) {
        const int pix = base + k * 256;
        w[k][0] = w[k][1] = w[k][2] = w[k][3] = 0u;
        if (pix < npix) {
            const int yy = (int)__umulhi((unsigned)pix, wp_magic), y = yy - 1, x = pix - yy * Wp - 1;
            if (y >= 0 && 2 * y + 1 < H && x >= 0 && 2 * x + 1 < W) {
#pragma unroll
                for (int ci = 0; ci < 4; ci++) { /* the mode requires C <= 4 */
                    if (ci < C) {
                        if (src_nhwc) { /* channel-innermost source: pixel (yy, xx) channel ci at (yy * W + xx) * C + ci */
                            const uint8_t *r0 = src + ((long long)(2 * y) * W + 2 * x) * C + ci;
                            w[k][ci] = (uint32_t)r0[0] | ((uint32_t)r0[C] << 8) | ((uint32_t)r0[(long long)W * C] << 16) | ((uint32_t)r0[(long long)W * C + C] << 24);
                        } else {
                            const uint8_t *r0 = src + ((long long)ci * H + 2 * y) * W + 2 * x;
                            w[k][ci] = (uint32_t)*reinterpret_cast<const uint16_t *>(r0) | ((uint32_t)*reinterpret_cast<const uint16_t *>(r0 + W) << 16);
                        }
                    }
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < PPT; k++) {
        const int pix = base + k * 256;
        if (pix < npix) dst[pix] = make_uint4(w[k][0], w[k][1], w[k][2], w[k][3]);
    }
}
/* OIHW 6x6 weights -> [t = ky2*2 + pair][Co_pad][32]: K byte k = (pixel kx2 = 2*pair + k/16, channel byte c' = k%16) */
__global__ void k_repack_s2d(const int8_t *w, int8_t *dst, int Co, int Co_pad, int Ci, int ohwi) {
    const long long total = 6ll * Co_pad * 32;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(i % 32), co = (int)((i / 32) % Co_pad), t = (int)(i / (32ll * Co_pad));
        const int ky2 = t >> 1, kx2 = 2 * (t & 1) + (k >> 4), cp = k & 15, ci = cp >> 2, py = (cp >> 1) & 1, px = cp & 1;
        int8_t v = 0;
        if (co < Co && ci < Ci && kx2 < 3) v = ohwi ? w[(((long long)co * 6 + (2 * ky2 + py)) * 6 + (2 * kx2 + px)) * Ci + ci]
                                                    : w[(((long long)co * Ci + ci) * 6 + (2 * ky2 + py)) * 6 + (2 * kx2 + px)];
        dst[i] = v;
    }
}
/* OIHW rows (Kt bytes) -> [Co_pad][Kp], zero padded */
__global__ void k_repack_rows(const int8_t *w, int8_t *dst, int Co, int Co_pad, int Kt, int Kp) {
    long long total = (long long)Co_pad * Kp;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        int k = (int)(i % Kp), co = (int)(i / Kp);
        dst[i] = (co < Co && k < Kt) ? w[(long long)co * Kt + k] : (int8_t)0;
    }
}
/* OIHW -> [tap][Co_pad][Cip], rows beyond Co and columns beyond Ci zero */
__global__ void k_repack_weights(const int8_t *w, int8_t *dst, int Co, int Co_pad, int Ci, int Cip, int ntaps, int ohwi) {
    long long total = (long long)ntaps * Co_pad * Cip; /* Cip >= Ci: K extent per tap, columns beyond Ci zero */
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        int ci = (int)(i % Cip);
        long long r = i / Cip;
        int co = (int)(r % Co_pad), tap = (int)(r / Co_pad);
        dst[i] = (co < Co && ci < Ci) ? (ohwi ? w[((long long)co * ntaps + tap) * Ci + ci] : w[((long long)co * Ci + ci) * ntaps + tap]) : (int8_t)0;
    }
}

/* ---- host side ------------------------------------------------------------------ */
typedef void (*TcKernel)(const CUtensorMap, const CUtensorMap, const TcParams);
struct TcPlanImpl {
    CUtensorMap mapA, mapB, mapA_linked;
    bool tst = false;      /* plane stores through shared memory (the space-to-depth stem) */
    bool has_linked = false;
    TcParams p;
    int prepass = 0;
    int rq = 0;     /* requantisation variant of the epilogue (requant_pair) */
    bool tab = false; /* the epilogue looks its byte up in the per-lane word table */
    int C = 0, Cp = 0, H = 0, W = 0, npix = 0; /* Cp: bytes per pixel of the channel-innermost copy */
    PixelCopy copy; /* prepass 1 / 2 */
    const uint8_t *src_slot0 = nullptr; /* input tensor in slot 0 */
    uint8_t *scratch = nullptr;
    size_t scratch_stride = 0, slot_stride = 0;
    int8_t *d_wr = nullptr;     /* repacked weights */
    uint32_t *d_lutw = nullptr; /* epilogue word table */
    int nst = 0;                /* NCHW streams stored */
    int stream_byte[4] = {-1, -1, -1, -1}; /* table byte of stream Z / S / Y (plain conv: Y is stream 0) / the forwarded copy, -1 = not in the table */
    int nhwc_stream = -1;              /* stream whose value also fills table byte 3 (side output), -1 = none */
    TcKernel kernel = nullptr;
    size_t smem = 0;
    int ctas_per_sm = 2;
    int epi = 8; /* epilogue warps per CTA */
    int sms = 0; /* multiprocessors of the device the plan was built on */
    int nhwc_in = 0;  /* channel-innermost activations / OHWI weights (OP_CONV_I8_NHWC) */
    bool gather_direct = false; /* gather mode reads the input tensor in the arena itself (no private copy needed) */
};

EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)sym;
    }
    return fn;
}

bool make_map3(CUtensorMap *m, void *base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t s1, uint64_t s2, uint32_t b0, uint32_t b1,
               CUtensorMapSwizzle sw) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return false;
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {s1, s2};
    cuuint32_t box[3] = {b0, b1, 1};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_last_error("cuTensorMapEncodeTiled failed: %d (dims %llu %llu %llu strides %llu %llu box %u %u)", (int)r,
                       (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2, (unsigned long long)s1,
                       (unsigned long long)s2, b0, b1);
        return false;
    }
    return true;
}

bool make_map4(CUtensorMap *m, void *base, uint64_t C, uint64_t W, uint64_t H, uint64_t N, uint64_t img_stride, uint32_t bc, uint32_t bw,
               uint32_t bh, uint32_t es, CUtensorMapSwizzle sw) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return false;
    cuuint64_t dims[4] = {C, W, H, N};
    cuuint64_t strides[3] = {C, W * C, img_stride};
    cuuint32_t box[4] = {bc, bw, bh, 1};
    cuuint32_t estr[4] = {1, es, es, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_last_error("cuTensorMapEncodeTiled (4-d) failed: %d (dims %llu %llu %llu %llu box %u %u %u stride %u)", (int)r, (unsigned long long)C,
                       (unsigned long long)W, (unsigned long long)H, (unsigned long long)N, bc, bw, bh, es);
        return false;
    }
    return true;
}

int tc_n_tile(int oc) {
    const int co_pad = round_up(oc, 16);
    return co_pad <= 256 ? co_pad : (co_pad % 256 == 0 ? 256 : 128);
}
int tc_n_tiles(int oc) { return (round_up(oc, 16) + tc_n_tile(oc) - 1) / tc_n_tile(oc); }
int tc_bk(int kbytes) { return kbytes % 128 == 0 ? 128 : (kbytes % 64 == 0 ? 64 : 32); }
uint32_t tc_umma_layout(int bk) { return bk == 128 ? 2u : (bk == 64 ? 4u : 6u); }
CUtensorMapSwizzle tc_swizzle(int bk) { return bk == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (bk == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B); }
int tc_sm_count() {
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms > 0 ? sms : 148;
}

PixelCopy pixel_copy(const Op &o) {
    PixelCopy c;
    if (o.sh < 1 || o.sh > 2 || o.pl >= o.kw || o.pt >= o.kh) return c;
    c.pt = o.pt; c.pl = o.pl;
    if (o.sh == 1) {
        c.Wp = o.iw + o.kw - 1; c.plane = o.ih * c.Wp; c.npix = c.plane;
    } else {
        /* phase plane: rows a = 0 .. , pitch Wp >= ow + (k-1)/2; enough zero rows below that the
         * deepest tap of the last output row stays inside its own plane */
        c.Wp = o.ow + (o.kw - 1) / 2;
        const int rows = std::max((o.ih - 1 + o.pt) / 2 + 1, o.oh + (o.kh - 1) / 2);
        c.plane = rows * c.Wp; c.npix = 4 * c.plane;
    }
    if (o.ow > c.Wp) return PixelCopy();
    c.mode = o.sh;
    return c;
}

/* Row pitch of the space-to-depth stem's bordered pixel index.  The stem's NCHW streams leave through a shared-memory staging
 * block (TST: the stem writes the largest planes next to a side output and is the one layer class where staging pays, -7 %;
 * profiles/r02l_staged_stores.txt), copied out in 16-pixel pieces of one row.  So when the output rows are a multiple of 16
 * pixels the pitch is rounded up to one as well: every 128-pixel tile then starts on a 16-pixel boundary of its row.  The extra
 * pad columns are computed and discarded; the rounding is skipped when they would add more than 20 % to the layer. */
static int store_pitch(int wp_min, int ow) {
    constexpr int max_waste = 20; /* percent */
    if (ow % 16 || wp_min % 16 == 0) return wp_min;
    const int wp = (wp_min + 15) / 16 * 16;
    return (wp - wp_min) * 100 <= max_waste * wp_min ? wp : wp_min;
}

/* geometry shared by tc_scratch_need and tc_plan */
struct TcGeom {
    bool ok = false;
    int prepass = 0; /* 4: space-to-depth copy with 16-byte pixels (stem); 0: A from the arena (1x1); 1: NHWC copy, rows padded (stride 1); 2: NHWC 2x2 phase split (stride 2);
                        3: gather -- A rows built in shared memory from a private NCHW copy of the input (small Ci);
                        5: NHWC 1x1 -- flat tiles, A rows = the arena tensor's pixels; 6: NHWC kxk -- rect tiles, one 4-d TMA box per tap */
    int Wp = 0, npix = 0, ntaps = 0, Kp = 0;
    PixelCopy copy; /* prepass 1 / 2 */
    int kpad = 0; /* prepass 0 with Ci not a multiple of 32: K extent padded with zeros (TMA fills the missing channel rows, the repacked weights hold zeros) */
    int tw_shift = 0, PH = 0, PWW = 0, dx = 0; /* gather: M tile shape and input patch geometry */
    int rtw = 0, rth = 0; /* rect mode (prepass 6): output pixels per tile row / tile rows, rtw * rth <= 128 */
    size_t scratch_bytes = 0;
};
/* the YOLOv5 stem shape: 6x6 stride 2 pad 0 / 2 over <= 4 channels == 3x3 stride 1 over the 2x2 space-to-depth image (prepass 4,
 * the same copy for NCHW and channel-innermost inputs); fills *g when the op has that shape */
static bool stem_geometry(const Op &o, TcGeom *g) {
    if (!(o.sh == 2 && o.sw == 2 && o.kh == 6 && o.kw == 6 && (o.pt == 0 || o.pt == 2) && (o.pl == 0 || o.pl == 2) && o.ic <= 4 &&
          o.ih % 2 == 0 && o.iw % 2 == 0 && o.oh <= o.ih / 2 && o.ow <= o.iw / 2 && round_up(o.oc, 16) <= 128 && (long long)o.oh * o.ow >= 4096))
        return false;
    g->prepass = 4; g->Wp = store_pitch(o.iw / 2 + 2, o.ow); g->npix = (o.ih / 2 + 2) * g->Wp; g->ntaps = 6; g->Kp = 32;
    g->scratch_bytes = (size_t)g->npix * 16;
    g->ok = true;
    return true;
}
static TcGeom tc_geometry(const Op &o) {
    TcGeom g;
    if (o.kind == OP_CONV_I8_NHWC) { /* channel-innermost activations and OHWI weights (reference src/mars/mxu_conv.c:713-757) */
        if (o.mode != EXEC_PARALLEL || o.xlat) return g;
        if (o.oc < 16 || o.sh != o.sw || o.sh < 1 || o.sh > 2 || o.kh < 1 || o.kh != o.kw) return g;
        if (o.oh <= 0 || o.ow <= 0 || o.ih <= 0 || o.iw <= 0 || o.ic <= 0 || round_up(o.oc, 16) > TC_MAX_CO) return g;
        if (o.pt < 0 || o.pl < 0 || o.pt >= o.kh || o.pl >= o.kw) return g;
        g.ntaps = o.kh * o.kw;
        if (g.ntaps > TC_MAX_TAPS) return g;
        if (stem_geometry(o, &g)) return g;
        if (o.ic < 32 || o.ic % 32) return g; /* K rows are the pixels' channel vectors: whole 32-byte k-steps only */
        if (o.kh == 1 && o.sh == 1 && o.pt == 0 && o.pl == 0 && o.oh <= o.ih && o.ow == o.iw) {
            g.prepass = 5; g.Wp = o.iw; /* 1x1: flat 128-pixel tiles, A rows straight from the arena tensor (or a private copy) */
            g.scratch_bytes = (size_t)o.ic * o.ih * o.iw;
        } else {
            /* kxk / strided: an M tile is tw x th output pixels; a tap is one 4-d TMA box with OOB zero fill.  Least waste wins */
            long long best = -1;
            for (int tw = 2; tw <= 128 && tw <= o.ow + 15; tw++) {
                const int th = 128 / tw;
                if (tw * o.sh > 256 || th * o.sh > 256 || th < 1) continue;
                const long long tiles = (long long)((o.ow + tw - 1) / tw) * ((o.oh + th - 1) / th);
                if (best < 0 || tiles < best) { best = tiles; g.rtw = tw; g.rth = th; }
            }
            if (best < 0) return g;
            g.prepass = 6; g.Wp = o.ow;
            g.scratch_bytes = (size_t)o.ic * o.ih * o.iw; /* private copy of the input when a fused output overwrites it */
        }
        g.ok = true;
        return g;
    }
    if (o.kind != OP_CONV_I8_NCHW || o.mode != EXEC_PARALLEL || o.xlat) return g;
    if (o.oc < 16 || o.sh != o.sw || o.sh < 1 || o.kh < 1 || o.kw < 1) return g;
    if (o.oh <= 0 || o.ow <= 0 || o.ih <= 0 || o.iw <= 0 || o.ic <= 0) return g;
    if (round_up(o.oc, 16) > TC_MAX_CO) return g;
    /* 1x1 stride-1 conv straight from the NCHW planes with any channel count >= 16 (ShuffleNet-style 58 / 116 / 232 / 464):
     * the channel rows a k-step reads beyond Ci do not exist in the tensor map and arrive as zeros */
    if (o.ic >= 16 && o.ic % 32 && o.kh == 1 && o.kw == 1 && o.sh == 1 && o.pt == 0 && o.pl == 0 && o.oh <= o.ih && o.ow == o.iw) {
        g.ntaps = 1; g.Wp = o.iw;
        g.kpad = o.ic > 64 ? round_up(o.ic, 128) : round_up(o.ic, 32);
        if (((long long)o.ih * o.iw) % 16 == 0) g.prepass = 0;
        else { /* planes that TMA cannot address (stride not a multiple of 16 bytes, e.g. 10 x 10): channel-innermost copy, kpad bytes per pixel */
            g.copy = pixel_copy(o);
            g.prepass = 1; g.npix = g.copy.npix;
            g.scratch_bytes = (size_t)g.npix * g.kpad;
        }
        g.ok = true;
        return g;
    }
    if (o.ic < 32 || o.ic % 32 || o.kh != o.kw) {
        auto small_k = [&]() -> bool {
        if (stem_geometry(o, &g)) return true;
        /* small / odd channel counts: one 128-byte K row per pixel, built in shared memory from a staged input patch */
        const int Kt = o.ic * o.kh * o.kw;
        if (Kt > 128 || o.kh > 255 || o.kw > 255 || (long long)o.oh * o.ow < 4096 || round_up(o.oc, 16) > 256) return false;
        if (o.iw % 4 || o.pl < 0 || o.pt < 0) return false;
        /* M tile = tw x (128/tw) output pixels: least padding, then the widest */
        long long best = -1;
        for (int sh = 7; sh >= 4; sh--) {
            const int tw = 1 << sh, th = 128 >> sh;
            if ((tw * o.sh) % 4) continue;
            const int dx = ((-o.pl) % 4 + 4) % 4;
            const int PH = (th - 1) * o.sh + o.kh, PWW = (dx + (tw - 1) * o.sw + o.kw + 3) / 4;
            if ((long long)o.ic * PH * PWW > 1024) continue;
            const long long padded = (long long)((o.ow + tw - 1) / tw) * tw * ((o.oh + th - 1) / th) * th;
            if (best < 0 || padded < best) { best = padded; g.tw_shift = sh; g.PH = PH; g.PWW = PWW; g.dx = dx; }
        }
        if (best < 0) return false;
        g.prepass = 3; g.Kp = 128; g.ntaps = 1; g.Wp = o.ow; g.npix = o.oh * o.ow;
        g.scratch_bytes = (size_t)o.ic * o.ih * o.iw;
        g.ok = true;
        return true;
            };
        if (small_k()) return g;
        /* larger K with a channel count that is not a multiple of 32: the general paths below over a channel-innermost copy
         * whose pixels are padded to kpad bytes (zero channels), weights repacked with zero columns */
        if (o.kh != o.kw || o.ic < 8) return TcGeom();
        g = TcGeom();
        g.kpad = round_up(o.ic, 32);
    }
    g.ntaps = o.kh * o.kw;
    if (g.ntaps > TC_MAX_TAPS) return g;
    if (!g.kpad && o.kh == 1 && o.sh == 1 && o.pt == 0 && o.pl == 0 && o.oh <= o.ih && o.ow == o.iw && ((long long)o.ih * o.iw) % 16 == 0) {
        g.prepass = 0; g.Wp = o.iw;
    } else {
        g.copy = pixel_copy(o);
        if (!g.copy.mode) return g;
        g.prepass = g.copy.mode; g.Wp = g.copy.Wp; g.npix = g.copy.npix;
    }
    g.scratch_bytes = g.prepass ? (size_t)g.npix * (g.kpad ? g.kpad : o.ic) : 0;
    g.ok = true;
    return g;
}

size_t tc_scratch_need(const Op &o) {
    TcGeom g = tc_geometry(o);
    return g.ok ? g.scratch_bytes : 0;
}
bool tc_supported(const Op &o) {
    if (!tc_geometry(o).ok) return false;
    return true; /* any Co up to TC_MAX_CO: above 256 the N tiles are 256 or 128 wide and the last one may be ragged (weight rows
                  * beyond Co_pad do not exist in the tensor map and arrive as zeros; the epilogue skips their columns) */
}
bool tc_uses_copy(const Op &o) { return tc_geometry(o).prepass != 0; } /* (NHWC layers: a private copy on demand, see tc_plan) */
bool tc_linkable(const Op &o) { const TcGeom g = tc_geometry(o); return g.ok && (g.prepass == 1 || g.prepass == 2) && !g.kpad; }

/* the word table of the epilogue: index = r + 128 (r = the clamped conv output); byte k = value of output stream k, byte 3 =
 * the side-output stream.  Stream order: a fused conv stores [Z, S, Y] (Z = SiLU product, the stream almost every consumer
 * reads, sits in the low byte), a plain conv stores [Y]. */
static void build_lutw(const Op &o, const uint8_t *h_cpool, const int stream_byte[4], int nhwc_stream, uint32_t *t) {
    const int8_t *ls = o.lut_s >= 0 ? reinterpret_cast<const int8_t *>(h_cpool + o.lut_s) : nullptr;
    const int8_t *lz = o.lut_z >= 0 ? reinterpret_cast<const int8_t *>(h_cpool + o.lut_z) : nullptr;
    for (int idx = 0; idx < 256; idx++) {
        int y = idx - 128;
        if (o.post_relu && y < 0) y = 0;
        /* stream values: fused conv = {Z, S, Y}, plain conv = {Y} */
        uint8_t val[3] = {(uint8_t)y, 0, 0};
        if (o.fused_layers > 0) { val[0] = (uint8_t)(lz ? lz[y + 128] : 0); val[1] = (uint8_t)(ls ? ls[y + 128] : 0); val[2] = (uint8_t)y; }
        uint32_t w = 0;
        for (int k = 0; k < 3; k++)
            if (stream_byte[k] >= 0) w |= (uint32_t)val[k] << (8 * stream_byte[k]);
        if (stream_byte[3] >= 0) w |= (uint32_t)val[o.fused_layers > 0 ? o.fwd_stream : 0] << (8 * stream_byte[3]); /* Op::fwd_out: a second copy of one stream */
        if (nhwc_stream >= 0) w |= (uint32_t)val[nhwc_stream] << 24; /* at most 3 stored streams use bytes 0..2 */
        t[idx] = w;
    }
}

/* Is floor(fl(sc + 0.5f)) the reference's (int32)(sc + (sc >= 0 ? 0.5f : -0.5f)) (src/mars/mxu_conv.c:663-666) for every
 * t = acc + bias with |t| <= bound, sc = fl((float)t * cs)?  For sc >= 0 both are floor(fl(sc + 0.5f)).  For sc < 0 the sum
 * sc + 0.5f is exact, and the two differ exactly when sc is a tie -(n + 0.5) (half-away gives -(n + 1), half-up -n; equal after
 * the clamp for n >= 128) or sc = -pred(0.5), where the reference's fl(sc - 0.5f) rounds to -1.0.  Those 129 floats are
 * enumerated and the integers t around c / cs tested. */
static bool halfup_requant_ok(float cs, long long bound) {
    if (!(fabsf(cs) > 0.0f)) return true; /* sc is always +-0 */
    /* the round-down add of 1.5 * 2^23 must stay inside [2^23, 2^24): |sc| + 0.5 < 2^22 */
    if (!((double)bound * fabs((double)cs) < 4194300.0)) return false;
    for (int n = -1; n <= 127; n++) {
        const float c = n < 0 ? -nextafterf(0.5f, 0.0f) : -((float)n + 0.5f);
        const double t0 = (double)c / (double)cs;
        if (fabs(t0) > (double)bound + 8.0) continue;
        const double ulp = (double)(nextafterf(fabsf(c), 1e30f) - fabsf(c));
        const double span = 2.0 * ulp / fabs((double)cs) + 3.0;
        if (span > 4096.0) return false;
        const long long tc = llround(t0), W = (long long)span;
        for (long long t = tc - W; t <= tc + W; t++) {
            if (std::llabs(t) > bound) continue;
            volatile float sc = (float)t * cs;
            if (sc == c) return false;
        }
    }
    return true;
}

/* max |acc + bias| over all output channels, from the real weights (int32 accumulation: K * 127 * 128 stays far below 2^31) */
static long long acc_bound(const Op &o, const ArenaGeom &ag) {
    const int8_t *w = reinterpret_cast<const int8_t *>(ag.h_weights + o.w);
    const long long K = (long long)o.ic * o.kh * o.kw;
    long long bound = 0;
    for (int co = 0; co < o.oc; co++) {
        long long sum = 0;
        for (long long k = 0; k < K; k++) sum += std::abs((int)w[co * K + k]);
        long long b = 0;
        if (o.bias >= 0) { int32_t bv; memcpy(&bv, ag.h_weights + o.bias + 4 * (size_t)co, 4); b = std::llabs((long long)bv); }
        bound = std::max(bound, sum * 128 + b);
    }
    return bound;
}

/* the reference's requantisation of t = acc + bias (src/mars/mxu_conv.c:663-666), x86 float -> int rule included */
static int ref_requant(int32_t t, float cs) {
    volatile float sc = (float)t * cs;
    volatile float h = sc + (sc >= 0 ? 0.5f : -0.5f);
    const float hv = h;
    const int32_t r = !(hv > -2147483904.0f && hv < 2147483648.0f) ? INT32_MIN : (int32_t)hv;
    return r > 127 ? 127 : (r < -128 ? -128 : r);
}

/* RQ 3: integers (m, s, c) with clamp(floor((t * m + c) / 2^(32 + s))) == ref_requant(t, cs) for EVERY |t| <= tmax, or false.
 * Both sides are monotone step functions of t (cs > 0), so they agree everywhere iff they agree on the two points either side of
 * each of the reference's steps: with theta_k the first t whose reference value is >= k (bisection),
 *     theta_k * m + c >= k * 2^(32+s)      and      (theta_k - 1) * m + c <= k * 2^(32+s) - 1        for k = -127 .. 127
 * (plus the two range ends).  For a given m the valid c form the interval [lo(m), hi(m)]; hi - lo is concave in m, so the best m
 * is found by ternary search around cs * 2^(32+s).  The second degree of freedom matters: the float product fl(t * cs) rounds
 * values just below a tie n + 0.5 up to it on BOTH sides of zero (the reference then rounds away from zero), which a slightly
 * larger multiplier reproduces and a rounding addend alone cannot.  What remains unfittable are scales where that rounding,
 * constant per binade, and the linear tilt disagree on some integer t -- the caller then keeps a float variant. */
static bool int_requant_fit(float cs, long long tmax, int *m_out, int *s_out, long long *c_out) {
    if (!(cs > 0.0f) || !(cs < 0.49f) || tmax < 1 || tmax > 2147483647ll) return false;
    int sh = 0;
    while (sh < 24 && ldexp((double)cs, 32 + sh + 1) < 2147483647.0) sh++;
    const long long m0 = llround(ldexp((double)cs, 32 + sh));
    const int lo_r = ref_requant((int32_t)-tmax, cs), hi_r = ref_requant((int32_t)tmax, cs);
    if (lo_r > hi_r || m0 < 1) return false;
    typedef __int128 i128;
    const i128 S = (i128)1 << (32 + sh);
    struct Con { long long t; int k; };
    std::vector<Con> ge, le; /* ge: t * m + c >= k * S;  le: t * m + c <= k * S - 1 */
    for (int k = -127; k <= 127; k++) {
        if (k <= lo_r) ge.push_back({-tmax, k});      /* the reference is >= k on the whole range */
        else if (k > hi_r) le.push_back({tmax, k});   /* ... < k on the whole range */
        else {
            long long a = -tmax, b = tmax; /* ref(a) < k <= ref(b) */
            while (b - a > 1) {
                const long long mid = a + (b - a) / 2;
                if (ref_requant((int32_t)mid, cs) >= k) b = mid; else a = mid;
            }
            ge.push_back({b, k});
            le.push_back({b - 1, k});
        }
    }
    auto slack = [&](long long m, i128 *lo, i128 *hi) -> i128 {
        i128 l = -((i128)1 << 120), h = (i128)1 << 120;
        for (const Con &c : ge) l = std::max(l, (i128)c.k * S - (i128)c.t * m);
        for (const Con &c : le) h = std::min(h, (i128)c.k * S - 1 - (i128)c.t * m);
        if (lo) *lo = l;
        if (hi) *hi = h;
        return h - l;
    };
    long long a = std::max(1ll, m0 - (1ll << 20)), b = std::min(2147483647ll, m0 + (1ll << 20));
    while (b - a > 2) {
        const long long m1 = a + (b - a) / 3, m2 = b - (b - a) / 3;
        if (slack(m1, nullptr, nullptr) < slack(m2, nullptr, nullptr)) a = m1; else b = m2;
    }
    long long m = a;
    for (long long q = a + 1; q <= b; q++) if (slack(q, nullptr, nullptr) > slack(m, nullptr, nullptr)) m = q;
    i128 cl, ch;
    if (slack(m, &cl, &ch) < 0) return false;
    const i128 c = cl + (ch - cl) / 2;
    /* the sum t * m + c64 (c64 = bias * m + c, |t - bias| + |bias| <= 2 tmax) must stay inside int64 */
    const i128 cabs = c < 0 ? -c : c;
    if (cabs > ((i128)1 << 61) || (i128)2 * tmax * m + cabs >= ((i128)1 << 62)) return false;
    /* belt and braces: both sides evaluated around every step and at the range ends */
    auto g = [&](long long t) { i128 x = ((i128)t * m + c) >> (32 + sh); return (int)(x > 127 ? 127 : (x < -128 ? -128 : x)); };
    for (const Con &cn : ge) for (long long t = cn.t - 2; t <= cn.t + 2; t++)
        if (t >= -tmax && t <= tmax && g(t) != ref_requant((int32_t)t, cs)) return false;
    if (g(-tmax) != lo_r || g(tmax) != hi_r) return false;
    *m_out = (int)m; *s_out = sh; *c_out = (long long)c;
    return true;
}

/* requantisation variant of the epilogue (requant_pair / requant_int) for conv scale cs and bound = max |acc + bias| over all
 * output channels (acc_bound):
 *   3  the integer form reproduces the reference on |t| <= bound (int_requant_fit fills m / s / c);
 *   2  else, when |cs| < 512 and bound < 2^22 (the magic-number int -> float conversion is exact and |sc| < 2^31) and no t in range
 *      lands on a negative tie (halfup_requant_ok);
 *   1  else, under the same two limits;
 *   0  otherwise: huge, infinite or NaN scales, accumulators from 2^22 up (int32 wrap-around of acc + bias included). */
static int select_requant(float cs, long long bound, int *m, int *s, long long *c) {
    if (int_requant_fit(cs, std::max(1ll, bound), m, s, c)) return 3;
    if (!(fabsf(cs) < 512.0f) || bound >= (1ll << 22)) return 0; /* also rejects NaN */
    return halfup_requant_ok(cs, bound) ? 2 : 1;
}

/* kernel variants: requantisation x GATHER producer x word table x number of stored streams x output mode (0 NCHW planes,
 * 1 + side copy, 2 channel-innermost tensors) x TST (staged plane stores: only the space-to-depth stem, i.e. EPI 8, no
 * gather, output mode 0 / 1, at least one stream).  Without a table (plain conv, no byte-ReLU) there is one stream at most. */
template <int RQ, bool GATHER, int EPI, bool TST>
static TcKernel pick_kernel2(bool tab, int nst, int out) {
    if (out == 2) {
        if (GATHER || TST) return nullptr;
        if (!tab) return nst == 1 ? k_conv_tc<RQ, false, false, 1, 2, EPI> : nullptr;
        switch (nst) {
            case 1: return k_conv_tc<RQ, false, true, 1, 2, EPI>;
            case 2: return k_conv_tc<RQ, false, true, 2, 2, EPI>;
            case 3: return k_conv_tc<RQ, false, true, 3, 2, EPI>;
            default: return nullptr;
        }
    }
    if (TST && nst == 0) return nullptr;
    if (!tab) {
        switch (nst * 2 + out) {
            case 0: return k_conv_tc<RQ, GATHER, false, 0, 0, EPI, false>;
            case 1: return k_conv_tc<RQ, GATHER, false, 0, 1, EPI, false>;
            case 2: return k_conv_tc<RQ, GATHER, false, 1, 0, EPI, TST>;
            default: return k_conv_tc<RQ, GATHER, false, 1, 1, EPI, TST>;
        }
    }
    switch (nst * 2 + out) {
        case 0: return k_conv_tc<RQ, GATHER, true, 0, 0, EPI, false>;
        case 1: return k_conv_tc<RQ, GATHER, true, 0, 1, EPI, false>;
        case 2: return k_conv_tc<RQ, GATHER, true, 1, 0, EPI, TST>;
        case 3: return k_conv_tc<RQ, GATHER, true, 1, 1, EPI, TST>;
        case 4: return k_conv_tc<RQ, GATHER, true, 2, 0, EPI, TST>;
        case 5: return k_conv_tc<RQ, GATHER, true, 2, 1, EPI, TST>;
        case 6: return k_conv_tc<RQ, GATHER, true, 3, 0, EPI, TST>;
        default: return k_conv_tc<RQ, GATHER, true, 3, 1, EPI, TST>;
    }
}
/* gather mode always runs two CTAs per SM (N tile <= 256 columns of TMEM in total), i.e. 8 epilogue warps */
template <int RQ>
static TcKernel pick_kernel1(bool gather, bool tab, int nst, int out, int epi, bool tst) {
    if (gather) return pick_kernel2<RQ, true, 8, false>(tab, nst, out);
    if (tst) return epi == 8 ? pick_kernel2<RQ, false, 8, true>(tab, nst, out) : nullptr;
    if (epi == 16) return pick_kernel2<RQ, false, 16, false>(tab, nst, out);
    return pick_kernel2<RQ, false, 8, false>(tab, nst, out);
}
static TcKernel pick_kernel(int rq, bool gather, bool tab, int nst, int out, int epi, bool tst) {
    if (rq == 3) return pick_kernel1<3>(gather, tab, nst, out, epi, tst);
    if (rq == 2) return pick_kernel1<2>(gather, tab, nst, out, epi, tst);
    if (rq == 1) return pick_kernel1<1>(gather, tab, nst, out, epi, tst);
    return pick_kernel1<0>(gather, tab, nst, out, epi, tst);
}

bool tc_plan(const Op &o, const ArenaGeom &ag, uint8_t *scratch, size_t scratch_stride, uint8_t *linked, size_t linked_stride,
             const Op *consumer, TcPlan *plan) {
    TcGeom g = tc_geometry(o);
    if (!g.ok || !encode_tiled()) return false;
    if (o.in0 < (int64_t)ag.W || o.out < (int64_t)ag.W || o.w >= (int64_t)ag.W) return false;
    if (g.scratch_bytes > scratch_stride) return false;
    TcPlanImpl *t = new TcPlanImpl();
    TcParams &p = t->p;
    memset(&p, 0, sizeof p);
    const bool gather = g.prepass == 3, s2d = g.prepass == 4, rect = g.prepass == 6;
    const int nhwc_in = o.kind == OP_CONV_I8_NHWC ? 1 : 0;
    t->nhwc_in = nhwc_in;
    const int ci_eff = (gather || s2d) ? g.Kp : (g.kpad ? g.kpad : o.ic); /* K extent of one tap */
    p.Co = o.oc; p.Ho = o.oh; p.Wo = o.ow; p.Wp = g.Wp; p.mflat = o.oh * g.Wp; p.plane = o.oh * o.ow;
    const int co_pad = round_up(o.oc, 16);
    p.n_tile = tc_n_tile(o.oc);
    p.n_tiles = tc_n_tiles(o.oc);
    p.bk = tc_bk(ci_eff);
    p.ksteps_per_tap = ci_eff / p.bk;
    p.ntaps = g.ntaps;
    p.a_tile_bytes = (uint32_t)(TC_BM * p.bk);
    p.a_row_bytes = s2d ? 16 : p.bk;
    p.toep = s2d ? 1 : 0;
    p.b_stage_bytes = (uint32_t)round_up(p.n_tile * p.bk, 1024);
    /* Accumulators in TMEM: two CTAs per SM share the 512 columns when a double-buffered accumulator group fits into 256.
     * Narrow N tiles are processed in groups of several M tiles per pipeline step: the per-step cost of the single-thread
     * producer / MMA loops and of the barrier hand-overs (measured: ~0.7 us per step, whatever the tile holds) is then
     * paid once per group. */
    t->ctas_per_sm = 2 * p.n_tile > 256 ? 1 : 2;
    p.tmem_cols = t->ctas_per_sm == 1 ? 512 : 256;
    p.grp = 1;
    if (p.n_tiles == 1 && t->ctas_per_sm == 2) {
        while (p.grp < 4 && 2 * (p.grp * 2) * p.n_tile <= p.tmem_cols) p.grp *= 2; /* up to four M tiles per group */
    }
    p.acc_bufs = std::max(2, std::min(4, p.tmem_cols / (p.grp * p.n_tile)));
    p.a_stage_bytes = p.grp * p.a_tile_bytes;
    p.tx_bytes = p.a_stage_bytes + (uint32_t)(p.n_tile * p.bk);
    /* the op needs the word table when it has fused followers or a byte-ReLU (plain conv: the byte is r itself).  The table is
     * replicated per lane group in shared memory ([256][rep] words, lane l reads copy l % rep): rep = 32 makes the lookups
     * conflict free; 16 or 8 (two / four lanes per bank) when the stages, the halo region or the resident weights need the room */
    t->tab = o.fused_layers > 0 || o.post_relu;
    /* output streams: the values the op produces per element, in table-byte order (see build_lutw); the ones the
     * planner keeps are compacted to table bytes 0..nst-1 */
    int64_t stream_off[4] = {-1, -1, -1, -1};
    if (o.fused_layers > 0) {
        stream_off[0] = o.store_z ? o.out_z : -1; stream_off[1] = o.out_s; stream_off[2] = o.store_y ? o.out : -1;
    } else stream_off[0] = o.store_y ? o.out : -1;
    if (o.fwd_out >= 0 && o.fwd_stream >= 0 && o.fwd_stream <= 2) stream_off[3] = o.fwd_out;
    t->nst = 0;
    for (int k = 0; k < 4; k++) t->stream_byte[k] = -1;
    for (int k = 0; k < 3; k++) p.out_off[k] = 0;
    for (int k = 0; k < 4; k++)
        if (stream_off[k] >= 0) {
            if (t->nst == 3) { delete t; return false; } /* the planner forwards only when a table byte is free */
            t->stream_byte[k] = t->nst; p.out_off[t->nst++] = stream_off[k] - (int64_t)ag.W;
        }
    if (t->nst > 1) t->tab = true; /* a plain conv with a forwarded second copy: the bytes of the streams come from the (identity) table */
    /* TST (the NCHW space-to-depth stem, see store_pitch): the NCHW streams leave through a shared-memory staging block, copied out
     * by the threads in 16-byte pieces of one row, instead of one byte per lane and channel.  Needs rows and pitch in whole 16-pixel
     * pieces and 16-byte aligned stream bases */
    t->tst = s2d && !nhwc_in && t->nst >= 1 && o.ow % 16 == 0 && g.Wp % 16 == 0;
    for (int k = 0; k < t->nst; k++) if (p.out_off[k] % 16) t->tst = false;
    const int epi_warps = (!gather && t->ctas_per_sm == 1) ? 16 : 8;
    const int stg_bytes = t->tst ? (epi_warps / 4) * 2 * t->nst * 2048 : 0;
    t->rq = select_requant(o.f0, acc_bound(o, ag), &p.q_m, &p.q_s, &p.q_c);
    const int cm64_bytes = t->rq == 3 ? 8 * p.n_tiles * p.n_tile : 0; /* RQ 3: per-channel int64 addends behind the table */
    const int nsteps = g.ntaps * p.ksteps_per_tap;
    int grp0 = p.grp, acc0 = p.acc_bufs;
    uint32_t a_stage0 = p.a_stage_bytes;
    bool plan_ok = true, over = false; /* over: even the two-stage minimum does not fit the budget (a second CTA would not be resident) */
    /* dynamic shared memory of a CTA: stages + weights + table (+ 1 KiB alignment slack); 227 KiB per SM, ~7 KiB static */
    auto plan_smem = [&](int tab_bytes) {
        const int budget = (t->ctas_per_sm == 1 ? 200 * 1024 : 104 * 1024) - tab_bytes;
        p.grp = grp0; p.acc_bufs = acc0; p.a_stage_bytes = a_stage0; p.halo = 0; p.halo_wide = 0; p.b_resident = 0; plan_ok = true;
        if (gather) { /* + 3 x 4 KiB patch ring + 8 KiB patch-word tables */
            if (p.grp > 2) { p.grp = 2; p.a_stage_bytes = p.grp * p.a_tile_bytes; p.acc_bufs = std::max(2, std::min(4, p.tmem_cols / (p.grp * p.n_tile))); }
            p.stages = std::max(2, std::min(8, (budget - (int)p.b_stage_bytes - 20480 - 1024) / (int)p.a_stage_bytes));
            t->smem = 1024 + (size_t)p.stages * p.a_stage_bytes + p.b_stage_bytes + 20480;
        } else {
            /* small weight matrices stay resident in shared memory for the whole (persistent) launch: one TMA per k-step */
            const size_t b_all = (size_t)nsteps * p.b_stage_bytes;
            p.b_resident = (p.n_tiles == 1 && b_all <= (size_t)budget / 2) ? 1 : 0;
            /* kxk stride 1 over the padded channel-innermost copy: every tap is a row shift of the same pixel rows, so one
             * load of the tile's rows plus its halo (128 + (kh-1)*Wp + kw-1 rows) serves all taps of a k block */
            if (s2d && !p.b_resident) { plan_ok = false; return; }
            if ((g.prepass == 1 && p.b_resident && g.ntaps > 1) || s2d) {
                /* s2d: the copy has a one-pixel zero border, so tap (ky2, pair) of output pixel q = oh*Wp + ow starts at row
                 * q + (ky2 + 1 - pt/2)*Wp + (2*pair + 1 - pl/2) and reads two pixels; taps that leave the image hit the border, the
                 * next row's border column, or rows beyond the copy (zero-filled by TMA) */
                const int s2d_min = (1 - o.pt / 2) * g.Wp + (1 - o.pl / 2);
                const int smin = s2d ? s2d_min : -o.pt * g.Wp, smax = s2d ? s2d_min + 2 * g.Wp + 3 : (o.kh - 1 - o.pt) * g.Wp + o.kw - 1;
                if (s2d && g.npix % 16 == 0 && (p.grp * TC_BM) % 16 == 0) {
                    /* the region starts on a 16-pixel boundary and travels as 256-byte rows: same shared-memory image, 1/16 of the rows */
                    const int smin_al = (smin >= 0 ? smin / 16 : -((-smin + 15) / 16)) * 16;
                    const int R16 = (p.grp * TC_BM + smax - smin_al + 15) / 16;
                    const int nb = (R16 + 255) / 256, rb = (R16 + nb - 1) / nb;
                    const uint32_t bytes = (uint32_t)round_up(nb * rb * 256, 1024);
                    if ((size_t)2 * bytes + b_all <= (size_t)budget) {
                        p.halo = 1; p.halo_min = smin_al; p.halo_rb = rb; p.halo_nb = nb; p.halo_wide = 1;
                        p.a_stage_bytes = bytes;
                    }
                }
                const int R = p.grp * TC_BM + smax - smin;
                const int nb = (R + 255) / 256, rb = round_up((R + nb - 1) / nb, 8);
                const uint32_t bytes = (uint32_t)round_up(nb * rb * p.a_row_bytes, 1024);
                if (!p.halo && rb <= 256 && (size_t)2 * bytes + b_all <= (size_t)budget) {
                    p.halo = 1; p.halo_min = smin; p.halo_rb = rb; p.halo_nb = nb;
                    p.a_stage_bytes = bytes;
                }
            }
            if (s2d && !p.halo) { plan_ok = false; return; }
            if (p.b_resident) {
                p.stages = std::max(2, std::min(8, (budget - (int)b_all) / (int)p.a_stage_bytes));
                t->smem = 1024 + (size_t)p.stages * p.a_stage_bytes + b_all;
            } else {
                const int stage_bytes = (int)(p.a_stage_bytes + p.b_stage_bytes);
                p.stages = std::max(2, std::min(8, budget / stage_bytes));
                t->smem = 1024 + (size_t)p.stages * stage_bytes;
            }
        }
        over = (long long)t->smem - 1024 > (long long)budget;
    };
    int rep = t->tab ? 8 : 0;
    plan_smem(rep * 1024 + cm64_bytes + stg_bytes);
    while (plan_ok && over && grp0 > 1 && !gather) { /* fewer M tiles per pipeline step rather than one CTA per SM */
        grp0 /= 2; a_stage0 = grp0 * p.a_tile_bytes; acc0 = std::max(2, std::min(4, p.tmem_cols / (grp0 * p.n_tile)));
        plan_smem(rep * 1024 + cm64_bytes + stg_bytes);
    }
    if (!plan_ok) { delete t; return false; }
    if (t->tab) { /* widen the replication while the pipeline keeps its shape (resident weights, halo loads, >= 3 stages) */
        const int res8 = p.b_resident, halo8 = p.halo, st8 = p.stages, grp8 = p.grp;
        for (int r2 = 32; r2 > 8; r2 >>= 1) {
            plan_smem(r2 * 1024 + cm64_bytes + stg_bytes);
            if (plan_ok && !over && p.b_resident == res8 && p.halo == halo8 && p.grp == grp8 && p.stages >= std::min(st8, 3)) { rep = r2; break; }
        }
        if (rep == 8) plan_smem(8 * 1024 + cm64_bytes + stg_bytes);
        p.tab_rep = (uint32_t)rep;
        p.tab_off = (uint32_t)round_up((int)(t->smem - 1024), 128); /* the table copies sit behind everything else */
        t->smem = 1024 + (size_t)p.tab_off + (size_t)rep * 1024;
    }
    if (cm64_bytes) {
        p.cm_off = (uint32_t)round_up((int)(t->smem - 1024), 128);
        t->smem = 1024 + (size_t)p.cm_off + (size_t)cm64_bytes;
    }
    if (stg_bytes) {
        p.stg_off = (uint32_t)round_up((int)(t->smem - 1024), 128);
        t->smem = 1024 + (size_t)p.stg_off + (size_t)stg_bytes;
    }
    /* keep residency at ctas_per_sm: a further CTA would fit the registers but stall in tcgen05.alloc */
    t->smem = std::max<size_t>(t->smem, t->ctas_per_sm == 1 ? 120 * 1024 : 80 * 1024);
    /* cute/arch/mma_sm100_desc.hpp InstrDescriptor: c=S32, a=b=signed 8 bit, A MN-major, B K-major, N>>3, M>>4 */
    p.idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.n_tile >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
    p.b_layout = tc_umma_layout(p.bk);
    p.a_kmajor = g.prepass != 0;
    if (!p.a_kmajor) p.idesc |= 1u << 15; /* A MN-major */
    if (s2d) for (int t6 = 0; t6 < 6; t6++) p.a_shift[t6] = ((t6 >> 1) + 1 - o.pt / 2) * g.Wp + 2 * (t6 & 1) + 1 - o.pl / 2;
    for (int kh = 0; kh < ((gather || s2d) ? (s2d ? 0 : 1) : o.kh); kh++)
        for (int kw = 0; kw < (gather ? 1 : o.kw); kw++) {
            const int tap = kh * o.kw + kw;
            if (g.prepass == 0 || g.prepass == 5 || gather) p.a_shift[tap] = 0;
            else if (rect) p.a_shift[tap] = (kh << 16) | kw;
            else p.a_shift[tap] = g.copy.tap_shift(kh, kw);
        }
    p.bias = o.bias >= 0 ? reinterpret_cast<const int32_t *>(ag.d_weights + o.bias) : nullptr;
    if (o.bias >= 0 && (o.bias % 4 || o.bias + 4 * (int64_t)o.oc > (int64_t)ag.W)) { delete t; return false; }
    p.cs = o.f0;
    p.slot_stride = ag.slot_stride;
    p.m_tiles = (p.mflat + TC_BM - 1) / TC_BM;
    p.m_groups = (p.m_tiles + p.grp - 1) / p.grp;
    p.wp_magic = (unsigned)((1ull << 32) / (unsigned)g.Wp) + 1u;
    /* (+ 2 rows: the s2d pre-pass divides pixel indices of the bordered image by Wp with the same multiply-high trick) */
    if ((unsigned long long)(p.mflat + 2 * g.Wp) * (unsigned)g.Wp >= (1ull << 32) || (long long)p.m_tiles * p.n_tiles * ag.capacity >= (1ll << 31)) { delete t; return false; }
    p.a_tx_bytes = p.a_stage_bytes;
    if (rect) {
        p.rect = 1; p.tw = g.rtw; p.th = g.rth; p.rs = o.sh; p.rpt = o.pt; p.rpl = o.pl;
        p.tw_magic = (unsigned)((1ull << 32) / (unsigned)g.rtw) + 1u;
        p.tiles_x = (o.ow + g.rtw - 1) / g.rtw;
        p.m_tiles = p.tiles_x * ((o.oh + g.rth - 1) / g.rth);
        p.m_groups = (p.m_tiles + p.grp - 1) / p.grp;
        p.a_tx_bytes = (uint32_t)(p.grp * p.bk * g.rtw * g.rth);
    }
    if (nhwc_in) p.onhwc_vec = (o.oc % 16 == 0) ? 1 : 0;
    if (gather) {
        const int tw = 1 << g.tw_shift, th = TC_BM >> g.tw_shift;
        p.tw_shift = g.tw_shift;
        p.tiles_x = (o.ow + tw - 1) / tw;
        p.m_tiles = p.tiles_x * ((o.oh + th - 1) / th);
        p.m_groups = (p.m_tiles + p.grp - 1) / p.grp;
        p.gPH = g.PH; p.gPWW = g.PWW; p.gdx = g.dx;
        p.g_align2 = (o.sh % 2 == 0 && o.kw % 2 == 0 && g.dx % 2 == 0) ? 1 : 0;
    }
    p.dbg = getenv("MARS_TC_DEBUG") ? atoi(getenv("MARS_TC_DEBUG")) : 0; /* read by the kernels only in a -DMARS_TC_TUNING build */
    p.nhwc_sel = -1;
    if (consumer && linked) { /* this op's epilogue also writes the consumer's channel-innermost input copy */
        const TcGeom cg = tc_geometry(*consumer);
        const int sidx = o.fused_layers > 0 ? o.nhwc_stream : 0; /* stream index in {Z,S,Y} order; a plain conv only has Y = 0 */
        if (!cg.ok || !cg.copy.mode || sidx < 0 || sidx > 2 || consumer->ic != o.oc) { delete t; return false; }
        t->nhwc_stream = sidx; /* its value goes into the top byte of every table word */
        p.nhwc_sel = 3;
        p.nhwc_mode = cg.copy.mode; p.nhwc_Wp = cg.copy.Wp; p.nhwc_plane = cg.copy.plane; p.nhwc_pt = cg.copy.pt; p.nhwc_pl = cg.copy.pl;
        p.nhwc_C = consumer->ic;
        p.nhwc_base = linked + consumer->copy_off;
        p.nhwc_stride = linked_stride;
        /* the side output leaves in 32-byte pieces (two 16-channel units of a pixel per store) */
        if (consumer->ic % 32 || p.n_tile % 32 || consumer->copy_off % 32 || linked_stride % 32 || ((uintptr_t)linked % 32)) { delete t; return false; }
    }
    t->prepass = g.prepass; t->C = o.ic; t->Cp = ci_eff; t->H = o.ih; t->W = o.iw; t->npix = g.npix; t->copy = g.copy;
    t->src_slot0 = ag.d_slots + (o.in0 - (int64_t)ag.W);
    t->scratch = scratch; t->scratch_stride = scratch_stride; t->slot_stride = ag.slot_stride;
    if (gather) {
        /* the private input copy is only needed when a stored output stream overwrites the input tensor (round-robin work
         * buffers, SURVEY C.2) while other tiles still have to read it */
        const int64_t in_lo = o.in0 - (int64_t)ag.W, in_hi = in_lo + (int64_t)o.ic * o.ih * o.iw;
        t->gather_direct = true;
        for (int k = 0; k < t->nst; k++)
            if (p.out_off[k] < in_hi && in_lo < p.out_off[k] + (int64_t)o.oc * o.oh * o.ow) t->gather_direct = false;
        p.g_src = scratch; p.g_stride = scratch_stride;
        p.gC = o.ic; p.gH = o.ih; p.gW = o.iw; p.gS = o.sh; p.gpt = o.pt; p.gpl = o.pl; p.gKH = o.kh; p.gKW = o.kw;
        p.gKt = o.ic * o.kh * o.kw;
    }

    if (rect || g.prepass == 5) {
        /* read the arena tensor itself unless a stored stream overwrites it while other tiles still need it (round-robin work
         * buffers, SURVEY C.2).  A 1x1 layer with Ci == Co and one N tile may write onto its own input: every CTA has read the
         * pixels it overwrites (same bytes) before its epilogue starts. */
        const int64_t in_lo = o.in0 - (int64_t)ag.W, in_hi = in_lo + (int64_t)o.ic * o.ih * o.iw;
        t->gather_direct = true;
        for (int k = 0; k < t->nst; k++) {
            if (!(p.out_off[k] < in_hi && in_lo < p.out_off[k] + (int64_t)o.oc * o.oh * o.ow)) continue;
            const bool own_pixels = g.prepass == 5 && p.out_off[k] == in_lo && o.ic == o.oc && p.n_tiles == 1;
            if (!own_pixels) t->gather_direct = false;
        }
    }
    if (nhwc_in && t->nst == 0) { delete t; return false; } /* nothing to store: not a case the planner produces */

    /* weights: [tap][co_pad][Ci] K-major, and the epilogue table */
    const size_t wr_bytes = (size_t)g.ntaps * co_pad * ci_eff;
    uint32_t lutw[256];
    build_lutw(o, ag.h_cpool, t->stream_byte, t->nhwc_stream, lutw);
    if (cudaMalloc(&t->d_wr, wr_bytes) != cudaSuccess || cudaMalloc(&t->d_lutw, sizeof lutw) != cudaSuccess) {
        cudaFree(t->d_wr); delete t; return false;
    }
    cudaMemcpy(t->d_lutw, lutw, sizeof lutw, cudaMemcpyHostToDevice);
    p.lutw = t->d_lutw;
    if (s2d)
        k_repack_s2d<<<64, 256>>>(reinterpret_cast<const int8_t *>(ag.d_weights + o.w), t->d_wr, o.oc, co_pad, o.ic, nhwc_in);
    else if (gather)
        k_repack_rows<<<256, 256>>>(reinterpret_cast<const int8_t *>(ag.d_weights + o.w), t->d_wr, o.oc, co_pad, o.ic * o.kh * o.kw, g.Kp);
    else
        k_repack_weights<<<256, 256>>>(reinterpret_cast<const int8_t *>(ag.d_weights + o.w), t->d_wr, o.oc, co_pad, o.ic, ci_eff, g.ntaps, nhwc_in);
    bool ok = cudaDeviceSynchronize() == cudaSuccess;

    const CUtensorMapSwizzle ksw = tc_swizzle(p.bk);
    if (ok && g.prepass == 0) /* the NCHW planes in the arena */
        ok = make_map3(&t->mapA, (void *)t->src_slot0, (uint64_t)o.ih * o.iw, (uint64_t)o.ic, (uint64_t)ag.capacity,
                       (uint64_t)o.ih * o.iw, ag.slot_stride, TC_BM, (uint32_t)p.bk, CU_TENSOR_MAP_SWIZZLE_128B);
    else if (ok && s2d) /* 16-byte pixels, linear rows (no swizzle): the MMA reads them as overlapping 32-byte K rows */
        ok = p.halo_wide ? make_map3(&t->mapA, scratch, 256, (uint64_t)g.npix / 16, (uint64_t)ag.capacity, 256, scratch_stride, 256, (uint32_t)p.halo_rb,
                                     CU_TENSOR_MAP_SWIZZLE_NONE)
                         : make_map3(&t->mapA, scratch, 16, (uint64_t)g.npix, (uint64_t)ag.capacity, 16, scratch_stride, 16, (uint32_t)p.halo_rb,
                                     CU_TENSOR_MAP_SWIZZLE_NONE);
    else if (ok && g.prepass == 5) /* the arena tensor's pixels are the K rows: dims (C, pixels, images), K-major box {bk, 128} */
        ok = make_map3(&t->mapA, t->gather_direct ? (void *)t->src_slot0 : (void *)scratch, (uint64_t)o.ic, (uint64_t)o.ih * o.iw, (uint64_t)ag.capacity,
                       (uint64_t)o.ic, t->gather_direct ? ag.slot_stride : scratch_stride, (uint32_t)p.bk, TC_BM, ksw);
    else if (ok && rect)
        ok = make_map4(&t->mapA, t->gather_direct ? (void *)t->src_slot0 : (void *)scratch, (uint64_t)o.ic, (uint64_t)o.iw, (uint64_t)o.ih,
                       (uint64_t)ag.capacity, t->gather_direct ? ag.slot_stride : scratch_stride, (uint32_t)p.bk, (uint32_t)(g.rtw * o.sh),
                       (uint32_t)(g.rth * o.sh), (uint32_t)o.sh, ksw);
    else if (ok && !gather) /* NHWC copy: dims (C, pixels, images), K-major box {bk, 128} */
        ok = make_map3(&t->mapA, scratch, (uint64_t)ci_eff, (uint64_t)g.npix, (uint64_t)ag.capacity, (uint64_t)ci_eff,
                       scratch_stride, (uint32_t)p.bk, p.halo ? (uint32_t)p.halo_rb : TC_BM, ksw);
    else if (ok) t->mapA = CUtensorMap(); /* unused in gather mode */
    if (ok && o.copy_from >= 0 && linked && !gather && g.prepass != 0) {
        ok = make_map3(&t->mapA_linked, linked + o.copy_off, (uint64_t)ci_eff, (uint64_t)g.npix, (uint64_t)ag.capacity, (uint64_t)ci_eff,
                       linked_stride, (uint32_t)p.bk, p.halo ? (uint32_t)p.halo_rb : TC_BM, ksw);
        t->has_linked = ok;
    }
    ok = ok && make_map3(&t->mapB, t->d_wr, (uint64_t)ci_eff, (uint64_t)co_pad, (uint64_t)g.ntaps, (uint64_t)ci_eff,
                         (uint64_t)co_pad * ci_eff, (uint32_t)p.bk, (uint32_t)p.n_tile, ksw);
    t->sms = tc_sm_count();
    t->epi = epi_warps;
    t->kernel = pick_kernel(t->rq, gather, t->tab, t->nst, nhwc_in ? 2 : (p.nhwc_sel >= 0 ? 1 : 0), t->epi, t->tst);
    ok = ok && t->kernel != nullptr;
    ok = ok && cudaFuncSetAttribute((const void *)t->kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 210 * 1024) == cudaSuccess;
    if (!ok) { cudaFree(t->d_wr); cudaFree(t->d_lutw); delete t; return false; }
    if (getenv("MARS_TC_VERBOSE"))
        fprintf(stderr, "tc_plan layer %d: %dx%d k%d s%d ci %d co %d | n_tile %d grp %d acc %d stages %d bk %d halo %d b_res %d ctas %d epi %d | rq %d tab %d rep %u nst %d side %d tst %d smem %zu\n",
                o.layer, o.oh, o.ow, o.kh, o.sh, o.ic, o.oc, p.n_tile, p.grp, p.acc_bufs, p.stages, p.bk, p.halo, p.b_resident, t->ctas_per_sm, t->epi,
                t->rq, (int)t->tab, p.tab_rep, t->nst, p.nhwc_sel >= 0, (int)t->tst, t->smem);
    plan->i8 = t;
    return true;
}

bool tc_launch(const TcPlan &plan, uint8_t *slots_base, int first, int n, bool use_linked, cudaStream_t s, uint64_t *launches) {
    TcPlanImpl *t = plan.i8;
    if (!t) return false;
    const uint8_t *src = t->src_slot0 + (size_t)first * t->slot_stride;
    uint8_t *scr = t->scratch + (size_t)first * t->scratch_stride;
    if (t->prepass == 3 && !t->gather_direct) {
        /* private copy of the input tensor: the fused outputs may overwrite the input's work buffer (SURVEY C.2) */
        if (cudaMemcpy2DAsync(scr, t->scratch_stride, src, t->slot_stride, (size_t)t->C * t->H * t->W, (size_t)n,
                              cudaMemcpyDeviceToDevice, s) != cudaSuccess) return false;
    } else if (t->prepass == 4) {
        k_s2d16<<<dim3((t->npix + 1023) / 1024, n), 256, 0, s>>>(src, (unsigned long long)t->slot_stride, scr, (unsigned long long)t->scratch_stride, t->C, t->H, t->W, t->p.Wp, t->npix, t->nhwc_in);
        (*launches)++;
    } else if (t->prepass == 6 || t->prepass == 5) {
        if (!t->gather_direct && cudaMemcpy2DAsync(scr, t->scratch_stride, src, t->slot_stride, (size_t)t->C * t->H * t->W, (size_t)n,
                                                  cudaMemcpyDeviceToDevice, s) != cudaSuccess) return false;
    } else if (t->prepass && t->prepass != 3 && !(use_linked && t->has_linked)) {
        dim3 g((t->npix + 31) / 32, (t->Cp + 31) / 32, n);
        k_to_nhwc<<<g, 256, 0, s>>>(src, (unsigned long long)t->slot_stride, scr, (unsigned long long)t->scratch_stride, t->C, t->Cp, t->H, t->W,
                                    t->copy.Wp, t->copy.plane, t->npix, (int)(t->copy.mode == 2), t->copy.pt, t->copy.pl);
        (*launches)++;
    }
    TcParams p = t->p;
    p.out_base = slots_base + (size_t)first * t->slot_stride;
    p.img0 = first;
    p.n_img = n;
    if (t->prepass == 3) {
        if (t->gather_direct) { p.g_src = src; p.g_stride = t->slot_stride; }
        else p.g_src = scr;
    }
    if (p.nhwc_sel >= 0) p.nhwc_base += (size_t)first * p.nhwc_stride;
    const long long total_tiles = (long long)p.m_groups * p.n_tiles * n;
    const unsigned grid = (unsigned)std::min<long long>(total_tiles, (long long)t->sms * t->ctas_per_sm);
    t->kernel<<<grid, (t->epi + (t->prepass == 3 ? 5 : 2)) * 32, t->smem, s>>>((use_linked && t->has_linked) ? t->mapA_linked : t->mapA, t->mapB, p);
    (*launches)++;
    return cudaGetLastError() == cudaSuccess;
}

int tc_rq(const TcPlan &plan) { return plan.i8 ? plan.i8->rq : -1; }

void tc_release(std::vector<TcPlan> &plans) {
    for (auto &pl : plans) {
        if (TcPlanImpl *t = pl.i8) { cudaFree(t->d_wr); cudaFree(t->d_lutw); delete t; }
        tf32_release(pl.f32);
    }
    plans.clear();
}

} // namespace marsb200

extern "C" {
int mars_b200_requant_fit(float scale, long long tmax, int *m, int *s, long long *c) {
    int mm = 0, ss = 0; long long cc = 0;
    if (!marsb200::int_requant_fit(scale, tmax, &mm, &ss, &cc)) return 0;
    if (m) *m = mm;
    if (s) *s = ss;
    if (c) *c = cc;
    return 1;
}
int mars_b200_requant_ref(int t, float scale) { return marsb200::ref_requant((int32_t)t, scale); }
int mars_b200_requant_variant(float scale, long long bound) {
    int m = 0, s = 0; long long c = 0;
    return marsb200::select_requant(scale, bound, &m, &s, &c);
}
}
