/*
 * tools/epi_bench.cu -- instruction-throughput microbenchmark of candidate conv epilogues (sm_100a).
 *
 * Measures, per variant, how many output elements per clock one SM sustains when 16 warps run the per-element
 * sequence of the int8 conv epilogue (reference arithmetic: src/mars/mxu_conv.c:663-666) on accumulators read from
 * shared memory (16 bytes per lane per load, standing in for tcgen05.ld):
 *   old    : round-1 sequence -- magic int->float, |sc|+0.5, min, RZ add, sign merge, 512-entry sign/magnitude word table
 *            (bank conflicts), one STG.U8 per element into an NCHW plane
 *   new    : packed FADD2/FMUL2, copysign + FADD + F2I.S8, lane-replicated 256-entry word table (conflict free),
 *            STS.U8 into a [channel][pixel] staging block, 16-byte copy-out per 16 pixels
 *   new_sh : `new` with a plain (not replicated) 256-entry table
 *   new_nt : `new` without the table (plain conv: the byte is the clamped value itself)
 *   new_c  : `new` + the channel-innermost side output (3 PRMT per 4 elements, one 16-byte store per 16 channels)
 * build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 --fmad=false -o /tmp/epi_bench tools/epi_bench.cu
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "../thingino-accel_b200/csrc/tc_common.cuh"

using namespace marsb200;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(1); } } while (0)

__device__ __forceinline__ uint32_t old_index(int32_t t, float cs) {
    const float f = __fsub_rn(__int_as_float(t), 12582912.0f);
    const float sc = __fmul_rn(f, cs);
    const float m = fminf(__fadd_rn(fabsf(sc), 0.5f), 128.0f);
    const float u = __fadd_rz(m, 8388608.0f);
    return (__float_as_uint(u) - 0x4B000000u) | ((__float_as_uint(sc) >> 23) & 0x100u);
}
/* two accumulators (bias and the int->float magic already added) -> two clamped int8 values, sign extended */
__device__ __forceinline__ void new_pair(int32_t t0, int32_t t1, float cs, int &r0, int &r1) {
    unsigned long long p, q, c2;
    asm("mov.b64 %0, {%1, %2};" : "=l"(p) : "r"(t0), "r"(t1));
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(q) : "l"(p), "l"(0xCB400000CB400000ull));
    asm("mov.b64 %0, {%1, %1};" : "=l"(c2) : "f"(cs));
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(p) : "l"(q), "l"(c2));
    float s0, s1;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(s0), "=f"(s1) : "l"(p));
    const float h0 = __fadd_rn(s0, copysignf(0.5f, s0)), h1 = __fadd_rn(s1, copysignf(0.5f, s1));
    asm("cvt.rzi.s8.f32 %0, %1;" : "=r"(r0) : "f"(h0));
    asm("cvt.rzi.s8.f32 %0, %1;" : "=r"(r1) : "f"(h1));
}

/* round-half-up variant: floor(fl(sc + 0.5)); equals the reference's trunc(fl(sc +- 0.5)) unless a reachable sc is a negative
 * exact tie or one of a few special floats -- the host checks that per layer */
__device__ __forceinline__ void halfup_pair(int32_t t0, int32_t t1, float cs, int &r0, int &r1) {
    unsigned long long p, q, c2;
    asm("mov.b64 %0, {%1, %2};" : "=l"(p) : "r"(t0), "r"(t1));
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(q) : "l"(p), "l"(0xCB400000CB400000ull));
    asm("mov.b64 %0, {%1, %1};" : "=l"(c2) : "f"(cs));
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(p) : "l"(q), "l"(c2));
    float s0, s1; /* scalar adds: ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 (one rounding), which is not the reference */
    asm("mov.b64 {%0, %1}, %2;" : "=f"(s0), "=f"(s1) : "l"(p));
    const float h0 = __fadd_rn(s0, 0.5f), h1 = __fadd_rn(s1, 0.5f);
    asm("cvt.rmi.s8.f32 %0, %1;" : "=r"(r0) : "f"(h0));
    asm("cvt.rmi.s8.f32 %0, %1;" : "=r"(r1) : "f"(h1));
}

/* conversion-free round-half-up: floor via a round-down add of 1.5 * 2^23, clamp on the integer pattern */
__device__ __forceinline__ void halfup_nocvt_pair(int32_t t0, int32_t t1, float cs, int &r0, int &r1) {
    unsigned long long p, q, c2;
    asm("mov.b64 %0, {%1, %2};" : "=l"(p) : "r"(t0), "r"(t1));
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(q) : "l"(p), "l"(0xCB400000CB400000ull));
    asm("mov.b64 %0, {%1, %1};" : "=l"(c2) : "f"(cs));
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(p) : "l"(q), "l"(c2));
    float s0, s1;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(s0), "=f"(s1) : "l"(p));
    const float h0 = __fadd_rn(s0, 0.5f), h1 = __fadd_rn(s1, 0.5f);
    const int i0 = __float_as_int(__fadd_rd(h0, 12582912.0f)), i1 = __float_as_int(__fadd_rd(h1, 12582912.0f));
    r0 = min(max(i0, 0x4B400000 - 128), 0x4B400000 + 127) - 0x4B400000;
    r1 = min(max(i1, 0x4B400000 - 128), 0x4B400000 + 127) - 0x4B400000;
}

constexpr int WARPS = 16, UNITS = 8; /* 16 warps x 32 lanes, 8 units of 16 channels per "tile" (128 channels) */

/* MATH: 0 = round-1 sequence (sign/magnitude index), 1 = packed + F2I.S8, 2 = scalar FADD/FMUL + F2I.S8
 * TAB : 0 = none, 1 = lane-replicated 256 words, 2 = plain 256 words, 3 = round-1 512-word sign/magnitude table
 * ST  : 0 = none (xor into a register), 1 = STG.U8 per element into NCHW planes, 2 = STS.U8 staging + 16-byte copy-out
 * SIDE: channel-innermost side output (PRMT packing + one 16-byte store per 16 channels) */
template <int MATH, int TAB, int ST, int SIDE>
__global__ void __launch_bounds__(WARPS * 32, 1) k_epi(const int32_t *acc_src, const uint32_t *lut512, const uint32_t *lut256, uint8_t *out,
                                                        uint8_t *side, float cs, int iters, long long plane, unsigned long long *cycles) {
    extern __shared__ __align__(16) uint8_t sm[];
    uint32_t *s_tab = reinterpret_cast<uint32_t *>(sm);               /* 32 KB: [256][32] replicated, or the plain tables */
    int32_t *s_cm = reinterpret_cast<int32_t *>(sm + 32768);          /* 512 B */
    uint8_t *s_stage = sm + 32768 + 1024;                             /* 2 x 128 ch x 144 B */
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (TAB == 3) { for (int i = threadIdx.x; i < 512; i += blockDim.x) s_tab[i] = lut512[i]; }
    else if (TAB == 2) { for (int i = threadIdx.x; i < 256; i += blockDim.x) s_tab[i] = lut256[i]; }
    else { for (int i = threadIdx.x; i < 8192; i += blockDim.x) s_tab[i] = lut256[i >> 5]; }
    for (int i = threadIdx.x; i < 128; i += blockDim.x) s_cm[i] = 0x4B400000 + (i * 37 % 200) - 100;
    __syncthreads();
    const int quad = warp & 3, part = warp >> 2; /* 4 parts x 4 quadrants */
    const int r = quad * 32 + lane;
    const uint32_t sa_cm = smem_u32(s_cm), sa_tab = smem_u32(s_tab);
    const uint32_t tab_lane = sa_tab + 128u * 128u + 4u * lane; /* entry r = 0 of this lane's table copy */
    const uint32_t tab_plain = sa_tab + 4u * 128u;
    uint8_t *obase = out + (size_t)blockIdx.x * 128 * plane + r;
    uint8_t *sbase = side + ((size_t)blockIdx.x * 128 + r) * 128;
    int32_t vreg[16];
#pragma unroll
    for (int k = 0; k < 16; k++) vreg[k] = acc_src[(blockIdx.x * 8192 + threadIdx.x * 16 + k) & 0xFFFFF];
    uint32_t sink = 0;
    unsigned long long t0 = clock64();
    for (int it = 0; it < iters; it++) {
        uint8_t *stage = s_stage + (it & 1) * (128 * 144);
        for (int u = part; u < UNITS; u += 4) {
            const uint32_t cm = sa_cm + 64u * ((u + it) & 7);
            uint8_t *o = obase + (size_t)(u * 16) * plane + (size_t)(it & 7) * 128;
            uint8_t *st = ST == 3 ? s_stage + warp * 512 + lane : stage + (u * 16) * 144 + r;
            uint32_t pk[4];
#pragma unroll
            for (int j4 = 0; j4 < 4; j4++) {
                int4 c4;
                asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(c4.x), "=r"(c4.y), "=r"(c4.z), "=r"(c4.w) : "r"(cm + 16u * j4));
                const int cc[4] = {c4.x, c4.y, c4.z, c4.w};
                uint32_t w[4];
#pragma unroll
                for (int k = 0; k < 4; k += 2) {
                    const int32_t ta = vreg[4 * j4 + k] + cc[k], tb = vreg[4 * j4 + k + 1] + cc[k + 1];
                    int r0, r1;
                    if (MATH == 0) { r0 = (int)old_index(ta, cs); r1 = (int)old_index(tb, cs); }
                    else if (MATH == 1) new_pair(ta, tb, cs, r0, r1);
                    else if (MATH == 3) halfup_pair(ta, tb, cs, r0, r1);
                    else if (MATH == 4) halfup_nocvt_pair(ta, tb, cs, r0, r1);
                    else {
                        const float s0 = __fmul_rn(__fsub_rn(__int_as_float(ta), 12582912.0f), cs), s1 = __fmul_rn(__fsub_rn(__int_as_float(tb), 12582912.0f), cs);
                        const float h0 = __fadd_rn(s0, copysignf(0.5f, s0)), h1 = __fadd_rn(s1, copysignf(0.5f, s1));
                        asm("cvt.rzi.s8.f32 %0, %1;" : "=r"(r0) : "f"(h0));
                        asm("cvt.rzi.s8.f32 %0, %1;" : "=r"(r1) : "f"(h1));
                    }
                    if (TAB == 0) { w[k] = (uint32_t)r0; w[k + 1] = (uint32_t)r1; }
                    else {
                        uint32_t a0 = TAB == 3 ? sa_tab + 4u * r0 : (TAB == 2 ? tab_plain + 4u * r0 : tab_lane + 128u * r0);
                        uint32_t a1 = TAB == 3 ? sa_tab + 4u * r1 : (TAB == 2 ? tab_plain + 4u * r1 : tab_lane + 128u * r1);
                        if (TAB == 4) { asm("mad.lo.s32 %0, %1, 128, %2;" : "=r"(a0) : "r"(r0), "r"(tab_lane)); asm("mad.lo.s32 %0, %1, 128, %2;" : "=r"(a1) : "r"(r1), "r"(tab_lane)); }
                        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w[k]) : "r"(a0));
                        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w[k + 1]) : "r"(a1));
                    }
                }
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    if (ST == 0) sink ^= w[k];
                    else if (ST == 1) { *o = (uint8_t)w[k]; o += plane; }
                    else if (ST == 4) o[(long long)(4 * j4 + k) * (int)plane] = (uint8_t)w[k];
                    else if (ST == 5) o[(4 * j4 + k) * 1024] = (uint8_t)w[k];
                    else if (ST == 2) st[(4 * j4 + k) * 144] = (uint8_t)w[k];
                    else st[(4 * j4 + k) * 32] = (uint8_t)w[k];
                }
                if (SIDE) {
                    const uint32_t p01 = __byte_perm(w[0], w[1], 0x0073), p23 = __byte_perm(w[2], w[3], 0x0073);
                    pk[j4] = __byte_perm(p01, p23, 0x5410);
                }
            }
            if (ST == 3) { /* per-warp staging: 16 channels x 32 pixels, lane -> (channel = lane / 2, half = lane % 2): 16 bytes each */
                __syncwarp();
                const uint4 d = *reinterpret_cast<const uint4 *>(s_stage + warp * 512 + lane * 16);
                *reinterpret_cast<uint4 *>(out + ((size_t)blockIdx.x * 128 + u * 16 + (lane >> 1)) * plane + (size_t)(it & 7) * 128 + quad * 32 + (lane & 1) * 16) = d;
                __syncwarp();
            }
            if (SIDE) *reinterpret_cast<uint4 *>(sbase + (size_t)(it & 7) * 16 + u * 16) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
        if (ST == 2) {
            asm volatile("bar.sync 1, %0;" ::"r"(WARPS * 32) : "memory");
            /* copy-out: 128 rows (channels) x 8 chunks of 16 pixels, 16 warps: warp w takes rows 8w .. 8w+7; 4 rows per pass */
            const int chunk = lane & 7;
#pragma unroll
            for (int p = 0; p < 2; p++) {
                const int row = warp * 8 + p * 4 + (lane >> 3);
                const uint4 d = *reinterpret_cast<const uint4 *>(stage + row * 144 + chunk * 16);
                *reinterpret_cast<uint4 *>(out + ((size_t)blockIdx.x * 128 + row) * plane + (size_t)(it & 7) * 128 + chunk * 16) = d;
            }
        }
#pragma unroll
        for (int k = 0; k < 16; k++) vreg[k] += 3; /* one more integer add per element than the real epilogue */
    }
    unsigned long long t1 = clock64();
    if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
    if (sink == 0x12345678u) out[0] = 1;
}

template <int MATH, int TAB, int ST, int SIDE>
static void run(const char *name, const int32_t *acc, const uint32_t *l512, const uint32_t *l256, uint8_t *out, uint8_t *side, unsigned long long *cyc, int sms) {
    const int iters = 2000;
    const size_t smem = 32768 + 1024 + 2 * 128 * 144;
    CK(cudaFuncSetAttribute(k_epi<MATH, TAB, ST, SIDE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long plane = 1024;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    k_epi<MATH, TAB, ST, SIDE><<<sms, WARPS * 32, smem>>>(acc, l512, l256, out, side, 0.0123f, 50, plane, cyc);
    CK(cudaDeviceSynchronize());
    cudaEventRecord(e0);
    k_epi<MATH, TAB, ST, SIDE><<<sms, WARPS * 32, smem>>>(acc, l512, l256, out, side, 0.0123f, iters, plane, cyc);
    cudaEventRecord(e1);
    CK(cudaDeviceSynchronize());
    float ms;
    cudaEventElapsedTime(&ms, e0, e1);
    unsigned long long h[256];
    CK(cudaMemcpy(h, cyc, sizeof(unsigned long long) * sms, cudaMemcpyDeviceToHost));
    double avg = 0;
    for (int i = 0; i < sms; i++) avg += (double)h[i];
    avg /= sms;
    const double elems = (double)iters * 128 * 128; /* per SM */
    printf("%-28s %8.3f ms %6.2f elements/clk/SM  %6.2f cycles per warp-element per SMSP  -> %6.2f ms per 26.4 G elements\n",
           name, ms, elems / avg, avg / (elems / 32 / 4), 26.4e9 / (elems * sms / (ms * 1e-3)) * 1e3);
}

int main() {
    int sms = 0;
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
    int32_t *acc; uint32_t *l512, *l256; uint8_t *out, *side; unsigned long long *cyc;
    CK(cudaMalloc(&acc, 4 << 20)); CK(cudaMalloc(&l512, 2048)); CK(cudaMalloc(&l256, 1024));
    CK(cudaMalloc(&out, (size_t)sms * 128 * 1024 + 4096)); CK(cudaMalloc(&side, (size_t)sms * 128 * 128 + 4096)); CK(cudaMalloc(&cyc, 8 * 256));
    int32_t *h = (int32_t *)malloc(4 << 20);
    srand(1);
    for (int i = 0; i < (1 << 20); i++) { /* accumulators whose requantised value is roughly N(0, 35) at cs = 0.0123 */
        double g = 0; for (int k = 0; k < 12; k++) g += rand() / (double)RAND_MAX; g -= 6.0;
        h[i] = (int32_t)(g * 35.0 / 0.0123);
    }
    CK(cudaMemcpy(acc, h, 4 << 20, cudaMemcpyHostToDevice));
    uint32_t t[512];
    for (int i = 0; i < 512; i++) t[i] = (uint32_t)(i * 2654435761u);
    CK(cudaMemcpy(l512, t, 2048, cudaMemcpyHostToDevice)); CK(cudaMemcpy(l256, t, 1024, cudaMemcpyHostToDevice));
    printf("SMs %d; 16 warps per SM; element = one int8 conv output (requant + table + store)\n", sms);
    run<0, 0, 0, 0>("old math only", acc, l512, l256, out, side, cyc, sms);
    run<1, 0, 0, 0>("packed+F2I math only", acc, l512, l256, out, side, cyc, sms);
    run<2, 0, 0, 0>("scalar+F2I math only", acc, l512, l256, out, side, cyc, sms);
    run<0, 3, 0, 0>("old math + table512", acc, l512, l256, out, side, cyc, sms);
    run<1, 1, 0, 0>("new math + replicated table", acc, l512, l256, out, side, cyc, sms);
    run<1, 2, 0, 0>("new math + plain table256", acc, l512, l256, out, side, cyc, sms);
    run<0, 3, 1, 0>("OLD: old+table512+STG.U8", acc, l512, l256, out, side, cyc, sms);
    run<1, 1, 1, 0>("new+repl table+STG.U8", acc, l512, l256, out, side, cyc, sms);
    run<1, 1, 2, 0>("NEW: new+repl table+staging", acc, l512, l256, out, side, cyc, sms);
    run<1, 0, 2, 0>("new, no table, staging", acc, l512, l256, out, side, cyc, sms);
    run<1, 1, 2, 1>("NEW + side output", acc, l512, l256, out, side, cyc, sms);
    run<0, 3, 1, 1>("OLD + side output", acc, l512, l256, out, side, cyc, sms);
    run<1, 1, 0, 1>("new, side output only", acc, l512, l256, out, side, cyc, sms);
    run<3, 0, 0, 0>("half-up packed math only", acc, l512, l256, out, side, cyc, sms);
    run<3, 1, 0, 0>("half-up + repl table (LEA)", acc, l512, l256, out, side, cyc, sms);
    run<3, 4, 0, 0>("half-up + repl table (IMAD)", acc, l512, l256, out, side, cyc, sms);
    run<3, 4, 3, 0>("half-up+table+warp staging", acc, l512, l256, out, side, cyc, sms);
    run<1, 4, 3, 0>("new+table+warp staging", acc, l512, l256, out, side, cyc, sms);
    run<3, 0, 3, 0>("half-up, no table, warp staging", acc, l512, l256, out, side, cyc, sms);
    run<3, 4, 3, 1>("half-up+table+warp staging+side", acc, l512, l256, out, side, cyc, sms);
    run<3, 4, 1, 0>("half-up+table+STG.U8", acc, l512, l256, out, side, cyc, sms);
    run<4, 0, 0, 0>("nocvt half-up math only", acc, l512, l256, out, side, cyc, sms);
    run<4, 4, 0, 0>("nocvt half-up + repl table", acc, l512, l256, out, side, cyc, sms);
    run<4, 4, 4, 0>("nocvt half-up+table+STG (IMAD.WIDE)", acc, l512, l256, out, side, cyc, sms);
    run<4, 4, 5, 0>("nocvt half-up+table+STG (imm plane)", acc, l512, l256, out, side, cyc, sms);
    run<3, 4, 5, 0>("F2I half-up+table+STG (imm plane)", acc, l512, l256, out, side, cyc, sms);
    run<4, 0, 5, 0>("nocvt half-up, no table, STG imm", acc, l512, l256, out, side, cyc, sms);
    run<4, 4, 5, 1>("nocvt half-up+table+STG imm+side", acc, l512, l256, out, side, cyc, sms);
    run<0, 3, 5, 0>("old math+table512+STG imm", acc, l512, l256, out, side, cyc, sms);
    return 0;
}
