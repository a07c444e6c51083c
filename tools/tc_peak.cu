/*
 * tools/tc_peak.cu -- measured ceiling of tcgen05.mma.kind::i8 on this chip (SURVEY 6.3: "the build must record its own
 * kind::i8 peak microbenchmark").
 *
 * One CTA per SM (or two), operands resident in shared memory (K-major, 128-byte swizzle, random bytes), no loads and no
 * epilogue inside the timed loop: `lanes` threads of one warp issue back-to-back M=128 x N x K=32 MMAs, lane g into its own
 * TMEM accumulator, `chain` MMAs per commit.  Prints TOP/s per N and issue configuration.
 * build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o /tmp/tc_peak tools/tc_peak.cu
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "../thingino-accel_b200/csrc/tc_common.cuh"

using namespace marsb200;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(1); } } while (0)

/* smem: A = 128 rows x 128 B (4 K=32 slices), B = N rows x 128 B, both in the canonical SW128 K-major layout (content is random:
 * the layout does not matter for timing, the power draw of random operands does) */
__global__ void __launch_bounds__(128) k_peak(int N, int lanes, int chain, int rounds, int tmem_cols, const uint8_t *rnd, unsigned long long *cycles) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar[16];
    __shared__ uint32_t tmem_slot;
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *al = smem_raw + (base - smem_u32(smem_raw));
    for (int i = threadIdx.x; i < (128 + 256) * 128 / 16; i += blockDim.x) reinterpret_cast<uint4 *>(al)[i] = reinterpret_cast<const uint4 *>(rnd)[i];
    if (threadIdx.x == 0) { for (int i = 0; i < 16; i++) mbar_init(smem_u32(&bar[i]), 1); mbar_fence_init(); }
    if (threadIdx.x < 32) tmem_alloc(smem_u32(&tmem_slot), (uint32_t)tmem_cols);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_d = tmem_slot;
    unsigned long long t0 = 0, t1 = 0;
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        if (lane < lanes) {
            const uint32_t hi = ((8u * 128u) >> 4) | (1u << 14) | (2u << 29); /* SBO = 1024 B, version 1, SW128 */
            const uint32_t a_lo = (base >> 4) | (1u << 16), b_lo = ((base + 128 * 128) >> 4) | (1u << 16);
            const uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
            const uint32_t acc = tmem_d + (uint32_t)(lane * N);
            const uint32_t mybar = smem_u32(&bar[2 * lane]); /* two barriers per lane: round r commits on barrier r & 1 */
            t0 = clock64();
            uint32_t ph[2] = {0, 0};
            for (int r = 0; r < rounds; r++) {
                if (r >= 2) { mbar_wait(mybar + 8u * (r & 1), ph[r & 1]); ph[r & 1] ^= 1; } /* one commit per barrier in flight */
                for (int c = 0; c < chain; c++) umma_i8(acc, a_lo + 2u * (c & 3), hi, b_lo + 2u * (c & 3), hi, idesc, (uint32_t)(c != 0));
                umma_commit(mybar + 8u * (r & 1));
            }
            for (int r = rounds > 2 ? rounds - 2 : 0; r < rounds; r++) { mbar_wait(mybar + 8u * (r & 1), ph[r & 1]); ph[r & 1] ^= 1; }
            t1 = clock64();
        }
        __syncwarp();
    }
    if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
    tcgen05_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) {
        tcgen05_fence_after();
        tmem_dealloc(tmem_d, (uint32_t)tmem_cols);
    }
}

int main(int argc, char **argv) {
    int sms = 0, clk = 0;
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
    CK(cudaDeviceGetAttribute(&clk, cudaDevAttrClockRate, 0));
    uint8_t *rnd; unsigned long long *cyc;
    const size_t nb = (128 + 256) * 128;
    CK(cudaMalloc(&rnd, nb)); CK(cudaMalloc(&cyc, 8 * 1024));
    uint8_t *h = (uint8_t *)malloc(nb);
    srand(7);
    for (size_t i = 0; i < nb; i++) h[i] = (uint8_t)(rand() >> 7);
    CK(cudaMemcpy(rnd, h, nb, cudaMemcpyHostToDevice));
    const size_t smem = nb + 2048;
    CK(cudaFuncSetAttribute(k_peak, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    printf("tcgen05.mma.cta_group::1.kind::i8, M=128, K=32 per instruction, operands resident in shared memory; %d SMs, max SM clock %d MHz\n", sms, clk / 1000);
    printf("%4s %5s %5s %5s %6s | %9s %12s %10s %9s\n", "N", "ctas", "lanes", "chain", "rounds", "ms", "cyc/MMA/lane", "TOP/s", "of 4500");
    const int Ns[] = {32, 64, 128, 256};
    for (int ctas = 1; ctas <= 2; ctas++)
        for (int ni = 0; ni < 4; ni++) {
            const int N = Ns[ni];
            const int tmem_cols = ctas == 1 ? 512 : 256;
            const int lane_opts[] = {1, 2, 4, 8};
            for (int li = 0; li < 4; li++) {
                const int lanes = lane_opts[li];
                if (lanes * N > tmem_cols) continue;
                for (int chain = 4; chain <= 36; chain *= 3) { /* 4, 12, 36 MMAs per commit */
                    const int rounds = 20000 / chain;
                    cudaEvent_t e0, e1;
                    cudaEventCreate(&e0); cudaEventCreate(&e1);
                    k_peak<<<sms * ctas, 128, smem>>>(N, lanes, chain, 64, tmem_cols, rnd, cyc);
                    CK(cudaDeviceSynchronize());
                    cudaEventRecord(e0);
                    k_peak<<<sms * ctas, 128, smem>>>(N, lanes, chain, rounds, tmem_cols, rnd, cyc);
                    cudaEventRecord(e1);
                    CK(cudaDeviceSynchronize());
                    float ms;
                    cudaEventElapsedTime(&ms, e0, e1);
                    unsigned long long hc[512];
                    CK(cudaMemcpy(hc, cyc, 8 * sms * ctas, cudaMemcpyDeviceToHost));
                    double avg = 0;
                    for (int i = 0; i < sms * ctas; i++) avg += (double)hc[i];
                    avg /= sms * ctas;
                    const double mmas = (double)rounds * chain; /* per lane */
                    const double ops = 2.0 * 128 * N * 32 * mmas * lanes * sms * ctas;
                    printf("%4d %5d %5d %5d %6d | %9.3f %12.1f %10.1f %8.1f%%\n", N, ctas, lanes, chain, rounds, ms, avg / mmas, ops / (ms * 1e-3) / 1e12,
                           100.0 * ops / (ms * 1e-3) / 4.5e15);
                    cudaEventDestroy(e0); cudaEventDestroy(e1);
                }
            }
        }
    return 0;
}
