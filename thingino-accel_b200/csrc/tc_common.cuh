/*
 * tc_common.cuh -- device-side building blocks of the tcgen05 convolutions (conv_tc.cu, conv_tf32.cu) and their microbenchmarks:
 * inline-PTX wrappers for mbarriers, TMA loads, UMMA issue / commit, TMEM management and loads, the persistent tile walk, and
 * the source pixel of a row of the padded / phase-split channel-innermost input copy.  Device code only: the host-side
 * planning helpers are in conv_tc.h.
 */
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace marsb200 {

/* ---- PTX wrappers ------------------------------------------------------------- */
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
/* makes the initialised barriers visible to the other threads and to the async proxy (TMA, tcgen05.commit) */
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t" /* suspend-time hint: the warp sleeps in the */
        "@p bra WAIT_DONE;\n\t"                                          /* barrier unit instead of spinning through */
        "bra WAIT_LOOP;\n\t"                                              /* issue slots the epilogue warps need     */
        "WAIT_DONE:\n\t"
        "}\n" ::"r"(bar), "r"(parity), "r"(0x989680u) : "memory");
}
/* wait used by warps that are not on the critical path (epilogue, gather producers): back off between polls so the
 * spin does not take issue slots from the warps doing the work */
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity) {
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}\n" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (done) break;
        __nanosleep(64);
    }
}
/* one non-blocking probe */
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    return done != 0;
}

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}

/* shared-memory accesses through a 32-bit shared address kept in a register (the generic->shared conversion of a
 * __shared__ object is otherwise re-materialised at every use in the epilogue's hot loop) */
__device__ __forceinline__ void sts_u8(uint32_t addr, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ int4 lds_v4(uint32_t addr) {
    int4 v;
    asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}

/* D[tmem] (+)= A[smem] * B[smem]; the two 64-bit shared-memory matrix descriptors are given as 32-bit halves (the high
 * halves are loop invariants of the issuing thread).  UMMA shared-memory matrix descriptor (cute/arch/mma_sm100_desc.hpp):
 * [0,14) start>>4, [16,30) LBO>>4, [32,46) SBO>>4, [46,48) version=1, [61,64) layout type (2 = SW128, 4 = SW64, 6 = SW32) */
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                        uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], da, db, %5, {%7, %7, %7, %7}, p;\n\t"
        "}\n" ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "mov.b64 da, {%1, %2};\n\t"
        "mov.b64 db, {%3, %4};\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %5, {%7, %7, %7, %7}, p;\n\t"
        "}\n" ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
/* arrives on the mbarrier when every MMA this thread issued before has retired */
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

/* ---- tensor memory ------------------------------------------------------------ */
/* warp-wide: allocate `cols` TMEM columns (address written to shared memory at `slot`) and give up the right to allocate
 * more, so that a co-resident CTA's allocation does not wait on this one */
__device__ __forceinline__ void tmem_alloc(uint32_t slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
/* warp-wide, by the allocating warp */
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
/* order tcgen05 operations before / after a thread synchronisation (barrier, mbarrier hand-over) */
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
/* split form of a 16-column TMEM load: issue the load, and later wait for it; the wait takes the destination registers as
 * in/out operands so that no use of them can be scheduled before it */
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&v)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]),
                   "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
                 :: "memory");
}

/* walks the tiles b, b + G, b + 2G, ... of a launch as (image, tile inside the image) without divisions in the loop */
struct TileIter {
    int img, rem, tpi, step_img, step_rem;
    __device__ __forceinline__ TileIter(int first, int G, int tiles_per_img) : tpi(tiles_per_img) {
        img = first / tpi; rem = first - img * tpi;
        step_img = G / tpi; step_rem = G - step_img * tpi;
    }
    __device__ __forceinline__ void next() {
        img += step_img; rem += step_rem;
        if (rem >= tpi) { rem -= tpi; img++; }
    }
};

/* source pixel (ih, iw) of row `pix` of the channel-innermost input copy (PixelCopy, conv_tc.h); outside the image = zeros:
 *   stride 1 (mode 1): ih = pix / Wp, iw = pix % Wp - pl                          (rows padded to Wp)
 *   stride 2 (mode 2): ph = pix / plane, a = (pix % plane) / Wp, b = .. % Wp, ih = 2a + ph/2 - pt, iw = 2b + ph%2 - pl */
__device__ __forceinline__ void copy_src_pixel(int pix, bool stride2, int Wp, int plane, int pt, int pl, int &ih, int &iw) {
    if (stride2) {
        int ph = pix / plane, r = pix - ph * plane, a = r / Wp, b = r - a * Wp;
        ih = 2 * a + (ph >> 1) - pt; iw = 2 * b + (ph & 1) - pl;
    } else {
        ih = pix / Wp; iw = pix - ih * Wp - pl;
    }
}

} // namespace marsb200
