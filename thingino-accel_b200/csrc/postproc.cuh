/*
 * postproc.cuh -- YOLO decode + class-wise NMS kernels (SURVEY §8a rows 18-21).
 *
 *  k_parse_output : parse_output() of reference src/mars/mars_yolo_test.c:80-104 --
 *                   per-row objectness/class decode through host-built libm tables,
 *                   ORDER-PRESERVING compaction with the reference's hard cap;
 *  k_nms_sort_warp, k_nms_suppress / k_nms_center :
 *                   nms() of reference src/mars/mars_yolo_test.c:107-130 -- the exchange
 *                   sort is emulated pass by pass (its permutation under ties is NOT a
 *                   stable sort, SURVEY A.4) by one warp per image, then greedy same-class
 *                   suppression through per-class member bitsets and a bit matrix (256
 *                   threads per image for large batches, 1024 for small ones);
 *  k_head_decode  : anchor-grid decode (mgk-decompiler/test_yolo_inference.py:136-202) of one head level, reading the raw
 *                   head convolution where the program leaves it (OP_YOLO_HEAD, mars_b200_set_yolo_heads);
 *  k_gfl_decode   : GFL decode of one NanoDet head level (ours; OP_GFL_HEAD, mars_b200_set_gfl_heads), the same placement;
 *  k_nms_corner_batch : nms() of reference examples/yolo_detect.cpp:152-173 (corner boxes), with the letterbox inverse;
 *  k_merge_rois   : the boxes of a frame's regions (tiled detection; ours, the reference does not tile) shifted into the frame and
 *                   merged by the same corner NMS (nms_corner_image, shared with k_nms_corner_batch);
 *  k_scale_detections : the letterbox inverse alone (reference examples/yolo_detect.cpp:208-227).
 * The host-pointer entry points (seam.inc) run these kernels on a batch of one image.
 * One thread block per image; blocks are independent (images shard with no exchange).
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <cub/block/block_radix_sort.cuh>

#include "kernels_exact.cuh"

namespace marsb200 {

#define MARS_MAX_DETS 1024

/* tables built on the host with the host libm (bit-exact w.r.t. the reference's expf) */
struct DecodeTables {
    float obj[256];  /* 1/(1+expf(-(v*scale)))                      mars_yolo_test.c:84 */
    float den[257];  /* 1+expf(-(v*scale)); [256] = the "no class beat -1e9f" case  :92 */
};

/* block-wide exclusive scan of one int per thread (blockDim.x <= 1024, multiple of 32) */
__device__ __forceinline__ int block_excl_scan(int v, int *total, int *warp_sums /* [32] shared */) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
        int s = lane < nw ? warp_sums[lane] : 0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int y = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += y;
        }
        warp_sums[lane] = s; /* inclusive over warps */
    }
    __syncthreads();
    int base = wid ? warp_sums[wid - 1] : 0;
    *total = warp_sums[nw - 1];
    __syncthreads();
    return base + x - v;
}

/* data: int8 [npred][85] per image at data + img*img_stride; dets: [maxd] per image */
__global__ void __launch_bounds__(256) k_parse_output(const int8_t *data, size_t img_stride, int npred, float scale,
                                                      const DecodeTables *tab, mars_det_t *dets, int32_t *counts,
                                                      int maxd, int det_stride) {
    __shared__ int warp_sums[32];
    const int8_t *rows = data + (size_t)blockIdx.x * img_stride;
    mars_det_t *out = dets + (size_t)blockIdx.x * det_stride;
    int cnt = 0;
    for (int base = 0; base < npred && cnt < maxd; base += blockDim.x) {
        int i = base + threadIdx.x;
        int pass = 0, best_c = 0;
        float conf = 0.0f;
        const int8_t *p = rows + (size_t)i * 85;
        if (i < npred) {
            float obj = tab->obj[(int)p[4] + 128];
            if (!(obj < 0.25f)) {
                float best_s = -1e9f;
                int best_v = 256 - 128; /* -> den[256] */
                for (int c = 0; c < 80; c++) {
                    int v = p[5 + c];
                    float s = __fmul_rn((float)v, scale);
                    if (s > best_s) { best_s = s; best_c = c; best_v = v; }
                }
                conf = __fdiv_rn(obj, tab->den[best_v + 128]);
                pass = !(conf < 0.25f);
            }
        }
        int total;
        int rank = cnt + block_excl_scan(pass, &total, warp_sums);
        if (pass && rank < maxd) {
            mars_det_t d;
            d.x = __fmul_rn((float)p[0], scale); d.y = __fmul_rn((float)p[1], scale);
            d.w = __fmul_rn((float)p[2], scale); d.h = __fmul_rn((float)p[3], scale);
            d.conf = conf; d.cls = best_c;
            out[rank] = d;
        }
        cnt += total;
    }
    if (threadIdx.x == 0) counts[blockIdx.x] = cnt < maxd ? cnt : maxd;
}

/* reference src/mars/mars_yolo_test.c:115-121, every operation rounded separately */
__device__ __forceinline__ float iou_center(const mars_det_t &a, const mars_det_t &b) {
    float ahw = __fdiv_rn(a.w, 2.0f), ahh = __fdiv_rn(a.h, 2.0f), bhw = __fdiv_rn(b.w, 2.0f), bhh = __fdiv_rn(b.h, 2.0f);
    float x1 = fmaxf(__fsub_rn(a.x, ahw), __fsub_rn(b.x, bhw));
    float y1 = fmaxf(__fsub_rn(a.y, ahh), __fsub_rn(b.y, bhh));
    float x2 = fminf(__fadd_rn(a.x, ahw), __fadd_rn(b.x, bhw));
    float y2 = fminf(__fadd_rn(a.y, ahh), __fadd_rn(b.y, bhh));
    float inter = __fmul_rn(fmaxf(0.0f, __fsub_rn(x2, x1)), fmaxf(0.0f, __fsub_rn(y2, y1)));
    float u = __fadd_rn(__fsub_rn(__fadd_rn(__fmul_rn(a.w, a.h), __fmul_rn(b.w, b.h)), inter), 1e-6f);
    return __fdiv_rn(inter, u);
}

/* reference examples/yolo_detect.cpp:138-149 */
__device__ __forceinline__ float iou_corner(const mars_box_t &a, const mars_box_t &b) {
    float x0 = fmaxf(a.x0, b.x0), y0 = fmaxf(a.y0, b.y0), x1 = fminf(a.x1, b.x1), y1 = fminf(a.y1, b.y1);
    float inter = __fmul_rn(fmaxf(0.0f, __fsub_rn(x1, x0)), fmaxf(0.0f, __fsub_rn(y1, y0)));
    float aa = __fmul_rn(__fsub_rn(a.x1, a.x0), __fsub_rn(a.y1, a.y0));
    float ab = __fmul_rn(__fsub_rn(b.x1, b.x0), __fsub_rn(b.y1, b.y0));
    return __fdiv_rn(inter, __fadd_rn(__fsub_rn(__fadd_rn(aa, ab), inter), 1e-6f));
}

/*
 * Exchange-sort emulation, one WARP per image and no barriers.  Pass i of `for i: for j>i: if d[j].conf > d[i].conf swap`
 * (reference src/mars/mars_yolo_test.c:108-110) walks the strict prefix-maximum records r0 = i < r1 < ... < rk of key[i..n):
 * afterwards position r0 holds the element of rk and every other record position holds the previous record's element
 * (SURVEY A.4; NOT a stable sort).
 *
 * Lane L holds positions [32L, 32L+32) in registers (key k[], input index x[]); the 32 positions of the lane that
 * contains the current pass index i are spread one per lane (Bk, Bx: "the block"), so that the hand d[i] is a shuffle
 * from lane i % 32 and nothing is indexed dynamically.  Pass i rotates the chain of strict prefix-maximum records of d[i..n):
 * every record takes its predecessor's element, the first record takes the hand and position i takes the last record's
 * element.  The chain is found in two levels:
 *   block    : prefix max over the 32 lanes (retired positions hold -inf and are inert);
 *   registers: each lane keeps the first-occurrence maximum (lm, lmx) of its 32 positions; a prefix max over the lanes
 *              (seeded with the block's outgoing maximum) tells which lanes contain records and what enters them, and those
 *              lanes walk their registers with the literal compare-and-swap of the C loop.
 * The element leaving the last record is final: it is written to order[i] and never looked at again.
 * NaN keys never compare greater (never records); a NaN hand makes every comparison fail, so the pass moves nothing.
 */
/* passes [i0, i1) over a layout in which lane L holds the R consecutive positions base + L*R .. (R = 32, 16, 8 or 4; i0 - base
 * is a multiple of 32).  A block of 32 positions is 32/R lanes wide. */
template <int R>
__device__ __forceinline__ void nms_sort_passes(float (&k)[R], int (&x)[R], int base, int i0, int i1, uint16_t *order, int lane) {
    const float NEG_INF = -__int_as_float(0x7f800000), POS_INF = __int_as_float(0x7f800000);
    const unsigned FULL = 0xffffffffu;
    constexpr int LPB = 32 / R; /* lanes per block */
    float lm = NEG_INF, Bk = NEG_INF;
    int lmx = 0, Bx = 0;
    const unsigned below = (1u << lane) - 1u;
    for (int i = i0; i < i1; i++) {
        const int t = (i - base) & 31;
        if (t == 0) {
            /* the next 32 positions become the block; the lanes that held them are dead from now on */
            const int l0 = ((i - base) >> 5) * LPB;
#pragma unroll
            for (int sub = 0; sub < LPB; sub++) {
#pragma unroll
                for (int u = 0; u < R; u++) {
                    const float vk = __shfl_sync(FULL, k[u], l0 + sub);
                    const int vx = __shfl_sync(FULL, x[u], l0 + sub);
                    if (lane == sub * R + u) { Bk = vk; Bx = vx; }
                }
            }
            if (lane >= l0 && lane < l0 + LPB) {
#pragma unroll
                for (int u = 0; u < R; u++) k[u] = NEG_INF;
            }
            if (i == i0) { /* first-occurrence maxima of the register lanes of this phase */
                lm = NEG_INF;
#pragma unroll
                for (int u = 0; u < R; u++)
                    if (k[u] > lm) { lm = k[u]; lmx = x[u]; }
            } else if (lane >= l0 && lane < l0 + LPB) lm = NEG_INF;
        }
        /* The pass is one dependent chain (scan -> who holds records -> walk -> next pass's maxima), so it is written for
         * latency: both prefix-max scans run interleaved and start before the hand is known (only their seeds depend on it),
         * and the walk keeps four independent one-operation chains (running key, running index, new maximum, its index). */
        const float hk = __shfl_sync(FULL, Bk, t);
        const int hx = __shfl_sync(FULL, Bx, t);
        if (lane == t) Bk = NEG_INF; /* position i retires */
        float inc = (Bk == Bk) ? Bk : NEG_INF; /* block: records among the 32 spread positions */
        float inc2 = lm;                       /* register lanes: which lanes hold records */
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const float y = __shfl_up_sync(FULL, inc, d);
            const float y2 = __shfl_up_sync(FULL, inc2, d);
            if (lane >= d) { inc = fmaxf(inc, y); inc2 = fmaxf(inc2, y2); }
        }
        float exc = __shfl_up_sync(FULL, inc, 1);
        float e2 = __shfl_up_sync(FULL, inc2, 1);
        const float bmax = __shfl_sync(FULL, inc, 31); /* maximum of the whole block */
        const float run0 = (hk != hk) ? POS_INF : hk;
        exc = fmaxf(lane ? exc : NEG_INF, run0);
        const float ok = fmaxf(bmax, run0); /* key that leaves the block: its last record's, or the hand's */
        e2 = fmaxf(lane ? e2 : NEG_INF, ok);
        const bool brec = Bk > exc;
        const bool has = lm > e2;
        const unsigned bm = __ballot_sync(FULL, brec);
        const unsigned hm = __ballot_sync(FULL, has);
        const int blast = bm ? 31 - __clz(bm) : 0;
        const unsigned blower = bm & below;
        const int bsrc = blower ? 31 - __clz(blower) : 0;
        int ox = __shfl_sync(FULL, Bx, blast);
        const float pk = __shfl_sync(FULL, Bk, bsrc);
        const int px = __shfl_sync(FULL, Bx, bsrc);
        if (!bm) ox = hx; /* the hand itself leaves the block */
        if (brec) { Bk = blower ? pk : hk; Bx = blower ? px : hx; }
        int wx = ox;
        if (hm) { /* uniform */
            const unsigned hlower = hm & below;
            const int hsrc = hlower ? 31 - __clz(hlower) : 0;
            const int ix = __shfl_sync(FULL, lmx, hsrc);
            float run_k = e2;
            int run_x = hlower ? ix : ox;
            float nlm = NEG_INF;
            int nlx = 0;
#pragma unroll
            for (int u = 0; u < R; u++) {
                const float ku = k[u];
                const int xu = x[u];
                const bool sw = ku > run_k;          /* the C loop's comparison (false for NaN) */
                const float nk = sw ? run_k : ku;
                const int nx = sw ? run_x : xu;
                run_k = fmaxf(run_k, ku);            /* == sw ? ku : run_k; run_k is never NaN and fmaxf ignores a NaN ku */
                run_x = sw ? xu : run_x;
                k[u] = nk; x[u] = nx;
                const bool q = nk > nlm;
                nlm = fmaxf(nlm, nk);
                nlx = q ? nx : nlx;
            }
            lm = nlm; lmx = nlx;
            wx = __shfl_sync(FULL, run_x, 31 - __clz(hm));
        }
        if (lane == 0) order[i] = (uint16_t)wx;
    }
}

/* all passes from position `base` on, starting with R positions per lane: the first half of what is left is sorted with this
 * layout, then the surviving upper 16 lanes are spread over the whole warp (R/2 positions per lane: the walk, the largest
 * part of a pass, shrinks with the data) and the rest follows recursively */
template <int R>
__device__ __forceinline__ void nms_sort_from(float (&k)[R], int (&x)[R], int base, int n, uint16_t *order, int lane) {
    constexpr int RMIN = 4;
    const int stop = (R > RMIN) ? min(n, base + 16 * R) : n;
    nms_sort_passes<R>(k, x, base, base, stop, order, lane);
    if constexpr (R > RMIN) {
        if (n > stop) { /* uniform */
            float nk[R / 2];
            int nx[R / 2];
            const int src = 16 + (lane >> 1);
#pragma unroll
            for (int u = 0; u < R / 2; u++) {
                const float a = __shfl_sync(0xffffffffu, k[u], src), b = __shfl_sync(0xffffffffu, k[u + R / 2], src);
                const int ax = __shfl_sync(0xffffffffu, x[u], src), bx = __shfl_sync(0xffffffffu, x[u + R / 2], src);
                nk[u] = (lane & 1) ? b : a;
                nx[u] = (lane & 1) ? bx : ax;
            }
            nms_sort_from<R / 2>(nk, nx, base + 16 * R, n, order, lane);
        }
    }
}

template <int R>
__device__ __forceinline__ void nms_sort_image(const mars_det_t *in, int n, uint16_t *order, int lane) {
    const float NEG_INF = -__int_as_float(0x7f800000);
    float k[R];
    int x[R];
#pragma unroll
    for (int u = 0; u < R; u++) {
        const int p = lane * R + u;
        k[u] = p < n ? in[p].conf : NEG_INF;
        x[u] = p;
    }
    nms_sort_from<R>(k, x, 0, n, order, lane);
}

__global__ void __launch_bounds__(32) k_nms_sort_warp(const mars_det_t *dets_in, const int32_t *counts_in, int det_stride,
                                                      unsigned *scratch, size_t scratch_stride_words) {
    const int img = blockIdx.x, lane = threadIdx.x;
    const mars_det_t *in = dets_in + (size_t)img * det_stride;
    uint16_t *order = reinterpret_cast<uint16_t *>(scratch + (size_t)img * scratch_stride_words + (size_t)MARS_MAX_DETS * 32);
    int n = counts_in[img];
    if (n > MARS_MAX_DETS) n = MARS_MAX_DETS;
    /* fewest positions per lane that hold the image: short lists do not pay for a 1024-position layout */
    if (n <= 128) nms_sort_image<4>(in, n, order, lane);
    else if (n <= 256) nms_sort_image<8>(in, n, order, lane);
    else if (n <= 512) nms_sort_image<16>(in, n, order, lane);
    else nms_sort_image<32>(in, n, order, lane);
}

/* words of per-image scratch: the suppression bit matrix, the sorted order (uint16 per position), and the per-class member
 * bitsets of k_nms_suppress (NMS_CLASS_ROWS x 32 words) */
#define NMS_CLASS_ROWS 128 /* class ids -1..126 get a member bitset; anything else takes the dense pair loop */
#define NMS_SCRATCH_WORDS ((size_t)MARS_MAX_DETS * 32 + MARS_MAX_DETS / 2 + NMS_CLASS_ROWS * 32)

#define NMS_THREADS 1024 /* threads of k_nms_center: one per sorted position */

/* the sorted elements of one image as the centre-box suppression reads them: corners, area and class id */
struct NmsBoxes {
    float x0[MARS_MAX_DETS], y0[MARS_MAX_DETS], x1[MARS_MAX_DETS], y1[MARS_MAX_DETS], area[MARS_MAX_DETS];
    int cls[MARS_MAX_DETS];
};

/* dynamic shared memory of k_nms_center */
struct NmsShared {
    NmsBoxes b;
    unsigned members[NMS_CLASS_ROWS][32]; /* bit j of row c: sorted element j has class c - 1 */
    unsigned removed[32];
    int warp_sums[32];
    int dense;
};

/* IoU of reference src/mars/mars_yolo_test.c:115-121 from the per-element corners and areas (each operation rounded
 * separately, exactly as when it is evaluated per pair: the corner and area expressions only involve one box) */
__device__ __forceinline__ float iou_pre(float ax0, float ay0, float ax1, float ay1, float aarea, float bx0, float by0, float bx1,
                                         float by1, float barea) {
    const float x1 = fmaxf(ax0, bx0), y1 = fmaxf(ay0, by0), x2 = fminf(ax1, bx1), y2 = fminf(ay1, by1);
    const float inter = __fmul_rn(fmaxf(0.0f, __fsub_rn(x2, x1)), fmaxf(0.0f, __fsub_rn(y2, y1)));
    return __fdiv_rn(inter, __fadd_rn(__fsub_rn(__fadd_rn(aarea, barea), inter), 1e-6f));
}

/* sorted element j is d: the corner and area terms of iou_pre (d by value: the caller's loads all issue before these stores) */
__device__ __forceinline__ void nms_set_box(NmsBoxes &b, int j, const mars_det_t d) {
    const float hw = __fdiv_rn(d.w, 2.0f), hh = __fdiv_rn(d.h, 2.0f);
    b.x0[j] = __fsub_rn(d.x, hw); b.x1[j] = __fadd_rn(d.x, hw);
    b.y0[j] = __fsub_rn(d.y, hh); b.y1[j] = __fadd_rn(d.y, hh);
    b.area[j] = __fmul_rn(d.w, d.h);
    b.cls[j] = d.cls;
}

/* sorted element j has class cls: bit j of the class's member row members[(cls + 1) * 32 + word] (rows zeroed beforehand), or
 * *dense = 1 when the class has no row */
__device__ __forceinline__ void nms_add_member(unsigned *members, int cls, int j, int *dense) {
    const unsigned c = (unsigned)(cls + 1);
    if (c < NMS_CLASS_ROWS) atomicOr(&members[c * 32 + (j >> 5)], 1u << (j & 31));
    else *dense = 1;
}

/* rows i = row0, row0 + rstep, ... of the suppression bit matrix, one warp per row: bit j of row i is set when sorted element
 * j > i has i's class and IoU(i, j) > thresh.  Only same-class pairs can suppress: the member row of i's class turns row i
 * into "members of i's class behind i" -- one word per lane -- and each lane evaluates the IoU of the few bits set in its
 * word.  With dense set (class ids without a member row) every pair behind i is tested, lane = bit. */
__device__ __forceinline__ void nms_build_rows(const NmsBoxes &b, const unsigned *members, bool dense, int n, float thresh,
                                               unsigned *mask, int row0, int rstep, int lane) {
    const int nwords = (n + 31) >> 5;
    if (!dense) {
        for (int i = row0; i < n; i += rstep) {
            const int w0 = i >> 5;
            unsigned cand = (lane >= w0 && lane < nwords) ? members[(b.cls[i] + 1) * 32 + lane] : 0u;
            if (lane == w0) cand &= ~((2u << (i & 31)) - 1u); /* only elements behind i */
            unsigned bits = 0u;
            if (__any_sync(0xffffffffu, cand != 0u)) {
                const float ax0 = b.x0[i], ay0 = b.y0[i], ax1 = b.x1[i], ay1 = b.y1[i], aarea = b.area[i];
                while (cand) {
                    const int q = __ffs(cand) - 1;
                    cand &= cand - 1u;
                    const int jj = lane * 32 + q;
                    if (iou_pre(ax0, ay0, ax1, ay1, aarea, b.x0[jj], b.y0[jj], b.x1[jj], b.y1[jj], b.area[jj]) > thresh) bits |= 1u << q;
                }
            }
            if (lane >= w0 && lane < nwords) mask[i * 32 + lane] = bits;
        }
    } else {
        for (int i = row0; i < n; i += rstep) {
            const float ax0 = b.x0[i], ay0 = b.y0[i], ax1 = b.x1[i], ay1 = b.y1[i], aarea = b.area[i];
            const int acls = b.cls[i];
            for (int w = i >> 5; w < nwords; w++) {
                const int jj = w * 32 + lane;
                bool sup = false;
                if (jj > i && jj < n && b.cls[jj] == acls)
                    sup = iou_pre(ax0, ay0, ax1, ay1, aarea, b.x0[jj], b.y0[jj], b.x1[jj], b.y1[jj], b.area[jj]) > thresh;
                const unsigned bits = __ballot_sync(0xffffffffu, sup);
                if (lane == 0) mask[i * 32 + w] = bits;
            }
        }
    }
}

/* The greedy walk of one warp over the bit matrix: i ascending, row i is ORed into the removed set iff i is still alive -- the
 * same result as the sequential double loop.  Returns lane w's removed bits (sorted elements [32w, 32w+32)).  The walk is
 * serial in i but the rows do not depend on it: they are fetched CH at a time (independent L2 loads in flight together), the
 * next CH while these are used. */
template <int CH>
__device__ __forceinline__ unsigned nms_walk(const unsigned *mask, int n, int lane) {
    const int nwords = (n + 31) >> 5;
    unsigned removed = 0u;
    unsigned cur_rows[CH], nxt_rows[CH];
    auto fetch = [&](unsigned (&rows)[CH], int base) {
#pragma unroll
        for (int q = 0; q < CH; q++) {
            const int i = base + q;
            rows[q] = (i < n && lane >= (i >> 5) && lane < nwords) ? mask[i * 32 + lane] : 0u;
        }
    };
    fetch(cur_rows, 0);
    for (int base = 0; base < n; base += CH) {
        fetch(nxt_rows, base + CH);
#pragma unroll
        for (int q = 0; q < CH; q++) {
            const int i = base + q; /* rows beyond n are zero */
            const unsigned word = __shfl_sync(0xffffffffu, removed, (i >> 5) & 31);
            if (!((word >> (i & 31)) & 1u)) removed |= cur_rows[q];
        }
#pragma unroll
        for (int q = 0; q < CH; q++) cur_rows[q] = nxt_rows[q];
    }
    return removed;
}

/* lane w publishes its removed bits (removed[w]) and the exclusive prefix of the per-word removed counts (before[w]: removed
 * elements in words 0..w-1); lane 31 writes the kept count of the n elements to *kept */
__device__ __forceinline__ void nms_publish_removed(unsigned removed, int n, int lane, unsigned *removed_out, int *before, int32_t *kept) {
    const int cnt = __popc(removed);
    int incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += y;
    }
    removed_out[lane] = removed;
    before[lane] = incl - cnt;
    if (lane == 31) *kept = n - incl;
}

/* dets_in/dets_out: [det_stride] per image; counts in/out per image.  blockDim.x = NMS_THREADS, dynamic smem = sizeof(NmsShared);
 * mask_scratch: NMS_SCRATCH_WORDS per image: the MARS_MAX_DETS x 32 words of the bit matrix (kept in global memory,
 * L2-resident, written and read once, so that two blocks fit one SM), then the sorted order written by k_nms_sort_warp.
 * Greedy suppression (mars_yolo_test.c:113-123) as a bit matrix (nms_build_rows) and its walk (nms_walk). */
__global__ void __launch_bounds__(NMS_THREADS, 2) k_nms_center(const mars_det_t *dets_in, const int32_t *counts_in,
                                                               mars_det_t *dets_out, int32_t *counts_out, int det_stride,
                                                               float thresh, unsigned *mask_scratch) {
    extern __shared__ __align__(16) uint8_t nms_smem[];
    NmsShared &sh = *reinterpret_cast<NmsShared *>(nms_smem);
    const mars_det_t *in = dets_in + (size_t)blockIdx.x * det_stride;
    mars_det_t *out = dets_out + (size_t)blockIdx.x * det_stride;
    unsigned *const mask = mask_scratch + (size_t)blockIdx.x * NMS_SCRATCH_WORDS;
    const uint16_t *order = reinterpret_cast<const uint16_t *>(mask + (size_t)MARS_MAX_DETS * 32);
    int n = counts_in[blockIdx.x];
    if (n > MARS_MAX_DETS) n = MARS_MAX_DETS;
    const int j = threadIdx.x, lane = j & 31, wid = j >> 5;
    /* sorted position j holds input element src (k_nms_sort_warp) */
    const int src = j < n ? order[j] : j;
    for (int q = j; q < NMS_CLASS_ROWS * 32; q += NMS_THREADS) (&sh.members[0][0])[q] = 0u;
    if (j == 0) sh.dense = 0;
    mars_det_t me;
    if (j < n) {
        me = in[src];
        nms_set_box(sh.b, j, me);
    }
    __syncthreads();
    if (j < n) nms_add_member(&sh.members[0][0], me.cls, j, &sh.dense);
    __syncthreads();
    nms_build_rows(sh.b, &sh.members[0][0], sh.dense, n, thresh, mask, wid, NMS_THREADS / 32, lane);
    __syncthreads();
    if (wid == 0) sh.removed[lane] = nms_walk<16>(mask, n, lane);
    __syncthreads();
    /* ordered compaction */
    const int keep = j < n && !((sh.removed[wid] >> lane) & 1u);
    int total;
    const int r = block_excl_scan(keep, &total, sh.warp_sums);
    if (keep) out[r] = me;
    if (j == 0) counts_out[blockIdx.x] = total;
}

/* ---- suppression for presorted images: 256 threads per image, ~24 KiB of shared memory ----------------------------------
 * The algorithm of k_nms_center sized so that eight images share an SM and a whole 1024-image batch is resident at once: the
 * per-class member bitsets live in the image's global scratch (L2), each thread owns four sorted positions, and the compaction
 * rank comes from population counts over the removed set instead of a block scan. */
#define NMS_SUP_THREADS 256
struct NmsSupShared {
    NmsBoxes b;
    unsigned removed[32];
    int removed_before[32]; /* removed elements in words 0..w-1 */
    int dense;
};

__global__ void __launch_bounds__(NMS_SUP_THREADS, 8) k_nms_suppress(const mars_det_t *dets_in, const int32_t *counts_in,
                                                                     mars_det_t *dets_out, int32_t *counts_out, int det_stride,
                                                                     float thresh, unsigned *scratch) {
    __shared__ NmsSupShared sh;
    const mars_det_t *in = dets_in + (size_t)blockIdx.x * det_stride;
    mars_det_t *out = dets_out + (size_t)blockIdx.x * det_stride;
    unsigned *const mask = scratch + (size_t)blockIdx.x * NMS_SCRATCH_WORDS;
    const uint16_t *order = reinterpret_cast<const uint16_t *>(mask + (size_t)MARS_MAX_DETS * 32);
    unsigned *const members = mask + (size_t)MARS_MAX_DETS * 32 + MARS_MAX_DETS / 2; /* [NMS_CLASS_ROWS][32] */
    int n = counts_in[blockIdx.x];
    if (n > MARS_MAX_DETS) n = MARS_MAX_DETS;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    constexpr int NW = NMS_SUP_THREADS / 32, PER = MARS_MAX_DETS / NMS_SUP_THREADS;
    for (int q = tid; q < NMS_CLASS_ROWS * 32; q += NMS_SUP_THREADS) members[q] = 0u;
    if (tid == 0) sh.dense = 0;
    /* thread tid owns the sorted positions j = tid + k * 256 */
#pragma unroll
    for (int k = 0; k < PER; k++) {
        const int j = tid + k * NMS_SUP_THREADS;
        if (j < n) nms_set_box(sh.b, j, in[order[j]]);
    }
    __syncthreads(); /* members zeroed (global writes of this block are visible to it after the barrier), dense flag reset */
#pragma unroll
    for (int k = 0; k < PER; k++) {
        const int j = tid + k * NMS_SUP_THREADS;
        if (j < n) nms_add_member(members, sh.b.cls[j], j, &sh.dense);
    }
    __syncthreads();
    nms_build_rows(sh.b, members, sh.dense, n, thresh, mask, wid, NW, lane);
    __syncthreads();
    if (wid == 0) nms_publish_removed(nms_walk<8>(mask, n, lane), n, lane, sh.removed, sh.removed_before, &counts_out[blockIdx.x]);
    __syncthreads();
    /* ordered compaction: a kept element moves up by the number of removed elements in front of it */
#pragma unroll
    for (int k = 0; k < PER; k++) {
        const int j = tid + k * NMS_SUP_THREADS;
        if (j < n) {
            const unsigned word = sh.removed[j >> 5];
            if (!((word >> (j & 31)) & 1u)) out[j - sh.removed_before[j >> 5] - __popc(word & ((1u << (j & 31)) - 1u))] = in[order[j]];
        }
    }
}

static inline cudaError_t launch_nms_center(const mars_det_t *dets_in, const int32_t *counts_in, mars_det_t *dets_out,
                                            int32_t *counts_out, int det_stride, float thresh, int n_img, unsigned *scratch /* NMS_SCRATCH_WORDS per image */,
                                            cudaStream_t s) {
    static unsigned long long attr = 0; /* function attributes are per device */
    if (first_time_on_device(&attr)) {
        cudaError_t e = cudaFuncSetAttribute(k_nms_center, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(NmsShared));
        if (e != cudaSuccess) return e;
    }
    k_nms_sort_warp<<<n_img, 32, 0, s>>>(dets_in, counts_in, det_stride, scratch, NMS_SCRATCH_WORDS);
    /* many images: eight 256-thread blocks per SM keep the whole batch resident (throughput); few images: 1024 threads
     * per image finish each one sooner (latency) */
    if (n_img > 2 * 296) k_nms_suppress<<<n_img, NMS_SUP_THREADS, 0, s>>>(dets_in, counts_in, dets_out, counts_out, det_stride, thresh, scratch);
    else k_nms_center<<<n_img, NMS_THREADS, sizeof(NmsShared), s>>>(dets_in, counts_in, dets_out, counts_out, det_stride, thresh, scratch);
    return cudaGetLastError();
}

/* ---- letterbox inverse of reference examples/yolo_detect.cpp:208-227 (mo_scale_detections), one rounding per operation ---- */
struct Letterbox { float sc, px, py, wmax, hmax; };

/* the scale and padding that letterboxed an orig_w x orig_h frame into the net_w x net_h input, and the frame's last pixel */
__device__ __forceinline__ Letterbox letterbox_params(int orig_w, int orig_h, int net_w, int net_h) {
    Letterbox l;
    l.sc = fminf(__fdiv_rn((float)net_w, (float)orig_w), __fdiv_rn((float)net_h, (float)orig_h));
    l.px = __fdiv_rn(__fsub_rn((float)net_w, __fmul_rn((float)orig_w, l.sc)), 2.0f);
    l.py = __fdiv_rn(__fsub_rn((float)net_h, __fmul_rn((float)orig_h, l.sc)), 2.0f);
    l.wmax = __fsub_rn((float)orig_w, 1.0f); l.hmax = __fsub_rn((float)orig_h, 1.0f);
    return l;
}

/* a box in input pixels -> frame pixels, clamped to the frame */
__device__ __forceinline__ mars_box_t letterbox_inverse(mars_box_t b, const Letterbox &l) {
    b.x0 = fmaxf(0.0f, fminf(__fdiv_rn(__fsub_rn(b.x0, l.px), l.sc), l.wmax));
    b.y0 = fmaxf(0.0f, fminf(__fdiv_rn(__fsub_rn(b.y0, l.py), l.sc), l.hmax));
    b.x1 = fmaxf(0.0f, fminf(__fdiv_rn(__fsub_rn(b.x1, l.px), l.sc), l.wmax));
    b.y1 = fmaxf(0.0f, fminf(__fdiv_rn(__fsub_rn(b.y1, l.py), l.sc), l.hmax));
    return b;
}

__global__ void k_scale_detections(mars_box_t *d, int n, int orig_w, int orig_h, int net_w, int net_h) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] = letterbox_inverse(d[i], letterbox_params(orig_w, orig_h, net_w, net_h));
}

/* ---- YOLOv5 Detect heads ------------------------------------------------------------------------------------------------ */
#define HEAD_MAX_CAND 1000 /* candidates per image over the three levels (yolo_detect.cpp keeps an uncapped vector) */

/* Anchor-grid decode of one level for every image of the launch: the head of image b is at head + b * img_stride, element
 * (anchor a, channel c, cell p = y * gw + x) at a * astride + c * cstride + p * pstride (NCHW: cstride = gh * gw, pstride = 1, so a
 * warp reads one byte plane across adjacent x; NHWC: cstride = 1, pstride = 3 (5 + nc)); sig[v+128] =
 * 1/(1+expf(-(v*scale))) from the host.  Candidates go to boxes[b][...] in (anchor, y, x) order, ordered compaction after the
 * image's running count when `append` is set (else from 0), capped at maxd. */
__global__ void __launch_bounds__(256) k_head_decode(const int8_t *head, size_t img_stride, int gh, int gw, int nc, int astride, int cstride,
                                                     int pstride, const float *sig, float stride, HeadAnchors anc, float conf_thresh,
                                                     int append, mars_box_t *boxes, int32_t *counts, int box_stride, int maxd) {
    __shared__ int warp_sums[32];
    const int8_t *hb = head + (size_t)blockIdx.x * img_stride;
    mars_box_t *out = boxes + (size_t)blockIdx.x * box_stride;
    const int P = gh * gw, ncell = 3 * P;
    int cnt = append ? min(counts[blockIdx.x], maxd) : 0;
    __syncthreads(); /* every thread has read the count before thread 0 rewrites it */
    for (int base = 0; base < ncell && cnt < maxd; base += blockDim.x) {
        const int i = base + threadIdx.x;
        int pass = 0, best = 0, a = 0, cell = 0;
        float conf = 0.0f;
        const int8_t *p = hb;
        if (i < ncell) {
            a = i / P; cell = i - a * P;
            p = hb + (size_t)a * astride + (size_t)cell * pstride;
            const float obj = sig[(int)p[4 * cstride] + 128];
            if (!(obj < conf_thresh)) {
                int bv = p[5 * cstride];
                for (int c = 1; c < nc; c++) {
                    const int v = p[(size_t)(5 + c) * cstride];
                    if (v > bv) { bv = v; best = c; }
                }
                conf = __fmul_rn(obj, sig[bv + 128]);
                pass = !(conf < conf_thresh);
            }
        }
        int total;
        const int rank = cnt + block_excl_scan(pass, &total, warp_sums);
        if (pass && rank < maxd) {
            const int y = cell / gw, x = cell - y * gw;
            const float aw = anc.wh[2 * a], ah = anc.wh[2 * a + 1];
            const float cx = __fmul_rn(__fadd_rn(__fsub_rn(__fmul_rn(sig[(int)p[0] + 128], 2.0f), 0.5f), (float)x), stride);
            const float cy = __fmul_rn(__fadd_rn(__fsub_rn(__fmul_rn(sig[(int)p[cstride] + 128], 2.0f), 0.5f), (float)y), stride);
            const float tw = __fmul_rn(sig[(int)p[2 * cstride] + 128], 2.0f), th = __fmul_rn(sig[(int)p[3 * cstride] + 128], 2.0f);
            const float w = __fmul_rn(__fmul_rn(tw, tw), aw), h = __fmul_rn(__fmul_rn(th, th), ah);
            const float hw = __fdiv_rn(w, 2.0f), hh = __fdiv_rn(h, 2.0f);
            mars_box_t d;
            d.x0 = __fsub_rn(cx, hw); d.y0 = __fsub_rn(cy, hh); d.x1 = __fadd_rn(cx, hw); d.y1 = __fadd_rn(cy, hh);
            d.confidence = conf; d.class_id = best;
            out[rank] = d;
        }
        cnt += total;
    }
    if (threadIdx.x == 0) counts[blockIdx.x] = min(cnt, maxd);
}

/* ---- NanoDet GFL heads (ours: the reference has no NanoDet code) --------------------------------------------------------
 * GFL decode of one level for every image of the launch: the head of image b is at head + b * img_stride, element (channel c, cell
 * p = y * gw + x) at c * cstride + p * pstride (NCHW: cstride = gh * gw, pstride = 1, so a warp reads each class plane across
 * adjacent x; NHWC: cstride = 1, pstride = C).  tab = sig[256] (sig[v+128] = 1/(1+expf(-(v*scale)))) then E[256] (E[d] =
 * expf(-(d*scale))), both from the host.  Per cell, every operation one float32 rounding:
 *   score = max_c sig[v_c], label = the first c with that score (floats compared: the table saturates); candidate when score >
 *   conf_thresh;
 *   side s (left, top, right, bottom): bins v_j (j = 0..R), e_j = E[vmax - v_j] (the softmax numerators), den = sum e_j and
 *   dist = sum j * (e_j / den), both in j order; distance = dist * stride;
 *   cx = (x + off) * stride; box (max(cx - l, 0), max(cy - t, 0), min(cx + r, net_w), min(cy + b, net_h)).
 * The distribution bins are read only for candidates.  Candidates go to boxes[b][...] in (y, x) order, ordered compaction after
 * the image's running count when `append` is set (else from 0), capped at maxd. */
/* one side's distance: the expectation of the softmax of its nb bins q[j * cstride], times the stride */
__device__ __forceinline__ float gfl_distance(const int8_t *q, int nb, int cstride, const float *E, float stride) {
    int vmax = q[0];
    for (int j = 1; j < nb; j++) vmax = max(vmax, (int)q[(size_t)j * cstride]);
    float den = E[vmax - q[0]];
    for (int j = 1; j < nb; j++) den = __fadd_rn(den, E[vmax - q[(size_t)j * cstride]]);
    float dist = 0.0f;
    for (int j = 0; j < nb; j++) dist = __fadd_rn(dist, __fmul_rn((float)j, __fdiv_rn(E[vmax - q[(size_t)j * cstride]], den)));
    return __fmul_rn(dist, stride);
}

__global__ void __launch_bounds__(256) k_gfl_decode(const int8_t *head, size_t img_stride, int gh, int gw, int nc, int reg_max, int cstride,
                                                    int pstride, const float *tab, float stride, float off, float net_w, float net_h,
                                                    float conf_thresh, int append, mars_box_t *boxes, int32_t *counts, int box_stride,
                                                    int maxd) {
    __shared__ int warp_sums[32];
    __shared__ float sig[256], E[256];
    const int8_t *hb = head + (size_t)blockIdx.x * img_stride;
    mars_box_t *out = boxes + (size_t)blockIdx.x * box_stride;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) { sig[i] = tab[i]; E[i] = tab[256 + i]; }
    const int P = gh * gw, nb = reg_max + 1;
    int cnt = append ? min(counts[blockIdx.x], maxd) : 0;
    __syncthreads(); /* the tables are in place and every thread has read the count before thread 0 rewrites it */
    for (int base = 0; base < P && cnt < maxd; base += blockDim.x) {
        const int cell = base + threadIdx.x;
        int pass = 0, label = 0;
        float score = 0.0f;
        const int8_t *p = hb + (size_t)cell * pstride;
        if (cell < P) {
            score = sig[(int)p[0] + 128];
            for (int c = 1; c < nc; c++) {
                const float s = sig[(int)p[(size_t)c * cstride] + 128];
                if (s > score) { score = s; label = c; }
            }
            pass = score > conf_thresh;
        }
        int total;
        const int rank = cnt + block_excl_scan(pass, &total, warp_sums);
        if (pass && rank < maxd) {
            const int8_t *q = p + (size_t)nc * cstride;
            const size_t side = (size_t)nb * cstride;
            const float dl = gfl_distance(q, nb, cstride, E, stride), dt = gfl_distance(q + side, nb, cstride, E, stride);
            const float dr = gfl_distance(q + 2 * side, nb, cstride, E, stride), db = gfl_distance(q + 3 * side, nb, cstride, E, stride);
            const int y = cell / gw, x = cell - y * gw;
            const float cx = __fmul_rn(__fadd_rn((float)x, off), stride), cy = __fmul_rn(__fadd_rn((float)y, off), stride);
            mars_box_t b;
            b.x0 = fmaxf(__fsub_rn(cx, dl), 0.0f); b.y0 = fmaxf(__fsub_rn(cy, dt), 0.0f);
            b.x1 = fminf(__fadd_rn(cx, dr), net_w); b.y1 = fminf(__fadd_rn(cy, db), net_h);
            b.confidence = score; b.class_id = label;
            out[rank] = b;
        }
        cnt += total;
    }
    if (threadIdx.x == 0) counts[blockIdx.x] = min(cnt, maxd);
}

/* Corner-box NMS of reference examples/yolo_detect.cpp:152-173 for every image of the launch, one CTA per image.
 *   order : descending confidence, equal confidences in input order, -0 == +0, NaN after every number: a block radix sort of
 *           (confidence key << 10 | input index), unique keys, so no stability question arises;
 *   test  : same class and IoU (iou_corner) > thresh, one row of a suppression bit matrix per sorted element (warp per row,
 *           lane per bit) in the image's global scratch, then the greedy walk (nms_walk);
 *   output: kept boxes in sorted order; for an image with a frame size (frames[b].x > 0 and frames[b].y > 0) the letterbox
 *           inverse is applied on the way out. */
#define NMSB_THREADS 256
#define NMSB_ITEMS (MARS_MAX_DETS / NMSB_THREADS)
struct NmsBatchShared {
    union {
        typename cub::BlockRadixSort<unsigned long long, NMSB_THREADS, NMSB_ITEMS>::TempStorage sort;
        struct { float x0[MARS_MAX_DETS], y0[MARS_MAX_DETS], x1[MARS_MAX_DETS], y1[MARS_MAX_DETS]; } box;
    };
    uint16_t order[MARS_MAX_DETS];
    int cls[MARS_MAX_DETS];
    unsigned removed[32];
    int removed_before[32];
};

/* the 32-bit sort key of a confidence: ascending key = descending confidence, -0 == +0 (a tie, as the comparison sort sees it),
 * NaN last */
__device__ __forceinline__ unsigned nms_conf_key(float c) {
    if (c != c) return 0xFFFFFFFFu;
    const unsigned b = __float_as_uint(__fadd_rn(c, 0.0f));
    const unsigned asc = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
    return ~asc;
}

/* The corner NMS of one image by one NMSB_THREADS block, shared by k_nms_corner_batch and k_merge_rois: input element j < n
 * (n <= MARS_MAX_DETS) is load(j), a mars_box_t; kept element r (sorted order) goes out as emit(r, box); the kept count to
 * *count_out.  mask = the image's NMS_SCRATCH_WORDS of global scratch. */
template <class Load, class Emit>
__device__ __forceinline__ void nms_corner_image(NmsBatchShared &sh, int n, float thresh, unsigned *mask, int32_t *count_out, Load load,
                                                 Emit emit) {
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    unsigned long long key[NMSB_ITEMS];
#pragma unroll
    for (int k = 0; k < NMSB_ITEMS; k++) {
        const int j = tid * NMSB_ITEMS + k;
        const unsigned u = j < n ? nms_conf_key(load(j).confidence) : 0xFFFFFFFFu; /* padding sorts last */
        key[k] = ((unsigned long long)u << 10) | (unsigned)j;
    }
    cub::BlockRadixSort<unsigned long long, NMSB_THREADS, NMSB_ITEMS>(sh.sort).Sort(key, 0, 42);
#pragma unroll
    for (int k = 0; k < NMSB_ITEMS; k++) sh.order[tid * NMSB_ITEMS + k] = (uint16_t)(key[k] & 1023u);
    __syncthreads(); /* the sort's storage is reused for the sorted boxes */
    for (int j = tid; j < n; j += NMSB_THREADS) {
        const mars_box_t b = load(sh.order[j]);
        sh.box.x0[j] = b.x0; sh.box.y0[j] = b.y0; sh.box.x1[j] = b.x1; sh.box.y1[j] = b.y1;
        sh.cls[j] = b.class_id;
    }
    __syncthreads();
    const int nwords = (n + 31) >> 5;
    for (int i = wid; i < n; i += NMSB_THREADS / 32) {
        mars_box_t a;
        a.x0 = sh.box.x0[i]; a.y0 = sh.box.y0[i]; a.x1 = sh.box.x1[i]; a.y1 = sh.box.y1[i];
        const int acls = sh.cls[i];
        for (int w = i >> 5; w < nwords; w++) {
            const int j = w * 32 + lane;
            bool sup = false;
            if (j > i && j < n && sh.cls[j] == acls) {
                mars_box_t b;
                b.x0 = sh.box.x0[j]; b.y0 = sh.box.y0[j]; b.x1 = sh.box.x1[j]; b.y1 = sh.box.y1[j];
                sup = iou_corner(a, b) > thresh;
            }
            const unsigned bits = __ballot_sync(0xffffffffu, sup);
            if (lane == 0) mask[i * 32 + w] = bits;
        }
    }
    __syncthreads();
    if (wid == 0) nms_publish_removed(nms_walk<8>(mask, n, lane), n, lane, sh.removed, sh.removed_before, count_out);
    __syncthreads();
    for (int j = tid; j < n; j += NMSB_THREADS) {
        const unsigned word = sh.removed[j >> 5];
        if ((word >> (j & 31)) & 1u) continue;
        emit(j - sh.removed_before[j >> 5] - __popc(word & ((1u << (j & 31)) - 1u)), load(sh.order[j]));
    }
}

__global__ void __launch_bounds__(NMSB_THREADS) k_nms_corner_batch(const mars_box_t *in_all, const int32_t *counts_in, mars_box_t *out_all,
                                                                  int32_t *counts_out, int box_stride, float thresh, unsigned *scratch,
                                                                  const int2 *frames, int net_w, int net_h) {
    __shared__ NmsBatchShared sh;
    const mars_box_t *in = in_all + (size_t)blockIdx.x * box_stride;
    mars_box_t *out = out_all + (size_t)blockIdx.x * box_stride;
    const int n = min(counts_in[blockIdx.x], MARS_MAX_DETS);
    const int2 fr = frames[blockIdx.x];
    const bool inv = fr.x > 0 && fr.y > 0;
    const Letterbox lb = inv ? letterbox_params(fr.x, fr.y, net_w, net_h) : Letterbox{1.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    nms_corner_image(sh, n, thresh, scratch + (size_t)blockIdx.x * NMS_SCRATCH_WORDS, &counts_out[blockIdx.x],
                     [in](int j) { return in[j]; },
                     [out, inv, &lb](int r, mars_box_t b) { out[r] = inv ? letterbox_inverse(b, lb) : b; });
}

/* ---- merge of the regions of a frame (mars_b200_merge_rois_resident) ----------------------------------------------------
 * The candidates of frame f are the kept boxes of its regions' slots, concatenated in region order, each shifted into frame
 * coordinates by its region's origin (one float add per coordinate).  The first MERGE_CAP of them by (confidence key, position
 * in the concatenation) are selected without materialising the union: a radix select over the 32-bit key, 8 bits per pass,
 * finds the key T of the MERGE_CAP-th; every candidate with a smaller key and the first ones equal to T (in concatenation order)
 * are compacted in concatenation order.  Compaction keeps that order, so the (key, position) sort of nms_corner_image over the
 * selection orders ties exactly as a stable sort of the whole union would.  One block per frame.
 *   tab: [n_frames + 1] region starts (frame f has regions [tab[f], tab[f + 1]) of the call), then (x, y) per region;
 *   boxes / counts: the kept boxes of the call's slots (region r in slot r), box_stride apart. */
#define MERGE_CAP HEAD_MAX_CAND
struct MergeShared {
    NmsBatchShared nms;
    int cand[MARS_MAX_DETS]; /* selected candidate: region << 10 | index in the region's slot */
    int warp_sums[32];
    unsigned hist[256];
    unsigned prefix;
    int need;
};

__global__ void __launch_bounds__(NMSB_THREADS) k_merge_rois(const mars_box_t *boxes, const int32_t *counts, int box_stride, const int *tab,
                                                            int n_frames, mars_box_t *out_all, int32_t *counts_out, float thresh, unsigned *scratch) {
    __shared__ MergeShared sh;
    const int f = blockIdx.x, tid = threadIdx.x;
    const int r0 = tab[f], r1 = tab[f + 1];
    const int *org = tab + n_frames + 1; /* (x, y) of region r at org[2r], org[2r + 1]: 4-byte aligned only */
    auto key_of = [&](int r, int k) { return nms_conf_key(boxes[(size_t)r * box_stride + k].confidence); };
    int total = 0;
    for (int r = r0; r < r1; r++) total += min(counts[r], MARS_MAX_DETS);
    /* select: candidates with key < thr, then the first `need` with key == thr */
    unsigned thr = 0xFFFFFFFFu;
    int need = 0x7FFFFFFF;
    if (total > MERGE_CAP) {
        unsigned prefix = 0u;
        need = MERGE_CAP;
        for (int shift = 24; shift >= 0; shift -= 8) {
            const unsigned hi = shift == 24 ? 0u : 0xFFFFFFFFu << (shift + 8);
            sh.hist[tid] = 0u;
            __syncthreads();
            for (int r = r0; r < r1; r++) {
                const int c = min(counts[r], MARS_MAX_DETS);
                for (int k = tid; k < c; k += NMSB_THREADS) {
                    const unsigned u = key_of(r, k);
                    if ((u & hi) == prefix) atomicAdd(&sh.hist[(u >> shift) & 255u], 1u);
                }
            }
            __syncthreads();
            const int h = (int)sh.hist[tid];
            int sum;
            const int before = block_excl_scan(h, &sum, sh.warp_sums);
            if (before < need && before + h >= need) { sh.prefix = prefix | ((unsigned)tid << shift); sh.need = need - before; }
            __syncthreads();
            prefix = sh.prefix;
            need = sh.need;
        }
        thr = prefix;
    }
    /* ordered compaction of the selection */
    int eq_seen = 0, taken = 0;
    for (int r = r0; r < r1; r++) {
        const int c = min(counts[r], MARS_MAX_DETS);
        for (int base = 0; base < c; base += NMSB_THREADS) {
            const int k = base + tid;
            const unsigned u = k < c ? key_of(r, k) : 0xFFFFFFFFu;
            const bool eq = k < c && u == thr;
            int n_eq, n_take;
            const int eq_rank = eq_seen + block_excl_scan(eq ? 1 : 0, &n_eq, sh.warp_sums);
            const bool take = k < c && (u < thr || (eq && eq_rank < need));
            const int pos = taken + block_excl_scan(take ? 1 : 0, &n_take, sh.warp_sums);
            if (take) sh.cand[pos] = (r << 10) | k;
            eq_seen += n_eq;
            taken += n_take;
        }
    }
    __syncthreads();
    mars_box_t *out = out_all + (size_t)f * MARS_MAX_DETS;
    nms_corner_image(
        sh.nms, taken, thresh, scratch + (size_t)f * NMS_SCRATCH_WORDS, &counts_out[f],
        [&](int j) {
            const int c = sh.cand[j], r = c >> 10;
            mars_box_t b = boxes[(size_t)r * box_stride + (c & 1023)];
            const float ox = (float)org[2 * r], oy = (float)org[2 * r + 1];
            b.x0 = __fadd_rn(b.x0, ox); b.y0 = __fadd_rn(b.y0, oy);
            b.x1 = __fadd_rn(b.x1, ox); b.y1 = __fadd_rn(b.y1, oy);
            return b;
        },
        [out](int r, mars_box_t b) { out[r] = b; });
}

} // namespace marsb200
