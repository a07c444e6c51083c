/*
 * track.cuh -- per-stream multi-object tracking on the device (ours; include/mars_b200.h, mars_b200_set_tracking).
 *
 *  k_track : one CTA per entry of a call.  Entry i is the next frame of stream streams[i]: its detections are the corner boxes
 *            boxes[i * box_stride ...], counts[i] of them (the kept boxes of a heads step, or a host upload); the stream's live
 *            tracks (at most MARS_B200_MAX_TRACKS, kept in track_id order) and its frame counter live in HBM between calls.
 * ByteTrack's schedule and Kalman filter with greedy matching, float32 with one rounding per operation: the definition is written
 * out in tests/track_oracle.c and the device equals it bit for bit.
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "postproc.cuh"

namespace marsb200 {

#define TRK_THREADS MARS_B200_MAX_TRACKS /* thread t owns live track t */
#define TRK_MAX_DETS HEAD_MAX_CAND      /* detections read per frame: the heads path keeps at most this many */
#define TRK_DPT ((TRK_MAX_DETS + TRK_THREADS - 1) / TRK_THREADS) /* detections per thread: thread t owns j = t + k * TRK_THREADS */

enum { TRK_TRACKED = 0, TRK_LOST = 1 };
enum { DET_NONE = 0, DET_HIGH = 1, DET_LOW = 2 };

/* one live track: the Kalman state (cx, cy, a, h and their velocities; per coordinate k the covariance block (p00, p01, p11)),
 * and what the last matched detection said */
struct TrackSlot {
    float mean[8];
    float p00[4], p01[4], p11[4];
    float conf;
    int32_t class_id, track_id, det_index, last, state, activated, pad;
};
/* per stream: frames seen, track IDs issued, live tracks (all zero = a fresh stream) */
struct TrackMeta {
    int32_t frame, issued, live, pad;
};

#define TRK_WP 0.05f
#define TRK_WV 0.00625f

/* measurement (cx, cy, a, h) of a corner box */
__device__ __forceinline__ void trk_measure(const mars_box_t &b, float z[4]) {
    const float w = __fsub_rn(b.x1, b.x0), h = __fsub_rn(b.y1, b.y0);
    z[0] = __fadd_rn(b.x0, __fdiv_rn(w, 2.0f));
    z[1] = __fadd_rn(b.y0, __fdiv_rn(h, 2.0f));
    z[2] = __fdiv_rn(w, h);
    z[3] = h;
}

/* corner box of a track's mean */
__device__ __forceinline__ mars_box_t trk_box(const TrackSlot &t) {
    mars_box_t b;
    const float w = __fmul_rn(t.mean[2], t.mean[3]);
    b.x0 = __fsub_rn(t.mean[0], __fdiv_rn(w, 2.0f));
    b.y0 = __fsub_rn(t.mean[1], __fdiv_rn(t.mean[3], 2.0f));
    b.x1 = __fadd_rn(b.x0, w);
    b.y1 = __fadd_rn(b.y0, t.mean[3]);
    b.confidence = t.conf;
    b.class_id = t.class_id;
    return b;
}

__device__ __forceinline__ void trk_initiate(TrackSlot &t, const float z[4]) {
    const float h = z[3];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const float sp = k == 2 ? 1e-2f : __fmul_rn(2.0f * TRK_WP, h), sv = k == 2 ? 1e-5f : __fmul_rn(10.0f * TRK_WV, h);
        t.mean[k] = z[k];
        t.mean[4 + k] = 0.0f;
        t.p00[k] = __fmul_rn(sp, sp);
        t.p01[k] = 0.0f;
        t.p11[k] = __fmul_rn(sv, sv);
    }
}

__device__ __forceinline__ void trk_predict(TrackSlot &t) {
    if (t.state == TRK_LOST) t.mean[7] = 0.0f;
    const float h = t.mean[3];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const float qp = k == 2 ? 1e-2f : __fmul_rn(TRK_WP, h), qv = k == 2 ? 1e-5f : __fmul_rn(TRK_WV, h);
        t.mean[k] = __fadd_rn(t.mean[k], t.mean[4 + k]);
        const float s = __fadd_rn(t.p01[k], t.p11[k]);
        t.p00[k] = __fadd_rn(__fadd_rn(__fadd_rn(t.p00[k], t.p01[k]), s), __fmul_rn(qp, qp));
        t.p01[k] = s;
        t.p11[k] = __fadd_rn(t.p11[k], __fmul_rn(qv, qv));
    }
}

__device__ __forceinline__ void trk_update(TrackSlot &t, const float z[4]) {
    const float h = t.mean[3];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const float r = k == 2 ? 1e-1f : __fmul_rn(TRK_WP, h);
        const float p00 = t.p00[k], p01 = t.p01[k], p11 = t.p11[k];
        const float S = __fadd_rn(p00, __fmul_rn(r, r)), K0 = __fdiv_rn(p00, S), K1 = __fdiv_rn(p01, S), y = __fsub_rn(z[k], t.mean[k]);
        t.mean[k] = __fadd_rn(t.mean[k], __fmul_rn(K0, y));
        t.mean[4 + k] = __fadd_rn(t.mean[4 + k], __fmul_rn(K1, y));
        t.p00[k] = __fsub_rn(p00, __fmul_rn(K0, p00));
        t.p01[k] = __fsub_rn(p01, __fmul_rn(K0, p01));
        t.p11[k] = __fsub_rn(p11, __fmul_rn(K1, p01));
    }
}

struct TrackShared {
    mars_box_t det[TRK_MAX_DETS];      /* the frame's detections */
    int16_t dmatch[TRK_MAX_DETS];      /* matched track index, -1 */
    uint8_t dcat[TRK_MAX_DETS];        /* DET_NONE / HIGH / LOW */
    float4 tbox[MARS_B200_MAX_TRACKS]; /* track boxes (predicted for the pool) */
    int tcls[MARS_B200_MAX_TRACKS];
    int16_t tmatch[MARS_B200_MAX_TRACKS]; /* matched detection, -1 */
    uint8_t trole[MARS_B200_MAX_TRACKS];  /* 1: pool Tracked, 2: pool Lost, 3: unconfirmed */
    unsigned long long tkey[MARS_B200_MAX_TRACKS]; /* best pair of a track in a round: sim bits << 32 | ~j */
    int warp_sums[32];
};

/* Greedy matching of the tracks with role in roles (bit mask) x the free detections of category cat, similarity IoU (* conf
 * when with_conf), gate g, as rounds of locally dominant pairs: every free track finds its best free admissible detection (larger
 * similarity, then smaller j), every free detection its best free admissible track (larger similarity, then smaller track index =
 * smaller track_id), and mutual choices are matched.  The order on pairs is strict, so each round matches the pairs the literal
 * greedy loop would take next in some order, and the result is the literal loop's. */
__device__ __forceinline__ void trk_match(TrackShared &sh, int nt, int nd, unsigned roles, int cat, bool with_conf, float g, bool class_aware) {
    const int tid = threadIdx.x, lane = tid & 31;
    for (;;) {
        if (tid < nt) sh.tkey[tid] = 0ull;
        __syncthreads();
        unsigned dbs[TRK_DPT];
        int dbt[TRK_DPT];
#pragma unroll
        for (int k = 0; k < TRK_DPT; k++) { dbs[k] = 0u; dbt[k] = -1; }
        for (int t = 0; t < nt; t++) {
            if (!((roles >> sh.trole[t]) & 1u) || sh.tmatch[t] >= 0) continue; /* uniform */
            const float4 q = sh.tbox[t];
            mars_box_t a;
            a.x0 = q.x; a.y0 = q.y; a.x1 = q.z; a.y1 = q.w;
            const int tc = sh.tcls[t];
            unsigned long long best = 0ull;
#pragma unroll
            for (int k = 0; k < TRK_DPT; k++) {
                const int j = tid + k * TRK_THREADS;
                if (j >= nd || sh.dcat[j] != cat || sh.dmatch[j] >= 0) continue;
                const mars_box_t &b = sh.det[j];
                if (class_aware && b.class_id != tc) continue;
                const float iou = iou_corner(a, b);
                const float sim = with_conf ? __fmul_rn(iou, b.confidence) : iou;
                if (!(sim > g)) continue; /* g >= 0: an admissible similarity is positive, its bits order like the float */
                const unsigned sb = __float_as_uint(sim);
                if (sb > dbs[k]) { dbs[k] = sb; dbt[k] = t; }
                const unsigned long long key = ((unsigned long long)sb << 32) | (0xFFFFFFFFu - (unsigned)j);
                if (key > best) best = key;
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                const unsigned long long o = __shfl_xor_sync(0xffffffffu, best, d);
                if (o > best) best = o;
            }
            if (lane == 0 && best) atomicMax(&sh.tkey[t], best);
        }
        __syncthreads();
        int matched = 0;
#pragma unroll
        for (int k = 0; k < TRK_DPT; k++) {
            const int j = tid + k * TRK_THREADS;
            if (dbt[k] >= 0 && (unsigned)(sh.tkey[dbt[k]] & 0xFFFFFFFFull) == 0xFFFFFFFFu - (unsigned)j) {
                sh.dmatch[j] = (int16_t)dbt[k];
                sh.tmatch[dbt[k]] = (int16_t)j;
                matched = 1;
            }
        }
        if (!__syncthreads_or(matched)) break;
    }
}

/* blockDim.x = TRK_THREADS.  out: [out_stride] records per entry, out_counts: one per entry */
__global__ void __launch_bounds__(TRK_THREADS) k_track(const mars_box_t *boxes, const int32_t *counts, int box_stride, const int32_t *streams,
                                                       TrackSlot *table, TrackMeta *meta, mars_b200_track_params_t p,
                                                       mars_b200_track_box_t *out_all, int32_t *out_counts, int out_stride) {
    __shared__ TrackShared sh;
    const int tid = threadIdx.x, e = blockIdx.x;
    const int s = streams[e];
    const TrackMeta m = meta[s];
    const int frame = m.frame + 1, nt = m.live;
    TrackSlot *tab = table + (size_t)s * MARS_B200_MAX_TRACKS;
    const mars_box_t *in = boxes + (size_t)e * box_stride;
    const int nd = max(0, min(counts[e], TRK_MAX_DETS));
    /* the detections and their classes */
    for (int j = tid; j < nd; j += TRK_THREADS) {
        const mars_box_t b = in[j];
        const bool ok = isfinite(b.x0) && isfinite(b.y0) && isfinite(b.x1) && isfinite(b.y1) && isfinite(b.confidence) &&
                        __fsub_rn(b.x1, b.x0) > 0.0f && __fsub_rn(b.y1, b.y0) > 0.0f;
        sh.det[j] = b;
        sh.dcat[j] = !ok ? DET_NONE : b.confidence > p.high_thresh ? DET_HIGH : (b.confidence > p.low_thresh && b.confidence < p.high_thresh) ? DET_LOW : DET_NONE;
        sh.dmatch[j] = -1;
    }
    /* the stream's tracks: the pool is predicted */
    TrackSlot tr;
    const bool have = tid < nt;
    int role = 0;
    if (have) {
        tr = tab[tid];
        role = tr.state == TRK_LOST ? 2 : tr.activated ? 1 : 3;
        if (role != 3) trk_predict(tr);
        const mars_box_t b = trk_box(tr);
        sh.tbox[tid] = make_float4(b.x0, b.y0, b.x1, b.y1);
        sh.tcls[tid] = tr.class_id;
        sh.tmatch[tid] = -1;
        sh.trole[tid] = (uint8_t)role;
    }
    __syncthreads();
    const bool ca = p.class_aware != 0;
    trk_match(sh, nt, nd, (1u << 1) | (1u << 2), DET_HIGH, true, p.sim_high, ca); /* stage 1: the pool x high */
    trk_match(sh, nt, nd, 1u << 1, DET_LOW, false, p.sim_low, ca);                /* stage 2: unmatched Tracked x low */
    trk_match(sh, nt, nd, 1u << 3, DET_HIGH, true, p.sim_unconfirmed, ca);        /* stage 3: unconfirmed x remaining high */
    /* the tracks' outcomes: keep5 = alive after the unconfirmed removal, keep = alive after the lost expiry */
    int keep5 = 0, keep = 0, shown = 0;
    if (have) {
        const int j = sh.tmatch[tid];
        if (j >= 0) {
            const mars_box_t &b = sh.det[j];
            float z[4];
            trk_measure(b, z);
            trk_update(tr, z);
            tr.state = TRK_TRACKED;
            tr.activated = 1;
            tr.conf = b.confidence;
            tr.class_id = b.class_id;
            tr.det_index = j;
            tr.last = frame;
        } else if (role == 1) {
            tr.state = TRK_LOST;
        }
        keep5 = j >= 0 || role != 3;
        keep = keep5 && !(tr.state == TRK_LOST && frame - tr.last > p.max_lost);
        shown = keep && tr.state == TRK_TRACKED && tr.activated;
    }
    int live5, kept, nshown;
    block_excl_scan(keep5, &live5, sh.warp_sums);
    const int rank = block_excl_scan(keep, &kept, sh.warp_sums);
    const int orank = block_excl_scan(shown, &nshown, sh.warp_sums);
    /* every thread holds its own track in registers and has passed the scans' barriers: the table can be rewritten in place */
    mars_b200_track_box_t *out = out_all + (size_t)e * out_stride;
    if (keep) tab[rank] = tr;
    if (shown) {
        const mars_box_t b = trk_box(tr);
        out[orank] = mars_b200_track_box_t{b.x0, b.y0, b.x1, b.y1, tr.conf, tr.class_id, tr.track_id, tr.det_index};
    }
    /* births: the unmatched high detections with conf >= new_thresh in j order, while fewer than MARS_B200_MAX_TRACKS are live */
    const int room = MARS_B200_MAX_TRACKS - live5;
    int born = 0;
#pragma unroll
    for (int k = 0; k < TRK_DPT; k++) {
        const int j = tid + k * TRK_THREADS;
        const bool nb = j < nd && sh.dcat[j] == DET_HIGH && sh.dmatch[j] < 0 && sh.det[j].confidence >= p.new_thresh;
        int total;
        const int r = born + block_excl_scan(nb ? 1 : 0, &total, sh.warp_sums);
        if (nb && r < room) {
            const mars_box_t &b = sh.det[j];
            TrackSlot t;
            float z[4];
            trk_measure(b, z);
            trk_initiate(t, z);
            t.conf = b.confidence;
            t.class_id = b.class_id;
            t.track_id = m.issued + 1 + r;
            t.det_index = j;
            t.last = frame;
            t.state = TRK_TRACKED;
            t.activated = frame == 1;
            t.pad = 0;
            tab[kept + r] = t;
            if (t.activated) {
                const mars_box_t q = trk_box(t);
                out[nshown + r] = mars_b200_track_box_t{q.x0, q.y0, q.x1, q.y1, t.conf, t.class_id, t.track_id, j};
            }
        }
        born += total;
    }
    born = min(born, max(room, 0));
    if (tid == 0) {
        meta[s] = TrackMeta{frame, m.issued + born, kept + born, 0};
        out_counts[e] = nshown + (frame == 1 ? born : 0);
    }
}

} // namespace marsb200
