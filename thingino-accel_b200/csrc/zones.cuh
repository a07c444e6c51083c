/*
 * zones.cuh -- line crossings, zone occupancy and zone events of tracked camera streams (ours; include/mars_b200.h,
 * mars_b200_set_zones).
 *
 *  k_zones : one CTA per entry of a tracker call, right after k_track on the compute stream.  Entry i is the frame k_track just
 *            processed for stream streams[i]: the stream's live track IDs (k_track's table, in track_id order), the entry's shown
 *            tracks (k_track's records, in track_id order), the stream's geometry, and its analytics state in HBM: at most
 *            MARS_B200_MAX_TRACKS ZoneTrack entries in track_id order and the line totals.
 * Float32 with one rounding per operation: the definition is written out in tests/zones_oracle.c and the device equals it byte for
 * byte.
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "track.cuh"

namespace marsb200 {

#define ZN_THREADS MARS_B200_MAX_TRACKS /* thread t owns old state entry t and shown record t */

/* the geometry of one stream (n_zones = n_lines = 0: analytics off) */
struct ZoneGeom {
    int32_t n_zones, n_lines, pad[2];
    mars_b200_zone_t zone[MARS_B200_MAX_ZONES];
    mars_b200_line_t line[MARS_B200_MAX_LINES];
};
/* the analytics state of one track that has been shown (64 bytes) */
struct ZoneTrack {
    int32_t track_id, class_id;          /* class at its last shown frame */
    float x0, y0, x1, y1;                /* tracked box at its last shown frame */
    uint32_t sigma;                      /* bit l: sigma of line l is +1; bit 8 + l: it is -1 */
    uint32_t zmask;                      /* bit z: inside zone z; bit 8 + z: DWELL emitted in this stay */
    int32_t entry[MARS_B200_MAX_ZONES];  /* entry frame per zone */
};
static_assert(sizeof(ZoneTrack) == 64, "ZoneTrack layout");
static_assert(sizeof(mars_b200_zone_frame_t) == 2152 && sizeof(mars_b200_zone_event_t) == 16, "zone record layout");
/* per stream: state entries, line totals */
struct ZoneMeta {
    int32_t n, pad[3];
    int32_t pos[MARS_B200_MAX_LINES], neg[MARS_B200_MAX_LINES];
};

__device__ __forceinline__ void zn_anchor(float x0, float y0, float x1, float y1, int anchor, float &px, float &py) {
    px = __fmul_rn(__fadd_rn(x0, x1), 0.5f);
    py = anchor == MARS_B200_ANCHOR_CENTRE ? __fmul_rn(__fadd_rn(y0, y1), 0.5f) : y1;
}

/* crossing number, even-odd rule */
__device__ __forceinline__ bool zn_inside(const mars_b200_zone_t &z, float px, float py) {
    bool c = false;
    for (int i = 0, n = z.n_verts; i < n; i++) {
        const int j = i ? i - 1 : n - 1;
        const float xi = z.x[i], yi = z.y[i], xj = z.x[j], yj = z.y[j];
        if ((yi > py) != (yj > py) && px < __fadd_rn(xi, __fdiv_rn(__fmul_rn(__fsub_rn(xj, xi), __fsub_rn(py, yi)), __fsub_rn(yj, yi)))) c = !c;
    }
    return c;
}

__device__ __forceinline__ int zn_side(const mars_b200_line_t &l, float px, float py) {
    const float v = __fsub_rn(__fmul_rn(__fsub_rn(l.x1, l.x0), __fsub_rn(py, l.y0)), __fmul_rn(__fsub_rn(l.y1, l.y0), __fsub_rn(px, l.x0)));
    return (v > 0.0f) - (v < 0.0f);
}

/* the step p -> q meets the closed segment a b: o_a and o_b are not both strictly of one sign */
__device__ __forceinline__ bool zn_meets(const mars_b200_line_t &l, float px, float py, float qx, float qy) {
    const float dx = __fsub_rn(qx, px), dy = __fsub_rn(qy, py);
    const float oa = __fsub_rn(__fmul_rn(dx, __fsub_rn(l.y0, py)), __fmul_rn(dy, __fsub_rn(l.x0, px)));
    const float ob = __fsub_rn(__fmul_rn(dx, __fsub_rn(l.y1, py)), __fmul_rn(dy, __fsub_rn(l.x1, px)));
    return !((oa > 0.0f && ob > 0.0f) || (oa < 0.0f && ob < 0.0f));
}

__device__ __forceinline__ bool zn_class(int geom_class, int cls) { return geom_class == -1 || geom_class == cls; }

/* a shown frame of a track (z: its state, fresh when first); the crossing, ENTER, DWELL and EXIT masks of this frame */
struct ZoneHits {
    uint32_t cp = 0, cn = 0, enter = 0, dwell = 0, exit = 0;
    __device__ int count() const { return __popc(cp) + __popc(cn) + __popc(enter) + __popc(dwell) + __popc(exit); }
};
__device__ __forceinline__ ZoneHits zn_shown(ZoneTrack &z, const mars_b200_track_box_t &r, const ZoneGeom &g, int frame, bool first,
                                            int *occ) {
    ZoneHits h;
    const int cls = r.class_id;
    /* the loops run to the limits so that the per-zone state stays in registers */
#pragma unroll
    for (int l = 0; l < MARS_B200_MAX_LINES; l++) {
        if (l >= g.n_lines) break;
        const mars_b200_line_t &L = g.line[l];
        float px, py, qx, qy;
        zn_anchor(z.x0, z.y0, z.x1, z.y1, L.anchor, px, py);
        zn_anchor(r.x0, r.y0, r.x1, r.y1, L.anchor, qx, qy);
        const int sq = zn_side(L, qx, qy);
        const int sig = (z.sigma >> l) & 1u ? 1 : (z.sigma >> (8 + l)) & 1u ? -1 : 0;
        if (!first && sq != 0 && sig == -sq && zn_class(L.class_id, cls) && zn_meets(L, px, py, qx, qy)) {
            if (sq > 0) h.cp |= 1u << l; else h.cn |= 1u << l;
        }
        if (sq != 0) z.sigma = (z.sigma & ~((1u << l) | (1u << (8 + l)))) | (sq > 0 ? 1u << l : 1u << (8 + l));
    }
#pragma unroll
    for (int k = 0; k < MARS_B200_MAX_ZONES; k++) {
        if (k >= g.n_zones) break;
        const mars_b200_zone_t &Z = g.zone[k];
        float qx, qy;
        zn_anchor(r.x0, r.y0, r.x1, r.y1, Z.anchor, qx, qy);
        const bool now = zn_class(Z.class_id, cls) && zn_inside(Z, qx, qy);
        const bool was = (z.zmask >> k) & 1u;
        if (now && !was) {
            h.enter |= 1u << k;
            z.entry[k] = frame;
            z.zmask = (z.zmask | (1u << k)) & ~(1u << (8 + k));
        }
        if (now && Z.min_dwell > 0 && !((z.zmask >> (8 + k)) & 1u) && frame - z.entry[k] + 1 >= Z.min_dwell) {
            h.dwell |= 1u << k;
            z.zmask |= 1u << (8 + k);
        }
        if (!now && was) {
            h.exit |= 1u << k;
            z.zmask &= ~((1u << k) | (1u << (8 + k)));
        }
        if (now) atomicAdd(&occ[k], 1);
    }
    z.class_id = cls;
    z.x0 = r.x0; z.y0 = r.y0; z.x1 = r.x1; z.y1 = r.y1;
    return h;
}

__device__ __forceinline__ int zn_lower_bound(const int32_t *a, int n, int x) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a[mid] < x) lo = mid + 1; else hi = mid;
    }
    return lo;
}

struct ZoneShared {
    ZoneGeom g;
    int32_t lid[MARS_B200_MAX_TRACKS];       /* live track IDs */
    int32_t sid[MARS_B200_MAX_TRACKS];       /* shown track IDs */
    int32_t oid[MARS_B200_MAX_TRACKS];       /* IDs of the old state entries */
    int32_t nid[MARS_B200_MAX_TRACKS];       /* IDs of the new entries, compacted */
    int32_t kpre[MARS_B200_MAX_TRACKS + 1];  /* survivors among old entries [0, i) */
    int32_t ev[2 * MARS_B200_MAX_TRACKS];    /* event counts, then offsets, in merged (track_id) order */
    int32_t occ[MARS_B200_MAX_ZONES];
    int32_t wcross[ZN_THREADS / 32][2 * MARS_B200_MAX_LINES]; /* crossings per warp of old entries: +1 per line, then -1 */
    int32_t tot[2 * MARS_B200_MAX_LINES];                     /* line totals before this frame: +1 per line, then -1 */
    int warp_sums[32];
};

/* blockDim.x = ZN_THREADS.  geom / state / zmeta null: no stream has geometry; out null: no records */
__global__ void __launch_bounds__(ZN_THREADS) k_zones(const int32_t *streams, const TrackSlot *table, const TrackMeta *meta,
                                                      const mars_b200_track_box_t *shown_all, const int32_t *shown_counts, int shown_stride,
                                                      const ZoneGeom *geom, ZoneTrack *state, ZoneMeta *zmeta, mars_b200_zone_frame_t *out_all) {
    __shared__ ZoneShared sh;
    const int tid = threadIdx.x, e = blockIdx.x, lane = tid & 31, wid = tid >> 5;
    const int s = streams[e];
    const TrackMeta tm = meta[s];
    const int frame = tm.frame;
    mars_b200_zone_frame_t *out = out_all ? out_all + e : nullptr;
    const bool on = geom && (geom[s].n_zones > 0 || geom[s].n_lines > 0);
    if (!on) {
        if (out) {
            if (tid < MARS_B200_MAX_ZONE_EVENTS) out->events[tid] = mars_b200_zone_event_t{0, 0, 0, 0, 0};
            if (tid < 2 + MARS_B200_MAX_ZONES + 2 * MARS_B200_MAX_LINES) (&out->frame)[tid] = tid == 0 ? frame : 0;
        }
        return;
    }
    {
        const int *src = reinterpret_cast<const int *>(geom + s);
        int *dst = reinterpret_cast<int *>(&sh.g);
        for (int i = tid; i < (int)(sizeof(ZoneGeom) / 4); i += ZN_THREADS) dst[i] = src[i];
    }
    const int n_old = zmeta[s].n;
    if (tid < 2 * MARS_B200_MAX_LINES) sh.tot[tid] = tid < MARS_B200_MAX_LINES ? zmeta[s].pos[tid] : zmeta[s].neg[tid - MARS_B200_MAX_LINES];
    ZoneTrack *st = state + (size_t)s * MARS_B200_MAX_TRACKS;
    const mars_b200_track_box_t *shown = shown_all + (size_t)e * shown_stride;
    const int n_live = tm.live, n_shown = max(0, min(shown_counts[e], MARS_B200_MAX_TRACKS));
    if (tid < n_live) sh.lid[tid] = table[(size_t)s * MARS_B200_MAX_TRACKS + tid].track_id;
    mars_b200_track_box_t r;
    if (tid < n_shown) { r = shown[tid]; sh.sid[tid] = r.track_id; }
    ZoneTrack o;
    const bool has_old = tid < n_old;
    if (has_old) { o = st[tid]; sh.oid[tid] = o.track_id; }
    if (tid < MARS_B200_MAX_ZONES) sh.occ[tid] = 0;
    __syncthreads();
    const ZoneGeom &g = sh.g;
    /* old entry tid: removed, shown (record si) or unchanged; shown record tid: new when it has no state */
    bool removed = false;
    int si = -1;
    if (has_old) {
        const int a = zn_lower_bound(sh.lid, n_live, o.track_id);
        removed = !(a < n_live && sh.lid[a] == o.track_id);
        const int b = zn_lower_bound(sh.sid, n_shown, o.track_id);
        if (b < n_shown && sh.sid[b] == o.track_id) si = b;
    }
    int lbo = 0;
    bool has_new = false;
    if (tid < n_shown) {
        lbo = zn_lower_bound(sh.oid, n_old, r.track_id);
        has_new = !(lbo < n_old && sh.oid[lbo] == r.track_id);
    }
    const bool keep = has_old && !removed;
    int n_new, n_keep;
    const int nrank = block_excl_scan(has_new ? 1 : 0, &n_new, sh.warp_sums);
    const int krank = block_excl_scan(keep ? 1 : 0, &n_keep, sh.warp_sums);
    if (has_new) sh.nid[nrank] = r.track_id;
    if (tid < n_old) sh.kpre[tid] = krank;
    if (tid == 0) sh.kpre[n_old] = n_keep;
    /* this frame's decisions */
    ZoneHits ho, hn;
    uint32_t gone = 0;
    int cls_old = has_old ? o.class_id : 0;
    if (keep && si >= 0) {
        ho = zn_shown(o, shown[si], g, frame, false, sh.occ);
        cls_old = o.class_id;
    } else if (removed) {
        gone = o.zmask & ((1u << g.n_zones) - 1u);
    }
    ZoneTrack nw;
    if (has_new) {
        nw.track_id = r.track_id;
        nw.x0 = r.x0; nw.y0 = r.y0; nw.x1 = r.x1; nw.y1 = r.y1;
        nw.sigma = 0u;
        nw.zmask = 0u;
#pragma unroll
        for (int k = 0; k < MARS_B200_MAX_ZONES; k++) nw.entry[k] = 0;
        hn = zn_shown(nw, r, g, frame, true, sh.occ);
    }
    /* crossings per warp (only old entries cross) */
    const int nl = g.n_lines, nz = g.n_zones;
    for (int l = 0; l < nl; l++) {
        const unsigned bp = __ballot_sync(0xffffffffu, (ho.cp >> l) & 1u), bn = __ballot_sync(0xffffffffu, (ho.cn >> l) & 1u);
        if (lane == 0) { sh.wcross[wid][l] = __popc(bp); sh.wcross[wid][MARS_B200_MAX_LINES + l] = __popc(bn); }
    }
    __syncthreads(); /* nid, kpre, wcross, occ complete */
    /* merged (track_id) order of old and new entries: positions, then offsets of their events */
    const int p_old = has_old ? tid + zn_lower_bound(sh.nid, n_new, o.track_id) : -1;
    const int p_new = has_new ? nrank + lbo : -1;
    const int c_old = has_old ? ho.count() + __popc(gone) : 0, c_new = has_new ? hn.count() : 0;
    if (has_old) sh.ev[p_old] = c_old;
    if (has_new) sh.ev[p_new] = c_new;
    const int n_merged = n_old + n_new;
    __syncthreads();
    const int v0 = 2 * tid < n_merged ? sh.ev[2 * tid] : 0, v1 = 2 * tid + 1 < n_merged ? sh.ev[2 * tid + 1] : 0;
    int n_events;
    const int base = block_excl_scan(v0 + v1, &n_events, sh.warp_sums);
    if (2 * tid < n_merged) sh.ev[2 * tid] = base;
    if (2 * tid + 1 < n_merged) sh.ev[2 * tid + 1] = base + v0;
    __syncthreads();
    /* the events */
    auto put = [&](int k, int id, int cls, int kind, int index, int value) {
        if (out && k < MARS_B200_MAX_ZONE_EVENTS) out->events[k] = mars_b200_zone_event_t{id, cls, (int16_t)kind, (int16_t)index, value};
    };
    int ko = has_old ? sh.ev[p_old] : 0;
    for (int l = 0; l < nl; l++) {
        const unsigned lt = (1u << lane) - 1u;
        const unsigned bp = __ballot_sync(0xffffffffu, (ho.cp >> l) & 1u), bn = __ballot_sync(0xffffffffu, (ho.cn >> l) & 1u);
        if ((ho.cp | ho.cn) >> l & 1u) {
            const bool pos = (ho.cp >> l) & 1u;
            const int col = (pos ? 0 : MARS_B200_MAX_LINES) + l;
            int before = sh.tot[col];
            for (int w = 0; w < wid; w++) before += sh.wcross[w][col];
            put(ko++, o.track_id, cls_old, pos ? MARS_B200_CROSS_POS : MARS_B200_CROSS_NEG, l, before + __popc((pos ? bp : bn) & lt) + 1);
        }
    }
    auto zone_events = [&](int k0, const ZoneTrack &z, const ZoneHits &h, uint32_t gone_mask, bool first) {
        int k = k0;
#pragma unroll
        for (int q = 0; q < MARS_B200_MAX_ZONES; q++) {
            if (q >= nz) break;
            if ((h.enter >> q) & 1u) put(k++, z.track_id, z.class_id, MARS_B200_ZONE_ENTER, q, first ? 1 : 0);
            if ((h.dwell >> q) & 1u) put(k++, z.track_id, z.class_id, MARS_B200_ZONE_DWELL, q, frame - z.entry[q] + 1);
            if ((h.exit >> q) & 1u) put(k++, z.track_id, z.class_id, MARS_B200_ZONE_EXIT, q, frame - z.entry[q]);
            if ((gone_mask >> q) & 1u) put(k++, z.track_id, z.class_id, MARS_B200_ZONE_GONE, q, frame - z.entry[q]);
        }
    };
    if (has_old) zone_events(ko, o, ho, gone, false);
    if (has_new) zone_events(sh.ev[p_new], nw, hn, 0u, true);
    /* the record */
    if (out) {
        if (tid >= n_events && tid < MARS_B200_MAX_ZONE_EVENTS) out->events[tid] = mars_b200_zone_event_t{0, 0, 0, 0, 0};
        if (tid == 0) { out->frame = frame; out->n_events = n_events; }
        if (tid < MARS_B200_MAX_ZONES) out->occupancy[tid] = tid < nz ? sh.occ[tid] : 0;
    }
    if (tid < 2 * MARS_B200_MAX_LINES) {
        const int l = tid & (MARS_B200_MAX_LINES - 1), neg = tid >= MARS_B200_MAX_LINES;
        int total = 0;
        if (l < nl) {
            total = sh.tot[tid];
            for (int w = 0; w < ZN_THREADS / 32; w++) total += sh.wcross[w][tid];
        }
        if (out) (neg ? out->crossed_neg : out->crossed_pos)[l] = total;
        (neg ? zmeta[s].neg : zmeta[s].pos)[l] = total;
    }
    if (tid == 0) zmeta[s].n = n_keep + n_new;
    /* the new state in track_id order, in place: every thread holds its entries in registers and has passed the barriers */
    if (keep) st[krank + zn_lower_bound(sh.nid, n_new, o.track_id)] = o;
    if (has_new) st[nrank + sh.kpre[lbo]] = nw;
}

} // namespace marsb200
