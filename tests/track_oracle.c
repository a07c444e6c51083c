/*
 * tests/track_oracle.c -- TEST INFRASTRUCTURE: the C statement of the multi-object tracker that k_track (track.cuh) is checked
 * against, one stream at a time.
 *
 * The tracker is this library's own definition (include/mars_b200.h, mars_b200_set_tracking): ByteTrack's schedule and Kalman
 * filter (Zhang et al., ECCV 2022) with greedy matching under a strict total order instead of an optimal assignment.  Everything
 * is written the literal way: the greedy matching takes the best admissible pair again and again.  float32, one rounding per
 * operation, left to right as written; tests/track_ref.py compiles this file with -ffp-contract=off into a temporary directory.
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

#define MAX_TRACKS 256
#define MAX_DETS 1000
#define WP 0.05f
#define WV 0.00625f
enum { TRACKED = 0, LOST = 1 };
enum { NONE = 0, HIGH = 1, LOW = 2 };

typedef struct { float x0, y0, x1, y1, confidence; int32_t class_id; } box_t;
typedef struct { float x0, y0, x1, y1, confidence; int32_t class_id, track_id, det_index; } track_box_t;
typedef struct { float high_thresh, low_thresh, new_thresh, sim_high, sim_low, sim_unconfirmed; int32_t max_lost, class_aware; } params_t;
typedef struct {
    float mean[8]; /* cx, cy, a, h, then their velocities */
    float p00[4], p01[4], p11[4];
    float conf;
    int32_t class_id, track_id, det_index, last, state, activated;
} track_t;
/* one stream; all zero = fresh (frame 0, no ID issued) */
typedef struct {
    int32_t frame, issued, live;
    track_t t[MAX_TRACKS]; /* the live tracks in track_id order */
} stream_t;

int trk_stream_bytes(void) { return (int)sizeof(stream_t); }

/* iou_corner of postproc.cuh (reference examples/yolo_detect.cpp:138-149) */
static float iou_corner(box_t a, box_t b) {
    float x0 = fmaxf(a.x0, b.x0), y0 = fmaxf(a.y0, b.y0), x1 = fminf(a.x1, b.x1), y1 = fminf(a.y1, b.y1);
    float inter = fmaxf(0.0f, x1 - x0) * fmaxf(0.0f, y1 - y0);
    float aa = (a.x1 - a.x0) * (a.y1 - a.y0);
    float ab = (b.x1 - b.x0) * (b.y1 - b.y0);
    return inter / (aa + ab - inter + 1e-6f);
}

static void measure(const box_t *b, float z[4]) {
    float w = b->x1 - b->x0, h = b->y1 - b->y0;
    z[0] = b->x0 + w / 2.0f;
    z[1] = b->y0 + h / 2.0f;
    z[2] = w / h;
    z[3] = h;
}

static box_t track_box(const track_t *t) {
    box_t b;
    float w = t->mean[2] * t->mean[3];
    b.x0 = t->mean[0] - w / 2.0f;
    b.y0 = t->mean[1] - t->mean[3] / 2.0f;
    b.x1 = b.x0 + w;
    b.y1 = b.y0 + t->mean[3];
    b.confidence = t->conf;
    b.class_id = t->class_id;
    return b;
}

static void initiate(track_t *t, const float z[4]) {
    float h = z[3];
    for (int k = 0; k < 4; k++) {
        float sp = k == 2 ? 1e-2f : (2.0f * WP) * h, sv = k == 2 ? 1e-5f : (10.0f * WV) * h;
        t->mean[k] = z[k];
        t->mean[4 + k] = 0.0f;
        t->p00[k] = sp * sp;
        t->p01[k] = 0.0f;
        t->p11[k] = sv * sv;
    }
}

static void predict(track_t *t) {
    if (t->state == LOST) t->mean[7] = 0.0f;
    float h = t->mean[3];
    for (int k = 0; k < 4; k++) {
        float qp = k == 2 ? 1e-2f : WP * h, qv = k == 2 ? 1e-5f : WV * h;
        t->mean[k] = t->mean[k] + t->mean[4 + k];
        float s = t->p01[k] + t->p11[k];
        t->p00[k] = t->p00[k] + t->p01[k] + s + qp * qp;
        t->p01[k] = s;
        t->p11[k] = t->p11[k] + qv * qv;
    }
}

static void update(track_t *t, const float z[4]) {
    float h = t->mean[3];
    for (int k = 0; k < 4; k++) {
        float r = k == 2 ? 1e-1f : WP * h;
        float p00 = t->p00[k], p01 = t->p01[k], p11 = t->p11[k];
        float S = p00 + r * r, K0 = p00 / S, K1 = p01 / S, y = z[k] - t->mean[k];
        t->mean[k] = t->mean[k] + K0 * y;
        t->mean[4 + k] = t->mean[4 + k] + K1 * y;
        t->p00[k] = p00 - K0 * p00;
        t->p01[k] = p01 - K0 * p01;
        t->p11[k] = p11 - K1 * p01;
    }
}

/* the literal greedy matching: tin[t] / din[j] mark the two sets, tm / dm the matches (-1 = free) */
static void greedy(const stream_t *s, const box_t *tb, const int *tin, int *tm, const box_t *det, const int *din, int *dm, int nd,
                   int with_conf, float g, int class_aware) {
    for (;;) {
        int bt = -1, bj = -1;
        float bs = 0.0f;
        for (int t = 0; t < s->live; t++) {
            if (!tin[t] || tm[t] >= 0) continue;
            for (int j = 0; j < nd; j++) {
                if (!din[j] || dm[j] >= 0) continue;
                if (class_aware && det[j].class_id != s->t[t].class_id) continue;
                float iou = iou_corner(tb[t], det[j]);
                float sim = with_conf ? iou * det[j].confidence : iou;
                if (!(sim > g)) continue;
                /* larger similarity, then smaller track_id (t ascending = track_id ascending), then smaller j */
                if (bt < 0 || sim > bs || (sim == bs && (s->t[t].track_id < s->t[bt].track_id ||
                                                         (s->t[t].track_id == s->t[bt].track_id && j < bj)))) {
                    bt = t; bj = j; bs = sim;
                }
            }
        }
        if (bt < 0) return;
        tm[bt] = bj;
        dm[bj] = bt;
    }
}

/* one frame of stream s: n detections (kept order); the tracked boxes go to out (track_id order); returns their count */
int trk_step(stream_t *s, const params_t *p, const box_t *boxes, int n, track_box_t *out) {
    static box_t det[MAX_DETS];
    int cat[MAX_DETS], dm[MAX_DETS], din[MAX_DETS];
    box_t tb[MAX_TRACKS];
    int role[MAX_TRACKS], tm[MAX_TRACKS], tin[MAX_TRACKS];
    const int frame = ++s->frame;
    if (n < 0) n = 0;
    if (n > MAX_DETS) n = MAX_DETS;
    for (int j = 0; j < n; j++) {
        box_t b = boxes[j];
        int ok = isfinite(b.x0) && isfinite(b.y0) && isfinite(b.x1) && isfinite(b.y1) && isfinite(b.confidence) && b.x1 - b.x0 > 0.0f &&
                 b.y1 - b.y0 > 0.0f;
        det[j] = b;
        cat[j] = !ok ? NONE : b.confidence > p->high_thresh ? HIGH : (b.confidence > p->low_thresh && b.confidence < p->high_thresh) ? LOW : NONE;
        dm[j] = -1;
    }
    /* 1. the pool (Tracked and activated, or Lost) is predicted; unconfirmed tracks are not */
    for (int t = 0; t < s->live; t++) {
        track_t *tr = &s->t[t];
        role[t] = tr->state == LOST ? 2 : tr->activated ? 1 : 3;
        if (role[t] != 3) predict(tr);
        tb[t] = track_box(tr);
        tm[t] = -1;
    }
    /* 2. the pool x high, IoU * conf */
    for (int t = 0; t < s->live; t++) tin[t] = role[t] == 1 || role[t] == 2;
    for (int j = 0; j < n; j++) din[j] = cat[j] == HIGH;
    greedy(s, tb, tin, tm, det, din, dm, n, 1, p->sim_high, p->class_aware);
    /* 3. unmatched Tracked tracks of the pool x low, IoU */
    for (int t = 0; t < s->live; t++) tin[t] = role[t] == 1 && tm[t] < 0;
    for (int j = 0; j < n; j++) din[j] = cat[j] == LOW;
    greedy(s, tb, tin, tm, det, din, dm, n, 0, p->sim_low, p->class_aware);
    /* 5. unconfirmed x the high detections left, IoU * conf */
    for (int t = 0; t < s->live; t++) tin[t] = role[t] == 3;
    for (int j = 0; j < n; j++) din[j] = cat[j] == HIGH && dm[j] < 0;
    greedy(s, tb, tin, tm, det, din, dm, n, 1, p->sim_unconfirmed, p->class_aware);
    /* updates; 4. unmatched Tracked pool tracks become Lost; 5. unmatched unconfirmed tracks are removed */
    track_t keep[MAX_TRACKS];
    int live = 0;
    for (int t = 0; t < s->live; t++) {
        track_t tr = s->t[t];
        if (tm[t] >= 0) {
            float z[4];
            measure(&det[tm[t]], z);
            update(&tr, z);
            tr.state = TRACKED;
            tr.activated = 1;
            tr.conf = det[tm[t]].confidence;
            tr.class_id = det[tm[t]].class_id;
            tr.det_index = tm[t];
            tr.last = frame;
        } else if (role[t] == 1) {
            tr.state = LOST;
        } else if (role[t] == 3) {
            continue;
        }
        keep[live++] = tr;
    }
    /* 6. births in j order while fewer than MAX_TRACKS are live */
    for (int j = 0; j < n; j++) {
        if (cat[j] != HIGH || dm[j] >= 0 || !(det[j].confidence >= p->new_thresh) || live >= MAX_TRACKS) continue;
        track_t tr;
        memset(&tr, 0, sizeof tr);
        float z[4];
        measure(&det[j], z);
        initiate(&tr, z);
        tr.conf = det[j].confidence;
        tr.class_id = det[j].class_id;
        tr.track_id = ++s->issued;
        tr.det_index = j;
        tr.last = frame;
        tr.state = TRACKED;
        tr.activated = frame == 1;
        keep[live++] = tr;
    }
    /* 7. lost tracks expire; 8. output */
    s->live = 0;
    int nout = 0;
    for (int t = 0; t < live; t++) {
        track_t *tr = &keep[t];
        if (tr->state == LOST && frame - tr->last > p->max_lost) continue;
        s->t[s->live++] = *tr;
        if (tr->state == TRACKED && tr->activated) {
            box_t b = track_box(tr);
            track_box_t o = {b.x0, b.y0, b.x1, b.y1, tr->conf, tr->class_id, tr->track_id, tr->det_index};
            out[nout++] = o;
        }
    }
    return nout;
}
