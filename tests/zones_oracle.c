/*
 * tests/zones_oracle.c -- TEST INFRASTRUCTURE: the C statement of the zone and line analytics that k_zones (zones.cuh) is checked
 * against, one stream at a time.
 *
 * The analytics are this library's own definition (include/mars_b200.h, mars_b200_set_zones).  Everything is written the literal
 * way: the old state and the frame's shown tracks are walked together in track_id order, each track's events are appended to one
 * list, and the line totals count up as the walk goes.  float32, one rounding per operation, left to right as written;
 * tests/zones_ref.py compiles this file with -ffp-contract=off into a temporary directory.
 */
#include <stdint.h>
#include <string.h>

#define MAX_TRACKS 256
#define MAX_ZONES 8
#define MAX_VERTS 16
#define MAX_LINES 8
#define MAX_EVENTS 128
enum { BOTTOM = 0, CENTRE = 1 };
enum { ENTER = 0, DWELL = 1, EXIT = 2, GONE = 3, CROSS_POS = 4, CROSS_NEG = 5 };

typedef struct { float x0, y0, x1, y1, confidence; int32_t class_id, track_id, det_index; } track_box_t;
typedef struct { float x[MAX_VERTS], y[MAX_VERTS]; int32_t n_verts, class_id, anchor, min_dwell; } zone_t;
typedef struct { float x0, y0, x1, y1; int32_t class_id, anchor; } line_t;
typedef struct { int32_t n_zones, n_lines; zone_t zone[MAX_ZONES]; line_t line[MAX_LINES]; } geom_t;
typedef struct { int32_t track_id, class_id; int16_t kind, index; int32_t value; } event_t;
typedef struct {
    int32_t frame, n_events, occupancy[MAX_ZONES], crossed_pos[MAX_LINES], crossed_neg[MAX_LINES];
    event_t events[MAX_EVENTS];
} zone_frame_t;
/* one track that has been shown */
typedef struct {
    int32_t track_id, class_id;
    float x0, y0, x1, y1;         /* tracked box at its last shown frame */
    int32_t sigma[MAX_LINES];     /* last non-zero side seen, 0 = none */
    int32_t inside[MAX_ZONES], dwelt[MAX_ZONES], entry[MAX_ZONES];
} ztrack_t;
/* one stream; all zero = fresh */
typedef struct {
    int32_t n, pos[MAX_LINES], neg[MAX_LINES];
    ztrack_t t[MAX_TRACKS]; /* in track_id order */
} zstream_t;

int zn_stream_bytes(void) { return (int)sizeof(zstream_t); }
int zn_geom_bytes(void) { return (int)sizeof(geom_t); }
int zn_frame_bytes(void) { return (int)sizeof(zone_frame_t); }

static event_t list[2 * MAX_TRACKS * (MAX_LINES + 2 * MAX_ZONES)];
static int n_list;

static void emit(int32_t id, int32_t cls, int kind, int index, int32_t value) {
    event_t e = {id, cls, (int16_t)kind, (int16_t)index, value};
    list[n_list++] = e;
}

static void anchor(float x0, float y0, float x1, float y1, int a, float *px, float *py) {
    *px = (x0 + x1) * 0.5f;
    *py = a == CENTRE ? (y0 + y1) * 0.5f : y1;
}

static int inside(const zone_t *z, float px, float py) {
    int c = 0;
    for (int i = 0; i < z->n_verts; i++) {
        int j = i == 0 ? z->n_verts - 1 : i - 1;
        float xi = z->x[i], yi = z->y[i], xj = z->x[j], yj = z->y[j];
        if ((yi > py) != (yj > py) && px < xi + ((xj - xi) * (py - yi)) / (yj - yi)) c = !c;
    }
    return c;
}

static int side(const line_t *l, float px, float py) {
    float v = (l->x1 - l->x0) * (py - l->y0) - (l->y1 - l->y0) * (px - l->x0);
    return v > 0.0f ? 1 : v < 0.0f ? -1 : 0;
}

static float cross(float ux, float uy, float vx, float vy) { return ux * vy - uy * vx; }

static int meets(const line_t *l, float px, float py, float qx, float qy) {
    float oa = cross(qx - px, qy - py, l->x0 - px, l->y0 - py);
    float ob = cross(qx - px, qy - py, l->x1 - px, l->y1 - py);
    return !((oa > 0.0f && ob > 0.0f) || (oa < 0.0f && ob < 0.0f));
}

static int matches(int32_t geom_class, int32_t cls) { return geom_class == -1 || geom_class == cls; }

/* a shown frame of track z (first: it has no state yet) */
static void shown_frame(zstream_t *s, const geom_t *g, int frame, ztrack_t *z, const track_box_t *r, int first, int32_t *occupancy) {
    for (int l = 0; l < g->n_lines; l++) {
        const line_t *L = &g->line[l];
        float px, py, qx, qy;
        anchor(z->x0, z->y0, z->x1, z->y1, L->anchor, &px, &py);
        anchor(r->x0, r->y0, r->x1, r->y1, L->anchor, &qx, &qy);
        int sq = side(L, qx, qy);
        if (!first && sq != 0 && z->sigma[l] == -sq && matches(L->class_id, r->class_id) && meets(L, px, py, qx, qy)) {
            if (sq > 0) emit(r->track_id, r->class_id, CROSS_POS, l, ++s->pos[l]);
            else emit(r->track_id, r->class_id, CROSS_NEG, l, ++s->neg[l]);
        }
        if (sq != 0) z->sigma[l] = sq;
    }
    for (int k = 0; k < g->n_zones; k++) {
        const zone_t *Z = &g->zone[k];
        float qx, qy;
        anchor(r->x0, r->y0, r->x1, r->y1, Z->anchor, &qx, &qy);
        int now = matches(Z->class_id, r->class_id) && inside(Z, qx, qy);
        if (now && !z->inside[k]) {
            emit(r->track_id, r->class_id, ENTER, k, first ? 1 : 0);
            z->inside[k] = 1;
            z->dwelt[k] = 0;
            z->entry[k] = frame;
        }
        if (now && Z->min_dwell > 0 && !z->dwelt[k] && frame - z->entry[k] + 1 >= Z->min_dwell) {
            emit(r->track_id, r->class_id, DWELL, k, frame - z->entry[k] + 1);
            z->dwelt[k] = 1;
        }
        if (!now && z->inside[k]) {
            emit(r->track_id, r->class_id, EXIT, k, frame - z->entry[k]);
            z->inside[k] = 0;
            z->dwelt[k] = 0;
        }
        if (now) occupancy[k]++;
    }
    z->class_id = r->class_id;
    z->x0 = r->x0; z->y0 = r->y0; z->x1 = r->x1; z->y1 = r->y1;
}

/* frame `frame` of stream s: live[n_live] the track IDs the tracker holds after this frame, shown[n_shown] its output of this
 * frame (both in track_id order) */
void zn_step(zstream_t *s, const geom_t *g, int frame, const int32_t *live, int n_live, const track_box_t *shown, int n_shown,
             zone_frame_t *out) {
    static ztrack_t next[MAX_TRACKS];
    memset(out, 0, sizeof *out);
    out->frame = frame;
    if (g->n_zones == 0 && g->n_lines == 0) return;
    n_list = 0;
    int nn = 0, i = 0, k = 0;
    while (i < s->n || k < n_shown) {
        if (i < s->n && (k >= n_shown || s->t[i].track_id <= shown[k].track_id)) {
            ztrack_t z = s->t[i++];
            int is_live = 0;
            for (int a = 0; a < n_live; a++) is_live |= live[a] == z.track_id;
            if (!is_live) { /* removed by the tracker */
                for (int q = 0; q < g->n_zones; q++)
                    if (z.inside[q]) emit(z.track_id, z.class_id, GONE, q, frame - z.entry[q]);
                continue;
            }
            if (k < n_shown && shown[k].track_id == z.track_id) shown_frame(s, g, frame, &z, &shown[k++], 0, out->occupancy);
            next[nn++] = z;
        } else { /* shown for the first time */
            ztrack_t z;
            memset(&z, 0, sizeof z);
            z.track_id = shown[k].track_id;
            shown_frame(s, g, frame, &z, &shown[k++], 1, out->occupancy);
            next[nn++] = z;
        }
    }
    s->n = nn;
    memcpy(s->t, next, (size_t)nn * sizeof(ztrack_t));
    out->n_events = n_list;
    memcpy(out->events, list, (size_t)(n_list < MAX_EVENTS ? n_list : MAX_EVENTS) * sizeof(event_t));
    for (int l = 0; l < g->n_lines; l++) {
        out->crossed_pos[l] = s->pos[l];
        out->crossed_neg[l] = s->neg[l];
    }
}
