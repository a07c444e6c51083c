/*
 * tests/gfl_oracle.c -- TEST INFRASTRUCTURE: the C statement of the NanoDet GFL head decode that k_gfl_decode is checked against.
 *
 * The decode is this library's own definition (the reference has no NanoDet code; include/mars_b200.h, mars_b200_set_gfl_heads).
 * tests/gfl_ref.py compiles this file with -ffp-contract=off into a temporary directory and binds it with ctypes.
 * head: int8 [gh, gw, nc + 4 (reg_max + 1)] dequantised with `scale`; centre 0 = cell centre (x + 0.5) * stride, 1 = cell corner
 * x * stride; appends to dets (corner boxes) up to maxd, order = y, x.  One float32 rounding per operation; the exponentials are
 * the host-libm tables the library builds (sigmoid of v * scale, expf(-(d * scale)) for d = 0..255).
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

typedef struct { float x0, y0, x1, y1, confidence; int32_t class_id; } gfl_box_t;

static float sigmoidf_1r(float x) { volatile float e = expf(-x); volatile float d = 1.0f + e; volatile float r = 1.0f / d; return r; }

int gfl_decode(const int8_t *head, int gh, int gw, int nc, int reg_max, float scale, int stride, int centre, int net_w, int net_h,
               float conf_thresh, gfl_box_t *dets, int cnt, int maxd) {
    float sig[256], E[256];
    for (int v = -128; v < 128; v++) { volatile float x = (float)v * scale; sig[v + 128] = sigmoidf_1r(x); }
    for (int d = 0; d < 256; d++) { volatile float x = (float)d * scale; volatile float e = expf(-x); E[d] = e; }
    const int nb = reg_max + 1, C = nc + 4 * nb;
    const float fs = (float)stride, off = centre == 0 ? 0.5f : 0.0f;
    for (int y = 0; y < gh; y++)
        for (int x = 0; x < gw; x++) {
            if (cnt >= maxd) return cnt;
            const int8_t *p = head + ((size_t)y * gw + x) * C;
            float score = sig[p[0] + 128];
            int label = 0;
            for (int c = 1; c < nc; c++) if (sig[p[c] + 128] > score) { score = sig[p[c] + 128]; label = c; }
            if (!(score > conf_thresh)) continue;
            float dist[4];
            for (int s = 0; s < 4; s++) {
                const int8_t *q = p + nc + s * nb;
                int vmax = q[0];
                for (int j = 1; j < nb; j++) if (q[j] > vmax) vmax = q[j];
                volatile float den = E[vmax - q[0]];
                for (int j = 1; j < nb; j++) den = den + E[vmax - q[j]];
                volatile float acc = 0.0f;
                for (int j = 0; j < nb; j++) { volatile float pr = E[vmax - q[j]] / den; volatile float t = (float)j * pr; acc = acc + t; }
                volatile float dd = acc * fs;
                dist[s] = dd;
            }
            volatile float cx0 = (float)x + off, cy0 = (float)y + off;
            volatile float cx = cx0 * fs, cy = cy0 * fs;
            volatile float x0 = cx - dist[0], y0 = cy - dist[1], x1 = cx + dist[2], y1 = cy + dist[3];
            dets[cnt].x0 = x0 > 0.0f ? x0 : 0.0f;
            dets[cnt].y0 = y0 > 0.0f ? y0 : 0.0f;
            dets[cnt].x1 = x1 < (float)net_w ? x1 : (float)net_w;
            dets[cnt].y1 = y1 < (float)net_h ? y1 : (float)net_h;
            dets[cnt].confidence = score; dets[cnt].class_id = label;
            cnt++;
        }
    return cnt;
}
