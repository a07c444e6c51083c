/*
 * preproc.cuh -- letterbox pre-processing on the GPU (SURVEY 8f2): the step in front of mars_run in the reference's
 * callers, load_image() of src/mars/mars_yolo_test.c:40-77 minus the file decode:
 *     scale = fminf(tw/ow, th/oh); nw = (int)(ow*scale); nh = (int)(oh*scale); px = (tw-nw)/2; py = (th-nh)/2;
 *     stbir_resize_uint8(img, ow, oh, 0, rsz, nw, nh, 0, 3);  out = -17 everywhere, (int8)(rsz - 128) inside, NCHW or NHWC.
 *
 * stbir_resize_uint8 is the vendored include/stb/stb_image_resize.h (v0.9x): linear colour space, clamp edges, default
 * filters -- Catmull-Rom when an axis is enlarged (ratio > 1), Mitchell otherwise -- horizontal pass first, float
 * intermediate, every product and sum rounded separately.  Whatever route it takes (gather when enlarging, scatter when
 * shrinking), an output sample is a sum of (input sample x coefficient) terms added onto 0.0f in ascending source order;
 * build_resize_taps() restates its coefficient construction (stb_image_resize.h:1008-1231) on the host and hands the
 * kernels one tap list per output index, in that order, so the device sums are bit-identical:
 *     k_pre_horizontal    : H[f][r][x][c] = sum_t (u8 / 255.0f) * wh[t]            (stb :1243-1282, :1441-1652)
 *     k_pre_vertical_pack : v = sum_t H[f][src_t][x][c] * wv[t]; u8 = (int)((double)(sat(v) * 255.0f) + 0.5);
 *                           out = (int8)(u8 - 128), border -17  -- or RGBA u8, border 114 (stb :1692-1760, :1866-2061)
 * Every frame of a launch has its own size, row pitch and tap lists (a table of PreFrame descriptors); the target size is
 * shared.  A uniform batch is a table of identical descriptors.
 *
 * A frame is RGB8 or NV12.  An NV12 frame is converted to RGB8 where k_pre_horizontal reads its source bytes (pre_nv12_rgb),
 * so it letterboxes to exactly the slot tensor of the RGB8 frame that conversion produces; no RGB copy is written.
 */
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <vector>

namespace marsb200 {

/* per output index o: taps [start[o], start[o+1]) = (source index already clamped to the image, coefficient) */
struct ResizeTaps {
    std::vector<int> start, src;
    std::vector<float> w;
};

/* the two default kernels (stb :810-836); x86-64 evaluates every operation in float */
static inline float pre_catmullrom(float x) {
    x = fabsf(x);
    if (x < 1.0f) return 1 - x * x * (2.5f - 1.5f * x);
    if (x < 2.0f) return 2 - x * (4 + x * (0.5f * x - 2.5f));
    return 0.0f;
}
static inline float pre_mitchell(float x) {
    x = fabsf(x);
    if (x < 1.0f) return (16 + x * x * (21 * x - 36)) / 18;
    if (x < 2.0f) return (32 + x * (-60 + x * (36 - 7 * x))) / 18;
    return 0.0f;
}

/* Coefficients live in one flat array of `width` floats per contributor, exactly as in the reference: a contributor with
 * width + 1 candidates spills its last (zero) candidate into its neighbour's first cell, which the neighbour then
 * overwrites -- kept, so that every read sees what the reference's read sees. */
static inline void build_resize_taps(int in_size, int out_size, ResizeTaps *t) {
    const float scale = ((float)out_size / in_size) / (1.0f - 0.0f);
    const float shift = 0.0f * out_size / (1.0f - 0.0f);
    const bool up = scale > 1;
    const float support = 2.0f; /* both default filters */
    const int width = (int)ceil(support * 2);
    t->start.assign(1, 0);
    t->src.clear();
    t->w.clear();
    auto clampi = [&](int v) { return v < 0 ? 0 : (v >= in_size ? in_size - 1 : v); };
    if (up) {
        /* one contributor per OUTPUT index: which input samples it gathers (stb :1008-1021, :1037-1085) */
        const int nc = out_size;
        std::vector<float> coef((size_t)nc * width + 16, 0.0f);
        std::vector<int> n0(nc), n1(nc);
        const float radius = support * scale;
        for (int n = 0; n < nc; n++) {
            const float center = (float)n + 0.5f;
            const float lo = center - radius, hi = center + radius;
            const float in_lo = (lo + shift) / scale, in_hi = (hi + shift) / scale;
            const float in_center = (center + shift) / scale;
            int first = (int)floor(in_lo + 0.5), last = (int)floor(in_hi - 0.5);
            float *g = &coef[(size_t)n * width];
            float total = 0;
            n0[n] = first; n1[n] = last;
            for (int i = 0; i <= last - first; i++) {
                const float pc = (float)(i + first) + 0.5f;
                g[i] = pre_catmullrom(in_center - pc);
                if (i == 0 && !g[i]) { /* a leading zero is dropped and the window slides */
                    n0[n] = ++first;
                    i--;
                    continue;
                }
                total += g[i];
            }
            const float fs = 1 / total;
            for (int i = 0; i <= last - first; i++) g[i] *= fs;
            for (int i = last - first; i >= 0; i--) {
                if (g[i]) break;
                n1[n] = n0[n] + i - 1;
            }
        }
        for (int o = 0; o < out_size; o++) {
            for (int k = n0[o]; k <= n1[o]; k++) {
                t->src.push_back(clampi(k));
                t->w.push_back(coef[(size_t)o * width + (k - n0[o])]);
            }
            t->start.push_back((int)t->src.size());
        }
    } else {
        /* one contributor per INPUT index (with a margin of clamped virtual samples either side): which output samples it
         * feeds (stb :1023-1035, :1087-1115), then the per-output normalisation and clean-up (stb :1117-1190) */
        const int pixel_width = (int)ceil(support * 2 / scale);
        const int margin = pixel_width / 2;
        const int nc = in_size + margin * 2;
        std::vector<float> coef((size_t)nc * width + 16, 0.0f);
        coef[(size_t)nc * width + 8] = 1.0f; /* stops a zero-skip that would otherwise run off the end */
        std::vector<int> n0(nc), n1(nc);
        const float radius = support / scale;
        for (int n = 0; n < nc; n++) {
            const int na = n - margin;
            const float center = (float)na + 0.5f;
            const float lo = center - radius, hi = center + radius;
            const float out_lo = lo * scale - shift, out_hi = hi * scale - shift;
            const float out_center = center * scale - shift;
            const int first = (int)floor(out_lo + 0.5), last = (int)floor(out_hi - 0.5);
            float *g = &coef[(size_t)n * width];
            n0[n] = first; n1[n] = last;
            for (int i = 0; i <= last - first; i++) {
                const float pc = (float)(i + first) + 0.5f;
                const float x = pc - out_center;
                g[i] = pre_mitchell(x) * scale;
            }
            for (int i = last - first; i >= 0; i--) {
                if (g[i]) break;
                n1[n] = n0[n] + i - 1;
            }
        }
        auto at = [&](int j, int c) -> float & { return coef[(size_t)width * j + c]; };
        for (int i = 0; i < out_size; i++) {
            float total = 0;
            for (int j = 0; j < nc; j++) {
                if (i >= n0[j] && i <= n1[j]) total += at(j, i - n0[j]);
                else if (i < n0[j]) break;
            }
            const float s = 1 / total;
            for (int j = 0; j < nc; j++) {
                if (i >= n0[j] && i <= n1[j]) at(j, i - n0[j]) *= s;
                else if (i < n0[j]) break;
            }
        }
        for (int j = 0; j < nc; j++) {
            int skip = 0;
            while (at(j, skip) == 0) skip++;
            n0[j] += skip;
            while (n0[j] < 0) { n0[j]++; skip++; }
            const int range = n1[j] - n0[j] + 1;
            const int mx = width < range ? width : range;
            for (int i = 0; i < mx; i++) {
                if (i + skip >= width) break;
                at(j, i) = at(j, i + skip);
            }
        }
        for (int j = 0; j < nc; j++) n1[j] = n1[j] < out_size - 1 ? n1[j] : out_size - 1;
        /* scatter order = ascending contributor; per output that is the order of its additions */
        std::vector<std::vector<int>> who(out_size);
        for (int j = 0; j < nc; j++)
            for (int k = n0[j]; k <= n1[j]; k++)
                if (k >= 0 && k < out_size) who[k].push_back(j);
        for (int o = 0; o < out_size; o++) {
            for (int j : who[o]) {
                t->src.push_back(clampi(j - margin));
                t->w.push_back(at(j, o - n0[j]));
            }
            t->start.push_back((int)t->src.size());
        }
    }
}

/* the caller's letterbox geometry (mars_yolo_test.c:46-49) */
struct LetterboxGeom {
    int ow, oh, tw, th, nw, nh, px, py;
};
static inline LetterboxGeom letterbox_geom(int ow, int oh, int tw, int th) {
    LetterboxGeom g;
    g.ow = ow; g.oh = oh; g.tw = tw; g.th = th;
    const float scale = fminf((float)tw / ow, (float)th / oh);
    g.nw = (int)(ow * scale);
    g.nh = (int)(oh * scale);
    g.px = (tw - g.nw) / 2;
    g.py = (th - g.nh) / 2;
    return g;
}

/* source formats of a frame */
enum { PRE_RGB8 = 0, PRE_NV12 = 1 };

/* NV12 -> RGB8 in 16.16 fixed point, per colour variant (mars_b200.h MARS_B200_YUV_*): y0, cy, crv, cgu, cgv, cbu.  With
 * Kg = 1 - Kr - Kb, each constant is floor(c * 65536 + 0.5) in double of cy = ys, crv = cs 2 (1 - Kr), cgu = cs 2 Kb (1 - Kb) / Kg,
 * cgv = cs 2 Kr (1 - Kr) / Kg, cbu = cs 2 (1 - Kb); limited range ys = 255/219, cs = 255/224, y0 = 16; full range ys = cs = 1,
 * y0 = 0.  BT.601 (Kr, Kb) = (0.299, 0.114), BT.709 (0.2126, 0.0722).  Every channel is within 0.5 + 2^-8 of the clamped
 * exact matrix over all 2^24 (Y, U, V), and |accumulator| < 2^26. */
#define PRE_YUV_COEF_INIT                                  \
    {                                                      \
        {16, 76309, 104597, 25675, 53279, 132201},  /* BT.601 limited */ \
        {16, 76309, 117489, 13975, 34925, 138438},  /* BT.709 limited */ \
        {0, 65536, 91881, 22553, 46802, 116130},    /* BT.601 full */    \
        {0, 65536, 103206, 12276, 30679, 121609},   /* BT.709 full */    \
    }
enum { PRE_YUV_VARIANTS = 4 };
static const int32_t PRE_YUV_COEF[PRE_YUV_VARIANTS][6] = PRE_YUV_COEF_INIT;
static __constant__ int32_t pre_yuv_coef[PRE_YUV_VARIANTS][6] = PRE_YUV_COEF_INIT;

/* One frame of a ragged batch as the kernels see it.  A launch covers a run of frames that share the target size; each has
 * its own source format, geometry, row pitches, tap lists and float rows.  Offsets are relative to the launch (chunk).
 * A region of a larger frame is the ow x oh pixels at (ox, oy) of the frame that src / uv point at: the kernels read row
 * oy + r and column ox + c of the full planes, so an NV12 region at an odd origin keeps the chroma of the frame's 2 x 2 blocks. */
struct PreFrame {
    const uint8_t *src;  /* row 0 of the RGB8 frame, or of the NV12 luma plane (device) */
    const uint8_t *uv;   /* NV12: row 0 of the chroma plane, ceil(h / 2) rows of ceil(w / 2) U,V pairs of the w x h frame (device) */
    size_t row_stride;   /* bytes from one row of src to the next (>= w * 3 for RGB8, >= w for NV12) */
    size_t uv_stride;    /* NV12: bytes from one chroma row to the next (>= 2 * ceil(w / 2)) */
    size_t hoff;         /* its first float in the H scratch: oh x nw x 3 floats */
    int ox, oy;          /* the region's origin in the frame (0, 0 for a whole frame) */
    int ow, oh, nw, nh, px, py;
    int hs, vs;          /* its first entry in the start list of the horizontal / vertical taps */
    int blk0;            /* its first block in the horizontal grid: blocks [blk0, blk0 + oh * ceil(nw / 128)) */
    int fmt, colour;     /* PRE_RGB8 / PRE_NV12; the NV12 colour variant (row of pre_yuv_coef) */
};

/* bytes of a frame staged tightly on the device: RGB8 rows ow * 3 apart; NV12 the luma plane (rows ow apart), then the
 * chroma plane (rows 2 * ceil(ow / 2) apart) */
static inline size_t pre_frame_bytes(int fmt, int ow, int oh) {
    return fmt == PRE_NV12 ? (size_t)ow * oh + (size_t)2 * ((ow + 1) / 2) * ((oh + 1) / 2) : (size_t)ow * oh * 3;
}

/* one NV12 sample -> R, G, B bytes; k = the variant's row of pre_yuv_coef.  Arithmetic shifts (floor), clamp to [0, 255]. */
__device__ __forceinline__ void pre_nv12_rgb(int Y, int U, int V, int y0, int cy, int crv, int cgu, int cgv, int cbu, int *r, int *g, int *b) {
    const int yy = cy * (Y - y0) + 32768, u = U - 128, v = V - 128;
    *r = min(max((yy + crv * v) >> 16, 0), 255);
    *g = min(max((yy - cgu * u - cgv * v) >> 16, 0), 255);
    *b = min(max((yy + cbu * u) >> 16, 0), 255);
}
/* the concatenated tap lists of a batch: taps of output o of a list beginning at s are [start[s + o], start[s + o + 1]),
 * indices straight into src / w */
struct PreTaps {
    const int *start, *src;
    const float *w;
};

/* one thread per resized column of one source row.  The blocks of every frame follow each other (no grid sized to the
 * largest frame); a block finds its frame by a binary search over the first blocks.  H[r][x][c] = sum_t (u8 / 255) * w[t],
 * u8 read from the RGB8 frame or converted from the NV12 frame's luma byte and U,V pair at each tap (the branch is
 * uniform over the block: a block belongs to one frame). */
__global__ void __launch_bounds__(128) k_pre_horizontal(const PreFrame *fr, int n, PreTaps t, float *H) {
    __shared__ float dec[256]; /* the decode step: (float)u8 / 255.0f, IEEE division */
    dec[threadIdx.x] = __fdiv_rn((float)threadIdx.x, 255.0f);
    dec[threadIdx.x + 128] = __fdiv_rn((float)(threadIdx.x + 128), 255.0f);
    __syncthreads();
    const int b = blockIdx.x;
    int lo = 0, hi = n - 1; /* the last frame whose first block is <= b */
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (fr[mid].blk0 <= b) lo = mid;
        else hi = mid - 1;
    }
    const PreFrame &d = fr[lo];
    const int nw = d.nw, bx = (nw + 127) >> 7, local = b - d.blk0, r = local / bx, x = (local - r * bx) * 128 + threadIdx.x;
    if (x >= nw) return;
    const int sy = d.oy + r;
    const uint8_t *row = d.src + (size_t)sy * d.row_stride;
    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f;
    const int k0 = t.start[d.hs + x], ke = t.start[d.hs + x + 1];
    if (d.fmt == PRE_NV12) {
        const uint8_t *crow = d.uv + (size_t)(sy >> 1) * d.uv_stride;
        const int *q = pre_yuv_coef[d.colour];
        const int y0 = q[0], cy = q[1], crv = q[2], cgu = q[3], cgv = q[4], cbu = q[5];
        const int ox = d.ox;
        for (int k = k0; k < ke; k++) {
            const int sx = ox + t.src[k];
            const uint8_t *p = crow + 2 * (sx >> 1);
            int c0, c1, c2;
            pre_nv12_rgb(row[sx], p[0], p[1], y0, cy, crv, cgu, cgv, cbu, &c0, &c1, &c2);
            const float c = t.w[k];
            a0 = __fadd_rn(a0, __fmul_rn(dec[c0], c));
            a1 = __fadd_rn(a1, __fmul_rn(dec[c1], c));
            a2 = __fadd_rn(a2, __fmul_rn(dec[c2], c));
        }
    } else {
        row += (size_t)d.ox * 3;
        for (int k = k0; k < ke; k++) {
            const uint8_t *p = row + (size_t)t.src[k] * 3;
            const float c = t.w[k];
            a0 = __fadd_rn(a0, __fmul_rn(dec[p[0]], c));
            a1 = __fadd_rn(a1, __fmul_rn(dec[p[1]], c));
            a2 = __fadd_rn(a2, __fmul_rn(dec[p[2]], c));
        }
    }
    float *o = H + d.hoff + ((size_t)r * nw + x) * 3;
    o[0] = a0; o[1] = a1; o[2] = a2;
}

/* the resized sample as stb stores it: (unsigned char)(int)((double)(saturate(v) * 255.0f) + 0.5) */
__device__ __forceinline__ int pre_encode_u8(float v) {
    const float s = v < 0 ? 0.0f : (v > 1 ? 1.0f : v);
    return (int)(unsigned char)__double2int_rz((double)__fmul_rn(s, 255.0f) + 0.5);
}

/* packing of the target frame: the two int8 tensor layouts of mars_yolo_test.c:62-72 (px - 128, border -17), or the RGBA
 * uint8 frame of examples/yolo_detect.cpp:104-124 (memset 114 -- alpha included -- then R, G, B, 0 inside the image) */
enum { PRE_NCHW_I8 = 0, PRE_NHWC_I8 = 1, PRE_RGBA_U8 = 2 };

/* one thread per target pixel: grid (ceil(tw/128), th, n); dst = target of frame 0 of the launch, frames slot_stride apart.
 * frame_size (may be null) receives each frame's (ow, oh), for the letterbox inverse of the heads decode. */
__global__ void __launch_bounds__(128) k_pre_vertical_pack(const float *H, const PreFrame *fr, int tw, int th, PreTaps t, int8_t *dst,
                                                           size_t slot_stride, int mode, int2 *frame_size) {
    const int dx = blockIdx.x * 128 + threadIdx.x, dy = blockIdx.y, f = blockIdx.z;
    const PreFrame &d = fr[f];
    if (frame_size && dx == 0 && dy == 0) frame_size[f] = make_int2(d.ow, d.oh);
    if (dx >= tw) return;
    const int x = dx - d.px, y = dy - d.py, nw = d.nw;
    const bool inside = x >= 0 && x < nw && y >= 0 && y < d.nh;
    int u0 = 0, u1 = 0, u2 = 0;
    if (inside) {
        const float *Hf = H + d.hoff;
        float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f;
        for (int k = t.start[d.vs + y], ke = t.start[d.vs + y + 1]; k < ke; k++) {
            const float *p = Hf + ((size_t)t.src[k] * nw + x) * 3;
            const float c = t.w[k];
            a0 = __fadd_rn(a0, __fmul_rn(p[0], c));
            a1 = __fadd_rn(a1, __fmul_rn(p[1], c));
            a2 = __fadd_rn(a2, __fmul_rn(p[2], c));
        }
        u0 = pre_encode_u8(a0); u1 = pre_encode_u8(a1); u2 = pre_encode_u8(a2);
    }
    int8_t *o = dst + (size_t)f * slot_stride;
    if (mode == PRE_RGBA_U8) {
        uchar4 px = inside ? make_uchar4((unsigned char)u0, (unsigned char)u1, (unsigned char)u2, 0) : make_uchar4(114, 114, 114, 114);
        reinterpret_cast<uchar4 *>(o)[(size_t)dy * tw + dx] = px;
        return;
    }
    const int r0 = inside ? u0 - 128 : -17, r1 = inside ? u1 - 128 : -17, r2 = inside ? u2 - 128 : -17;
    if (mode == PRE_NHWC_I8) {
        int8_t *q = o + ((size_t)dy * tw + dx) * 3;
        q[0] = (int8_t)r0; q[1] = (int8_t)r1; q[2] = (int8_t)r2;
    } else {
        const size_t ps = (size_t)tw * th, at = (size_t)dy * tw + dx;
        o[at] = (int8_t)r0; o[ps + at] = (int8_t)r1; o[2 * ps + at] = (int8_t)r2;
    }
}

/* the H scratch of one launch stays under this; a batch that needs more is split on frame boundaries */
static const size_t PRE_H_CHUNK_BYTES = (size_t)256 << 20;

/* Host side of a ragged batch: the descriptors, the concatenated tap lists (one copy per distinct (in, out) of an axis) and
 * the launches.  Packed into one blob -- [PreFrame x n][start][src][w][merge] -- that is copied to the device in one piece.
 * The entries of a table are frames, or regions of frames (then several entries read one staged frame). */
struct PreTable {
    int tw = 0, th = 0;
    std::vector<PreFrame> fr;
    std::vector<size_t> stage; /* byte offset of each source frame in a tightly packed staging buffer (pre_frame_bytes each) */
    std::vector<int> start, src;
    std::vector<float> w;
    std::vector<int> merge;         /* optional trailer carried in the same upload: the region merge table of k_merge_rois, or the
                                     * stream table of k_track */
    std::vector<int> first, blocks; /* launch k covers entries [first[k], first[k + 1]) with blocks[k] horizontal blocks */
    size_t h_floats = 0;            /* H scratch of the largest launch */
    size_t stage_bytes = 0;         /* staging of the largest launch (per_launch staging) or of every frame */

    size_t merge_offset() const { return fr.size() * sizeof(PreFrame) + (start.size() + src.size()) * sizeof(int) + w.size() * sizeof(float); }
    size_t bytes() const { return merge_offset() + merge.size() * sizeof(int); }
    void pack(void *out) const {
        uint8_t *p = (uint8_t *)out;
        memcpy(p, fr.data(), fr.size() * sizeof(PreFrame)); p += fr.size() * sizeof(PreFrame);
        memcpy(p, start.data(), start.size() * sizeof(int)); p += start.size() * sizeof(int);
        memcpy(p, src.data(), src.size() * sizeof(int)); p += src.size() * sizeof(int);
        memcpy(p, w.data(), w.size() * sizeof(float)); p += w.size() * sizeof(float);
        memcpy(p, merge.data(), merge.size() * sizeof(int));
    }
    /* where the tap lists sit in the device copy of the blob */
    PreTaps taps(const void *dev) const {
        const int *s = (const int *)((const uint8_t *)dev + fr.size() * sizeof(PreFrame));
        return PreTaps{s, s + start.size(), (const float *)(s + start.size() + src.size())};
    }
};

/* Builds the table for n entries (geometry g[f] from letterbox_geom, all into the same target; source format fmt[f], or all
 * RGB8 when fmt is null) whose source pointers, pitches, origins and colour variants the caller fills in afterwards.
 * taps_of(in, out) returns the ResizeTaps of one axis (the caller's cache).  Launches split where the cumulative H bytes
 * (oh * nw * 12 per entry) would pass PRE_H_CHUNK_BYTES. */
template <class TapsOf>
static inline void pre_table_build(const LetterboxGeom *g, const int *fmt, int n, TapsOf taps_of, PreTable *t) {
    *t = PreTable();
    if (n <= 0) return;
    t->tw = g[0].tw; t->th = g[0].th;
    t->fr.resize(n);
    std::vector<std::pair<std::pair<int, int>, int>> seen; /* (in, out) -> its first entry in start */
    auto list = [&](int in, int out) {
        for (auto &s : seen)
            if (s.first.first == in && s.first.second == out) return s.second;
        const ResizeTaps &rt = taps_of(in, out);
        const int at = (int)t->start.size(), base = (int)t->src.size();
        for (int o = 0; o <= out; o++) t->start.push_back(base + rt.start[o]);
        t->src.insert(t->src.end(), rt.src.begin(), rt.src.end());
        t->w.insert(t->w.end(), rt.w.begin(), rt.w.end());
        seen.push_back({{in, out}, at});
        return at;
    };
    size_t hbytes = 0, hfl = 0;
    int blk = 0;
    for (int f = 0; f < n; f++) {
        const LetterboxGeom &q = g[f];
        const size_t need = (size_t)q.oh * q.nw * 3 * sizeof(float);
        if (f == 0 || (hbytes > 0 && hbytes + need > PRE_H_CHUNK_BYTES) || f - t->first.back() >= 65535) {
            if (f > 0) t->blocks.push_back(blk);
            t->first.push_back(f);
            hbytes = 0; hfl = 0; blk = 0;
        }
        PreFrame &d = t->fr[f];
        d.src = nullptr; d.uv = nullptr; d.row_stride = 0; d.uv_stride = 0;
        d.fmt = fmt ? fmt[f] : PRE_RGB8; d.colour = 0;
        d.hoff = hfl;
        d.ox = 0; d.oy = 0;
        d.ow = q.ow; d.oh = q.oh; d.nw = q.nw; d.nh = q.nh; d.px = q.px; d.py = q.py;
        d.hs = list(q.ow, q.nw);
        d.vs = list(q.oh, q.nh);
        d.blk0 = blk;
        blk += q.oh * ((q.nw + 127) / 128);
        hbytes += need;
        hfl += need / sizeof(float);
        t->h_floats = std::max(t->h_floats, hfl);
    }
    t->blocks.push_back(blk);
    t->first.push_back(n);
}

/* staging offsets of the n_frames source frames (frame_bytes[f] = pre_frame_bytes each), packed back to back.  per_launch: the
 * entries are the frames themselves and each launch stages its own frames, so the offsets restart with every launch. */
static inline void pre_table_stage(PreTable *t, const size_t *frame_bytes, int n_frames, bool per_launch) {
    t->stage.assign(n_frames, 0);
    t->stage_bytes = 0;
    size_t soff = 0;
    for (int f = 0, k = 0; f < n_frames; f++) {
        if (per_launch && k + 1 < (int)t->first.size() && f == t->first[k]) { soff = 0; k++; }
        t->stage[f] = soff;
        soff += frame_bytes[f];
        t->stage_bytes = std::max(t->stage_bytes, soff);
    }
}

/* launch k of a table whose blob was copied to dev: frames [first[k], first[k+1]) -> dst + f * slot_stride (dst = target of
 * the table's frame 0), H = scratch of h_floats floats; frame_size (may be null) = that of the table's frame 0 */
static inline cudaError_t launch_letterbox(const PreTable &t, int k, const void *dev, float *H, int8_t *dst, size_t slot_stride,
                                           int mode, int2 *frame_size, cudaStream_t s) {
    const int f0 = t.first[k], c = t.first[k + 1] - f0;
    const PreFrame *fr = (const PreFrame *)dev + f0;
    const PreTaps taps = t.taps(dev);
    k_pre_horizontal<<<t.blocks[k], 128, 0, s>>>(fr, c, taps, H);
    k_pre_vertical_pack<<<dim3((t.tw + 127) / 128, t.th, c), 128, 0, s>>>(H, fr, t.tw, t.th, taps, dst + (size_t)f0 * slot_stride,
                                                                          slot_stride, mode, frame_size ? frame_size + f0 : nullptr);
    return cudaGetLastError();
}

} // namespace marsb200
