/*
 * render_core.cuh -- the per-env scene and the per-pixel colour of msoc_render_kernel (msoc.cu), all __host__ __device__
 * like step_core.cuh so that the host harness tests/hostsim/render_host.cu renders with the very same arithmetic.
 *
 * The picture is the one marl_soccer_b200/renderer.py scene() defines, 800 x 600 screen units, y down, back to front:
 * field (green), centre line, centre circle, penalty boxes, goals (all white), then per agent its body (blue for
 * agents 0-1, red for 2-3) and its nose (yellow), then the ball (white).  Each primitive is an exact test on the pixel
 * centre: pixel (r, c) of an H x W image has its centre at sx = (c + 0.5) 800 / W, sy = (r + 0.5) 600 / H.
 *
 * The output is a flat stream of RGB bytes, images one after another.  It is cut into segments of 32 pixels = 96 bytes
 * (a multiple of 16, so a segment that starts at pixel 32k of the stream starts on a 16-byte boundary); one thread
 * colours one segment, row piece by row piece (a segment may cross rows and images), as five bit masks over its 32
 * pixels: white, blue, red, yellow and "no image" (out-of-range env index: zero bytes).  The static background of a
 * row is a few column intervals; an agent or the ball is tested per pixel only where its screen bounding box meets the
 * piece.
 */
#pragma once
#include "step_core.cuh"

/* checked build: env index read by the render kernel, byte offset of every store inside the output */
enum { CHK_RENDER = CHK_LIST_COUNT + 1 };

namespace msoc {

constexpr int RENDER_SEG = 32;               /* pixels per segment (bit j of a mask = pixel j) */
constexpr int RENDER_SEG_WORDS = RENDER_SEG * 3 / 4; /* 24 words = 96 bytes */
constexpr int RENDER_MAX_SIDE = 4096;
/* renderer.py colours as 0x00BBGGRR (byte order R, G, B in memory) */
constexpr uint32_t RGB_FIELD = 0x228B22u, RGB_WHITE = 0xFFFFFFu, RGB_BLUE = 0xFF0000u, RGB_RED = 0x0000FFu,
                   RGB_NOSE = 0x00FFFFu;

/* Column interval [lo, hi] (inclusive, lo > hi: empty) */
struct ColSpan { int lo, hi; };

/* Per image size, computed once on the host in fp64: the fixed background intervals as column and row index ranges
   (the circle is the only curved one and is done per row). */
struct RenderGeom {
    int H, W;
    float sxs, sys;     /* screen units per pixel: 800 / W, 600 / H */
    float isx;          /* W / 800 */
    ColSpan goal_l, goal_r, box_l, box_r, box_l0, box_l1, box_r0, box_r1, line;
    int goal_r0, goal_r1, box_r0w, box_r1w, inner_r0, inner_r1, line_r0, line_r1, ring_r0, ring_r1;
};

/* the columns whose pixel centres (c + 0.5) 800 / W lie in [x0, x1] */
static inline ColSpan render_cols(double x0, double x1, int W)
{
    ColSpan s;
    s.lo = (int)ceil(x0 * W / 800.0 - 0.5);
    s.hi = (int)floor(x1 * W / 800.0 - 0.5);
    if (s.lo < 0) s.lo = 0;
    if (s.hi > W - 1) s.hi = W - 1;
    return s;
}
/* rows whose centres lie in [y0, y1] (strict: in (y0, y1)) */
static inline void render_rows(double y0, double y1, int H, bool strict, int &r0, int &r1)
{
    const double a = y0 * H / 600.0 - 0.5, b = y1 * H / 600.0 - 0.5;
    r0 = strict ? (int)floor(a) + 1 : (int)ceil(a);
    r1 = strict ? (int)ceil(b) - 1 : (int)floor(b);
}

static inline void render_geom(int H, int W, RenderGeom &G)
{
    G.H = H; G.W = W;
    G.sxs = (float)(800.0 / W); G.sys = (float)(600.0 / H); G.isx = (float)(W / 800.0);
    /* scene(): goals (0, 225, 10, 150) and (790, 225, 10, 150) filled */
    G.goal_l = render_cols(0.0, 10.0, W); G.goal_r = render_cols(790.0, 800.0, W);
    render_rows(225.0, 375.0, H, false, G.goal_r0, G.goal_r1);
    /* penalty boxes (10, 150, 120, 300) and (670, 150, 120, 300), outline of width 2: inside the rect and not strictly
       inside the rect inset by 2 -- whole width on rows outside (152, 448), the two side bands on rows inside it */
    G.box_l = render_cols(10.0, 130.0, W); G.box_r = render_cols(670.0, 790.0, W);
    G.box_l0 = render_cols(10.0, 12.0, W); G.box_l1 = render_cols(128.0, 130.0, W);
    G.box_r0 = render_cols(670.0, 672.0, W); G.box_r1 = render_cols(788.0, 790.0, W);
    render_rows(150.0, 450.0, H, false, G.box_r0w, G.box_r1w);
    render_rows(152.0, 448.0, H, true, G.inner_r0, G.inner_r1);
    /* centre line (400, 10) - (400, 590), width 2 */
    G.line = render_cols(399.0, 401.0, W);
    render_rows(10.0, 590.0, H, false, G.line_r0, G.line_r1);
    /* centre circle (400, 300), radius 70, width 2: rows with |sy - 300| <= 70 */
    render_rows(230.0, 370.0, H, false, G.ring_r0, G.ring_r1);
}

/* An agent or the ball as the kernel tests it: centre in screen units, cos / sin of the angle, and the pixel index
   bounding box (rows r0..r1, columns c0..c1; empty when r0 > r1 or c0 > c1). */
struct RenderBody { float cx, cy, cs, sn; int r0, r1, c0, c1; };
struct RenderScene { RenderBody b[5]; int valid; int pad[3]; };

/* the record an image shows: the one msoc_get_state reads (the current buffer, or the injected state) */
MSOC_HD const float4 *render_record(const Arrays &A, int step, int64_t e)
{
    const float4 *rec = A.pose[buf_cur(step)] + e * POSE_F4;
    if ((f2u(rec[7].z) & FLAG_INJECT) != 0u && A.inject != nullptr) rec = A.inject + e * POSE_F4;
    return rec;
}

MSOC_HD int render_floor_i(float x) { return (int)floorf(x); }
MSOC_HD int render_ceil_i(float x) { return (int)ceilf(x); }

MSOC_HD void render_bbox(const RenderGeom &G, float cx, float cy, float half, RenderBody &B)
{
    const float isy = (float)G.H / 600.0f;
    B.c0 = render_ceil_i((cx - half) * G.isx - 0.5f); B.c1 = render_floor_i((cx + half) * G.isx - 0.5f);
    B.r0 = render_ceil_i((cy - half) * isy - 0.5f);   B.r1 = render_floor_i((cy + half) * isy - 0.5f);
    B.c0 = B.c0 < 0 ? 0 : B.c0; B.c1 = B.c1 > G.W - 1 ? G.W - 1 : B.c1;
    B.r0 = B.r0 < 0 ? 0 : B.r0; B.r1 = B.r1 > G.H - 1 ? G.H - 1 : B.r1;
}

/* scene of one env from the first six float4 of its record (positions, agent angles); rec == null: no image */
MSOC_HD void render_scene(const RenderGeom &G, const float4 *rec, RenderScene &S)
{
    S.valid = rec != nullptr;
    if (rec == nullptr) {
        for (int i = 0; i < 5; i++) { S.b[i].cx = S.b[i].cy = S.b[i].cs = S.b[i].sn = 0.0f; S.b[i].r0 = S.b[i].c0 = 0; S.b[i].r1 = S.b[i].c1 = -1; }
        return;
    }
    const float4 a = rec[5];
    const float ang[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int i = 0; i < 4; i++) {
        RenderBody &B = S.b[i];
        const float4 p = rec[i];
        B.cx = p.x; B.cy = SCREEN_H - p.y;
#if defined(__CUDA_ARCH__)
        __sincosf(ang[i], &B.sn, &B.cs); /* angles are kept in [-pi, pi]: absolute error < 4e-7, far below a pixel */
#else
        sincosf(ang[i], &B.sn, &B.cs);
#endif
        /* half extent of the rotated 30 x 30 box, plus a margin far above the rounding of the tests */
        render_bbox(G, B.cx, B.cy, AGENT_HALF * (fabsf(B.cs) + fabsf(B.sn)) + 0.01f, B);
    }
    RenderBody &B = S.b[4];
    const float4 p = rec[4];
    B.cx = p.x; B.cy = SCREEN_H - p.y; B.cs = 1.0f; B.sn = 0.0f;
    render_bbox(G, B.cx, B.cy, BALL_R + 0.01f, B);
}

/* bits of the columns of [s.lo, s.hi] among the `len` columns from c0 (bit 0 = column c0) */
MSOC_HD uint32_t render_span_bits(int lo, int hi, int c0, int len)
{
    const int a = lo > c0 ? lo : c0, b = hi < c0 + len - 1 ? hi : c0 + len - 1;
    if (a > b) return 0u;
    return (0xFFFFFFFFu >> (31 - (b - a))) << (a - c0);
}
MSOC_HD uint32_t render_span_bits(const ColSpan &s, int c0, int len) { return render_span_bits(s.lo, s.hi, c0, len); }

/* white (line) pixels of the static background among columns c0..c0+len-1 of row `row` */
MSOC_HD uint32_t render_background(const RenderGeom &G, int row, int c0, int len)
{
    uint32_t m = 0u;
    if (row >= G.goal_r0 && row <= G.goal_r1) m |= render_span_bits(G.goal_l, c0, len) | render_span_bits(G.goal_r, c0, len);
    if (row >= G.box_r0w && row <= G.box_r1w) {
        if (row >= G.inner_r0 && row <= G.inner_r1)
            m |= render_span_bits(G.box_l0, c0, len) | render_span_bits(G.box_l1, c0, len) | render_span_bits(G.box_r0, c0, len) |
                 render_span_bits(G.box_r1, c0, len);
        else
            m |= render_span_bits(G.box_l, c0, len) | render_span_bits(G.box_r, c0, len);
    }
    if (row >= G.line_r0 && row <= G.line_r1) m |= render_span_bits(G.line, c0, len);
    if (row >= G.ring_r0 && row <= G.ring_r1) {
        /* ring 68 <= d <= 70: |sx - 400| in [b, a], a = sqrt(70^2 - dy^2), b = sqrt(68^2 - dy^2) (b = 0 when |dy| >= 68) */
        const float dy = fabsf((row + 0.5f) * G.sys - 300.0f);
        const float a = sqrtf(fmaxf((70.0f - dy) * (70.0f + dy), 0.0f));
        const float b = dy < 68.0f ? sqrtf((68.0f - dy) * (68.0f + dy)) : -1.0f;
        const int ol = render_ceil_i((400.0f - a) * G.isx - 0.5f), orr = render_floor_i((400.0f + a) * G.isx - 0.5f);
        if (b < 0.0f) {
            m |= render_span_bits(ol, orr, c0, len);
        } else {
            m |= render_span_bits(ol, render_floor_i((400.0f - b) * G.isx - 0.5f), c0, len);
            m |= render_span_bits(render_ceil_i((400.0f + b) * G.isx - 0.5f), orr, c0, len);
        }
    }
    return m;
}

/* Colour masks of one segment: `count` pixels (1..32) of the flat stream starting at column `col` of row `row` of
   image `img` (an index into `scenes`).  wm / bm / rm / ym / zm: white, blue, red, yellow (nose), zero (no image);
   every other pixel is the field's green.  The masks are disjoint. */
MSOC_HD void render_segment_masks(const RenderGeom &G, const RenderScene *scenes, int img, int row, int col, int count,
                                  uint32_t &wm, uint32_t &bm, uint32_t &rm, uint32_t &ym, uint32_t &zm)
{
    wm = bm = rm = ym = zm = 0u;
    int j = 0;
    while (j < count) {
        const int len = count - j < G.W - col ? count - j : G.W - col;
        const RenderScene &S = scenes[img];
        const uint32_t piece = (0xFFFFFFFFu >> (32 - len)) << j;
        if (!S.valid) {
            zm |= piece;
        } else {
            wm |= render_background(G, row, col, len) << j;
            const float sy = (row + 0.5f) * G.sys;
#pragma unroll 1
            for (int k = 0; k < 5; k++) {
                const RenderBody &B = S.b[k];
                if (row < B.r0 || row > B.r1) continue;
                const int a = B.c0 > col ? B.c0 : col, b = B.c1 < col + len - 1 ? B.c1 : col + len - 1;
                if (a > b) continue;
                const float dys = sy - B.cy;
                uint32_t body = 0u, nose = 0u;
                if (k < 4) {
                    /* agent frame: (u, v) = R(-theta) (world - centre), world y = 600 - sy */
                    const float u_row = -B.sn * dys, v_row = -B.cs * dys;
                    for (int c = a; c <= b; c++) {
                        const float dxs = (c + 0.5f) * G.sxs - B.cx;
                        const float u = fmaf(B.cs, dxs, u_row), v = fmaf(-B.sn, dxs, v_row);
                        const uint32_t bit = 1u << (c - col + j);
                        if (fabsf(u) <= AGENT_HALF && fabsf(v) <= AGENT_HALF) body |= bit;
                        if (u >= 0.5f * AGENT_HALF && fabsf(v) <= AGENT_HALF - u) nose |= bit;
                    }
                    const uint32_t other = body & ~nose;
                    if (k < 2) { bm |= other; rm &= ~other; } else { rm |= other; bm &= ~other; }
                    wm &= ~body; ym = (ym & ~body) | nose;
                } else {
                    for (int c = a; c <= b; c++) {
                        const float dxs = (c + 0.5f) * G.sxs - B.cx;
                        if (fmaf(dxs, dxs, dys * dys) <= BALL_R * BALL_R) body |= 1u << (c - col + j);
                    }
                    wm |= body; bm &= ~body; rm &= ~body; ym &= ~body;
                }
            }
        }
        j += len; col += len;
        if (col == G.W) { col = 0; if (++row == G.H) { row = 0; img++; } }
    }
}

MSOC_HD uint32_t render_perm(uint32_t x, uint32_t y, uint32_t s)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(x, y, s);
#else
    const uint64_t v = (uint64_t)x | ((uint64_t)y << 32);
    uint32_t r = 0;
    for (int i = 0; i < 4; i++) r |= (uint32_t)((v >> (8 * ((s >> (4 * i)) & 7u))) & 0xFFu) << (8 * i);
    return r;
#endif
}

/* the 96 bytes of a segment from its masks; four pixels 0x00BBGGRR -> three words R0G0B0R1 G1B1R2G2 B2R3G3B3 */
MSOC_HD void render_pack(uint32_t wm, uint32_t bm, uint32_t rm, uint32_t ym, uint32_t zm, uint32_t w[RENDER_SEG_WORDS])
{
    const bool plain = (bm | rm | ym | zm) == 0u; /* the common case: field and lines only */
#pragma unroll
    for (int q = 0; q < RENDER_SEG / 4; q++) {
        uint32_t p[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int j = 4 * q + i;
            uint32_t c = ((wm >> j) & 1u) ? RGB_WHITE : RGB_FIELD;
            if (!plain) {
                c = ((bm >> j) & 1u) ? RGB_BLUE : c;
                c = ((rm >> j) & 1u) ? RGB_RED : c;
                c = ((ym >> j) & 1u) ? RGB_NOSE : c;
                c = ((zm >> j) & 1u) ? 0u : c;
            }
            p[i] = c;
        }
        w[3 * q] = render_perm(p[0], p[1], 0x4210u);
        w[3 * q + 1] = render_perm(p[1], p[2], 0x5421u);
        w[3 * q + 2] = render_perm(p[2], p[3], 0x6542u);
    }
}

/* Pixels per tile of the kernel (a tile is a multiple of 32 pixels and spans at most RENDER_MAX_SPAN images, whose
   scenes a block keeps in shared memory) */
constexpr int RENDER_BLOCK = 128, RENDER_SEGS_PER_THREAD = 4, RENDER_MAX_SPAN = 40;
static inline int64_t render_tile_px(int64_t hw)
{
    int64_t t = ((RENDER_MAX_SPAN - 2) * hw + 1) / RENDER_SEG * RENDER_SEG;
    const int64_t cap = (int64_t)RENDER_BLOCK * RENDER_SEG * RENDER_SEGS_PER_THREAD;
    return t < RENDER_SEG ? RENDER_SEG : t > cap ? cap : t;
}

} /* namespace msoc */
