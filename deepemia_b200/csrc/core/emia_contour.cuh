// emia_contour.cuh — external-contour extraction on a bit-packed crop (host/device).
//
// Replaces (reference call sites): cv2.findContours(mask, RETR_EXTERNAL, CHAIN_APPROX_SIMPLE) at
// src/functions/inference.py:1164-1167 (measurement loop) and :2605 (compactness pre-filter of
// deduplicate_masks_smart); cv2.contourArea at :1175 / src/utils/measurements.py:134 and cv2.arcLength at
// inference.py:2607 / measurements.py:135,163.
//
// Algorithm = Suzuki-Abe border following as OpenCV implements it (raster scan; an outer border starts at an
// unmarked foreground pixel whose left neighbour is background; in RETR_EXTERNAL mode the start is accepted
// only if the nearest already-marked pixel to its left on the same row is a "right-exit" pixel (negative
// label) or there is none; the border is followed with the 8-neighbour clockwise/counter-clockwise search and
// every visited pixel is labelled +2, or -126 when its east neighbour was examined and found empty).
// CHAIN_APPROX_SIMPLE keeps a point whenever the chain direction changes.
// State per pixel is held in two extra bit planes (marked / negative) instead of OpenCV's int8 image, so
// the scan for start pixels is word-parallel.
#pragma once
#include "emia_common.cuh"

#define EMIA_PACK_PT(x, y) ((uint32_t)(x) | ((uint32_t)(y) << 16))
#define EMIA_PT_X(p) ((int)((p) & 0xFFFFu))
#define EMIA_PT_Y(p) ((int)((p) >> 16))

struct EmiaContourOut {
    uint32_t* pts;     // packed vertices (frame coordinates), contours stored back-to-back in DISCOVERY order
    int cap_pts;
    int* cstart;       // cstart[k]..cstart[k+1] = vertex range of k-th discovered contour; size cap_contours+1
    int cap_contours;
    int n_contours;
    int n_pts;
    int overflow;      // set when a capacity was exceeded (results invalid)
    int store;         // 0: count only (pts / cstart untouched, capacities ignored)
    // optional running cv2.arcLength of the contour being followed (track != 0): perim_last = arcLength(closed) of the most
    // recently completed contour, i.e. of contours[0] in OpenCV's (reverse discovery) order once the crop is done
    int track;
    const float* diag; // table of fl32(sqrt(2 k^2)) or nullptr
    double per, perim_last;
    int first_x, first_y, last_x, last_y, cur_n;
};

#define EMIA_DIAG_TABLE 128
// length of one closed-polygon segment as cv2.arcLength computes it: sqrtf((float)dx * dx + (float)dy * dy) in float32.
// Segments of a CHAIN_APPROX_SIMPLE contour are axial runs (exactly k for k < 4096) or diagonal runs (diag[k] when the table
// is given); every other case goes through sqrtf, so the value is bit-identical to the plain formula for ANY segment.
EMIA_HD float emia_seg_len(int dx, int dy, const float* diag) {
    dx = dx < 0 ? -dx : dx; dy = dy < 0 ? -dy : dy;
    if ((dx == 0 || dy == 0) && (dx | dy) < 4096) return (float)(dx | dy);
    if (diag && dx == dy && dx < EMIA_DIAG_TABLE) return diag[dx];
    const float fx = (float)dx, fy = (float)dy;
    const float dx2 = fx * fx;
    const float dy2 = fy * fy;
    return sqrtf(dx2 + dy2);
}

EMIA_HD void emia_contour_emit(EmiaContourOut& o, int fx, int fy) {
    if (o.store) {
        if (o.n_pts < o.cap_pts) o.pts[o.n_pts] = EMIA_PACK_PT(fx, fy);
        else o.overflow = 1;
    }
    o.n_pts++;
    if (o.track) {
        // every term is a float32 >= 1 (a multiple of 2^-23) and the sum stays below 2^20, so the double accumulation is exact
        // and independent of the order in which cv2.arcLength adds the same terms
        if (o.cur_n == 0) { o.first_x = fx; o.first_y = fy; }
        else o.per += (double)emia_seg_len(fx - o.last_x, fy - o.last_y, o.diag);
        o.last_x = fx; o.last_y = fy; o.cur_n++;
    }
}
// a contour is complete
EMIA_HD void emia_contour_close(EmiaContourOut& o) {
    if (o.track) {
        if (o.cur_n > 1) o.per += (double)emia_seg_len(o.first_x - o.last_x, o.first_y - o.last_y, o.diag);
        o.perim_last = o.per;
        o.per = 0.0; o.cur_n = 0;
    }
}

struct EmiaMarks {
    uint32_t* mk;   // marked plane   (h * wwords words)
    uint32_t* ng;   // negative plane (h * wwords words)
    int wwords;
};
EMIA_HD int emia_marked(const EmiaMarks& m, int lx, int ly) {
    return (m.mk[ly * m.wwords + (lx >> 5)] >> (lx & 31)) & 1u;
}
EMIA_HD void emia_mark(const EmiaMarks& m, int lx, int ly, int negative) {
    const int w = ly * m.wwords + (lx >> 5);
    const uint32_t b = 1u << (lx & 31);
    m.mk[w] |= b;
    if (negative) m.ng[w] |= b;
}

// 8-neighbourhood, direction s: 0=E 1=NE 2=N 3=NW 4=W 5=SW 6=S 7=SE (y grows downwards); (delta + 1) packed 4 bits each
#define EMIA_DX(s) ((int)((0x21000122u >> (4 * (s))) & 0xFu) - 1)
#define EMIA_DY(s) ((int)((0x22210001u >> (4 * (s))) & 0xFu) - 1)

// All external contours of the crop, in discovery (raster) order.  OpenCV returns them in REVERSE discovery order;
// consumers iterate k = n_contours-1 .. 0.  mk/ng must hold h*wwords words each.
//
// The algorithm is a two-phase state machine — SCAN for the next start pixel / one border-FOLLOWING step — exposed as
// resumable step functions, so that a kernel can keep the 32 instances of a warp in ONE flat loop (every lane executes the
// same branch-free following step: 3x3 neighbour mask -> rotate -> count-trailing-zeros picks the next direction) and hand a
// lane its next instance inside that same loop (k_contour_trace_slab).  emia_find_external_contours is the plain driver.
struct EmiaTraceState {
    EmiaBitView v;
    uint32_t* mk;
    uint32_t* ng;
    EmiaContourOut o;
    // scan position (row, word).  A trace without marks never scans: while it follows the seeded contour, the row holds wleft,
    // the border-start candidates (foreground pixels whose west neighbour is background) not yet accounted for; every step
    // whose examined-empty arc contains W takes one off (see emia_trace_begin_seeded)
    union { int y; int wleft; };
    int c;
    uint32_t done_mask;       // bits of the current word already examined
    int x0, y0, x1, y1, x3, y3, s, prev_s;
    // 3 x 64-pixel window of the crop around the border pixel being followed: rows wy-1, wy, wy+1, word columns wc, wc+1
    // (wc = (x - 1) >> 5, i.e. -1 when x == 0; words outside the crop read as 0).  A border step moves by one pixel, so the next
    // step reuses two of the three rows (or all of them) instead of re-loading six words.
    uint32_t wu0, wu1, wm0, wm1, wd0, wd1;
    int wc, wy;
    // the row that enters the window on a vertical move is loaded when the move is known but rotated in only when the window
    // is next used (wpend = dy, 0 = nothing pending): nothing depends on the load until then
    uint32_t wn0, wn1;
    int wpend;
};
#define EMIA_TRACE_SCAN 0
#define EMIA_TRACE_FOLLOW 1
#define EMIA_TRACE_DONE 2
#define EMIA_TRACE_START 3    // a border starts at (x0, y0): emia_trace_start

// Seed of a crop (emia_trace_seed): the first foreground pixel in raster order and the crop's candidate count, packed into one
// int64; negative values are the two cases without a seeded start
#define EMIA_SEED_PACK(x, y, ncand) ((int64_t)(x) | ((int64_t)(y) << 16) | ((int64_t)(ncand) << 32))
#define EMIA_SEED_X(s) ((int)((s) & 0xFFFF))
#define EMIA_SEED_Y(s) ((int)(((s) >> 16) & 0xFFFF))
#define EMIA_SEED_NCAND(s) ((int)((s) >> 32))
#define EMIA_SEED_EMPTY ((int64_t)-1)      // no foreground pixel: no contour
#define EMIA_SEED_CLASSIC ((int64_t)-2)    // the crop's extent does not fit the packing: trace with the full scan
// x < 2^16 and y < 2^16; the candidate count (at most half the pixels) then stays below 2^31
#define EMIA_SEED_FITS(ch, cw) ((ch) <= 0xFFFF && (cw) <= 0x7FF)

EMIA_HD void emia_trace_begin(EmiaTraceState& T) {
    T.o.n_contours = 0; T.o.n_pts = 0; T.o.overflow = 0;
    T.o.per = 0.0; T.o.perim_last = 0.0; T.o.cur_n = 0;
    if (T.o.store) T.o.cstart[0] = 0;
    T.y = 0; T.c = 0; T.done_mask = 0u;
    T.x0 = T.y0 = T.x1 = T.y1 = T.x3 = T.y3 = T.s = T.prev_s = 0;
    T.wu0 = T.wu1 = T.wm0 = T.wm1 = T.wd0 = T.wd1 = 0u;
    T.wc = -2; T.wy = -4; T.wpend = 0;          // no window yet
    T.wn0 = T.wn1 = 0u;
}

EMIA_HD void emia_win_load_row(const EmiaBitView& v, int ly, int c, uint32_t* w0, uint32_t* w1) {
    if ((unsigned)ly >= (unsigned)v.h) { *w0 = 0u; *w1 = 0u; return; }
    const uint32_t* row = v.bits + (size_t)ly * v.pitch_words;
    *w0 = (c >= 0) ? row[c] : 0u;
    *w1 = (c + 1 < v.wwords) ? row[c + 1] : 0u;
}
// Centre the window on local pixel (x, y); called as soon as the next pixel is known, so that the loads are in flight while the
// other lanes of the warp take their turn.
EMIA_HD void emia_win_settle(EmiaTraceState& T) {
    if (T.wpend == 0) return;
    const bool down = T.wpend > 0;
    const uint32_t m0 = T.wm0, m1 = T.wm1;
    T.wm0 = down ? T.wd0 : T.wu0; T.wm1 = down ? T.wd1 : T.wu1;
    T.wu0 = down ? m0 : T.wn0;    T.wu1 = down ? m1 : T.wn1;
    T.wd0 = down ? T.wn0 : m0;    T.wd1 = down ? T.wn1 : m1;
    T.wpend = 0;
}
EMIA_HD void emia_win_move(EmiaTraceState& T, int x, int y) {
    emia_win_settle(T);
    const int c = (x - 1) >> 5;
    const int dy = y - T.wy;
    if (c == T.wc) {
        if (dy == 0) return;
        if (dy == 1 || dy == -1) {
            // one row enters the window: a single load site for both directions (SIMT: the lanes that moved up and the lanes
            // that moved down execute it together)
            emia_win_load_row(T.v, y + dy, c, &T.wn0, &T.wn1);
            T.wpend = dy;
            T.wy = y;
            return;
        }
    }
    emia_win_load_row(T.v, y - 1, c, &T.wu0, &T.wu1);
    emia_win_load_row(T.v, y, c, &T.wm0, &T.wm1);
    emia_win_load_row(T.v, y + 1, c, &T.wd0, &T.wd1);
    T.wc = c; T.wy = y;
}
EMIA_HD uint32_t emia_win_row3(uint32_t w0, uint32_t w1, int sh) {
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(w0, w1, sh) & 7u;
#else
    return (uint32_t)(((((uint64_t)w1) << 32) | w0) >> sh) & 7u;
#endif
}
// 8-bit neighbour mask of the pixel the window is centred on: bit s set <=> the neighbour in direction s is foreground
EMIA_HD uint32_t emia_win_nbr8(EmiaTraceState& T, int x) {
    emia_win_settle(T);
    const int sh = (x - 1) & 31;
    const uint32_t up = emia_win_row3(T.wu0, T.wu1, sh), mid = emia_win_row3(T.wm0, T.wm1, sh), dn = emia_win_row3(T.wd0, T.wd1, sh);
    return ((mid >> 2) & 1u) | (((up >> 2) & 1u) << 1) | (((up >> 1) & 1u) << 2) | ((up & 1u) << 3) | ((mid & 1u) << 4) |
           ((dn & 1u) << 5) | (((dn >> 1) & 1u) << 6) | (((dn >> 2) & 1u) << 7);
}
// Mark-plane update of a followed border pixel.  On the device it is a fire-and-forget reduction (RED.OR): the old value is
// not needed, so the step does not wait for a load; the thread's own later reads of the word (scan phase) are ordered behind
// it by same-address program order.
EMIA_HD void emia_mark_or(uint32_t* word, uint32_t bit) {
#if defined(__CUDA_ARCH__) && !defined(EMIA_MARK_PLAIN)
    atomicOr(word, bit);
#else
    *word |= bit;
#endif
}

// Mark-plane update of a followed border pixel; a trace without marks (mk == nullptr, the seeded first contour) skips it.
EMIA_HD void emia_trace_mark(const EmiaTraceState& T, int x, int y, int negative) {
    if (!T.mk) return;
    const int wi = y * T.v.wwords + (x >> 5);
    const uint32_t bit = 1u << (x & 31);
    emia_mark_or(&T.mk[wi], bit);
    if (negative) emia_mark_or(&T.ng[wi], bit);
}

// Start following the outer border whose start pixel is (x0, y0) (local).  Returns the next phase.
EMIA_HD int emia_trace_start(EmiaTraceState& T) {
    const EmiaBitView& v = T.v;
    EmiaContourOut& o = T.o;
    const int x = T.x0, y = T.y0;
    if (o.store && o.n_contours >= o.cap_contours) { o.overflow = 1; return EMIA_TRACE_DONE; }
    emia_win_move(T, x, y);
    const uint32_t N8 = emia_win_nbr8(T, x);
    // first neighbour clockwise from W: directions 3,2,1,0,7,6,5 -> bit k of M
    const uint32_t M = ((N8 >> 3) & 1u) | (((N8 >> 2) & 1u) << 1) | (((N8 >> 1) & 1u) << 2) | ((N8 & 1u) << 3) |
                       (((N8 >> 7) & 1u) << 4) | (((N8 >> 6) & 1u) << 5) | (((N8 >> 5) & 1u) << 6);
    if (M == 0u) {   // isolated pixel: its W neighbour is examined and found empty once
        emia_trace_mark(T, x, y, 1);
        if (!T.mk) T.wleft--;
        emia_contour_emit(o, v.x_origin + x, v.y_origin + y);
        emia_contour_close(o);
        o.n_contours++;
        if (o.store) o.cstart[o.n_contours] = o.n_pts;
        return o.overflow ? EMIA_TRACE_DONE : EMIA_TRACE_SCAN;
    }
    T.s = (3 - emia_ctz(M)) & 7;
    T.x1 = x + EMIA_DX(T.s); T.y1 = y + EMIA_DY(T.s);
    T.x3 = x; T.y3 = y;
    T.prev_s = T.s ^ 4;
    return EMIA_TRACE_FOLLOW;
}

// One scan step: walks the rest of the current row for a start candidate.  Returns the next phase (EMIA_TRACE_START with the
// candidate in (x0, y0) when a border starts there).
EMIA_HD int emia_trace_scan_step(EmiaTraceState& T) {
    const EmiaBitView& v = T.v;
    const int ww = v.wwords;
    if (T.y >= v.h) return EMIA_TRACE_DONE;
    const uint32_t* row = v.bits + (size_t)T.y * v.pitch_words;
    const uint32_t* mrow = T.mk + T.y * ww;
    uint32_t cand = 0u;
    if (ww <= 4) {
        // narrow crops (the common case): all words of the row and of its mark row are loaded at once (independent loads, one
        // exposed latency per row instead of one per word), the candidates are then found in registers
        uint32_t F[4], Mk[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) { F[c] = (c < ww) ? row[c] : 0u; Mk[c] = (c < ww) ? mrow[c] : 0u; }
        int first_c = ww;
#pragma unroll
        for (int c = 3; c >= 0; --c) {
            const uint32_t left = (F[c] << 1) | (c > 0 ? (F[c > 0 ? c - 1 : 0] >> 31) : 0u);
            uint32_t cd = F[c] & ~left & ~Mk[c];
            if (c < T.c) cd = 0u;
            if (c == T.c) cd &= ~T.done_mask;
            if (cd) { cand = cd; first_c = c; }
        }
        if (cand && first_c != T.c) T.done_mask = 0u;
        T.c = first_c;
    } else {
        for (; T.c < ww; ++T.c, T.done_mask = 0u) {
            const uint32_t F = row[T.c];
            const uint32_t left = (F << 1) | (T.c > 0 ? (row[T.c - 1] >> 31) : 0u);
            cand = F & ~left & ~mrow[T.c] & ~T.done_mask;
            if (cand) break;
        }
    }
    if (!cand) { T.c = 0; ++T.y; T.done_mask = 0u; return EMIA_TRACE_SCAN; }
    const int c = T.c, y = T.y;
    const int b = emia_ctz(cand);
    T.done_mask |= (b == 31) ? 0xFFFFFFFFu : ((2u << b) - 1u);
    const int x = c * 32 + b;
    // RETR_EXTERNAL: nearest marked pixel strictly left of x on this row must carry a negative label (or not exist)
    {
        int cc = c;
        uint32_t mw = mrow[cc] & ((b == 0) ? 0u : ((1u << b) - 1u));
        while (mw == 0u && cc > 0) { --cc; mw = mrow[cc]; }
        if (mw != 0u) {
            const int hb = emia_msb(mw);
            if (!((T.ng[y * ww + cc] >> hb) & 1u)) return EMIA_TRACE_SCAN;   // inside an already-followed outer border
        }
    }
    T.x0 = x; T.y0 = y;
    return EMIA_TRACE_START;
}

// One border-following step.  Returns the next phase.
EMIA_HD int emia_trace_follow_step(EmiaTraceState& T) {
    const EmiaBitView& v = T.v;
    EmiaContourOut& o = T.o;
    const uint32_t N8 = emia_win_nbr8(T, T.x3);                    // the window was centred on (x3, y3) by the previous step
    const int s_end = T.s;
    const int r = (s_end + 1) & 7;
    const uint32_t rot = ((N8 >> r) | (N8 << (8 - r))) & 0xFFu;
    const int e = emia_ctz(rot);                                    // neighbours examined and found empty: s_end+1 .. s_end+e
    const int s = (s_end + 1 + e) & 7;                              // next foreground neighbour counter-clockwise
    // label +2, or -126 when the east neighbour was examined empty
    emia_trace_mark(T, T.x3, T.y3, (unsigned)(s - 1) < (unsigned)s_end);
    if (!T.mk) T.wleft -= ((3 - s_end) & 7) < e;                    // the west neighbour was examined empty
    if (s != T.prev_s) {
        emia_contour_emit(o, v.x_origin + T.x3, v.y_origin + T.y3);
        T.prev_s = s;
    }
    const int x4 = T.x3 + EMIA_DX(s), y4 = T.y3 + EMIA_DY(s);
    if (x4 == T.x0 && y4 == T.y0 && T.x3 == T.x1 && T.y3 == T.y1) {
        emia_contour_close(o);
        o.n_contours++;
        if (o.store) o.cstart[o.n_contours] = o.n_pts;
        T.s = s;
        return o.overflow ? EMIA_TRACE_DONE : EMIA_TRACE_SCAN;
    }
    T.x3 = x4; T.y3 = y4;
    T.s = (s + 4) & 7;
    emia_win_move(T, x4, y4);
    return EMIA_TRACE_FOLLOW;
}

EMIA_HD int emia_trace_step(EmiaTraceState& T, int phase) {
    return phase == EMIA_TRACE_SCAN ? emia_trace_scan_step(T) : phase == EMIA_TRACE_START ? emia_trace_start(T) : emia_trace_follow_step(T);
}

// marks_zeroed != 0: the caller cleared both planes already (the kernels clear the whole buffer with coalesced stores).
EMIA_HD_NOINLINE void emia_find_external_contours(const EmiaBitView& v, uint32_t* mk, uint32_t* ng, EmiaContourOut& o, int marks_zeroed = 0) {
    const int nw = v.h * v.wwords;
    if (!marks_zeroed) for (int i = 0; i < nw; ++i) { mk[i] = 0u; ng[i] = 0u; }
    EmiaTraceState T;
    T.v = v; T.mk = mk; T.ng = ng; T.o = o;
    emia_trace_begin(T);
    int phase = EMIA_TRACE_SCAN;
    while (phase != EMIA_TRACE_DONE) phase = emia_trace_step(T, phase);
    o = T.o;
}

// ---- seeded trace: the first contour without the row scan ------------------------------------------------------------
// In RETR_EXTERNAL mode a border can start only at a candidate (a foreground pixel whose west neighbour is background), and a
// marked candidate starts nothing.  So:
//  - the first border starts at the first foreground pixel in raster order (nothing is marked yet, nothing lies to its left);
//  - following a border examines the west neighbour of each of its candidates, once per candidate (T.wleft counts these
//    examinations down from the crop's candidate count).  When the first border closes with wleft == 0, every candidate is
//    marked, the scan would start nothing more, and the crop has exactly one external contour.  The border is then followed
//    without reading or writing the mark planes at all.
// Otherwise (a hole, a second component) the crop is traced again from row 0 with marks (emia_trace_restart).

// Seed of a crop (the serial form of k_trace_seed).
EMIA_HD int64_t emia_trace_seed(const EmiaBitView& v) {
    if (!EMIA_SEED_FITS(v.h, v.wwords)) return EMIA_SEED_CLASSIC;
    int64_t first = -1, ncand = 0;
    for (int y = 0; y < v.h; ++y) {
        const uint32_t* row = v.bits + (size_t)y * v.pitch_words;
        for (int c = 0; c < v.wwords; ++c) {
            const uint32_t F = row[c];
            const uint32_t left = (F << 1) | (c > 0 ? (row[c - 1] >> 31) : 0u);
            ncand += emia_popc(F & ~left);
            if (F && first < 0) first = EMIA_SEED_PACK(c * 32 + emia_ctz(F), y, 0);
        }
    }
    return first < 0 ? EMIA_SEED_EMPTY : first | EMIA_SEED_PACK(0, 0, ncand);
}

// Begin a trace from its seed without marks (T.mk == nullptr).  Returns the next phase; EMIA_TRACE_SCAN with T.mk == nullptr
// means the seeded part is over: the crop is done when T.wleft == 0, and is traced again with emia_trace_restart otherwise.
EMIA_HD int emia_trace_begin_seeded(EmiaTraceState& T, int64_t seed) {
    T.mk = nullptr; T.ng = nullptr;
    emia_trace_begin(T);
    if (seed < 0) { T.wleft = (seed == EMIA_SEED_EMPTY) ? 0 : -1; return EMIA_TRACE_SCAN; }
    T.wleft = EMIA_SEED_NCAND(seed);
    T.x0 = EMIA_SEED_X(seed); T.y0 = EMIA_SEED_Y(seed);
    return EMIA_TRACE_START;
}

// The classic trace from row 0 with marks: clears the two planes (h * wwords words each) and resets the output.
EMIA_HD void emia_trace_restart(EmiaTraceState& T, uint32_t* mk, uint32_t* ng) {
    const int nw = T.v.h * T.v.wwords;
    for (int i = 0; i < nw; ++i) { mk[i] = 0u; ng[i] = 0u; }
    T.mk = mk; T.ng = ng;
    emia_trace_begin(T);
}

// Plain driver of the seeded trace; same result as emia_find_external_contours.  *fast = 1 when the seeded contour was the
// only one (no restart).
EMIA_HD_NOINLINE void emia_find_external_contours_seeded(const EmiaBitView& v, int64_t seed, uint32_t* mk, uint32_t* ng,
                                                          EmiaContourOut& o, int* fast) {
    EmiaTraceState T;
    T.v = v; T.o = o;
    int phase = emia_trace_begin_seeded(T, seed);
    *fast = 1;
    while (phase != EMIA_TRACE_DONE) {
        if (phase == EMIA_TRACE_SCAN && !T.mk) {
            if (T.wleft == 0) break;
            emia_trace_restart(T, mk, ng);
            *fast = 0;
        }
        phase = emia_trace_step(T, phase);
    }
    o = T.o;
}

// cv2.contourArea on integer vertices: |shoelace| / 2 (exact; OpenCV accumulates integer-valued doubles).
EMIA_HD double emia_contour_area(const uint32_t* pts, int n) {
    if (n == 0) return 0.0;
    long long a = 0;
    int px = EMIA_PT_X(pts[n - 1]), py = EMIA_PT_Y(pts[n - 1]);
#pragma unroll 4
    for (int i = 0; i < n; ++i) {
        const int x = EMIA_PT_X(pts[i]), y = EMIA_PT_Y(pts[i]);
        a += (long long)px * y - (long long)py * x;
        px = x; py = y;
    }
    if (a < 0) a = -a;
    return (double)a * 0.5;
}

// cv2.arcLength(c, closed=True): per-segment float32 sqrt of float32 (dx*dx+dy*dy), accumulated in double,
// starting with the closing segment (last -> first).
// The segments of a CHAIN_APPROX_SIMPLE contour are runs in one of the 8 chain directions, so almost every term is
// either an axial run (sqrtf(k*k) == k exactly for k < 4096) or a diagonal run (fl32(sqrt(2 k^2)), taken from `diag`
// when the caller provides the table: diag[k] = sqrtf((float)(2*k*k)), k < EMIA_DIAG_TABLE); anything else goes through
// sqrtf, so the result is bit-identical to the plain loop for ANY vertex list.
EMIA_HD double emia_arc_length_closed(const uint32_t* pts, int n, const float* diag = nullptr) {
    if (n <= 1) return 0.0;
    double per = 0.0;
    int px = EMIA_PT_X(pts[n - 1]), py = EMIA_PT_Y(pts[n - 1]);
#pragma unroll 4
    for (int i = 0; i < n; ++i) {
        const int x = EMIA_PT_X(pts[i]), y = EMIA_PT_Y(pts[i]);
        per += (double)emia_seg_len(x - px, y - py, diag);
        px = x; py = y;
    }
    return per;
}
