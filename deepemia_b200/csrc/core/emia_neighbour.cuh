// emia_neighbour.cuh — relations between the particles of one image (neighbours_results.csv; definitions in oracle/neighbours.py):
// the exact squared distance between two bit-packed masks, the centroid nearest-neighbour ring search and the closest-mask search
// over a uniform grid, and the union-find of the touching graph.  Host/device: the kernels of emia_neighbour_kernels.cuh run this
// source on sm_100a, tests/hostsim/hostsim_neighbour.cpp runs it serially on the CPU.
//
// Grid.  Cell (c, cx, cy) = entries ((c * gy + cy) * gx + cx) of cell_off / ent: class key c, cell_size-pixel squares.  A listed
// instance is entered in EVERY cell its tight bbox covers, so a cell lists each instance whose bbox meets it.  Its centroid lies in
// its bbox, so the centroid search finds each instance in the cell of its centroid and counts it there only.
#pragma once
#include <limits.h>
#include "emia_common.cuh"

#define EMIA_NB_F 4      // double per instance: centroid x, centroid y, nearest-neighbour distance, edge distance (NaN: none)
#define EMIA_NB_I 6      // int32 per instance: listed, nearest neighbour, closest neighbour (-1: none), touching, agglomerate, size

struct EmiaNbGrid {
    int cs, gx, gy;      // cell size in pixels, cells per row / column (one plane per class key)
};

// one bit-packed crop: rows [ry0, ry0 + ch) x frame word columns [wc0, wc0 + cw)
struct EmiaNbCrop {
    const uint32_t* w;
    int ry0, wc0, ch, cw;
};

// smallest set pixel x' >= x of a crop row, INT_MAX when there is none
EMIA_HD int emia_nb_next_set(const uint32_t* row, int wc0, int cw, int x) {
    const int xb = wc0 * 32;
    if (x < xb) x = xb;
    int k = (x - xb) >> 5;
    if (k >= cw) return INT_MAX;
    uint32_t w = row[k] & (0xffffffffu << ((x - xb) & 31));
    for (;;) {
        if (w) return xb + 32 * k + emia_ctz(w);
        if (++k >= cw) return INT_MAX;
        w = row[k];
    }
}
// smallest clear pixel x' >= x of a crop row (the crop's end when the row is set up to it)
EMIA_HD int emia_nb_next_clear(const uint32_t* row, int wc0, int cw, int x) {
    const int xb = wc0 * 32;
    int k = (x - xb) >> 5;
    if (k >= cw) return xb + 32 * cw;
    uint32_t w = ~row[k] & (0xffffffffu << ((x - xb) & 31));
    for (;;) {
        if (w) return xb + 32 * k + emia_ctz(w);
        if (++k >= cw) return xb + 32 * cw;
        w = ~row[k];
    }
}
// largest set pixel x' <= x of a crop row, INT_MIN when there is none
EMIA_HD int emia_nb_prev_set(const uint32_t* row, int wc0, int cw, int x) {
    const int xb = wc0 * 32;
    if (x < xb) return INT_MIN;
    if (x >= xb + 32 * cw) x = xb + 32 * cw - 1;
    int k = (x - xb) >> 5;
    const int b = (x - xb) & 31;
    uint32_t w = row[k] & (b == 31 ? 0xffffffffu : ((2u << b) - 1u));
    for (;;) {
        if (w) return xb + 32 * k + emia_msb(w);
        if (--k < 0) return INT_MIN;
        w = row[k];
    }
}

// least |x - x'| between a set pixel x of row ra (crop a) and a set pixel x' of row rb (crop b); INT_MAX when either row is empty.
// In one dimension the least gap is attained at the end of a run of a, so each run [s, e] of ra asks rb for its nearest set pixel
// at or after s and before s.
EMIA_HD int emia_nb_row_gap(const uint32_t* ra, int wca, int cwa, const uint32_t* rb, int wcb, int cwb) {
    int best = INT_MAX;
    int s = emia_nb_next_set(ra, wca, cwa, wca * 32);
    while (s != INT_MAX) {
        const int e = emia_nb_next_clear(ra, wca, cwa, s) - 1;
        const int q = emia_nb_next_set(rb, wcb, cwb, s);
        if (q <= e) return 0;
        if (q != INT_MAX && q - e < best) best = q - e;
        const int p = emia_nb_prev_set(rb, wcb, cwb, s);
        if (p != INT_MIN && s - p < best) best = s - p;
        if (q == INT_MAX) break;                       // rb has nothing right of this run: later runs are only farther from p
        s = emia_nb_next_set(ra, wca, cwa, e + 1);
    }
    return best;
}

// min over set pixels p of a, p' of b of (x - x')^2 + (y - y')^2, exact when it is below `limit`; otherwise some value >= limit.
// Row pairs with (y - y')^2 >= the best so far are never looked at; rows of b are visited outward from the row of a.
EMIA_HD long long emia_nb_pair_d2(const EmiaNbCrop& a, const EmiaNbCrop& b, long long limit) {
    // shared pixel: D2 = 0
    const int y0 = emia_max(a.ry0, b.ry0), y1 = emia_min(a.ry0 + a.ch, b.ry0 + b.ch);
    const int c0 = emia_max(a.wc0, b.wc0), c1 = emia_min(a.wc0 + a.cw, b.wc0 + b.cw);
    for (int y = y0; y < y1; ++y)
        for (int c = c0; c < c1; ++c)
            if (emia_popc(a.w[(size_t)(y - a.ry0) * a.cw + c - a.wc0] & b.w[(size_t)(y - b.ry0) * b.cw + c - b.wc0])) return 0;
    long long best = limit;
    const int bl = b.ry0, bh = b.ry0 + b.ch - 1;
    for (int ya = a.ry0; ya < a.ry0 + a.ch; ++ya) {
        const long long dmin = ya < bl ? bl - ya : ya > bh ? ya - bh : 0;
        if (dmin * dmin >= best) continue;
        const uint32_t* ra = a.w + (size_t)(ya - a.ry0) * a.cw;
        const int start = ya < bl ? bl : ya > bh ? bh : ya;
        for (int dir = 0; dir < 2; ++dir) {
            for (int yb = dir ? start - 1 : start; yb >= bl && yb <= bh; yb += dir ? -1 : 1) {
                const long long dy = yb - ya;
                if (dy * dy >= best) break;
                const int g = emia_nb_row_gap(ra, a.wc0, a.cw, b.w + (size_t)(yb - b.ry0) * b.cw, b.wc0, b.cw);
                if (g == INT_MAX) continue;
                const long long d = dy * dy + (long long)g * g;
                if (d < best) best = d;
            }
        }
    }
    return best;
}

EMIA_HD int emia_nb_cell_of(double c, int cs, int g) {
    const int v = (int)floor(c) / cs;
    return v < g ? v : g - 1;
}

// least squared distance, in the computed binary64 d2 = dx * dx + dy * dy, that a centroid outside rings 0..r around the query's
// cell can have.  Such a centroid lies in a cell column or row r + 1 or more away: |dx| or |dy| > r * cs exactly, and rounding is
// monotone, so its computed d2 is >= (r * cs)^2, which is an exact double.  The search stops only when this exceeds the best d2:
// a candidate at exactly the best d2 may still be ahead and have a lower index.
EMIA_HD bool emia_nb_ring_done(int r, int cs, double best_d2) {
    const double lb = (double)r * (double)cs;
    return lb * lb > best_d2;
}

// centroid nearest neighbour of listed instance i: the candidate of least d2, ties to the lowest index; -1 when there is none.
// Centroid k is (cent[stride * k], cent[stride * k + 1]).
EMIA_HD int emia_nb_nearest(int i, const double* cent, int stride, const int32_t* key, const int64_t* cell_off, const int32_t* ent,
                            EmiaNbGrid g, double* d2_out) {
    const double cx = cent[(int64_t)stride * i], cy = cent[(int64_t)stride * i + 1];
    const int qx = emia_nb_cell_of(cx, g.cs, g.gx), qy = emia_nb_cell_of(cy, g.cs, g.gy);
    const int64_t plane = (int64_t)key[i] * g.gx * g.gy;
    int best_k = -1;
    double best = 0.0;
    const int rmax = emia_max(emia_max(qx, g.gx - 1 - qx), emia_max(qy, g.gy - 1 - qy));
    for (int r = 0; r <= rmax; ++r) {
        for (int y = qy - r; y <= qy + r; ++y) {
            if (y < 0 || y >= g.gy) continue;
            const bool edge_row = y == qy - r || y == qy + r;
            for (int x = qx - r; x <= qx + r; x += edge_row ? 1 : 2 * r) {
                if (x >= 0 && x < g.gx) {
                    const int64_t c = plane + (int64_t)y * g.gx + x;
                    for (int64_t e = cell_off[c]; e < cell_off[c + 1]; ++e) {
                        const int k = ent[e];
                        if (k == i) continue;
                        const double kx = cent[(int64_t)stride * k], ky = cent[(int64_t)stride * k + 1];
                        if (emia_nb_cell_of(kx, g.cs, g.gx) != x || emia_nb_cell_of(ky, g.cs, g.gy) != y) continue;
                        const double dx = kx - cx, dy = ky - cy;
                        const double d2 = dx * dx + dy * dy;
                        if (best_k < 0 || d2 < best || (d2 == best && k < best_k)) { best = d2; best_k = k; }
                    }
                }
                if (r == 0) break;
            }
        }
        if (best_k >= 0 && emia_nb_ring_done(r, g.cs, best)) break;
    }
    *d2_out = best;
    return best_k;
}

EMIA_HD EmiaNbCrop emia_nb_crop(const uint32_t* crops, const int32_t* meta, const int64_t* crop_off, int k) {
    const int32_t* m = meta + 8 * (int64_t)k;
    EmiaNbCrop c;
    c.w = crops + crop_off[k]; c.ry0 = m[0]; c.wc0 = m[1]; c.ch = m[2]; c.cw = m[3];
    return c;
}

// least integer s with s * s >= v
EMIA_HD int emia_nb_ceil_sqrt(long long v) {
    long long s = (long long)sqrt((double)v);
    while (s * s < v) ++s;
    while (s > 0 && (s - 1) * (s - 1) >= v) --s;
    return (int)s;
}

// closest mask of listed instance i, given its centroid nearest neighbour nn (>= 0): least D2, ties to the lowest index; counts the
// candidates with D2 <= 2 and calls touch(k) for each.  D2(i, nn) bounds the search: a candidate that beats or ties it is at most
// R = ceil(sqrt(D2(i, nn))) pixels from i's bbox along both axes, so its bbox meets i's bbox grown by R, and its bbox gap (an exact
// lower bound of D2) decides whether its pixels are looked at.  Each candidate is seen once: in the first grid cell of the query
// rectangle that its bbox covers.
template <class Touch>
EMIA_HD int emia_nb_closest(int i, int nn, const uint32_t* crops, const int32_t* meta, const int64_t* crop_off, const int32_t* bbox,
                            const int32_t* key, const int64_t* cell_off, const int32_t* ent, EmiaNbGrid g, long long* d2_out,
                            int* touching, Touch touch) {
    const EmiaNbCrop a = emia_nb_crop(crops, meta, crop_off, i);
    const int ay0 = bbox[4 * i], ax0 = bbox[4 * i + 1], ay1 = bbox[4 * i + 2], ax1 = bbox[4 * i + 3];
    long long best = emia_nb_pair_d2(a, emia_nb_crop(crops, meta, crop_off, nn), LLONG_MAX);
    int best_k = nn, nt = 0;
    const int R = emia_max(emia_nb_ceil_sqrt(best), 1);
    const int qx0 = emia_max(ax0 - R, 0) / g.cs, qy0 = emia_max(ay0 - R, 0) / g.cs;
    const int qx1 = emia_min((ax1 + R) / g.cs, g.gx - 1), qy1 = emia_min((ay1 + R) / g.cs, g.gy - 1);
    const int64_t plane = (int64_t)key[i] * g.gx * g.gy;
    for (int y = qy0; y <= qy1; ++y)
        for (int x = qx0; x <= qx1; ++x) {
            const int64_t c = plane + (int64_t)y * g.gx + x;
            for (int64_t e = cell_off[c]; e < cell_off[c + 1]; ++e) {
                const int k = ent[e];
                if (k == i) continue;
                const int* kb = bbox + 4 * (int64_t)k;
                if (emia_max(kb[1] / g.cs, qx0) != x || emia_max(kb[0] / g.cs, qy0) != y) continue;
                const long long gx = emia_max(emia_max(kb[1] - ax1, ax0 - kb[3]), 0);
                const long long gy = emia_max(emia_max(kb[0] - ay1, ay0 - kb[2]), 0);
                const long long lim = best > 2 ? best : 2;
                if (gx * gx + gy * gy > lim) continue;
                long long limit = k < best_k ? best + 1 : best;
                if (limit < 3) limit = 3;
                const long long d = emia_nb_pair_d2(a, emia_nb_crop(crops, meta, crop_off, k), limit);
                if (d < best || (d == best && k < best_k)) { best = d; best_k = k; }
                if (d <= 2) { ++nt; touch(k); }
            }
        }
    *d2_out = best;
    *touching = nt;
    return best_k;
}

// ---- union-find over the touching edges (ECL-CC style): a root is hooked under the LOWER root only, so parent[x] <= x always and
// every component's root is its lowest member, whatever order the edges come in.
EMIA_HD int emia_nb_cas(int32_t* p, int32_t cmp, int32_t val) {
#if defined(__CUDA_ARCH__)
    return atomicCAS((int*)p, cmp, val);
#else
    const int32_t old = *p;
    if (old == cmp) *p = val;
    return old;
#endif
}

EMIA_HD int emia_nb_find(int32_t* parent, int x) {
    for (;;) {
        const int p = ((volatile int32_t*)parent)[x];
        if (p == x) return x;
        const int gp = ((volatile int32_t*)parent)[p];
        if (gp != p) parent[x] = gp;                   // path halving: x is not a root, so no hook can target it
        x = gp;
    }
}

EMIA_HD void emia_nb_unite(int32_t* parent, int a, int b) {
    for (;;) {
        a = emia_nb_find(parent, a);
        b = emia_nb_find(parent, b);
        if (a == b) return;
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = emia_nb_cas(parent + b, b, a);
        if (old == b) return;
        b = old;
    }
}
