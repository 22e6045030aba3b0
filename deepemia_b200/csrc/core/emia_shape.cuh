// emia_shape.cuh — shape descriptors of one external contour (host/device): area, convex hull area and perimeter, solidity,
// convexity, largest and smallest caliper (Feret) diameter, direction of the largest one, centroid.
//
// No reference counterpart: these are the opt-in columns after "File name" in measurements_results.csv, and oracle/shape.py states
// their definitions in numpy + OpenCV.  Every value is exact up to correctly rounded sqrt / division (and atan2 for the angle):
//   area, hull area        : integer shoelace (emia_contour_area), i.e. cv2.contourArea
//   hull perimeter         : cv2.arcLength on the canonical hull (emia_arc_length_closed: float32 segments, double sum starting with
//                            the closing segment) — the hull is rotated to start at its smallest (y, x) vertex, because the start
//                            changes the rounding of the sum and cv2.convexHull's start is not a function of the coordinates alone
//   Feret diameters        : int64 squared distances / cross products over the hull vertices
//   centroid               : cv2.moments' contourMoments — a00, a10, a01 are exact integers, scaled by +-1/2 and +-1/6
#pragma once
#include "emia_common.cuh"
#include "emia_contour.cuh"
#include "emia_hull.cuh"

enum EmiaShapeField {
    EMIA_S_AREA = 0,             // "Area"                (A * u) * u
    EMIA_S_CONVEX_AREA = 1,      // "Convex area"         (Ah * u) * u
    EMIA_S_SOLIDITY = 2,         // "Solidity"            A / Ah
    EMIA_S_CONVEX_PERIMETER = 3, // "Convex perimeter"    Ph * u
    EMIA_S_CONVEXITY = 4,        // "Convexity"           Ph / P
    EMIA_S_MAX_FERET = 5,        // "Max Feret diameter"  sqrt(D2) * u
    EMIA_S_MIN_FERET = 6,        // "Min Feret diameter"  min over hull edges of the farthest hull vertex from the edge's line, * u
    EMIA_S_FERET_ANGLE = 7,      // "Feret angle"         degrees in [0, 180) of the max-Feret direction, y up
    EMIA_S_CENTROID_X = 8,       // "Centroid X"          m10 / m00, frame pixels
    EMIA_S_CENTROID_Y = 9,       // "Centroid Y"          m01 / m00, frame pixels
    EMIA_S_COUNT = 10
};

// Fill out[EMIA_S_COUNT] for one contour of n >= 1 vertices (OpenCV order).  scratch: 28 n + 8 bytes, 8-byte aligned — the carve-up of
// emia_measure_contour, so a contour's emia_measure_scratch_bytes(n) sub-block serves both.
EMIA_HD_NOINLINE void emia_shape_contour(const uint32_t* pts, int n, double um_pix, void* scratch, double* out) {
    const double area = emia_contour_area(pts, n);
    const double perimeter = emia_arc_length_closed(pts, n);

    long long a00 = 0, a10 = 0, a01 = 0;
    int px = EMIA_PT_X(pts[n - 1]), py = EMIA_PT_Y(pts[n - 1]);
    for (int i = 0; i < n; ++i) {
        const int x = EMIA_PT_X(pts[i]), y = EMIA_PT_Y(pts[i]);
        const long long dxy = (long long)px * y - (long long)x * py;
        a00 += dxy;
        a10 += dxy * (px + x);
        a01 += dxy * (py + y);
        px = x; py = y;
    }
    const double s2 = a00 > 0 ? 0.5 : -0.5, s6 = a00 > 0 ? 0.16666666666666666 : -0.16666666666666666;
    const double m00 = (double)a00 * s2;

    uint64_t* keys = (uint64_t*)scratch;               // 8n   (later: the canonical hull, packed)
    int* stack = (int*)(keys + 2 * n);                 // 4(n+2)
    int* hull = stack + (n + 2);                       // 4n
    int* tmp = hull + n;                               // 4n
    const int nh = emia_convex_hull(pts, n, /*clockwise=*/0, keys, stack, hull, tmp);
    int s = 0;
    for (int i = 1; i < nh; ++i) {
        const uint32_t a = pts[hull[i]], b = pts[hull[s]];
        if (EMIA_PT_Y(a) < EMIA_PT_Y(b) || (EMIA_PT_Y(a) == EMIA_PT_Y(b) && EMIA_PT_X(a) < EMIA_PT_X(b))) s = i;
    }
    uint32_t* h = (uint32_t*)keys;
    for (int i = 0; i < nh; ++i) h[i] = pts[hull[s + i < nh ? s + i : s + i - nh]];
    const double harea = emia_contour_area(h, nh);
    const double hperim = emia_arc_length_closed(h, nh);

    // largest squared distance between hull vertices; among the pairs that reach it, the direction (dx, -dy) turned into
    // [0, 180) degrees with the smallest angle (exact: sign of the integer cross product), so that no vertex order matters
    long long d2max = 0;
    long long vx = 1, vy = 0;
    for (int i = 0; i < nh; ++i) {
        const long long xi = EMIA_PT_X(h[i]), yi = EMIA_PT_Y(h[i]);
        for (int j = i + 1; j < nh; ++j) {
            const long long dx = (long long)EMIA_PT_X(h[j]) - xi, dy = (long long)EMIA_PT_Y(h[j]) - yi;
            const long long d2 = dx * dx + dy * dy;
            if (d2 < d2max) continue;
            long long ux = dx, uy = -dy;
            if (uy < 0 || (uy == 0 && ux < 0)) { ux = -ux; uy = -uy; }
            if (d2 > d2max || ux * vy - uy * vx > 0) { d2max = d2; vx = ux; vy = uy; }
        }
    }
    // smallest caliper width: over the hull edges, the distance of the farthest hull vertex from the edge's line
    double wmin = -1.0;
    for (int e = 0; e < nh; ++e) {
        const uint32_t a = h[e], b = h[e + 1 < nh ? e + 1 : 0];
        const long long ax = EMIA_PT_X(a), ay = EMIA_PT_Y(a);
        const long long ex = (long long)EMIA_PT_X(b) - ax, ey = (long long)EMIA_PT_Y(b) - ay;
        const long long l2 = ex * ex + ey * ey;
        if (l2 == 0) continue;
        long long cmax = 0;
        for (int k = 0; k < nh; ++k) {
            long long c = ex * ((long long)EMIA_PT_Y(h[k]) - ay) - ey * ((long long)EMIA_PT_X(h[k]) - ax);
            if (c < 0) c = -c;
            if (c > cmax) cmax = c;
        }
        const double w = (double)cmax / sqrt((double)l2);
        if (wmin < 0.0 || w < wmin) wmin = w;
    }
    if (wmin < 0.0) wmin = 0.0;

    out[EMIA_S_AREA] = (area * um_pix) * um_pix;
    out[EMIA_S_CONVEX_AREA] = (harea * um_pix) * um_pix;
    out[EMIA_S_SOLIDITY] = area / harea;
    out[EMIA_S_CONVEX_PERIMETER] = hperim * um_pix;
    out[EMIA_S_CONVEXITY] = hperim / perimeter;
    out[EMIA_S_MAX_FERET] = sqrt((double)d2max) * um_pix;
    out[EMIA_S_MIN_FERET] = wmin * um_pix;
    out[EMIA_S_FERET_ANGLE] = atan2((double)vy, (double)vx) * (180.0 / M_PI);
    out[EMIA_S_CENTROID_X] = ((double)a10 * s6) / m00;
    out[EMIA_S_CENTROID_Y] = ((double)a01 * s6) / m00;
}
