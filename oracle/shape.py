"""Oracle: the opt-in shape columns of measurements_results.csv (numpy/OpenCV; test infrastructure only).

A DEFINITION, not a restatement: the reference has no counterpart (it writes no area, hull, Feret or centroid column).  One row per
measured record: an external contour ``c`` (OpenCV vertex order) whose ``contourArea`` passes the measurement loop's area gate.
``A = cv2.contourArea(c)``, ``P = cv2.arcLength(c, True)``, ``u = um_pix``; float64 unless noted.

  Area                (A * u) * u
  Convex area         (Ah * u) * u,  Ah = cv2.contourArea(h)
  Solidity            A / Ah
  Convex perimeter    Ph * u,        Ph = cv2.arcLength(h, True)
  Convexity           Ph / P
  Max Feret diameter  sqrt(D2) * u,  D2 = largest squared distance between two hull vertices (int64)
  Min Feret diameter  min over hull edges (a, b) of max_k |(b - a) x (h_k - a)| / sqrt(|b - a|^2), * u (int64 cross products)
  Feret angle         degrees in [0, 180) of the max-Feret direction with y up; ties between maximal pairs: each pair's (dx, -dy)
                      turned into the half-plane y > 0 or (y == 0 and x > 0), the one with the smallest angle (exact integer
                      comparison), then atan2(y, x) * (180 / pi)
  Centroid X, Y       m10 / m00, m01 / m00 of cv2.moments(c), frame pixels (not scaled by u)

The canonical hull ``h`` is cv2.convexHull(c) (default orientation, no collinear vertices) rotated to start at its smallest (y, x)
vertex: the start changes the rounding of Ph.
"""
import math

import cv2
import numpy as np

SHAPE_HEADER = ["Area", "Convex area", "Solidity", "Convex perimeter", "Convexity", "Max Feret diameter", "Min Feret diameter",
                "Feret angle", "Centroid X", "Centroid Y"]


def canonical_hull(c):
    """int64 [k, 2] vertices of cv2.convexHull(c), starting at the smallest (y, x)."""
    h = cv2.convexHull(np.asarray(c, np.int32).reshape(-1, 1, 2)).reshape(-1, 2).astype(np.int64)
    s = int(np.lexsort((h[:, 0], h[:, 1]))[0])
    return np.roll(h, -s, axis=0)


def feret(h):
    """(D2, (vx, vy), min width in pixels) of the canonical hull h (int64 [k, 2])."""
    d = h[:, None, :] - h[None, :, :]
    d2 = (d * d).sum(-1)
    D2 = int(d2.max())
    best = None
    for i, j in zip(*np.nonzero(np.triu(d2 == D2, 1))):
        dx, dy = int(h[j, 0] - h[i, 0]), int(h[j, 1] - h[i, 1])
        vx, vy = dx, -dy
        if vy < 0 or (vy == 0 and vx < 0):
            vx, vy = -vx, -vy
        if best is None or vx * best[1] - vy * best[0] > 0:
            best = (vx, vy)
    if best is None:
        best = (1, 0)
    wmin = None
    for e in range(len(h)):
        a, b = h[e], h[(e + 1) % len(h)]
        ex, ey = int(b[0] - a[0]), int(b[1] - a[1])
        l2 = ex * ex + ey * ey
        if l2 == 0:
            continue
        cross = np.abs(ex * (h[:, 1] - a[1]) - ey * (h[:, 0] - a[0]))
        w = float(int(cross.max())) / math.sqrt(float(l2))
        if wmin is None or w < wmin:
            wmin = w
    return D2, best, 0.0 if wmin is None else wmin


def shape_descriptors(c, um_pix=1.0):
    """The ten shape values (SHAPE_HEADER order, Python floats) of one contour c ([K, 2] or OpenCV's [K, 1, 2])."""
    c = np.asarray(c, np.int32).reshape(-1, 1, 2)
    u = float(um_pix)
    A = cv2.contourArea(c)
    P = cv2.arcLength(c, True)
    h = canonical_hull(c)
    hc = h.astype(np.int32).reshape(-1, 1, 2)
    Ah = cv2.contourArea(hc)
    Ph = cv2.arcLength(hc, True)
    D2, (vx, vy), wmin = feret(h)
    M = cv2.moments(c)
    return [(A * u) * u, (Ah * u) * u, A / Ah, Ph * u, Ph / P, math.sqrt(float(D2)) * u, wmin * u,
            math.atan2(float(vy), float(vx)) * (180.0 / math.pi), M["m10"] / M["m00"], M["m01"] / M["m00"]]
