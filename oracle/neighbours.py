"""Oracle: neighbours_results.csv (numpy/scipy; test infrastructure only).

A DEFINITION, not a restatement: the reference has no counterpart (it writes nothing about how particles sit relative to each other).

Per image, the LISTED instances are those with at least one measured record: exactly the instances with rows in
measurements_results.csv, so both files share ``Instance_ID``.  Two instances are CANDIDATES for each other when both are listed, are
not the same instance and have the same (Class, Class_Name) entry of the class table.  ``u = um_pix``; binary64, no fused
multiply-add.  One row per listed instance, in instance order:

  Centroid X, Y               m10 / m00, m01 / m00 of the mask (exact integer sums, one division), frame pixels
  Nearest neighbour           the candidate j of least d2 = dx * dx + dy * dy, dx = cx_j - cx_i, dy = cy_j - cy_i; ties to the lowest
                              index; empty without a candidate
  Nearest neighbour distance  sqrt(d2) * u; empty without a candidate
  Closest neighbour           the candidate of least D2, ties to the lowest index; D2 = least (x - x')^2 + (y - y')^2 (an integer)
                              between a pixel of this mask and a pixel of that mask; empty without a candidate
  Edge distance               sqrt(float(D2)) * u (0.0 when the masks share a pixel); empty without a candidate
  Touching neighbours         the number of candidates with D2 <= 2 (a shared pixel or 8-adjacent)
  Agglomerate                 the lowest-index member of the instance's connected component in the graph of D2 <= 2 edges
  Agglomerate size            the number of members of that component

An instance is given as a PIECE ``(y0, x0, m)``: the bool array ``m`` placed with its top-left pixel at frame (x0, y0).  The only
pruning used here is the bbox gap: g2 = gx^2 + gy^2 with gx, gy the gaps between the two tight bboxes along x and y, which is <= D2.
Results are arrays of the device layout: ``nbf`` float64 [n, 4] (centroid x, y, nearest-neighbour distance, edge distance; NaN for
empty) and ``nbi`` int64 [n, 6] (listed, nearest neighbour, closest neighbour (-1: none), touching, agglomerate (-1: not listed),
agglomerate size).
"""
import math

import numpy as np
from scipy import ndimage

NEIGHBOUR_HEADER = ["Instance_ID", "Class", "Class_Name", "Centroid X", "Centroid Y", "Nearest neighbour", "Nearest neighbour distance",
                    "Closest neighbour", "Edge distance", "Touching neighbours", "Agglomerate", "Agglomerate size", "Detected scale bar",
                    "File name"]


def tight(piece):
    """(y0, x0, m) -> the same piece cut to the tight bbox of its set pixels; bbox (y_min, x_min, y_max, x_max) inclusive."""
    y0, x0, m = piece
    ys, xs = np.nonzero(m)
    m = m[ys.min():ys.max() + 1, xs.min():xs.max() + 1]
    return (y0 + int(ys.min()), x0 + int(xs.min()), m)


def centroid(piece):
    y0, x0, m = piece
    ys, xs = np.nonzero(m)
    m00 = len(ys)
    m10 = int((xs.astype(np.int64) + x0).sum())
    m01 = int((ys.astype(np.int64) + y0).sum())
    return float(m10) / float(m00), float(m01) / float(m00)


def bbox_gap2(a, b):
    """Squared bbox gap of two tight pieces: a lower bound of their D2."""
    ay0, ax0, am = a
    by0, bx0, bm = b
    gx = max(bx0 - (ax0 + am.shape[1] - 1), ax0 - (bx0 + bm.shape[1] - 1), 0)
    gy = max(by0 - (ay0 + am.shape[0] - 1), ay0 - (by0 + bm.shape[0] - 1), 0)
    return gx * gx + gy * gy


def pair_d2(a, b):
    """D2 of two pieces: the exact Euclidean distance transform of the complement of b over the window of both bboxes gives each
    pixel its nearest pixel of b; D2 is the least integer squared offset to it over the pixels of a."""
    ay0, ax0, am = a
    by0, bx0, bm = b
    y0, x0 = min(ay0, by0), min(ax0, bx0)
    y1, x1 = max(ay0 + am.shape[0], by0 + bm.shape[0]), max(ax0 + am.shape[1], bx0 + bm.shape[1])
    B = np.zeros((y1 - y0, x1 - x0), bool)
    B[by0 - y0:by0 - y0 + bm.shape[0], bx0 - x0:bx0 - x0 + bm.shape[1]] = bm
    ys, xs = np.nonzero(am)
    ys = ys + (ay0 - y0)
    xs = xs + (ax0 - x0)
    if B[ys, xs].any():
        return 0
    iy, ix = ndimage.distance_transform_edt(~B, return_distances=False, return_indices=True)
    dy = ys.astype(np.int64) - iy[ys, xs]
    dx = xs.astype(np.int64) - ix[ys, xs]
    return int((dy * dy + dx * dx).min())


class Neighbours:
    """The relations of one image.  pieces: one per instance (None or an empty mask for an instance that is not listed);
    listed: bool per instance; class_idx: the class-table index per instance."""

    def __init__(self, pieces, listed, class_idx):
        self.n = len(pieces)
        self.listed = np.asarray(listed, bool).copy()
        self.cls = np.asarray(class_idx, np.int64)
        self.pieces = [tight(p) if ok else None for p, ok in zip(pieces, self.listed)]
        self.cent = np.full((self.n, 2), np.nan)
        self.box = np.zeros((self.n, 4), np.int64)
        for i, p in enumerate(self.pieces):
            if p is not None:
                self.cent[i] = centroid(p)
                self.box[i] = (p[0], p[1], p[0] + p[2].shape[0] - 1, p[1] + p[2].shape[1] - 1)
        self._touch = {}

    def candidates(self, i):
        return np.nonzero(self.listed & (self.cls == self.cls[i]) & (np.arange(self.n) != i))[0]

    def nearest(self, idx, chunk=2048):
        """(nearest neighbour, d2) of the listed instances idx, by brute force over every candidate, in chunks."""
        nn = np.full(len(idx), -1, np.int64)
        d2 = np.full(len(idx), np.nan)
        for a in range(0, len(idx), chunk):
            q = np.asarray(idx[a:a + chunk])
            dx = self.cent[None, :, 0] - self.cent[q, None, 0]
            dy = self.cent[None, :, 1] - self.cent[q, None, 1]
            d = dx * dx + dy * dy
            ok = self.listed[None, :] & (self.cls[None, :] == self.cls[q, None]) & (np.arange(self.n)[None, :] != q[:, None])
            d[~ok] = np.inf
            j = np.argmin(d, axis=1)                 # the first least value: the lowest index
            has = ok.any(1)
            nn[a:a + chunk] = np.where(has, j, -1)
            d2[a:a + chunk] = np.where(has, d[np.arange(len(q)), j], np.nan)
        return nn, d2

    def _gaps(self, i, cand):
        b = self.box[cand]
        gx = np.maximum(np.maximum(b[:, 1] - self.box[i, 3], self.box[i, 1] - b[:, 3]), 0)
        gy = np.maximum(np.maximum(b[:, 0] - self.box[i, 2], self.box[i, 0] - b[:, 2]), 0)
        return gx * gx + gy * gy

    def closest(self, i):
        """(closest neighbour, D2, touching candidates) of listed instance i; candidates in increasing bbox gap, stopped once the gap
        exceeds both the best D2 and 2."""
        cand = self.candidates(i)
        if len(cand) == 0:
            return -1, None, []
        g2 = self._gaps(i, cand)
        order = np.lexsort((cand, g2))
        best, best_k, touch = None, -1, []
        for j in order:
            k, g = int(cand[j]), int(g2[j])
            if best is not None and g > max(best, 2):
                break
            d = pair_d2(self.pieces[i], self.pieces[k])
            if best is None or d < best or (d == best and k < best_k):
                best, best_k = d, k
            if d <= 2:
                touch.append(k)
        self._touch[i] = touch
        return best_k, best, touch

    def touching(self, i):
        if i not in self._touch:
            cand = self.candidates(i)
            cand = cand[self._gaps(i, cand) <= 2]
            self._touch[i] = [int(k) for k in cand if pair_d2(self.pieces[i], self.pieces[k]) <= 2]
        return self._touch[i]

    def component(self, i):
        seen, todo = {i}, [i]
        while todo:
            for k in self.touching(todo.pop()):
                if k not in seen:
                    seen.add(k)
                    todo.append(k)
        return seen

    def rows(self, um_pix, idx=None):
        """(nbf, nbi) of the instances idx (default: all); rows of instances outside idx or not listed keep their defaults."""
        n = self.n
        nbf = np.full((n, 4), np.nan)
        nbi = np.zeros((n, 6), np.int64)
        nbi[:, 1:3] = -1
        nbi[:, 4] = -1
        nbi[:, 0] = self.listed
        nbf[:, :2] = self.cent
        idx = np.nonzero(self.listed)[0] if idx is None else np.asarray([i for i in idx if self.listed[i]], np.int64)
        nn, d2 = self.nearest(idx)
        for q, i in enumerate(idx):
            i = int(i)
            if nn[q] >= 0:
                nbi[i, 1] = nn[q]
                nbf[i, 2] = math.sqrt(d2[q]) * um_pix
                k, D2, touch = self.closest(i)
                nbi[i, 2] = k
                nbi[i, 3] = len(touch)
                nbf[i, 3] = math.sqrt(float(D2)) * um_pix
            comp = self.component(i)
            nbi[i, 4] = min(comp)
            nbi[i, 5] = len(comp)
        return nbf, nbi


def neighbours(pieces, listed, class_idx, um_pix=1.0, idx=None):
    """(nbf, nbi) of the definition above."""
    return Neighbours(pieces, listed, class_idx).rows(um_pix, idx)
