"""Mirror of the reference's src/utils/measurements.py::calculate_measurements (:114-233), computing in libemia.so.

Value types follow the reference as it executes under numpy 2.x (SURVEY Appendix A, Q14): the quantities derived from
``order_points`` (float32) are np.float32, the ellipse axes / Circularity / Chords Python floats, the rest np.float64."""
import numpy as np

from .. import engine

_F32 = ("Length", "Width", "Aspect_Ratio", "Roundness", "Feret_diam")
_PYFLOAT = ("major_axis_length", "minor_axis_length", "Circularity", "Chords")
_FIELDS = {"major_axis_length": engine.REC_MAJOR, "minor_axis_length": engine.REC_MINOR, "eccentricity": engine.REC_ECC,
           "Length": engine.REC_LENGTH, "Width": engine.REC_WIDTH, "CircularED": engine.REC_CED, "Aspect_Ratio": engine.REC_ASPECT,
           "Circularity": engine.REC_CIRC, "Chords": engine.REC_CHORDS, "Feret_diam": engine.REC_FERET, "Roundness": engine.REC_ROUND,
           "Sphericity": engine.REC_SPHER}
# the opt-in columns after "File name" (no reference counterpart): engine.shape_descriptors / core/emia_shape.cuh
SHAPE_HEADER = ["Area", "Convex area", "Solidity", "Convex perimeter", "Convexity", "Max Feret diameter", "Min Feret diameter",
                "Feret angle", "Centroid X", "Centroid Y"]
# the columns of the opt-in neighbours_results.csv (no reference counterpart): engine.neighbours / core/emia_neighbour.cuh
NEIGHBOUR_HEADER = ["Instance_ID", "Class", "Class_Name", "Centroid X", "Centroid Y", "Nearest neighbour", "Nearest neighbour distance",
                    "Closest neighbour", "Edge distance", "Touching neighbours", "Agglomerate", "Agglomerate size", "Detected scale bar",
                    "File name"]
KEY_ORDER = ["major_axis_length", "minor_axis_length", "eccentricity", "Length", "Width", "CircularED", "Aspect_Ratio", "Circularity",
             "Chords", "Feret_diam", "Roundness", "Sphericity", "contrast_d10", "contrast_d50", "contrast_d90"]


def record_to_dict(rec, n_vertices=None):
    """One 16-double record (engine.REC_* order) -> the reference's measurement dict (15 keys, :217-233)."""
    out = {}
    for k, f in _FIELDS.items():
        v = float(rec[f])
        if k in _F32:
            out[k] = np.float32(v)
        elif k in _PYFLOAT:
            out[k] = v
        else:
            out[k] = np.float64(v)
    nv = int(rec[engine.REC_NVERT]) if n_vertices is None else n_vertices
    if nv < 5:                                    # no ellipse fit below 5 points (:176): the reference stores int 0
        out["major_axis_length"] = out["minor_axis_length"] = out["eccentricity"] = 0
    out["contrast_d10"] = out["contrast_d50"] = out["contrast_d90"] = None
    return {k: out[k] for k in KEY_ORDER}


def calculate_measurements(c, single_im_mask, um_pix=1.0, pixelsPerMetric=1.0, original_image=None,
                           measure_contrast_distribution=False):
    """calculate_measurements (src/utils/measurements.py:114-233) for one OpenCV contour `c` ([K,1,2] int32)."""
    if pixelsPerMetric != 1 and pixelsPerMetric != 1.0:
        raise ValueError("pixelsPerMetric is always 1 in the reference (src/functions/inference.py:1174); other values are unsupported")
    rec = engine.measure_contours([np.asarray(c).reshape(-1, 2)], um_pix=um_pix)[0].cpu().numpy()
    out = record_to_dict(rec, n_vertices=len(c))
    if measure_contrast_distribution and original_image is not None:
        from .contrast import contrast_percentiles
        out["contrast_d10"], out["contrast_d50"], out["contrast_d90"] = contrast_percentiles(original_image, single_im_mask)
    return out


def shape_descriptors(c, um_pix=1.0):
    """The SHAPE_HEADER values of one OpenCV contour `c` ([K,1,2] or [K,2] int), as {column: float}: area, convex hull area and
    perimeter, solidity, convexity, max / min Feret diameter and the max-Feret angle (degrees in [0, 180), y up), centroid in pixels.
    Computed in libemia.so without an area gate; lengths and areas are scaled by um_pix."""
    vals = engine.shape_contours([np.asarray(c).reshape(-1, 2)], um_pix=um_pix)[0].cpu().numpy()
    return {k: float(v) for k, v in zip(SHAPE_HEADER, vals)}


# ---- colour -> wavelength helpers (src/utils/measurements.py:32-111; no caller in the reference, kept for API completeness) --------
def rgb_to_hsv(r, g, b):
    """src/utils/measurements.py:32-80: OpenCV-style HSV (hue halved to 0..180, s and v scaled to 0..255)."""
    MAX_PIXEL_VALUE = 255.0
    r = r / MAX_PIXEL_VALUE
    g = g / MAX_PIXEL_VALUE
    b = b / MAX_PIXEL_VALUE
    max_val = max(r, g, b)
    min_val = min(r, g, b)
    v = max_val
    if max_val == 0.0 or (max_val - min_val) == 0.0:
        s = 0
        h = 0
    else:
        s = (max_val - min_val) / max_val
        if max_val == r:
            h = 60 * ((g - b) / (max_val - min_val)) + 0
        elif max_val == g:
            h = 60 * ((b - r) / (max_val - min_val)) + 120
        else:
            h = 60 * ((r - g) / (max_val - min_val)) + 240
    if h < 0:
        h = h + 360.0
    return h / 2, s * MAX_PIXEL_VALUE, v * MAX_PIXEL_VALUE


def hue_to_wavelength(hue):
    """src/utils/measurements.py:83-96."""
    assert hue >= 0
    assert hue <= 270
    return 620 - 170 / 270 * hue


def rgb_to_wavelength(r, g, b):
    """src/utils/measurements.py:97-111."""
    h, s, v = rgb_to_hsv(r, g, b)
    return hue_to_wavelength(h)


def instance_wavelengths(iset, image_bgr):
    """Wavelength (nm) of the MEAN colour of the image pixels under every instance: the per-instance `Wavelength_nm` the
    reference's README advertises but no reference code computes (SURVEY Appendix A, Q9).  The colour sums come from the GPU
    as exact integers (engine.color_sums); empty masks give None."""
    sums = engine.color_sums(iset, image_bgr).cpu().numpy()
    out = []
    for sb, sg, sr, cnt in sums:
        out.append(None if cnt == 0 else rgb_to_wavelength(int(sr) / int(cnt), int(sg) / int(cnt), int(sb) / int(cnt)))
    return out
