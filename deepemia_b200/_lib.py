"""ctypes binding of libemia.so (include/emia.h).  There is NO CPU fallback: importing the product path without the
built CUDA library raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("EMIA_LIB_PATH") or os.path.join(_HERE, "libemia.so")     # override: kernel-variant experiments

c_void_p, c_int, c_int64, c_float, c_double, c_size_t = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float,
                                                         ctypes.c_double, ctypes.c_size_t)


class EmiaError(RuntimeError):
    pass


_SIGNATURES = {
    "emia_version": (c_int, []),
    "emia_last_error": (ctypes.c_char_p, []),
    "emia_scan_workspace_bytes": (c_size_t, [c_int64]),
    "emia_exclusive_scan_i64": (c_int, [c_void_p, c_int64, c_void_p, c_size_t, c_void_p]),
    "emia_paste_plan": (c_int, [c_void_p, c_int64, c_float, c_float, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "emia_paste_threshold_bitpack": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float, c_int, c_int,
                                             c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "emia_mask_bbox": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "emia_mask_pack": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "emia_mask_unpack": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p]),
    "emia_contour_count": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "emia_contour_measure": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_double,
                                     c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "emia_contour_store": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p]),
    "emia_contour_trace_plan": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "emia_contour_trace_slab": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "emia_list_measure_plan": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p]),
    "emia_contour_measure_list": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_double, c_double,
                                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "emia_list_measure_order": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "emia_contour_shape_list": (c_int, [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_double, c_void_p,
                                        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "emia_contour_measure_stored": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_double, c_double,
                                            c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "emia_group_workspace_bytes": (c_size_t, [c_void_p, c_int]),
    "emia_dedup_smart": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_double, c_double, c_void_p, c_void_p, c_void_p,
                                 c_size_t, c_void_p]),
    "emia_dedup_inorder": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                                   c_double, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "emia_dedup_sorted": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                  c_void_p, c_double, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "emia_overlap_rules": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_size_t,
                                   c_void_p]),
    "emia_containment_rules": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_double, c_void_p, c_void_p, c_void_p,
                                       c_size_t, c_void_p]),
    "emia_morph_scratch_words": (c_size_t, []),
    "emia_morph_plan": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "emia_morph_grow_plan": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "emia_morph": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "emia_overlap_first_come": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "emia_crop_stats": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "emia_group_filter_area": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "emia_column_gate": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p,
                                 c_void_p, c_void_p]),
    "emia_resize_place_plan": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p,
                                       c_void_p]),
    "emia_resize_nearest_place": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_void_p, c_int,
                                          c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_void_p]),
    "emia_group_filter_flag": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "emia_rle_count": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "emia_rle_encode": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "emia_rle_line_count": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "emia_rle_line_index": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "emia_rle_parse_count": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "emia_rle_parse_fill": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p]),
    "emia_rle_decode_plan": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p]),
    "emia_rle_decode": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "emia_csv_rle_count": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "emia_csv_rle_write": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "emia_csv_measure_count": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "emia_csv_measure_write": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                       c_void_p]),
    "emia_csv_measure_shape_count": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                             c_void_p, c_void_p]),
    "emia_csv_measure_shape_write": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                             c_void_p, c_void_p, c_void_p]),
    "emia_neighbour_plan": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int,
                                    c_void_p, c_void_p, c_void_p, c_void_p]),
    "emia_neighbour_search": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int,
                                      c_void_p, c_void_p, c_double, c_void_p, c_void_p, c_void_p, c_void_p]),
    "emia_csv_neighbour_count": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "emia_csv_neighbour_write": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                         c_void_p]),
    "emia_coco_ann_count": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_int64,
                                    c_void_p, c_void_p]),
    "emia_coco_ann_write": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_int64,
                                    c_void_p, c_void_p, c_void_p]),
    "emia_coco_counts_count": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "emia_coco_counts_fill": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "emia_cocoeval_order_workspace_bytes": (c_size_t, [c_int64]),
    "emia_cocoeval_order": (c_int, [c_void_p] * 4 + [c_int64, c_int, c_int64] + [c_void_p] * 4 + [c_size_t, c_void_p]),
    "emia_cocoeval_grid": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "emia_cocoeval_pair_count": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int]
                                 + [c_void_p] * 6 + [c_int, c_void_p, c_void_p]),
    "emia_cocoeval_pair_fill": (c_int, [c_void_p] * 13 + [c_int64, c_int, c_int, c_int, c_int] + [c_void_p] * 15),
    "emia_cocoeval_match": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64] + [c_void_p] * 7 + [c_int64] + [c_void_p] * 5),
    "emia_cocoeval_accumulate": (c_int, [c_void_p] * 7 + [c_int64, c_int] + [c_void_p] * 5),
    "emia_moments01": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "emia_moments": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "emia_color_sums": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "emia_overlay": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_void_p,
                             c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "emia_gray_hist": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "emia_image_gray_hist": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "emia_pair_counts": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "emia_group_filter_heads": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_float, c_int,
                                        c_void_p, c_void_p, c_void_p]),
    "emia_group_mark_members": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int64, c_void_p]),
    "emia_group_flatten": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p]),
    "emia_unit_broadcast_i32": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_int, c_void_p, c_void_p]),
    "emia_scale_f32": (c_int, [c_void_p, c_float, c_int64, c_void_p, c_void_p]),
    "emia_gather_plan": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "emia_gather_crops": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p]),
    "emia_gather_b32": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "emia_capacity_guard": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p]),
    "emia_scalebar_edges": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                    c_void_p]),
    "emia_hough_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "emia_hough_lines_p": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                   c_void_p, c_size_t, c_void_p]),
    "emia_line_mean": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
}

EXPORTS = tuple(_SIGNATURES)
_lib = None


def load():
    """Load libemia.so (once).  Raises EmiaError when the CUDA library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EmiaError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().emia_last_error()
        raise EmiaError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")
