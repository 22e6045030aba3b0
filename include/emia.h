/* emia.h — C ABI of libemia.so: the B200 (sm_100a) post-head hot path of deepEMIA.
 *
 * The reference (Deam0on/deepEMIA) is pure Python and has no FFI; the functions below are what a ctypes binding
 * inside the reference's own modules would call instead of numpy/OpenCV/scipy (see INTEGRATION.md).  Each entry
 * cites the reference code it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises the host;
 *   - no allocation, no global state: scratch comes from caller-provided workspaces sized by *_bytes() queries;
 *   - return value: 0 = OK, negative = error (EMIA_ERR_*); emia_last_error() gives a thread-local message;
 *   - masks are bit-packed: bit j (LSB first) of 32-bit word w of a row is pixel x = 32*w + j.
 *
 * Instance layout
 *   An "instance" is one mask.  Its bits live in a CROP: rows [ry0, ry0+ch) x frame word-columns [wc0, wc0+cw),
 *   stored contiguously (ch*cw words) at crops + crop_off[i].  Crops are word-aligned with the frame, so two
 *   crops intersect with plain AND of words.  Optionally the same bits are also written into a full
 *   H x pitch_words FRAME (the drop-in equivalent of Detectron2's N x H x W `pred_masks`).
 *   Instances are grouped (one group = one image / tile / de-dup call) by cap_off[G+1]; the members of group g
 *   that are currently alive are idx[cap_off[g] .. cap_off[g]+len[g]) (instance ids, in list order).
 */
#ifndef EMIA_H
#define EMIA_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EMIA_OK 0
#define EMIA_ERR_BAD_ARG (-1)
#define EMIA_ERR_UNSUPPORTED (-2)
#define EMIA_ERR_LAUNCH (-3)
#define EMIA_ERR_WORKSPACE (-4)

#define EMIA_MASK_SIDE 28   /* Mask R-CNN mask head resolution */
#define EMIA_PASTE_PROBS_F16 (1 << 16)
#define EMIA_REC_FIELDS 16  /* doubles per measurement record, see emia_rec_field */

typedef struct emia_inst_meta {
    int32_t ry0;     /* first frame row of the crop */
    int32_t wc0;     /* first frame word-column of the crop */
    int32_t ch;      /* crop rows */
    int32_t cw;      /* crop words per row */
    int32_t rx0;     /* first frame pixel column that may be set */
    int32_t rx1;     /* one past the last frame pixel column that may be set */
    int32_t valid;   /* 0: dropped by Boxes.nonempty() (detector_postprocess) */
    int32_t reserved;
} emia_inst_meta;

/* order of the doubles in one measurement record (CSV columns of src/functions/inference.py:987-1010 + extras) */
enum emia_rec_field {
    EMIA_REC_MAJOR_AXIS = 0, EMIA_REC_MINOR_AXIS = 1, EMIA_REC_ECCENTRICITY = 2, EMIA_REC_LENGTH = 3,
    EMIA_REC_WIDTH = 4, EMIA_REC_CIRCULAR_ED = 5, EMIA_REC_ASPECT = 6, EMIA_REC_CIRCULARITY = 7,
    EMIA_REC_CHORDS = 8, EMIA_REC_FERET = 9, EMIA_REC_ROUNDNESS = 10, EMIA_REC_SPHERICITY = 11,
    EMIA_REC_AREA = 12, EMIA_REC_PERIMETER = 13, EMIA_REC_NVERT = 14, EMIA_REC_MEASURED = 15
};

int emia_version(void);
const char* emia_last_error(void);

/* ---- utilities ------------------------------------------------------------------------------------------- */
/* in-place exclusive prefix sum of data[0..n) with the total stored at data[n] (n+1 entries).
 * workspace: emia_scan_workspace_bytes(n) bytes (may be NULL: slower single-CTA path). */
size_t emia_scan_workspace_bytes(int64_t n);
int emia_exclusive_scan_i64(int64_t* data, int64_t n, void* workspace, size_t workspace_bytes, void* stream);

/* abort_flag (optional device int32, may be NULL) on the three entry points that WRITE variable-size outputs — paste, contour
 * tracing, list measurement: when *abort_flag != 0 at kernel start the call writes nothing.  It lets a host enqueue a whole step
 * without reading sizes back: buffers are sized from the previous step, a device-side comparison of the new totals with those
 * capacities raises the flag, and the host looks at it once, when it consumes the results (engine.TilePipeline). */

/* ---- K1: paste + threshold + bit-pack ----------------------------------------------------------------------
 * Replaces Detectron2 0.6 detector_postprocess + paste_masks_in_image(threshold 0.5) reached through
 * `predictor(image)` at src/functions/inference.py:1395,1398,1507,1669,2107, the D2H of pred_masks at :1401,
 * `np.sum(mask)` at :1683,:1800,:2604 and get_mask_bbox at :2722-2733.
 * emia_paste_plan: box scale/clip/non-empty + sampling region -> meta[i], crop_words[i] = ch*cw (caller scans).
 * emia_paste_threshold_bitpack: writes crops (+ full frames when frames != NULL: instance i goes to frame slot
 *   i % frame_slots), bbox[i] = (y_min, x_min, y_max, x_max) inclusive or (-1,-1,-1,-1), area[i] = popcount.
 *   variant (bits 0-7): 0 = 128-bit streaming stores, 1 = bulk shared->global copies (TMA engine);
 *   bits 8-15 of the same argument: resident CTAs per SM of the persistent grid (0 = default 8 / 4) — a smaller grid
 *   leaves SM room for the contour / de-dup kernels of the previous tile batch running on another stream.
 *   bit 16 (EMIA_PASTE_PROBS_F16): `probs` holds IEEE half values (what the mask head emits under the reference's AMP autocast,
 *   inference.py:1392-1396); they are widened exactly to float32 before sampling, as torch's grid_sample autocast does.
 *   meta / crop_off / probs / boxes / bbox / area may point INTO larger arrays (a batch of a bigger plan): crop_off
 *   values are absolute word offsets into `crops`. */
int emia_paste_plan(const float* boxes, int64_t n, float scale_x, float scale_y, int H, int W,
                    emia_inst_meta* meta, int64_t* crop_words, void* stream);
int emia_paste_threshold_bitpack(const float* probs, const float* boxes, const emia_inst_meta* meta,
                                 const int64_t* crop_off, int64_t n, float scale_x, float scale_y, int H, int W,
                                 uint32_t* frames, int64_t frame_slots, int pitch_words, uint32_t* crops,
                                 int32_t* bbox, int32_t* area, int variant, const int32_t* abort_flag, void* stream);

/* ---- mask import: byte masks -> crops (for callers that already hold H x W masks) ---------------------------
 * Replaces the reference's list-of-H x W-numpy-arrays representation (src/functions/inference.py:1401-1403,
 * :2413-2416).  emia_mask_bbox: bbox/area of n byte masks (non-zero = set) + meta + crop_words (caller scans);
 * emia_mask_pack: bit-pack the bbox crops. */
int emia_mask_bbox(const uint8_t* masks, int64_t n, int H, int W, emia_inst_meta* meta, int64_t* crop_words,
                   int32_t* bbox, int32_t* area, void* stream);
int emia_mask_pack(const uint8_t* masks, int64_t n, int H, int W, const emia_inst_meta* meta,
                   const int64_t* crop_off, uint32_t* crops, void* stream);
/* crops -> byte masks (0/1), full frame, for the drop-in list-of-arrays surface */
int emia_mask_unpack(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off,
                     const int32_t* idx, int64_t n_idx, int H, int W, uint8_t* masks_out, void* stream);

/* ---- K5: external contours + morphometry --------------------------------------------------------------------
 * Replaces cv2.findContours(RETR_EXTERNAL, CHAIN_APPROX_SIMPLE) + imutils.grab_contours at
 * src/functions/inference.py:1164-1167 and :2605, cv2.contourArea :1175, the min-area gate :1178-1190,
 * calculate_measurements src/utils/measurements.py:114-233 and cv2.arcLength(contours[0]) at inference.py:2607.
 * Pass 1 (emia_contour_count) sizes the outputs; the caller scans n_contours / n_points / scratch sizes.
 *   marks: 2 * total_crop_words words of scratch.
 *   scratch_bytes[i] = bytes of per-instance hull scratch needed by pass 2.
 * Pass 2 (emia_contour_measure): pts (packed x | y<<16, frame coordinates), cstart (per instance n_contours+1
 *   entries at cont_off[i] + i, relative to pt_off[i], DISCOVERY order), records in OpenCV order (reverse
 *   discovery) at cont_off[i] + j, rec_inst (instance id per record), perim0[i] = arcLength of the first
 *   returned contour (0 if none).  records[..][EMIA_REC_MEASURED] = 1 when contourArea >= min_area; like the reference,
 *   which skips such a contour before calculate_measurements, a record below the gate carries only EMIA_REC_AREA,
 *   EMIA_REC_PERIMETER and EMIA_REC_NVERT (everything else 0).  Pass min_area = 0 to measure every contour. */
int emia_contour_count(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, int64_t n,
                       uint32_t* marks, int64_t* n_contours, int64_t* n_points, int64_t* scratch_bytes,
                       void* stream);
int emia_contour_measure(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, int64_t n,
                         uint32_t* marks, const int64_t* cont_off, const int64_t* pt_off,
                         const int64_t* scratch_off, double um_pix, double min_area, uint32_t* pts,
                         int32_t* cstart, double* records, int32_t* rec_inst, double* perim0, uint8_t* scratch,
                         void* stream);

/* Pass 2 without the records: vertex lists + perim0 only (the records then come from emia_contour_measure_list). */
int emia_contour_store(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, int64_t n,
                       uint32_t* marks, const int64_t* cont_off, const int64_t* pt_off, uint32_t* pts, int32_t* cstart,
                       double* perim0, void* stream);

/* Single-pass variant (the fast path of engine.trace): emia_contour_trace_plan gives per-instance vertex capacities
 * (caller scans them into pt_cap_off), emia_contour_trace_slab follows the borders once into those slabs
 * (cstart_slab: cap_contours + 1 ints per instance) and raises *overflow (caller-zeroed counter) when a capacity is
 * exceeded — the caller then falls back to emia_contour_count / emia_contour_measure; emia_contour_measure_stored
 * computes the records from stored vertices (cstart_stride = cap_contours + 1 for slabs, 0 for the packed layout).
 * emia_contour_trace_slab first writes a per-crop seed (first foreground pixel, candidate count) into n_contours and then
 * overwrites it with the contour count of every instance; crops with exactly one external contour are followed without
 * the mark planes, so `marks` (2 words per crop word) needs no initial contents and is left undefined. */
int emia_contour_trace_plan(const emia_inst_meta* meta, int64_t n, int64_t* pt_cap, void* stream);
int emia_contour_trace_slab(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, int64_t n,
                            uint32_t* marks, const int64_t* pt_cap_off, int32_t cap_contours, uint32_t* pts,
                            int32_t* cstart_slab, int64_t* n_contours, int64_t* scratch_bytes, int32_t* overflow,
                            double* perim0 /* optional: arcLength(contours[0]) per instance */, const int32_t* abort_flag,
                            void* stream);
int emia_contour_measure_stored(const emia_inst_meta* meta, int64_t n, const int64_t* cont_off, const int64_t* pt_off,
                                const int32_t* cstart, int32_t cstart_stride, const int64_t* scratch_off, double um_pix,
                                double min_area, const uint32_t* pts, double* records, int32_t* rec_inst, double* perim0,
                                uint8_t* scratch, void* stream);

/* Measure only the members of G lists — the reference measures what survived de-duplication and the spatial
 * constraints (measurement loop src/functions/inference.py:1148-1253 runs over the final mask list).
 * emia_list_measure_plan: per list slot s (total_cap slots): item_inst[s] = instance id (-1 for a dead slot),
 *   rec_cnt[s] / scr_cnt[s] = number of records / scratch bytes (caller scans both, total_cap + 1 entries).
 * emia_contour_measure_list: records of slot s at rec_off[s] + j (OpenCV contour order), rec_inst = instance id per record.
 *   inst_cont_off (per instance) is only needed for the packed cstart layout (cstart_stride == 0).  order (optional, n_items
 *   entries from emia_list_measure_order; NULL = list order): the order in which the slots are WORKED ON — the results do not depend
 *   on it.
 * emia_list_measure_order: order[] = the slots sorted by vertex count, longest first, dead slots last (a warp is as slow as its
 *   longest contour); bins = 128 int32 of workspace (cleared inside).
 * emia_contour_shape_list: after emia_contour_measure_list on the same list (same arguments, its records and its scratch, whose
 *   contents it overwrites), shape[r][10] = the shape descriptors of record r (core/emia_shape.cuh: area, convex area, solidity,
 *   convex perimeter, convexity, max / min Feret diameter, Feret angle, centroid x / y); NaN for records below the area gate. */
int emia_list_measure_plan(const int32_t* cap_off, int32_t G, int32_t total_cap, const int32_t* in_len,
                           const int32_t* in_idx, const int64_t* n_contours, const int64_t* scratch_bytes,
                           int32_t* item_inst, int64_t* rec_cnt, int64_t* scr_cnt, void* stream);
int emia_contour_measure_list(int64_t n_items, const int32_t* item_inst, const int64_t* rec_off, const int64_t* scr_off,
                              const int64_t* inst_cont_off, const int64_t* pt_off, const int32_t* cstart,
                              int32_t cstart_stride, double um_pix, double min_area, const uint32_t* pts, double* records,
                              int32_t* rec_inst, uint8_t* scratch, const int32_t* abort_flag, const int32_t* order, void* stream);
int emia_list_measure_order(int64_t n_items, const int32_t* item_inst, const int64_t* rec_off, const int64_t* inst_cont_off,
                            const int32_t* cstart, int32_t cstart_stride, int32_t* order, int32_t* bins, void* stream);
int emia_contour_shape_list(int64_t n_items, const int32_t* item_inst, const int64_t* rec_off, const int64_t* scr_off,
                            const int64_t* inst_cont_off, const int64_t* pt_off, const int32_t* cstart, int32_t cstart_stride,
                            double um_pix, const uint32_t* pts, const double* records, uint8_t* scratch, const int32_t* order,
                            double* shape, void* stream);

/* ---- K4: mask-IoU de-duplication and spatial constraints ----------------------------------------------------
 * All operate on G groups at once; see "Instance layout".  total_cap = cap_off[G] (the host knows it).
 * Workspace size: emia_group_workspace_bytes (pass exactly that many bytes: the tail is cleared per call).
 * max_cap = largest group capacity if the caller knows it (0 = unknown): groups of <= 1024 slots take the fast path — one
 *   CTA per group with the member tables, the suppression bit matrix and the candidate-pair queue in shared memory and
 *   eight lanes per candidate pair for the mask intersection; larger groups (the global de-dup of a whole micrograph,
 *   inference.py:2472) take the sparse path: rank by counting, x-sorted sweep with one warp per member, a sparse edge list and a
 *   fixed-point resolution of the greedy loop (csrc/emia_group_sparse.cuh).
 * emia_dedup_smart       : deduplicate_masks_smart, src/functions/inference.py:2552-2677 (+ :2680-2733), incl. the
 *                          artifact pre-filter (empty / aspect / compactness < 0.15) and quirks Q1, Q2, Q10.
 *                          Output in keep order (score descending).
 * emia_dedup_inorder     : greedy in-order de-dup with iou(), inference.py:1453-1459 (:422-435); also :2241-2246.
 * emia_overlap_rules     : filter_by_overlap_rules, src/utils/spatial_constraints.py:192-277.
 *                          rule_active[c] != 0 -> class c has an enforced rule with threshold rule_max_iou[c].
 * emia_containment_rules : filter_by_containment_rules, spatial_constraints.py:280-398 (rules applied in order). */
size_t emia_group_workspace_bytes(const int32_t* cap_off_host, int32_t G);
int emia_dedup_smart(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off,
                     const int32_t* bbox, const int32_t* area, const double* perim0, const int64_t* n_contours,
                     const float* scores, const int32_t* classes, const int32_t* cap_off, int32_t G,
                     int32_t total_cap, int32_t max_cap, const int32_t* in_len, const int32_t* in_idx, double iou_threshold, double max_aspect_ratio,
                     int32_t* out_len, int32_t* out_idx, void* workspace, size_t workspace_bytes, void* stream);
int emia_dedup_inorder(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off,
                       const int32_t* bbox, const int32_t* area, const int32_t* cap_off, int32_t G,
                       int32_t total_cap, int32_t max_cap, const int32_t* in_len, const int32_t* in_idx, double iou_threshold, int32_t* out_len,
                       int32_t* out_idx, void* workspace, size_t workspace_bytes, void* stream);
/* emia_dedup_sorted: score-sorted greedy de-dup with iou() (run_adaptive_multiscale_inference, inference.py:1964-1978) */
int emia_dedup_sorted(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, const int32_t* bbox,
                      const int32_t* area, const float* scores, const int32_t* cap_off, int32_t G, int32_t total_cap,
                      int32_t max_cap, const int32_t* in_len, const int32_t* in_idx, double iou_threshold, int32_t* out_len,
                      int32_t* out_idx, void* workspace, size_t workspace_bytes, void* stream);
int emia_overlap_rules(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off,
                       const int32_t* bbox, const int32_t* area, const float* scores, const int32_t* classes,
                       const int32_t* cap_off, int32_t G, int32_t total_cap, int32_t max_cap, const int32_t* in_len, const int32_t* in_idx,
                       const int32_t* rule_active, const double* rule_max_iou, int32_t num_classes,
                       int32_t* out_len, int32_t* out_idx, void* workspace, size_t workspace_bytes, void* stream);
int emia_containment_rules(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off,
                           const int32_t* bbox, const int32_t* area, const int32_t* classes,
                           const int32_t* cap_off, int32_t G, int32_t total_cap, int32_t max_cap, const int32_t* in_len, const int32_t* in_idx,
                           const int32_t* child_class_host, const int32_t* parent_class_host, int32_t n_rules,
                           double containment_threshold, int32_t* out_len, int32_t* out_idx, void* workspace,
                           size_t workspace_bytes, void* stream);

/* ---- K2: bit-packed clean-up morphology -------------------------------------------------------------------------
 * Replaces scipy.ndimage.binary_fill_holes + skimage erosion/dilation (3x3 cross, out-of-frame neighbours ignored) +
 * skimage.measure.label in postprocess_masks (src/utils/mask_utils.py:70-84), process_masks_parallel
 * (src/functions/inference.py:189-203) and postprocess_masks_universal (inference.py:1778-1806).
 * The work planes of an instance live in shared memory when its padded crop ((ch + 2) x (cw + 2) words) has at most 1024 words;
 * emia_morph_plan: global plane size of the LARGER instances only (0 for the others; caller scans -> pad_off);
 * work = emia_morph_scratch_words() + 3 * pad_off[n] words (the fixed part is one spare plane per resident warp for the rare
 * instances that need the hole test / flood).
 * emia_morph: applies n_ops (<= 4) operators in order (1 = fill holes, 2 = erode, 3 = dilate) to every crop.
 * emia_overlap_first_come: list member k loses the pixels of members 0..k-1 (in list order), then is zeroed when it has
 *   more than one 8-connected component (mask_utils.py:77-82); members keep their place in the list (Q6).
 * emia_crop_stats: recompute bbox / area after the masks changed. */
#define EMIA_MORPH_FILL 1
#define EMIA_MORPH_ERODE 2
#define EMIA_MORPH_DILATE 3
size_t emia_morph_scratch_words(void);
int emia_morph_plan(const emia_inst_meta* meta, int64_t n, int64_t* pad_words, void* stream);
/* meta_out / crop_off_out (NULL: the input geometry): geometry of the result.  A chain whose first structuring operator is a
 * dilation (closing, plain dilation) can grow a mask by one pixel — also a closing, next to the frame border, where the
 * erosion ignores out-of-frame neighbours — so its result needs the grown geometry of emia_morph_grow_plan (caller scans). */
int emia_morph_grow_plan(const emia_inst_meta* meta, int64_t n, int H, int W, emia_inst_meta* meta_out, int64_t* crop_words,
                         void* stream);
/* apply_flag (optional): instances with apply_flag[i] == 0 pass through unchanged (process_masks_parallel only runs on lists of
 * more than two masks, inference.py:1443; see emia_group_mark_members); n_ops in 5..8 gives a SECOND operator chain
 * ops_host[4..n_ops) that is applied to the instances with apply_flag[i] == 2 (postprocess_masks_universal: erosion only for small
 * classes, opening for the others, inference.py:1786-1796), ops_host[0..4) zero-padded being the chain of apply_flag 1.  bbox_out / area_out (optional): bbox / popcount of
 * the result (emia_overlap_first_come: of the list members only), which saves the emia_crop_stats pass. */
int emia_morph(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, int64_t n, int H, int W,
               const int32_t* ops_host, int32_t n_ops, const int64_t* pad_off, uint32_t* work,
               const emia_inst_meta* meta_out, const int64_t* crop_off_out, uint32_t* crops_out,
               const int32_t* apply_flag, int32_t* bbox_out, int32_t* area_out, void* stream);
int emia_overlap_first_come(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off,
                            const int32_t* bbox, const int32_t* cap_off, int32_t G, int32_t total_cap,
                            const int32_t* in_len, const int32_t* in_idx, const int64_t* pad_off, uint32_t* work,
                            uint32_t* crops_out, int32_t* bbox_out, int32_t* area_out, void* stream);
int emia_crop_stats(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, int64_t n,
                    int32_t* bbox, int32_t* area, void* stream);
/* list members with area >= min_area, list order kept (inference.py:1800 `np.sum(final_mask) >= min_crys_size`). */
int emia_group_filter_area(const int32_t* cap_off, int32_t G, const int32_t* in_len, const int32_t* in_idx,
                           const int32_t* area, int32_t min_area, int32_t* out_len, int32_t* out_idx, void* stream);
/* postprocess_masks' column gate (mask_utils.py:62-68): K = #frame columns whose total over all list members exceeds
 * min_size; the list is truncated to its first min(K, len) members. */
int emia_column_gate(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, const int32_t* cap_off,
                     int32_t G, const int32_t* in_len, const int32_t* in_idx, int W, int32_t min_size, int32_t* out_len,
                     int32_t* out_idx, void* stream);

/* ---- K3: nearest-neighbour back-projection of instances into a (larger) frame ------------------------------------------
 * Replaces the per-instance cv2.resize(mask, INTER_NEAREST) + is_edge_mask + zero-frame placement of the tile pipeline
 * (src/functions/inference.py:2399-2420, :2522-2549) and of the multi-scale pass (:2044-2054, offsets 0).
 * Source instances live in an Hs x Ws frame (the upscaled tile / scaled image); they are resized to th x tw (the tile /
 * original image) and placed at off_xy[i] = (x_offset, y_offset) (NULL: 0,0) of the Hd x Wd destination frame, clipped
 * like `global_mask[y:y_end, x:x_end] = downscaled[:y_end - y, :x_end - x]`.
 * emia_resize_place_plan: destination geometry + crop sizes (caller scans).  emia_resize_nearest_place: destination crops,
 * bbox, area and (optional) edge_flag[i] = is_edge_mask(downscaled mask, tile_size, overlap) with edge_width =
 * int(tile_size * overlap_ratio / 2) — evaluated on the UNCLIPPED tile-sized mask; empty => 1.
 * alive (optional, both calls): instances with alive[i] == 0 (no longer a member of any list) get an empty destination and edge
 * flag 1 without being resampled. */
int emia_resize_place_plan(const int32_t* src_bbox, int64_t n, int Hs, int Ws, int th, int tw, const int32_t* off_xy,
                           const int32_t* alive, int Hd, int Wd, emia_inst_meta* dst_meta, int64_t* dst_crop_words, void* stream);
int emia_resize_nearest_place(const uint32_t* src_crops, const emia_inst_meta* src_meta, const int64_t* src_crop_off,
                              const int32_t* src_bbox, int64_t n, int Hs, int Ws, int th, int tw, const int32_t* off_xy,
                              int Hd, int Wd, int edge_width, int tile_size, const emia_inst_meta* dst_meta,
                              const int64_t* dst_crop_off, uint32_t* dst_crops, int32_t* dst_bbox, int32_t* dst_area,
                              int32_t* edge_flag, const int32_t* alive, void* stream);
/* list members whose flag[inst] == keep_value, list order kept */
int emia_group_filter_flag(const int32_t* cap_off, int32_t G, const int32_t* in_len, const int32_t* in_idx,
                           const int32_t* flag, int32_t keep_value, int32_t* out_len, int32_t* out_idx, void* stream);

/* ---- K6: RLE wire format (rle_encoding, src/utils/mask_utils.py:17-35; R50_flip_results.csv "EncodedPixels") -----------
 * Column-major, 1-indexed (start, length) pairs.  emia_rle_count: runs per instance (caller scans);
 * emia_rle_encode: runs[2 * (run_off[i] + k)] = start, [.. + 1] = length.  H = frame height. */
int emia_rle_count(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, const int32_t* bbox,
                   int64_t n, int H, int64_t* n_runs, void* stream);
int emia_rle_encode(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, const int32_t* bbox,
                    int64_t n, int H, const int64_t* run_off, int64_t* runs, void* stream);

/* ---- K6 read-back: R50_flip_results.csv text -> runs -> instances (csrc/emia_rle_kernels.cuh, core/emia_rle.cuh) ------------------
 * Text -> runs, each step count / emia_exclusive_scan_i64 / fill:
 * emia_rle_line_count : chunk_lines[c] = number of '\n' in bytes [c * EMIA_RLE_TEXT_CHUNK, (c + 1) * EMIA_RLE_TEXT_CHUNK) of the
 *   text (caller scans the ceil(nbytes / EMIA_RLE_TEXT_CHUNK) counts).
 * emia_rle_line_index : line k of the text is bytes [line_off[k], line_off[k + 1]) (its '\n' included); line_off has
 *   chunk_off[last] + 2 entries, of which the last is only written (= nbytes) when the text does not end with '\n'.
 * emia_rle_parse_count: for the n_lines lines [line_off[j], line_off[j + 1]) (the caller skips the header): data_cnt[j] = 1 unless
 *   the line is empty (only blanks: ' ', '\r', '\n'), run_cnt[j] = runs of a well-formed data line (caller scans both, n_lines + 1).
 * emia_rle_parse_fill : per data line d (in line order): line_idx[d] = j, field[d] = byte range [begin, end) of its ImageId (the
 *   text before the LAST comma of the line, quotes included), status[d] = EMIA_RLE_* (0 = OK), run_off[d] (D + 1 entries) and the
 *   (start, length) values at runs[2 * run_off[d] ..].  An empty EncodedPixels field is an empty mask.
 * Runs -> instances (the exact inverse of emia_rle_encode; canonical tight-bbox geometry of emia_mask_bbox):
 * emia_rle_decode_plan: instance i = line rows[i] (rows NULL: i) of run_off / runs, in an H x W frame (1 <= H, W <= 65535): meta,
 *   crop_words (caller scans), bbox, area and status[i]; a rejected instance (status != 0) gets bbox -1, area 0 and no crop.
 * emia_rle_decode     : writes every crop word once (no zero pass needed). */
#define EMIA_RLE_TEXT_CHUNK 8192
#define EMIA_RLE_OK 0
#define EMIA_RLE_NO_SEPARATOR 1   /* no comma in a non-empty line */
#define EMIA_RLE_BAD_CHAR 2       /* EncodedPixels holds a character other than a digit or a blank */
#define EMIA_RLE_ODD_COUNT 3      /* odd number of values */
#define EMIA_RLE_LONG_VALUE 4     /* a value of more than 18 digits */
#define EMIA_RLE_BAD_RUN 5        /* start < 1 or length < 1 */
#define EMIA_RLE_PAST_END 6       /* a run past pixel H * W */
#define EMIA_RLE_UNSORTED 7       /* a run that starts at or before the end of the previous run */
#define EMIA_RLE_AREA 8           /* more than INT32_MAX pixels */
int emia_rle_line_count(const uint8_t* text, int64_t nbytes, int64_t* chunk_lines, void* stream);
int emia_rle_line_index(const uint8_t* text, int64_t nbytes, const int64_t* chunk_off, int64_t* line_off, void* stream);
int emia_rle_parse_count(const uint8_t* text, const int64_t* line_off, int64_t n_lines, int64_t* data_cnt, int64_t* run_cnt,
                         void* stream);
int emia_rle_parse_fill(const uint8_t* text, const int64_t* line_off, int64_t n_lines, const int64_t* data_off,
                        const int64_t* run_scan, int64_t* run_off, int64_t* runs, int64_t* field, int32_t* line_idx,
                        int32_t* status, void* stream);
int emia_rle_decode_plan(const int64_t* runs, const int64_t* run_off, const int32_t* rows, int64_t n, int H, int W,
                         emia_inst_meta* meta, int64_t* crop_words, int32_t* bbox, int32_t* area, int32_t* status, void* stream);
int emia_rle_decode(const int64_t* runs, const int64_t* run_off, const int32_t* rows, int64_t n, int H,
                    const emia_inst_meta* meta, const int64_t* crop_off, uint32_t* crops, void* stream);
/* ---- Result CSV text (csrc/emia_text_kernels.cuh, core/emia_text.cuh): byte for byte what csv.writer writes ----------------
 * Count -> exclusive scan of the n + 1 lengths (caller) -> write at the scanned offsets; the host renders every string field once
 * (csv.writer's QUOTE_MINIMAL rule) and the kernels only copy its bytes.
 * emia_csv_rle_count / _write: line i of R50_flip_results.csv for instance i of (run_off, runs) (emia_rle_encode's layout):
 *   prefix (the ImageId field and its comma, prefix_len bytes), the runs as "s1 l1 s2 l2 ...", "\r\n".
 * emia_csv_measure_count / _write: a measurements_results.csv row for every record r with records[r][15] (measured) == 1, none
 *   (length 0) for the others.  Fields: strs[0] instance + 1 strs[1] (Instance_ID), strs[3 + class_idx[rec_inst[r]]] (Class,
 *   Class_Name; class_idx[i] in [0, n_str - 3)), the 12 measurements (Python float / np.float64 repr, np.float32 str for C. Length,
 *   C. Width, Aspect ratio, Ferret diameter and Roundness, int 0 for the axes and the eccentricity below 5 contour points), the
 *   contrast d10 / d50 / d90 from contrast[inst][3] (NULL or NaN: empty), strs[2] (Detected scale bar,File name), "\r\n".
 *   String k is strs[str_off[k], str_off[k + 1]).
 * emia_csv_measure_shape_count / _write: the same rows with shape = NULL; otherwise strs[2] ends with ',' and the ten shape values
 *   shape[r][10] (emia_contour_shape_list) follow as Python float repr, the last one ending the row.  The two entry points above
 *   keep their signature for existing callers. */
int emia_csv_rle_count(const int64_t* runs, const int64_t* run_off, int64_t n, int64_t prefix_len, int64_t* line_len, void* stream);
int emia_csv_rle_write(const int64_t* runs, const int64_t* run_off, int64_t n, const uint8_t* prefix, int64_t prefix_len,
                       const int64_t* line_off, uint8_t* text, void* stream);
int emia_csv_measure_count(const double* records, const int32_t* rec_inst, int64_t n_rec, const int32_t* class_idx,
                           const double* contrast, const uint8_t* strs, const int64_t* str_off, int n_str, int64_t* row_len,
                           void* stream);
int emia_csv_measure_write(const double* records, const int32_t* rec_inst, int64_t n_rec, const int32_t* class_idx,
                           const double* contrast, const uint8_t* strs, const int64_t* str_off, int n_str, const int64_t* row_off,
                           uint8_t* text, void* stream);
int emia_csv_measure_shape_count(const double* records, const int32_t* rec_inst, int64_t n_rec, const int32_t* class_idx,
                                 const double* contrast, const double* shape, const uint8_t* strs, const int64_t* str_off, int n_str,
                                 int64_t* row_len, void* stream);
int emia_csv_measure_shape_write(const double* records, const int32_t* rec_inst, int64_t n_rec, const int32_t* class_idx,
                                 const double* contrast, const double* shape, const uint8_t* strs, const int64_t* str_off, int n_str,
                                 const int64_t* row_off, uint8_t* text, void* stream);
/* ---- neighbours_results.csv: relations between the particles of one image (no reference counterpart; definitions in
 * oracle/neighbours.py).  LISTED instances are those with a record whose EMIA_REC_MEASURED is 1; CANDIDATES are two listed
 * instances of the same class key class_idx[i] in [0, n_class).  Outputs per instance:
 *   nbf[i][4] (double): centroid x = m10 / m00, y = m01 / m00 (frame pixels), sqrt(d2) * um_pix of the centroid nearest neighbour,
 *     sqrt(D2) * um_pix of the closest mask (D2 = least integer squared pixel distance between the masks); NaN when none;
 *   nbi[i][6] (int32): listed, nearest neighbour, closest neighbour (-1: no candidate; ties to the lowest index), the number of
 *     candidates with D2 <= 2, the agglomerate (lowest member of the component of D2 <= 2 edges; -1 when not listed), its size.
 * Grid: cells of cell_size pixels, gx = ceil(W / cell_size), gy = ceil(H / cell_size), ncells = n_class * gx * gy.  bbox[i] (y_min,
 * x_min, y_max, x_max) must contain the instance's pixels.
 * emia_neighbour_plan: records / inst_cont_off as emia_contour_measure writes them, moments01 from emia_moments01; fills nbf / nbi
 *   for the listed flag and centroid, and cell_cnt[ncells + 1] (cleared inside) with the cells each listed bbox covers.  The caller
 *   scans cell_cnt (emia_exclusive_scan_i64) into cell_off; cell_off[ncells] entries of ent.
 * emia_neighbour_search: fills ent and the rest of nbf / nbi; work = n + ncells int32 of workspace.  The results do not depend on
 *   the order of the entries inside a cell. */
int emia_neighbour_plan(const double* records, const int64_t* inst_cont_off, const int32_t* bbox, const int64_t* moments01,
                        const int32_t* class_idx, int64_t n, int32_t n_class, int32_t H, int32_t W, int32_t cell_size, double* nbf,
                        int32_t* nbi, int64_t* cell_cnt, void* stream);
int emia_neighbour_search(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, const int32_t* bbox,
                          const int32_t* class_idx, int64_t n, int32_t n_class, int32_t H, int32_t W, int32_t cell_size,
                          const int64_t* cell_off, int32_t* ent, double um_pix, double* nbf, int32_t* nbi, int32_t* work, void* stream);
/* emia_csv_neighbour_count / _write: one row per listed instance of neighbours_results.csv, count -> scan -> write as the measurement
 *   rows: Instance_ID (strs[0] + index + 1 + strs[1], also for the three neighbour fields), Class,Class_Name (strs[3 + class_idx]),
 *   the values of nbf / nbi (Python float repr, decimal integers; empty without a candidate), strs[2] (Detected scale bar,File name),
 *   "\r\n".  Rows of instances that are not listed are empty. */
int emia_csv_neighbour_count(const double* nbf, const int32_t* nbi, int64_t n, const int32_t* class_idx, const uint8_t* strs,
                             const int64_t* str_off, int n_str, int64_t* row_len, void* stream);
int emia_csv_neighbour_write(const double* nbf, const int32_t* nbi, int64_t n, const int32_t* class_idx, const uint8_t* strs,
                             const int64_t* str_off, int n_str, const int64_t* row_off, uint8_t* text, void* stream);
/* ---- COCO instance JSON with compressed RLE (csrc/emia_coco_kernels.cuh, core/emia_coco.cuh; definition in oracle/coco.py) -------
 * emia_coco_ann_count / _write: the "annotations" entry of instance i of (run_off, runs) (emia_rle_encode's layout) in an H x W frame,
 *   count -> exclusive scan of the n + 1 lengths (caller) -> write, byte for byte json.dumps: id first_id + i, image_id, category_id
 *   category[i], segmentation {"size": [H, W], "counts": pycocotools' rleToString of the column-major counts}, area[i], bbox
 *   [x_min, y_min, width, height] from bbox[i] (y_min, x_min, y_max, x_max) as floats ([0.0, 0.0, 0.0, 0.0] when area[i] == 0),
 *   "iscrowd": 0, score[i] as a Python float; entries are followed by ", " except the last.
 * emia_coco_counts_count: string j = data[str_off[j], str_off[j + 1]) is the counts string of an H x W mask: run_cnt[j] = its
 *   non-empty foreground runs when well-formed (0 otherwise; caller scans the n + 1 entries into run_off), status[j] = EMIA_COCO_*.
 * emia_coco_counts_fill: the (start, length) runs of string j at runs[2 * run_off[j] ..] (1-indexed, column-major: the layout of
 *   emia_rle_encode, adjacent runs where a background count is 0), for emia_rle_decode_plan / emia_rle_decode. */
#define EMIA_COCO_OK 0
#define EMIA_COCO_BAD_CHAR 1      /* a character outside '0'..'o' */
#define EMIA_COCO_OPEN_VALUE 2    /* the string ends inside a value */
#define EMIA_COCO_RANGE 3         /* a count below 0 or above 2^31 - 1, or a value of more than 7 characters */
#define EMIA_COCO_SUM 4           /* the counts do not add up to H * W */
int emia_coco_ann_count(const int64_t* runs, const int64_t* run_off, int64_t n, const int32_t* bbox, const int32_t* area,
                        const double* score, const int32_t* category, int H, int W, int64_t image_id, int64_t first_id,
                        int64_t* ann_len, void* stream);
int emia_coco_ann_write(const int64_t* runs, const int64_t* run_off, int64_t n, const int32_t* bbox, const int32_t* area,
                        const double* score, const int32_t* category, int H, int W, int64_t image_id, int64_t first_id,
                        const int64_t* ann_off, uint8_t* text, void* stream);
int emia_coco_counts_count(const uint8_t* data, const int64_t* str_off, int64_t n, int H, int W, int64_t* run_cnt, int32_t* status,
                           void* stream);
int emia_coco_counts_fill(const uint8_t* data, const int64_t* str_off, int64_t n, int H, int W, const int64_t* run_off,
                          int64_t* runs, void* stream);
/* ---- COCO segm evaluation (csrc/emia_cocoeval_kernels.cuh, core/emia_cocoeval.cuh; definition in oracle/cocoeval.py) -----------
 * The evaluated detections (DT list, n_dt) and GTs (GT list) are sorted by (category, image, file order); cat_*_off[K + 1] and
 * seg_*_off[S + 1] bound the categories and the (category, image) segments in each list; dt_seg / img / cat are per DT list entry.
 * params_host: EMIA_CE_PARAMS doubles, min(iouThrs[t], 1 - 1e-10) x 10, recThrs x 101, the area ranges' lower bounds x 4 and upper
 * bounds x 4, np.spacing(1); max_dets_host: the three maxDets.  gt_flags: bit 0 iscrowd, bit 1 the GT's id is 0.
 * emia_cocoeval_order: stable radix sorts (O(n) per 8-bit pass) of the DT list: corder[cat_off[k] + p] = the DT at place p of
 *   category k by (score desc, image, file order); morder[seg_off[s] + r] = the DT of rank r of segment s by (score desc, file
 *   order) ("match position"); rank[i] = that place r of DT i.  workspace: emia_cocoeval_order_workspace_bytes(n_dt) bytes.
 * emia_cocoeval_grid (per frame size): cell_cnt[(gseg * gy + y) * gx + x] = GT boxes (gt_gseg[i] >= 0: a grid segment) covering the
 *   cell (cell_cnt has n_seg * gx * gy + 1 entries; caller scans it into cell_off).
 * emia_cocoeval_pair_count: fills the cell lists (ent, cursor: n_seg * gx * gy ints of scratch) and writes, for every local DT j with
 *   dt_eval[j] >= 0 and rank < max_det, pair_cnt[match position] = GTs of its grid segment whose box meets its box (caller zeroes
 *   pair_cnt[n_dt + 1] before the first frame size and scans it into pair_off after the last).
 * emia_cocoeval_pair_fill: those pairs at pair_off[match position]: GT list index, DT list index, flags (gt_flags | _ignore of area
 *   range a at bit 4 + a) and the IoU of maskApi.c rleIou.
 * emia_cocoeval_match: per segment and area range the greedy matching of evaluateImg at the 10 thresholds; state[a * n_dt + i] = tp
 *   bits 0..9 and fp bits 10..19 of DT i (matched: n_words * 40 words of scratch, wseg_off[s] = the segment's first bitmap word).
 * emia_cocoeval_accumulate: precision [10, 101, n_cat, 4, 3] and recall [10, n_cat, 4, 3] (float64, caller fills them with -1) as
 *   COCOeval.accumulate. */
size_t emia_cocoeval_order_workspace_bytes(int64_t n_dt);
int emia_cocoeval_order(const double* score, const int32_t* cat, const int32_t* dt_seg, const int64_t* seg_off, int64_t n_dt,
                        int32_t n_cat, int64_t n_seg, int32_t* rank, int32_t* corder, int32_t* morder, void* workspace,
                        size_t workspace_bytes, void* stream);
int emia_cocoeval_grid(const int32_t* gt_bbox, const int32_t* gt_gseg, int64_t n_gt, int32_t n_seg, int32_t H, int32_t W,
                       int32_t cell_size, int64_t* cell_cnt, void* stream);
int emia_cocoeval_pair_count(const int32_t* gt_bbox, const int32_t* gt_gseg, int64_t n_gt, const int32_t* dt_bbox, const int32_t* dt_eval,
                             const int32_t* dt_gseg, int64_t n_dt, int32_t n_seg, int32_t H, int32_t W, int32_t cell_size,
                             const int64_t* cell_off, int32_t* ent, int32_t* cursor, const int32_t* rank, const int32_t* dt_seg,
                             const int64_t* seg_dt_off, int32_t max_det, int64_t* pair_cnt, void* stream);
int emia_cocoeval_pair_fill(const uint32_t* gt_crops, const emia_inst_meta* gt_meta, const int64_t* gt_crop_off, const int32_t* gt_bbox,
                            const int32_t* gt_area, const int32_t* gt_eval, const uint32_t* dt_crops, const emia_inst_meta* dt_meta,
                            const int64_t* dt_crop_off, const int32_t* dt_bbox, const int32_t* dt_area, const int32_t* dt_eval,
                            const int32_t* dt_gseg, int64_t n_dt, int32_t n_seg, int32_t H, int32_t W, int32_t cell_size,
                            const int64_t* cell_off, const int32_t* ent, const int32_t* rank, const int32_t* dt_seg,
                            const int64_t* seg_dt_off, const double* gt_area_eval, const int32_t* gt_flags, const double* params_host,
                            const int32_t* max_dets_host, const int64_t* pair_off, int32_t* pair_g, int32_t* pair_d, int32_t* pair_f,
                            double* pair_iou, void* stream);
int emia_cocoeval_match(const int64_t* seg_dt_off, const int64_t* seg_gt_off, const int64_t* wseg_off, int64_t n_seg, int64_t n_words,
                        const int32_t* morder, const double* dt_area, const int64_t* pair_off, const int32_t* pair_g, const int32_t* pair_d,
                        const int32_t* pair_f, const double* pair_iou, int64_t n_dt, const double* params_host,
                        const int32_t* max_dets_host, uint32_t* matched, uint32_t* state, void* stream);
int emia_cocoeval_accumulate(const int32_t* corder, const int32_t* rank, const uint32_t* state, const int64_t* cat_dt_off,
                             const int64_t* cat_gt_off, const double* gt_area, const int32_t* gt_flags, int64_t n_dt, int32_t n_cat,
                             const double* params_host, const int32_t* max_dets_host, double* precision, double* recall, void* stream);
/* raw moments (m00, m10, m01) of every instance as exact integers: cv2.moments(mask) of src/functions/inference.py:1101-1104 */
int emia_moments01(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, int64_t n, int64_t* out,
                   void* stream);

/* all moments of cv2.moments(mask) (inference.py:1101): out[i][24] = m00 m10 m01 m20 m11 m02 m30 m21 m12 m03 (exact integer sums as
 * doubles), mu20 mu11 mu02 mu30 mu21 mu12 mu03, nu20 nu11 nu02 nu30 nu21 nu12 nu03 (OpenCV's completeMomentState arithmetic). */
#define EMIA_MOMENT_FIELDS 24
int emia_moments(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, int64_t n, double* out, void* stream);
/* colour sums of the H x W x 3 (BGR, uint8) image pixels under every instance: out[i] = {sum B, sum G, sum R, pixel count} — the
 * mean colour that rgb_to_wavelength (src/utils/measurements.py:32-111) turns into a wavelength. */
int emia_color_sums(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, int64_t n,
                    const uint8_t* image_bgr, int H, int W, int64_t* out, void* stream);

/* visualisation overlay of <name>_predictions.png (inference.py:1080-1100): for the n instances order[0..n) (NULL: 0..n-1), in that
 * order: every mask pixel <- saturate(rint(v + 0.5 * colour)) (cv2.addWeighted(vis, 1.0, colored_mask, 0.5, 0)), then the external
 * contours (vertex lists of emia_contour_trace_slab / emia_contour_store) drawn with the full colour (cv2.drawContours thickness 1).
 * image_bgr: H x W x 3 bytes, modified in place; colours_bgr[n_colors][3], class c uses colour c % n_colors (:972-981). */
int emia_overlay(uint8_t* image_bgr, int H, int W, const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off,
                 const int32_t* order, int64_t n, const int32_t* classes, const uint8_t* colors_bgr, int32_t n_colors,
                 const uint32_t* pts, const int64_t* pt_off, const int32_t* cstart, int32_t cstart_stride,
                 const int64_t* inst_cont_off, const int64_t* n_contours, void* stream);

/* 256-bin grey-level histogram of the image pixels under every instance (contrast d10/d50/d90, src/utils/measurements.py:
 * 195-215): image = H x W x channels bytes (3: BGR -> cv2's 8-bit BGR2GRAY fixed-point formula; 1: grey), hist[n][256]. */
int emia_gray_hist(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, int64_t n,
                   const uint8_t* image, int H, int W, int channels, int32_t* hist, void* stream);

/* 256-bin grey-level histogram of a whole H x W x channels image (same grey conversion as emia_gray_hist): the brightness / contrast
 * statistics of calculate_image_quality_score (src/functions/inference.py:256-283) follow exactly from the counts. */
int emia_image_gray_hist(const uint8_t* image, int H, int W, int channels, uint64_t* hist, void* stream);

/* ---- batched flows: list / unit plumbing and sync-free capacity guards (csrc/emia_flow_kernels.cuh) ---------------------------
 * The reference walks its flows one predictor call at a time (run_class_specific_inference src/functions/inference.py:1353-1461,
 * tile_based_inference_pipeline :2299-2485, run_ensemble_inference :1464-1598, run_adaptive_multiscale_inference :1833-1984); here
 * the head outputs of all units (tiles / images / scales / models) of a batch are processed by one launch per step.
 * emia_group_filter_heads : members with meta.valid (Boxes.nonempty()), class == target_class (< 0: any) and score >= min_score
 *   (inference.py:1411-1420, :1519-1523); zero_score_empties: a list still holding a score == 0 becomes empty (mask_utils.py:59).
 * emia_group_mark_members : flag[inst] = value for members of lists longer than min_len (inference.py:1443 `len > 2`); the other
 *   entries are cleared first unless keep != 0 (several calls can build one selector array).
 * emia_group_flatten      : output list s = members of the groups grp_list[seg_start[s] .. seg_start[s+1]) concatenated
 *   (`full_image_masks + all_tile_masks` :2452; `all_masks.extend` :1563, :1958); its slots start at out_cap_off[s]; id_add[g]
 *   (optional, per input group) is added to the member ids of group g.
 * emia_unit_broadcast_i32 : out[i*k + c] = vals[u*k + c] for unit_off[u] <= i < unit_off[u+1] (tile offsets :2411-2414).
 * emia_scale_f32          : out = in * w in float32 (`score * weight` :1553).
 * emia_gather_plan / emia_gather_crops / emia_gather_b32 : dst instance j = src instance idx[j] (idx NULL: identity); crop sizes
 *   for the caller's scan, then crop words + bbox + area; 32-bit payloads (scores, classes).
 * emia_capacity_guard     : if *total > capacity (or *abort_flag already set): *abort_flag = 1 and the ch / cw of poison_meta[0..n)
 *   are zeroed, so that no later kernel reads or writes crops of that set. */
int emia_group_filter_heads(const int32_t* cap_off, int32_t G, const int32_t* in_len, const int32_t* in_idx,
                            const emia_inst_meta* meta, const int32_t* classes, const float* scores, int32_t target_class,
                            float min_score, int32_t zero_score_empties, int32_t* out_len, int32_t* out_idx, void* stream);
int emia_group_mark_members(const int32_t* cap_off, int32_t G, int32_t total_cap, const int32_t* in_len, const int32_t* in_idx,
                            int32_t min_len, int32_t value, int32_t keep, int32_t* flag, int64_t n_inst, void* stream);
int emia_group_flatten(const int32_t* cap_off, int32_t G, const int32_t* in_len, const int32_t* in_idx, const int32_t* grp_list,
                       const int32_t* seg_start, int32_t S, const int32_t* id_add, const int32_t* out_cap_off, int32_t* out_len,
                       int32_t* out_idx, void* stream);
int emia_unit_broadcast_i32(const int32_t* unit_off, int32_t U, int64_t n, const int32_t* vals, int32_t k, int32_t* out,
                            void* stream);
int emia_scale_f32(const float* in, float w, int64_t n, float* out, void* stream);
int emia_gather_plan(const emia_inst_meta* src_meta, const int32_t* idx, int64_t k, emia_inst_meta* dst_meta,
                     int64_t* dst_crop_words, void* stream);
int emia_gather_crops(const uint32_t* src_crops, const int64_t* src_crop_off, const int32_t* src_bbox, const int32_t* src_area,
                      const int32_t* idx, int64_t k, const emia_inst_meta* dst_meta, const int64_t* dst_crop_off,
                      uint32_t* dst_crops, int32_t* dst_bbox, int32_t* dst_area, void* stream);
int emia_gather_b32(const void* src, const int32_t* idx, int64_t k, void* dst, void* stream);
int emia_capacity_guard(const int64_t* total, int64_t capacity, int32_t* abort_flag, emia_inst_meta* poison_meta,
                        int64_t poison_n, void* stream);

/* ---- row f3: scale-bar line detection for a batch of micrographs (csrc/emia_scalebar_kernels.cuh, core/emia_scalebar.cuh) -------
 * Replaces the OpenCV calls of detect_scale_bar (src/utils/scalebar_ocr.py:140 cv2.cvtColor(BGR2GRAY), :200 cv2.Canny(gray, 50, 150,
 * apertureSize=3), :207-214 cv2.HoughLinesP(edges, 1, pi/180, threshold=50, minLineLength=20, maxLineGap=10), :247-249 cv2.line(mask,
 * p1, p2, 255, 2) + cv2.mean(gray, mask)); results are bit-identical to OpenCV 4.x.  The OCR (EasyOCR) is not part of this library.
 * emia_scalebar_edges : images [B][H][W][channels] bytes (3: BGR, 1: grey); region (rx, ry, rw, rh) inside every image;
 *   gray [B][rh][rw] and edges [B][rh][rw] (0 / 255) are written.
 * emia_hough_lines_p  : edges [B][H][W]; trig[2a] = (float)(cos(a * theta) / rho), trig[2a+1] = (float)(sin(a * theta) / rho) for
 *   a < numangle; numrho = cvRound((2 (W + H) + 1) / rho); lines [B][max_lines][4] = (x1, y1, x2, y2) in OpenCV's output order;
 *   n_lines[b] = lines found (those beyond max_lines are dropped).  workspace: emia_hough_workspace_bytes().
 * emia_line_mean      : sum_count [B][max_lines][2] = {sum of gray, pixel count} under the thickness-2 line of every output line
 *   (end points inside the region, as HoughLinesP's are); cv2.mean(...)[0] = sum * (1.0 / count). */
int emia_scalebar_edges(const uint8_t* images, int32_t B, int32_t H, int32_t W, int32_t channels, int32_t rx, int32_t ry,
                        int32_t rw, int32_t rh, int32_t low, int32_t high, uint8_t* gray, uint8_t* edges, void* stream);
size_t emia_hough_workspace_bytes(int32_t B, int32_t H, int32_t W, int32_t numangle, int32_t numrho);
int emia_hough_lines_p(const uint8_t* edges, int32_t B, int32_t H, int32_t W, const float* trig, int32_t numangle,
                       int32_t numrho, int32_t threshold, int32_t min_line_length, int32_t max_line_gap, int32_t max_lines,
                       int32_t* lines, int32_t* n_lines, void* workspace, size_t workspace_bytes, void* stream);
int emia_line_mean(const uint8_t* gray, int32_t B, int32_t H, int32_t W, const int32_t* lines, const int32_t* n_lines,
                   int32_t max_lines, int64_t* sum_count, void* stream);

/* pairwise helpers (drop-in for iou / calculate_iou / calculate_containment on explicit pairs):
 * out[k] = {intersection, area_a, area_b} for pairs (pa[k], pb[k]). */
int emia_pair_counts(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off,
                     const int32_t* area, const int32_t* pa, const int32_t* pb, int64_t n_pairs, int64_t* out,
                     void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EMIA_H */
