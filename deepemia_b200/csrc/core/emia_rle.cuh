// emia_rle.cuh — host/device pieces of reading the RLE wire format back (R50_flip_results.csv "EncodedPixels"): the number
// parser of the text kernels, the per-run checks and bbox of the decode plan, and the canonical tight-bbox geometry that the
// decode plan shares with k_mask_bbox.  Compiled into the sm_100a kernels and into tests/hostsim.
#pragma once
#include "emia_common.cuh"
#include "../../../include/emia.h"

#define EMIA_RLE_MAX_DIGITS 18      // 10^18 - 1 < INT64_MAX, and start + length of two such values still fits

EMIA_HD bool emia_rle_is_digit(uint8_t c) { return c >= '0' && c <= '9'; }
EMIA_HD bool emia_rle_is_blank(uint8_t c) { return c == ' ' || c == '\r' || c == '\n'; }

// the decimal number whose first digit is s[0] (avail bytes readable): number of digits, or -1 when it has more than 18
EMIA_HD int emia_rle_parse_uint(const uint8_t* s, int64_t avail, int64_t* value) {
    int64_t v = 0;
    int k = 0;
    while (k < avail && emia_rle_is_digit(s[k])) {
        if (k == EMIA_RLE_MAX_DIGITS) return -1;
        v = v * 10 + (s[k] - '0');
        ++k;
    }
    *value = v;
    return k;
}

// run (start, length) of the 1-indexed column-major wire format after a run that ended at 1-indexed pixel prev_end (0 for the
// first run) in a frame of hw pixels: EMIA_RLE_OK or the rejection code
EMIA_HD int emia_rle_run_status(int64_t prev_end, int64_t start, int64_t length, int64_t hw) {
    if (start < 1 || length < 1) return EMIA_RLE_BAD_RUN;
    if (start > hw || length > hw - start + 1) return EMIA_RLE_PAST_END;
    if (start <= prev_end) return EMIA_RLE_UNSORTED;
    return EMIA_RLE_OK;
}

// rows and columns a valid run covers (flat index f = x * H + y, 0-indexed): columns x0..x1; a run over more than one column
// contains row H - 1 of its first column and row 0 of its last one
EMIA_HD void emia_rle_run_extent(int64_t start, int64_t length, int H, int* ymin, int* ymax, int* x0, int* x1) {
    const int64_t f0 = start - 1, f1 = start - 2 + length;
    *x0 = (int)(f0 / H);
    *x1 = (int)(f1 / H);
    if (*x0 == *x1) { *ymin = (int)(f0 - (int64_t)*x0 * H); *ymax = (int)(f1 - (int64_t)*x1 * H); }
    else { *ymin = 0; *ymax = H - 1; }
}

// canonical geometry of a mask with the given popcount and inclusive bbox: the tight crop of k_mask_bbox / from_masks
// (rx0 = x_min, rx1 = x_max + 1, word-aligned crop columns, valid = 1); an empty mask has a zero-size crop
EMIA_HD emia_inst_meta emia_meta_from_bbox(int64_t area, int ymin, int xmin, int ymax, int xmax) {
    emia_inst_meta mt;
    if (area > 0) {
        mt.ry0 = ymin; mt.ch = ymax - ymin + 1;
        mt.rx0 = xmin; mt.rx1 = xmax + 1;
        mt.wc0 = mt.rx0 >> 5; mt.cw = ((mt.rx1 - 1) >> 5) - mt.wc0 + 1;
    } else {
        mt.ry0 = mt.ch = mt.rx0 = mt.rx1 = mt.wc0 = mt.cw = 0;
    }
    mt.valid = 1; mt.reserved = 0;
    return mt;
}
