// emia_coco_kernels.cuh — COCO instance JSON with compressed RLE (part of emia_kernels.cu; string code: core/emia_coco.cuh).
// Write: the "annotations" entries of one image from the K6 runs, count -> emia_exclusive_scan_i64 -> write with one warp per
// instance, as k_csv_rle.  Read: "counts" strings -> (start, length) runs in the K6 layout, one warp per string, for
// emia_rle_decode_plan / emia_rle_decode.
#pragma once

#define EMIA_COCO_THREADS 128
#define EMIA_COCO_HEAD_LANES 6      // lanes 0..5: the text up to the counts string; lanes 6..12: the text after it
#define EMIA_COCO_FIXED_LANES 13

// ---- write: one annotation per instance ------------------------------------------------------------------------------------
// {"id": a, "image_id": img, "category_id": c, "segmentation": {"size": [H, W], "counts": "..."}, "area": A,
//  "bbox": [x, y, w, h], "iscrowd": 0, "score": s}  and ", " before the next one.  Fixed lane f writes key text f and its value.
__device__ __forceinline__ const char* emia_coco_key(int f, int* len) {
    const char* k = "";
    switch (f) {
        case 0: k = "{\"id\": "; break;
        case 1: k = ", \"image_id\": "; break;
        case 2: k = ", \"category_id\": "; break;
        case 3: k = ", \"segmentation\": {\"size\": ["; break;
        case 4: case 8: case 9: case 10: k = ", "; break;
        case 5: k = "], \"counts\": \""; break;
        case 6: k = "\"}, \"area\": "; break;
        case 7: k = ", \"bbox\": ["; break;
        case 11: k = "], \"iscrowd\": 0, \"score\": "; break;
        case 12: k = "}, "; break;
    }
    int n = 0;
    while (k[n]) ++n;
    *len = n;
    return k;
}

// a float as json.dumps writes it: repr, NaN / Infinity / -Infinity
__device__ __forceinline__ int emia_coco_json_f64(uint8_t* out, double v) {
    if (v == v && !isinf(v)) return emia_format_f64(out, v);
    const char* s = v != v ? "NaN" : v < 0 ? "-Infinity" : "Infinity";
    int n = 0;
    while (s[n]) { out[n] = (uint8_t)s[n]; ++n; }
    return n;
}

template <bool kWrite>
__global__ void __launch_bounds__(EMIA_COCO_THREADS) k_coco_ann(const int64_t* __restrict__ runs, const int64_t* __restrict__ run_off,
                                                                int64_t n, const int32_t* __restrict__ bbox,
                                                                const int32_t* __restrict__ area, const double* __restrict__ score,
                                                                const int32_t* __restrict__ category, int H, int W, int64_t image_id,
                                                                int64_t first_id, int64_t* __restrict__ ann_len,
                                                                const int64_t* __restrict__ ann_off, uint8_t* __restrict__ text) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= n) return;
    const int64_t r0 = run_off[i], nr = run_off[i + 1] - r0;
    const int64_t* rr = runs + 2 * r0;
    const int64_t hw = (int64_t)H * W;
    uint8_t* o = kWrite ? text + ann_off[i] : nullptr;

    // the fixed lanes: key text + value
    uint8_t num[EMIA_TEXT_NUM_MAX];
    int klen = 0, nlen = 0;
    const char* key = lane < EMIA_COCO_FIXED_LANES ? emia_coco_key(lane, &klen) : "";
    if (lane == 12 && i == n - 1) klen = 1;                            // no ", " after the last annotation
    const int a = area[i];
    const int32_t* bb = bbox + 4 * i;                                  // (y_min, x_min, y_max, x_max)
    switch (lane) {
        case 0: nlen = emia_write_i64(num, first_id + i); break;
        case 1: nlen = emia_write_i64(num, image_id); break;
        case 2: nlen = emia_write_i64(num, category[i]); break;
        case 3: nlen = emia_write_i64(num, H); break;
        case 4: nlen = emia_write_i64(num, W); break;
        case 6: nlen = emia_write_i64(num, a); break;
        case 7: nlen = emia_format_f64(num, a ? (double)bb[1] : 0.0); break;
        case 8: nlen = emia_format_f64(num, a ? (double)bb[0] : 0.0); break;
        case 9: nlen = emia_format_f64(num, a ? (double)(bb[3] - bb[1] + 1) : 0.0); break;
        case 10: nlen = emia_format_f64(num, a ? (double)(bb[2] - bb[0] + 1) : 0.0); break;
        case 11: nlen = emia_coco_json_f64(num, score[i]); break;
    }
    const int flen = klen + nlen;
    int finc = flen;
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(FULL, finc, d);
        if (lane >= d) finc += v;
    }
    const int head = __shfl_sync(FULL, finc, EMIA_COCO_HEAD_LANES - 1);
    const int fixed = __shfl_sync(FULL, finc, EMIA_COCO_FIXED_LANES - 1);
    auto put_fixed = [&](int64_t at) {
        uint8_t* p = o + at;
        for (int j = 0; j < klen; ++j) p[j] = (uint8_t)key[j];
        for (int j = 0; j < nlen; ++j) p[klen + j] = num[j];
    };
    if (kWrite && lane < EMIA_COCO_HEAD_LANES) put_fixed(finc - flen);

    // the counts: lane j of a window takes run k = base + j, i.e. count 2k (the gap before it) and 2k + 1 (its length)
    int64_t pos = head;
    int64_t c_end = 0, c_gap = 0, c_len = 0;                          // end, gap and length of the run before the window
    for (int64_t base = 0; base < nr; base += 32) {
        const int64_t k = base + lane;
        int64_t s = 0, l = 0;
        if (k < nr) { s = rr[2 * k]; l = rr[2 * k + 1]; }
        const int64_t end = s + l - 1;                                 // 1-indexed last pixel of the run
        int64_t pe = __shfl_up_sync(FULL, end, 1);
        if (lane == 0) pe = c_end;
        const int64_t gap = s - 1 - pe;
        int64_t pg = __shfl_up_sync(FULL, gap, 1), pl = __shfl_up_sync(FULL, l, 1);
        if (lane == 0) { pg = c_gap; pl = c_len; }
        const int64_t dg = k >= 2 ? gap - pg : gap, dl = k >= 1 ? l - pl : l;
        const int len = k < nr ? emia_coco_delta_len(dg, nullptr) + emia_coco_delta_len(dl, nullptr) : 0;
        int inc = len;
        for (int d = 1; d < 32; d <<= 1) {
            const int v = __shfl_up_sync(FULL, inc, d);
            if (lane >= d) inc += v;
        }
        if (kWrite && k < nr) {
            uint8_t* p = o + pos + inc - len;
            p += emia_coco_put_delta(p, dg);
            emia_coco_put_delta(p, dl);
        }
        pos += __shfl_sync(FULL, inc, 31);
        const int last = (int)min((int64_t)31, nr - 1 - base);
        c_end = __shfl_sync(FULL, end, last);
        c_gap = __shfl_sync(FULL, gap, last);
        c_len = __shfl_sync(FULL, l, last);
    }
    // the background after the last run (the whole frame for an empty mask): count 2 nr, written when not 0
    const int64_t tail = hw - c_end;
    const int64_t dt = nr >= 2 ? tail - c_gap : tail;
    const int tlen = tail > 0 ? emia_coco_delta_len(dt, nullptr) : 0;
    if (kWrite && lane == 0 && tail > 0) emia_coco_put_delta(o + pos, dt);
    pos += tlen;
    if (kWrite && lane >= EMIA_COCO_HEAD_LANES && lane < EMIA_COCO_FIXED_LANES) put_fixed(pos + finc - flen - head);
    if (!kWrite && lane == 0) ann_len[i] = pos + fixed - head;
}

static int emia_coco_ann_args(const char* what, const int64_t* runs, const int64_t* run_off, int64_t n, const int32_t* bbox,
                              const int32_t* area, const double* score, const int32_t* category, int H, int W, const void* out) {
    if (n < 0 || !emia_rle_frame_ok(H, W)) return emia_fail(EMIA_ERR_BAD_ARG, "%s: bad size (1 <= H, W <= 65535)", what);
    if (n && (!runs || !run_off || !bbox || !area || !score || !category || !out))
        return emia_fail(EMIA_ERR_BAD_ARG, "%s: null pointer", what);
    return EMIA_OK;
}

extern "C" int emia_coco_ann_count(const int64_t* runs, const int64_t* run_off, int64_t n, const int32_t* bbox, const int32_t* area,
                                   const double* score, const int32_t* category, int H, int W, int64_t image_id, int64_t first_id,
                                   int64_t* ann_len, void* stream) {
    if (int rc = emia_coco_ann_args("emia_coco_ann_count", runs, run_off, n, bbox, area, score, category, H, W, ann_len)) return rc;
    if (n == 0) return EMIA_OK;
    k_coco_ann<false><<<(unsigned)((n * 32 + EMIA_COCO_THREADS - 1) / EMIA_COCO_THREADS), EMIA_COCO_THREADS, 0, (cudaStream_t)stream>>>(
        runs, run_off, n, bbox, area, score, category, H, W, image_id, first_id, ann_len, nullptr, nullptr);
    return emia_check_launch("emia_coco_ann_count launch: %s");
}
extern "C" int emia_coco_ann_write(const int64_t* runs, const int64_t* run_off, int64_t n, const int32_t* bbox, const int32_t* area,
                                   const double* score, const int32_t* category, int H, int W, int64_t image_id, int64_t first_id,
                                   const int64_t* ann_off, uint8_t* text, void* stream) {
    if (int rc = emia_coco_ann_args("emia_coco_ann_write", runs, run_off, n, bbox, area, score, category, H, W, text)) return rc;
    if (n == 0) return EMIA_OK;
    if (!ann_off) return emia_fail(EMIA_ERR_BAD_ARG, "emia_coco_ann_write: %s", "null pointer");
    k_coco_ann<true><<<(unsigned)((n * 32 + EMIA_COCO_THREADS - 1) / EMIA_COCO_THREADS), EMIA_COCO_THREADS, 0, (cudaStream_t)stream>>>(
        runs, run_off, n, bbox, area, score, category, H, W, image_id, first_id, nullptr, ann_off, text);
    return emia_check_launch("emia_coco_ann_write launch: %s");
}

// ---- read: counts strings -> runs, one warp per string in windows of 32 characters ---------------------------------------------
// The lane at each value end (a character without 0x20) assembles its value from its characters; two parity-split scans undo the
// i > 2 delta coding and a third places the counts on the pixel axis.  Pass 1 (kFill = false) writes the runs of a well-formed
// string (0 otherwise) and its status; pass 2 repeats the walk and stores the runs of the strings with runs.  Errors are reported
// at the first bad character or value, in string order.
template <bool kFill>
__global__ void __launch_bounds__(EMIA_COCO_THREADS) k_coco_counts(const uint8_t* __restrict__ data, const int64_t* __restrict__ str_off,
                                                                   int64_t n, int64_t hw, int64_t* __restrict__ run_cnt,
                                                                   int32_t* __restrict__ status, const int64_t* __restrict__ run_off,
                                                                   int64_t* __restrict__ runs) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    const int64_t j = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (j >= n) return;
    const int64_t b = str_off[j], e = str_off[j + 1];
    if (kFill && run_off[j + 1] == run_off[j]) return;
    int64_t* out = kFill ? runs + 2 * run_off[j] : nullptr;
    int st = EMIA_COCO_OK;
    int64_t nv = 0, nrun = 0, last_end = b - 1;                        // values and runs so far, position of the last value end
    int64_t c_even = 0, c_odd = 0, c_pos = 0;                          // last even (index >= 2) / odd count, pixels so far
    for (int64_t w = b; w < e; w += 32) {
        const int64_t p = w + lane;
        const uint8_t c = p < e ? data[p] : (uint8_t)'0';
        const bool bad = p < e && !emia_coco_char_ok(c);
        const unsigned badm = __ballot_sync(FULL, bad);
        const unsigned endm = __ballot_sync(FULL, p < e && !bad && !emia_coco_char_more(c));
        const bool mine = (endm >> lane) & 1u;
        const unsigned before = endm & lt;
        const int64_t start = before ? w + 31 - __clz(before) + 1 : last_end + 1;
        const int64_t vi = nv + __popc(before);
        const int k = (int)(p - start + 1);
        bool range = mine && k > EMIA_COCO_MAX_CHARS;
        const int64_t x = mine && !range ? emia_coco_value(data + start, k) : 0;
        // counts: c0 = x0, c2 = x2, c(i) = x(i) + c(i - 2) for i > 2
        int64_t xe = mine && vi >= 2 && !(vi & 1) ? x : 0, xo = mine && (vi & 1) ? x : 0;
        for (int d = 1; d < 32; d <<= 1) {
            const int64_t ve = __shfl_up_sync(FULL, xe, d), vo = __shfl_up_sync(FULL, xo, d);
            if (lane >= d) { xe += ve; xo += vo; }
        }
        const int64_t cnt = !mine ? 0 : vi == 0 ? x : (vi & 1) ? c_odd + xo : c_even + xe;
        range |= mine && (cnt < 0 || cnt > INT32_MAX);
        const unsigned rangem = __ballot_sync(FULL, range);
        if (badm | rangem) {
            const int fb = badm ? __ffs(badm) - 1 : 32, fr = rangem ? __ffs(rangem) - 1 : 32;
            st = fb < fr ? EMIA_COCO_BAD_CHAR : EMIA_COCO_RANGE;
            break;
        }
        int64_t at = cnt;                                              // pixels before each value: exclusive scan of the counts
        for (int d = 1; d < 32; d <<= 1) {
            const int64_t v = __shfl_up_sync(FULL, at, d);
            if (lane >= d) at += v;
        }
        const unsigned runm = __ballot_sync(FULL, mine && (vi & 1) && cnt > 0);
        if (kFill && ((runm >> lane) & 1u)) {
            const int64_t r = nrun + __popc(runm & lt);
            out[2 * r] = c_pos + at - cnt + 1;
            out[2 * r + 1] = cnt;
        }
        nrun += __popc(runm);
        c_pos += __shfl_sync(FULL, at, 31);
        c_even += __shfl_sync(FULL, xe, 31);
        c_odd += __shfl_sync(FULL, xo, 31);
        if (endm) last_end = w + 31 - __clz(endm);
        nv += __popc(endm);
    }
    if (kFill || lane != 0) return;
    if (st == EMIA_COCO_OK && last_end != e - 1) st = EMIA_COCO_OPEN_VALUE;
    if (st == EMIA_COCO_OK && c_pos != hw) st = EMIA_COCO_SUM;
    run_cnt[j] = st == EMIA_COCO_OK ? nrun : 0;
    status[j] = st;
}

static int emia_coco_counts_args(const char* what, const uint8_t* data, const int64_t* str_off, int64_t n, int H, int W,
                                 const void* a, const void* b) {
    if (n < 0 || n > INT32_MAX || !emia_rle_frame_ok(H, W)) return emia_fail(EMIA_ERR_BAD_ARG, "%s: bad size (1 <= H, W <= 65535)", what);
    if (n && (!data || !str_off || !a || !b)) return emia_fail(EMIA_ERR_BAD_ARG, "%s: null pointer", what);
    return EMIA_OK;
}

extern "C" int emia_coco_counts_count(const uint8_t* data, const int64_t* str_off, int64_t n, int H, int W, int64_t* run_cnt,
                                      int32_t* status, void* stream) {
    if (int rc = emia_coco_counts_args("emia_coco_counts_count", data, str_off, n, H, W, run_cnt, status)) return rc;
    if (n == 0) return EMIA_OK;
    k_coco_counts<false><<<(unsigned)((n * 32 + EMIA_COCO_THREADS - 1) / EMIA_COCO_THREADS), EMIA_COCO_THREADS, 0, (cudaStream_t)stream>>>(
        data, str_off, n, (int64_t)H * W, run_cnt, status, nullptr, nullptr);
    return emia_check_launch("emia_coco_counts_count launch: %s");
}
extern "C" int emia_coco_counts_fill(const uint8_t* data, const int64_t* str_off, int64_t n, int H, int W, const int64_t* run_off,
                                     int64_t* runs, void* stream) {
    if (int rc = emia_coco_counts_args("emia_coco_counts_fill", data, str_off, n, H, W, run_off, runs)) return rc;
    if (n == 0) return EMIA_OK;
    k_coco_counts<true><<<(unsigned)((n * 32 + EMIA_COCO_THREADS - 1) / EMIA_COCO_THREADS), EMIA_COCO_THREADS, 0, (cudaStream_t)stream>>>(
        data, str_off, n, (int64_t)H * W, nullptr, nullptr, run_off, runs);
    return emia_check_launch("emia_coco_counts_fill launch: %s");
}
