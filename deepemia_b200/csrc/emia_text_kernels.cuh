// emia_text_kernels.cuh — the result CSV files as text on the device (part of emia_kernels.cu): the lines of R50_flip_results.csv
// from the K6 runs and the rows of measurements_results.csv from the K5 records, byte for byte what csv.writer writes for the
// values run_inference passes it (numbers: core/emia_text.cuh; strings are rendered once by the host and only copied here).
// Both follow count -> emia_exclusive_scan_i64 -> write: one warp per line / row, the same walk in both passes.
#pragma once

#define EMIA_CSV_THREADS 128
#define EMIA_CSV_SEP_LANES 17       // measurement lanes that end their field with ',' (the last one ends the row with "\r\n")

// ---- R50_flip_results.csv: `<ImageId>,<s1> <l1> <s2> <l2> ...\r\n`, one line per instance ------------------------------------
// prefix = the ImageId field and its comma.  Lanes take runs; run k is "s l" and a ' ' (the last one "\r\n"), placed by a warp scan.
template <bool kWrite>
__global__ void __launch_bounds__(EMIA_CSV_THREADS) k_csv_rle(const int64_t* __restrict__ runs, const int64_t* __restrict__ run_off,
                                                              int64_t n, const uint8_t* __restrict__ prefix, int prefix_len,
                                                              int64_t* __restrict__ line_len, const int64_t* __restrict__ line_off,
                                                              uint8_t* __restrict__ text) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= n) return;
    const int64_t r0 = run_off[i], nr = run_off[i + 1] - r0;
    const int64_t* rr = runs + 2 * r0;
    uint8_t* o = kWrite ? text + line_off[i] : nullptr;
    if (kWrite)
        for (int j = lane; j < prefix_len; j += 32) o[j] = prefix[j];
    int64_t pos = prefix_len;
    for (int64_t base = 0; base < nr; base += 32) {
        const int64_t k = base + lane;
        uint64_t s = 0, l = 0;
        int ds = 0, dl = 0, len = 0;
        if (k < nr) {
            s = (uint64_t)rr[2 * k]; l = (uint64_t)rr[2 * k + 1];
            ds = emia_u64_digits(s); dl = emia_u64_digits(l);
            len = ds + dl + (k == nr - 1 ? 3 : 2);
        }
        int inc = len;
        for (int d = 1; d < 32; d <<= 1) {
            const int v = __shfl_up_sync(FULL, inc, d);
            if (lane >= d) inc += v;
        }
        if (kWrite && k < nr) {
            uint8_t* p = o + pos + inc - len;
            emia_put_u64(p, s, ds);
            p[ds] = ' ';
            emia_put_u64(p + ds + 1, l, dl);
            if (k == nr - 1) { p[ds + dl + 1] = '\r'; p[ds + dl + 2] = '\n'; }
            else p[ds + dl + 1] = ' ';
        }
        pos += __shfl_sync(FULL, inc, 31);
    }
    if (lane == 0) {
        if (!kWrite) line_len[i] = nr ? pos : pos + 2;
        else if (!nr) { o[pos] = '\r'; o[pos + 1] = '\n'; }
    }
}

static int emia_csv_rle_args(const char* what, const int64_t* runs, const int64_t* run_off, int64_t n, int64_t prefix_len,
                             const void* out) {
    if (n < 0 || prefix_len < 0 || prefix_len > INT32_MAX) return emia_fail(EMIA_ERR_BAD_ARG, "%s: bad size", what);
    if (n && (!runs || !run_off || !out)) return emia_fail(EMIA_ERR_BAD_ARG, "%s: null pointer", what);
    return EMIA_OK;
}

extern "C" int emia_csv_rle_count(const int64_t* runs, const int64_t* run_off, int64_t n, int64_t prefix_len, int64_t* line_len,
                                  void* stream) {
    if (int rc = emia_csv_rle_args("emia_csv_rle_count", runs, run_off, n, prefix_len, line_len)) return rc;
    if (n == 0) return EMIA_OK;
    k_csv_rle<false><<<(unsigned)((n * 32 + EMIA_CSV_THREADS - 1) / EMIA_CSV_THREADS), EMIA_CSV_THREADS, 0, (cudaStream_t)stream>>>(
        runs, run_off, n, nullptr, (int)prefix_len, line_len, nullptr, nullptr);
    return emia_check_launch("emia_csv_rle_count launch: %s");
}
extern "C" int emia_csv_rle_write(const int64_t* runs, const int64_t* run_off, int64_t n, const uint8_t* prefix, int64_t prefix_len,
                                  const int64_t* line_off, uint8_t* text, void* stream) {
    if (int rc = emia_csv_rle_args("emia_csv_rle_write", runs, run_off, n, prefix_len, text)) return rc;
    if (n == 0) return EMIA_OK;
    if (!line_off || (prefix_len && !prefix)) return emia_fail(EMIA_ERR_BAD_ARG, "emia_csv_rle_write: %s", "null pointer");
    k_csv_rle<true><<<(unsigned)((n * 32 + EMIA_CSV_THREADS - 1) / EMIA_CSV_THREADS), EMIA_CSV_THREADS, 0, (cudaStream_t)stream>>>(
        runs, run_off, n, prefix, (int)prefix_len, nullptr, line_off, text);
    return emia_check_launch("emia_csv_rle_write launch: %s");
}

// ---- measurements_results.csv: one row per measured record ------------------------------------------------------------------
// Lane f writes field f: 0 Instance_ID (strs[0] + instance + 1 + strs[1]), 1 Class,Class_Name (strs[3 + class_idx]), 2..13 the
// measurements, 14..16 the contrast percentiles, 17 "Detected scale bar,File name" (strs[2]) and the line end — or, with the shape
// columns, a ',' and lanes 18..27 the ten shape values (repr of a Python float), the last one ending the row.
#define EMIA_CSV_SHAPE_LANE0 (EMIA_CSV_SEP_LANES + 1)
__device__ __forceinline__ int emia_csv_measure_field(int lane, const double* rec, const double* contrast, const double* shape,
                                                      uint8_t* num) {
    if (shape && lane >= EMIA_CSV_SHAPE_LANE0 && lane < EMIA_CSV_SHAPE_LANE0 + EMIA_S_COUNT)
        return emia_format_f64(num, shape[lane - EMIA_CSV_SHAPE_LANE0]);
    if (lane >= 2 && lane < 14) {
        const int c = lane - 2;                     // REC_MAJOR .. REC_SPHER
        if (c <= 2 && rec[14] < 5.0) { num[0] = '0'; return 1; }            // no ellipse below 5 contour points: int 0
        const bool f32 = c == 3 || c == 4 || c == 6 || c == 9 || c == 10;  // Length, Width, Aspect ratio, Feret, Roundness
        return f32 ? emia_format_f32(num, __double2float_rn(rec[c])) : emia_format_f64(num, rec[c]);
    }
    if (lane >= 14 && lane < 17 && contrast) {
        const double v = contrast[lane - 14];
        return v != v ? 0 : emia_format_f64(num, v);                      // NaN: None, an empty field
    }
    return 0;
}

template <bool kWrite>
__global__ void __launch_bounds__(EMIA_CSV_THREADS) k_csv_measure(const double* __restrict__ records, const int32_t* __restrict__ rec_inst,
                                                                  int64_t n_rec, const int32_t* __restrict__ class_idx,
                                                                  const double* __restrict__ contrast, const double* __restrict__ shape,
                                                                  const uint8_t* __restrict__ strs,
                                                                  const int64_t* __restrict__ str_off, int64_t* __restrict__ row_len,
                                                                  const int64_t* __restrict__ row_off, uint8_t* __restrict__ text) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= n_rec) return;
    const double* rec = records + r * 16;
    if (rec[15] != 1.0) {                           // REC_MEASURED: below the area gate, no row
        if (!kWrite && lane == 0) row_len[r] = 0;
        return;
    }
    const int inst = rec_inst[r];
    uint8_t num[EMIA_TEXT_NUM_MAX];
    int nlen = emia_csv_measure_field(lane, rec, contrast ? contrast + 3 * (int64_t)inst : nullptr,
                                      shape ? shape + r * EMIA_S_COUNT : nullptr, num);
    int s0 = -1, s1 = -1;                           // strings before / after the number
    if (lane == 0) { s0 = 0; s1 = 1; nlen = emia_write_i64(num, (int64_t)inst + 1); }
    else if (lane == 1) s0 = 3 + class_idx[inst];
    else if (lane == EMIA_CSV_SEP_LANES) s0 = 2;
    const int64_t a0 = s0 >= 0 ? str_off[s0] : 0, l0 = s0 >= 0 ? str_off[s0 + 1] - a0 : 0;
    const int64_t a1 = s1 >= 0 ? str_off[s1] : 0, l1 = s1 >= 0 ? str_off[s1 + 1] - a1 : 0;
    const int last = shape ? EMIA_CSV_SHAPE_LANE0 + EMIA_S_COUNT - 1 : EMIA_CSV_SEP_LANES;
    const int term = lane < last ? 1 : lane == last ? 2 : 0;
    const int64_t len = l0 + nlen + l1 + term;
    int64_t inc = len;
    for (int d = 1; d < 32; d <<= 1) {
        const int64_t v = __shfl_up_sync(FULL, inc, d);
        if (lane >= d) inc += v;
    }
    if (!kWrite) {
        if (lane == 31) row_len[r] = inc;
        return;
    }
    uint8_t* p = text + row_off[r] + inc - len;
    for (int64_t j = 0; j < l0; ++j) *p++ = strs[a0 + j];
    for (int j = 0; j < nlen; ++j) *p++ = num[j];
    for (int64_t j = 0; j < l1; ++j) *p++ = strs[a1 + j];
    if (term == 1) *p = ',';
    else if (term == 2) { p[0] = '\r'; p[1] = '\n'; }
}

static int emia_csv_measure_args(const char* what, const double* records, const int32_t* rec_inst, int64_t n_rec,
                                 const int32_t* class_idx, const uint8_t* strs, const int64_t* str_off, int n_str, const void* out) {
    if (n_rec < 0 || n_str < 3) return emia_fail(EMIA_ERR_BAD_ARG, "%s: bad size", what);
    if (n_rec && (!records || !rec_inst || !class_idx || !strs || !str_off || !out))
        return emia_fail(EMIA_ERR_BAD_ARG, "%s: null pointer", what);
    return EMIA_OK;
}

// shape: NULL, or float64 [n_rec][EMIA_S_COUNT] (emia_contour_shape_list) for the ten shape columns after "File name"
static int emia_csv_measure_launch(const char* what, bool write, const double* records, const int32_t* rec_inst, int64_t n_rec,
                                   const int32_t* class_idx, const double* contrast, const double* shape, const uint8_t* strs,
                                   const int64_t* str_off, int n_str, int64_t* row_len, const int64_t* row_off, uint8_t* text,
                                   void* stream) {
    if (int rc = emia_csv_measure_args(what, records, rec_inst, n_rec, class_idx, strs, str_off, n_str, write ? (const void*)text : row_len))
        return rc;
    if (n_rec == 0) return EMIA_OK;
    if (write && !row_off) return emia_fail(EMIA_ERR_BAD_ARG, "%s: null pointer", what);
    const unsigned grid = (unsigned)((n_rec * 32 + EMIA_CSV_THREADS - 1) / EMIA_CSV_THREADS);
    if (write)
        k_csv_measure<true><<<grid, EMIA_CSV_THREADS, 0, (cudaStream_t)stream>>>(records, rec_inst, n_rec, class_idx, contrast, shape, strs,
                                                                                 str_off, nullptr, row_off, text);
    else
        k_csv_measure<false><<<grid, EMIA_CSV_THREADS, 0, (cudaStream_t)stream>>>(records, rec_inst, n_rec, class_idx, contrast, shape, strs,
                                                                                  str_off, row_len, nullptr, nullptr);
    return emia_check_launch(write ? "emia_csv_measure_write launch: %s" : "emia_csv_measure_count launch: %s");
}

extern "C" int emia_csv_measure_count(const double* records, const int32_t* rec_inst, int64_t n_rec, const int32_t* class_idx,
                                      const double* contrast, const uint8_t* strs, const int64_t* str_off, int n_str, int64_t* row_len,
                                      void* stream) {
    return emia_csv_measure_launch("emia_csv_measure_count", false, records, rec_inst, n_rec, class_idx, contrast, nullptr, strs,
                                   str_off, n_str, row_len, nullptr, nullptr, stream);
}
extern "C" int emia_csv_measure_write(const double* records, const int32_t* rec_inst, int64_t n_rec, const int32_t* class_idx,
                                      const double* contrast, const uint8_t* strs, const int64_t* str_off, int n_str,
                                      const int64_t* row_off, uint8_t* text, void* stream) {
    return emia_csv_measure_launch("emia_csv_measure_write", true, records, rec_inst, n_rec, class_idx, contrast, nullptr, strs,
                                   str_off, n_str, nullptr, row_off, text, stream);
}
extern "C" int emia_csv_measure_shape_count(const double* records, const int32_t* rec_inst, int64_t n_rec, const int32_t* class_idx,
                                            const double* contrast, const double* shape, const uint8_t* strs, const int64_t* str_off,
                                            int n_str, int64_t* row_len, void* stream) {
    return emia_csv_measure_launch("emia_csv_measure_shape_count", false, records, rec_inst, n_rec, class_idx, contrast, shape, strs,
                                   str_off, n_str, row_len, nullptr, nullptr, stream);
}
extern "C" int emia_csv_measure_shape_write(const double* records, const int32_t* rec_inst, int64_t n_rec, const int32_t* class_idx,
                                            const double* contrast, const double* shape, const uint8_t* strs, const int64_t* str_off,
                                            int n_str, const int64_t* row_off, uint8_t* text, void* stream) {
    return emia_csv_measure_launch("emia_csv_measure_shape_write", true, records, rec_inst, n_rec, class_idx, contrast, shape, strs,
                                   str_off, n_str, nullptr, row_off, text, stream);
}
