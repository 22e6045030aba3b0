// emia_rle_kernels.cuh — reading the RLE wire format back (part of emia_kernels.cu): R50_flip_results.csv text -> runs -> instances.
// The inverse of K6 (emia_tile_kernels.cuh): the text is split into lines, every line is parsed by one warp (ballots over
// 32-byte windows find the number starts; the lane at each start parses its number), and the runs of an instance are decoded
// into its tight bbox crop by one CTA (one warp per crop word-column and row band, lanes on pixel columns).
#pragma once

// ---- text -> line table -------------------------------------------------------------------------------------------------
#define EMIA_RLE_LINE_THREADS 512
#define EMIA_RLE_LINE_BYTES (EMIA_RLE_TEXT_CHUNK / EMIA_RLE_LINE_THREADS)
static_assert(EMIA_RLE_LINE_THREADS == EMIA_SCAN_THREADS, "the line kernels use the CTA scan of the int64 prefix sum");

// one CTA per chunk; thread t owns bytes [t * 16, t * 16 + 16) of it.  kIndex: line_off[k + 1] = position after the k-th '\n'
template <bool kIndex>
__global__ void __launch_bounds__(EMIA_RLE_LINE_THREADS) k_rle_lines(const uint8_t* __restrict__ text, int64_t nbytes,
                                                                     int64_t* __restrict__ chunk_lines,
                                                                     const int64_t* __restrict__ chunk_off,
                                                                     int64_t* __restrict__ line_off) {
    __shared__ int64_t s_warp[EMIA_SCAN_THREADS / 32];
    const int64_t p0 = (int64_t)blockIdx.x * EMIA_RLE_TEXT_CHUNK + (int64_t)threadIdx.x * EMIA_RLE_LINE_BYTES;
    uint8_t b[EMIA_RLE_LINE_BYTES];
    if (p0 + EMIA_RLE_LINE_BYTES <= nbytes && ((uintptr_t)(text + p0) & 15) == 0) {
        const uint4 v = __ldg((const uint4*)(text + p0));
        memcpy(b, &v, sizeof(v));
    } else {
        for (int k = 0; k < EMIA_RLE_LINE_BYTES; ++k) b[k] = p0 + k < nbytes ? text[p0 + k] : 0;
    }
    int cnt = 0;
    for (int k = 0; k < EMIA_RLE_LINE_BYTES; ++k) cnt += b[k] == '\n';
    int64_t total;
    const int64_t ex = emia_block_exclusive_scan(cnt, s_warp, &total);
    if (!kIndex) {
        if (threadIdx.x == 0) chunk_lines[blockIdx.x] = total;
        return;
    }
    int64_t w = chunk_off[blockIdx.x] + ex + 1;
    for (int k = 0; k < EMIA_RLE_LINE_BYTES; ++k)
        if (b[k] == '\n') line_off[w++] = p0 + k + 1;
    if (blockIdx.x == 0 && threadIdx.x == 0) line_off[0] = 0;
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0 && text[nbytes - 1] != '\n') line_off[chunk_off[gridDim.x] + 1] = nbytes;
}

extern "C" int emia_rle_line_count(const uint8_t* text, int64_t nbytes, int64_t* chunk_lines, void* stream) {
    if (nbytes < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_rle_line_count: %s", "bad size");
    if (nbytes == 0) return EMIA_OK;
    if (!text || !chunk_lines) return emia_fail(EMIA_ERR_BAD_ARG, "emia_rle_line_count: %s", "null pointer");
    const int64_t chunks = (nbytes + EMIA_RLE_TEXT_CHUNK - 1) / EMIA_RLE_TEXT_CHUNK;
    k_rle_lines<false><<<(unsigned)chunks, EMIA_RLE_LINE_THREADS, 0, (cudaStream_t)stream>>>(text, nbytes, chunk_lines, nullptr, nullptr);
    return emia_check_launch("emia_rle_line_count launch: %s");
}
extern "C" int emia_rle_line_index(const uint8_t* text, int64_t nbytes, const int64_t* chunk_off, int64_t* line_off, void* stream) {
    if (nbytes < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_rle_line_index: %s", "bad size");
    if (nbytes == 0) return EMIA_OK;
    if (!text || !chunk_off || !line_off) return emia_fail(EMIA_ERR_BAD_ARG, "emia_rle_line_index: %s", "null pointer");
    const int64_t chunks = (nbytes + EMIA_RLE_TEXT_CHUNK - 1) / EMIA_RLE_TEXT_CHUNK;
    k_rle_lines<true><<<(unsigned)chunks, EMIA_RLE_LINE_THREADS, 0, (cudaStream_t)stream>>>(text, nbytes, nullptr, chunk_off, line_off);
    return emia_check_launch("emia_rle_line_index launch: %s");
}

// ---- lines -> runs: one warp per line --------------------------------------------------------------------------------------
// Pass 1 (kStore = false) counts; pass 2 repeats the same walk and stores.  The values of a line are only stored when pass 1
// gave it runs (status OK), so a malformed line never writes into its neighbour's range.
template <bool kStore>
__global__ void __launch_bounds__(128) k_rle_parse(const uint8_t* __restrict__ text, const int64_t* __restrict__ line_off, int64_t n_lines,
                                                   int64_t* __restrict__ data_cnt, int64_t* __restrict__ run_cnt,
                                                   const int64_t* __restrict__ data_off, const int64_t* __restrict__ run_scan,
                                                   int64_t* __restrict__ run_off, int64_t* __restrict__ runs, int64_t* __restrict__ field,
                                                   int32_t* __restrict__ line_idx, int32_t* __restrict__ status) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int64_t j = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (j >= n_lines) return;
    const int64_t b = line_off[j], e = line_off[j + 1];
    if (kStore && j == n_lines - 1 && lane == 0) run_off[data_off[n_lines]] = run_scan[n_lines];
    // the last comma separates ImageId from EncodedPixels (a quoted ImageId may hold commas, EncodedPixels never does)
    int64_t comma = -1;
    bool any = false;
    for (int64_t w = b; w < e; w += 32) {
        const int64_t p = w + lane;
        const uint8_t c = p < e ? text[p] : (uint8_t)' ';
        const unsigned cm = __ballot_sync(FULL, c == ',');
        any |= __ballot_sync(FULL, !emia_rle_is_blank(c)) != 0u;
        if (cm) comma = w + emia_msb(cm);
    }
    if (!any) {                                    // an empty line is no data line
        if (!kStore && lane == 0) { data_cnt[j] = 0; run_cnt[j] = 0; }
        return;
    }
    int st = EMIA_RLE_OK;
    int64_t nv = 0;
    const bool store = kStore && run_scan[j + 1] > run_scan[j];
    const int64_t vbase = kStore ? 2 * run_scan[j] : 0;
    if (comma < 0) {
        st = EMIA_RLE_NO_SEPARATOR;
    } else {
        unsigned carry = 0;                        // bit 0: the byte before the window is a digit
        for (int64_t w = comma + 1; w < e; w += 32) {
            const int64_t p = w + lane;
            const uint8_t c = p < e ? text[p] : (uint8_t)' ';
            const bool dig = emia_rle_is_digit(c);
            if (__ballot_sync(FULL, !dig && !emia_rle_is_blank(c))) { st = EMIA_RLE_BAD_CHAR; break; }
            const unsigned dm = __ballot_sync(FULL, dig);
            const unsigned starts = dm & ~((dm << 1) | carry);
            carry = dm >> 31;
            const bool mine = (starts >> lane) & 1u;
            int64_t v = 0;
            const bool too_long = mine && emia_rle_parse_uint(text + p, e - p, &v) < 0;
            if (__ballot_sync(FULL, too_long)) { st = EMIA_RLE_LONG_VALUE; break; }
            if (store && mine) runs[vbase + nv + emia_popc(starts & ((1u << lane) - 1u))] = v;
            nv += emia_popc(starts);
        }
        if (st == EMIA_RLE_OK && (nv & 1)) st = EMIA_RLE_ODD_COUNT;
    }
    if (lane != 0) return;
    if (!kStore) {
        data_cnt[j] = 1;
        run_cnt[j] = st == EMIA_RLE_OK ? nv / 2 : 0;
    } else {
        const int64_t d = data_off[j];
        run_off[d] = run_scan[j];
        field[2 * d] = b;
        field[2 * d + 1] = comma < 0 ? b : comma;
        line_idx[d] = (int32_t)j;
        status[d] = st;
    }
}

extern "C" int emia_rle_parse_count(const uint8_t* text, const int64_t* line_off, int64_t n_lines, int64_t* data_cnt, int64_t* run_cnt,
                                    void* stream) {
    if (n_lines < 0 || n_lines > INT32_MAX) return emia_fail(EMIA_ERR_BAD_ARG, "emia_rle_parse_count: %s", "bad line count");
    if (n_lines == 0) return EMIA_OK;
    if (!text || !line_off || !data_cnt || !run_cnt) return emia_fail(EMIA_ERR_BAD_ARG, "emia_rle_parse_count: %s", "null pointer");
    k_rle_parse<false><<<(unsigned)((n_lines * 32 + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        text, line_off, n_lines, data_cnt, run_cnt, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
    return emia_check_launch("emia_rle_parse_count launch: %s");
}
extern "C" int emia_rle_parse_fill(const uint8_t* text, const int64_t* line_off, int64_t n_lines, const int64_t* data_off,
                                   const int64_t* run_scan, int64_t* run_off, int64_t* runs, int64_t* field, int32_t* line_idx,
                                   int32_t* status, void* stream) {
    if (n_lines < 0 || n_lines > INT32_MAX) return emia_fail(EMIA_ERR_BAD_ARG, "emia_rle_parse_fill: %s", "bad line count");
    if (n_lines == 0) return EMIA_OK;
    if (!text || !line_off || !data_off || !run_scan || !run_off || !runs || !field || !line_idx || !status)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_rle_parse_fill: %s", "null pointer");
    k_rle_parse<true><<<(unsigned)((n_lines * 32 + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        text, line_off, n_lines, nullptr, nullptr, data_off, run_scan, run_off, runs, field, line_idx, status);
    return emia_check_launch("emia_rle_parse_fill launch: %s");
}

// ---- runs -> instances ---------------------------------------------------------------------------------------------------
// plan: one warp per instance, lanes over its runs; the first rejected run (in run order) names the status
__global__ void __launch_bounds__(128) k_rle_decode_plan(const int64_t* __restrict__ runs, const int64_t* __restrict__ run_off,
                                                         const int32_t* __restrict__ rows, int64_t n, int H, int W,
                                                         emia_inst_meta* __restrict__ meta, int64_t* __restrict__ crop_words,
                                                         int32_t* __restrict__ bbox, int32_t* __restrict__ area,
                                                         int32_t* __restrict__ status) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= n) return;
    const int64_t line = rows ? (int64_t)rows[i] : i;
    const int64_t r0 = run_off[line], nr = run_off[line + 1] - r0;
    const int64_t* rr = runs + 2 * r0;
    const int64_t hw = (int64_t)H * W;
    long long err = LLONG_MAX, a = 0;              // err: 16 * (first bad run) + code
    int ymin = INT_MAX, ymax = -1, xmin = INT_MAX, xmax = -1;
    for (int64_t k = lane; k < nr; k += 32) {
        const int64_t s = rr[2 * k], l = rr[2 * k + 1];
        const int64_t prev_end = k ? rr[2 * k - 2] + rr[2 * k - 1] - 1 : 0;
        const int code = emia_rle_run_status(prev_end, s, l, hw);
        if (code) { err = min(err, (long long)(16 * k + code)); continue; }
        int y0, y1, x0, x1;
        emia_rle_run_extent(s, l, H, &y0, &y1, &x0, &x1);
        a += l;
        ymin = min(ymin, y0); ymax = max(ymax, y1); xmin = min(xmin, x0); xmax = max(xmax, x1);
    }
    for (int o = 16; o; o >>= 1) {
        err = min(err, __shfl_xor_sync(FULL, err, o));
        a += __shfl_xor_sync(FULL, a, o);
        ymin = min(ymin, __shfl_xor_sync(FULL, ymin, o)); ymax = max(ymax, __shfl_xor_sync(FULL, ymax, o));
        xmin = min(xmin, __shfl_xor_sync(FULL, xmin, o)); xmax = max(xmax, __shfl_xor_sync(FULL, xmax, o));
    }
    if (lane) return;
    int code = err == LLONG_MAX ? EMIA_RLE_OK : (int)(err & 15);
    if (code == EMIA_RLE_OK && a > INT32_MAX) code = EMIA_RLE_AREA;
    if (code != EMIA_RLE_OK) a = 0;
    const emia_inst_meta mt = emia_meta_from_bbox(a, ymin, xmin, ymax, xmax);
    meta[i] = mt;
    crop_words[i] = (int64_t)mt.ch * mt.cw;
    ((int4*)bbox)[i] = a ? make_int4(ymin, xmin, ymax, xmax) : make_int4(-1, -1, -1, -1);
    area[i] = (int32_t)a;
    status[i] = code;
}

// decode: one CTA per instance; work item = (crop word-column, band of EMIA_RLE_BAND rows), one warp each.  Every lane finds the
// first run of its pixel column that ends at or after the band's first pixel by binary search, then the warp walks the rows: the
// runs are sorted and disjoint, so each row step advances a lane's run at most once.
#define EMIA_RLE_BAND 128
__global__ void __launch_bounds__(128) k_rle_decode(const int64_t* __restrict__ runs, const int64_t* __restrict__ run_off,
                                                    const int32_t* __restrict__ rows, int64_t n, int H,
                                                    const emia_inst_meta* __restrict__ meta, const int64_t* __restrict__ crop_off,
                                                    uint32_t* __restrict__ crops) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (int64_t inst = blockIdx.x; inst < n; inst += gridDim.x) {
        const emia_inst_meta m = meta[inst];
        if (m.ch <= 0 || m.cw <= 0) continue;
        const int64_t line = rows ? (int64_t)rows[inst] : inst;
        const int64_t r0 = run_off[line], nr = run_off[line + 1] - r0;
        const int64_t* rr = runs + 2 * r0;
        uint32_t* crop = crops + crop_off[inst];
        const int bands = (m.ch + EMIA_RLE_BAND - 1) / EMIA_RLE_BAND;
        const int items = m.cw * bands;
        for (int it = warp; it < items; it += nwarps) {
            const int band = it / m.cw, c = it - band * m.cw;
            const int y0 = band * EMIA_RLE_BAND, y1 = min(m.ch, y0 + EMIA_RLE_BAND);
            const int x = (m.wc0 + c) * 32 + lane;
            const bool live = x >= m.rx0 && x < m.rx1;
            int64_t f = (int64_t)x * H + m.ry0 + y0;             // 0-indexed flat index of the lane's pixel
            int64_t k = nr, s0 = 0, e0 = -1;                      // current run: flat indices [s0, e0]
            if (live) {
                int64_t lo = 0, hi = nr;
                while (lo < hi) {
                    const int64_t mid = (lo + hi) >> 1;
                    if (rr[2 * mid] + rr[2 * mid + 1] - 2 < f) lo = mid + 1;
                    else hi = mid;
                }
                k = lo;
                if (k < nr) { s0 = rr[2 * k] - 1; e0 = s0 + rr[2 * k + 1] - 1; }
            }
            for (int y = y0; y < y1; ++y, ++f) {
                if (k < nr && e0 < f && ++k < nr) { s0 = rr[2 * k] - 1; e0 = s0 + rr[2 * k + 1] - 1; }
                const unsigned word = __ballot_sync(FULL, k < nr && s0 <= f);
                if (lane == 0) crop[(size_t)y * m.cw + c] = word;
            }
        }
    }
}

static int emia_rle_frame_ok(int H, int W) { return H >= 1 && H <= 65535 && W >= 1 && W <= 65535; }

extern "C" int emia_rle_decode_plan(const int64_t* runs, const int64_t* run_off, const int32_t* rows, int64_t n, int H, int W,
                                    emia_inst_meta* meta, int64_t* crop_words, int32_t* bbox, int32_t* area, int32_t* status,
                                    void* stream) {
    if (n < 0 || !emia_rle_frame_ok(H, W)) return emia_fail(EMIA_ERR_BAD_ARG, "emia_rle_decode_plan: %s", "bad shape (1 <= H, W <= 65535)");
    if (n == 0) return EMIA_OK;
    if (!runs || !run_off || !meta || !crop_words || !bbox || !area || !status)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_rle_decode_plan: %s", "null pointer");
    k_rle_decode_plan<<<(unsigned)((n * 32 + 127) / 128), 128, 0, (cudaStream_t)stream>>>(runs, run_off, rows, n, H, W, meta, crop_words,
                                                                                         bbox, area, status);
    return emia_check_launch("emia_rle_decode_plan launch: %s");
}
extern "C" int emia_rle_decode(const int64_t* runs, const int64_t* run_off, const int32_t* rows, int64_t n, int H,
                               const emia_inst_meta* meta, const int64_t* crop_off, uint32_t* crops, void* stream) {
    if (n < 0 || H < 1 || H > 65535) return emia_fail(EMIA_ERR_BAD_ARG, "emia_rle_decode: %s", "bad shape (1 <= H <= 65535)");
    if (n == 0) return EMIA_OK;
    if (!runs || !run_off || !meta || !crop_off || !crops) return emia_fail(EMIA_ERR_BAD_ARG, "emia_rle_decode: %s", "null pointer");
    const unsigned grid = (unsigned)(n < 65535 ? n : 65535);
    k_rle_decode<<<grid, 128, 0, (cudaStream_t)stream>>>(runs, run_off, rows, n, H, meta, crop_off, crops);
    return emia_check_launch("emia_rle_decode launch: %s");
}
