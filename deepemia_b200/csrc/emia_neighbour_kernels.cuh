// emia_neighbour_kernels.cuh — neighbours_results.csv on the device (part of emia_kernels.cu): the listed instances of one image,
// their centroids, a class-keyed uniform grid built by counting sort, the centroid nearest neighbour, the closest mask, the touching
// count and the agglomerates (core/emia_neighbour.cuh), and the text of the rows.
#pragma once

#define EMIA_NB_THREADS 128

// listed flag, centroid and output defaults per instance; counts the grid cells its bbox covers
__global__ void __launch_bounds__(EMIA_NB_THREADS) k_nb_plan(const double* __restrict__ records, const int64_t* __restrict__ inst_cont_off,
                                                             const int32_t* __restrict__ bbox, const int64_t* __restrict__ mom,
                                                             const int32_t* __restrict__ class_idx, int64_t n, EmiaNbGrid g,
                                                             double* __restrict__ nbf, int32_t* __restrict__ nbi,
                                                             int64_t* __restrict__ cell_cnt) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int listed = 0;
    for (int64_t j = inst_cont_off[i]; j < inst_cont_off[i + 1] && !listed; ++j) listed = records[j * EMIA_REC_FIELDS + EMIA_REC_MEASURED] == 1.0;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    double* f = nbf + EMIA_NB_F * i;
    int32_t* o = nbi + EMIA_NB_I * i;
    f[0] = listed ? (double)mom[3 * i + 1] / (double)mom[3 * i] : nan;
    f[1] = listed ? (double)mom[3 * i + 2] / (double)mom[3 * i] : nan;
    f[2] = nan; f[3] = nan;
    o[0] = listed; o[1] = -1; o[2] = -1; o[3] = 0; o[4] = listed ? (int32_t)i : -1; o[5] = 0;
    if (!listed) return;
    const int32_t* b = bbox + 4 * i;
    const int64_t plane = (int64_t)class_idx[i] * g.gx * g.gy;
    for (int y = b[0] / g.cs; y <= b[2] / g.cs; ++y)
        for (int x = b[1] / g.cs; x <= b[3] / g.cs; ++x) atomicAdd((unsigned long long*)(cell_cnt + plane + (int64_t)y * g.gx + x), 1ull);
}

// cell lists: entries of a cell in any order (every result is a minimum with an index tie rule, or a count)
__global__ void __launch_bounds__(EMIA_NB_THREADS) k_nb_scatter(const int32_t* __restrict__ bbox, const int32_t* __restrict__ class_idx,
                                                                const int32_t* __restrict__ nbi, int64_t n, EmiaNbGrid g,
                                                                const int64_t* __restrict__ cell_off, int32_t* __restrict__ cursor,
                                                                int32_t* __restrict__ ent, int32_t* __restrict__ parent) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    parent[i] = (int32_t)i;
    if (!nbi[EMIA_NB_I * i]) return;
    const int32_t* b = bbox + 4 * i;
    const int64_t plane = (int64_t)class_idx[i] * g.gx * g.gy;
    for (int y = b[0] / g.cs; y <= b[2] / g.cs; ++y)
        for (int x = b[1] / g.cs; x <= b[3] / g.cs; ++x) {
            const int64_t c = plane + (int64_t)y * g.gx + x;
            ent[cell_off[c] + atomicAdd(cursor + c, 1)] = (int32_t)i;
        }
}

// one thread per instance: centroid nearest neighbour, then the closest mask seeded with it; touching pairs are united once (k > i)
__global__ void __launch_bounds__(EMIA_NB_THREADS) k_nb_search(const uint32_t* __restrict__ crops, const int32_t* __restrict__ meta,
                                                               const int64_t* __restrict__ crop_off, const int32_t* __restrict__ bbox,
                                                               const int32_t* __restrict__ class_idx, int64_t n, EmiaNbGrid g,
                                                               const int64_t* __restrict__ cell_off, const int32_t* __restrict__ ent,
                                                               double um_pix, double* __restrict__ nbf, int32_t* __restrict__ nbi,
                                                               int32_t* parent) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !nbi[EMIA_NB_I * i]) return;
    double d2;
    const int nn = emia_nb_nearest((int)i, nbf, EMIA_NB_F, class_idx, cell_off, ent, g, &d2);
    if (nn < 0) return;
    long long D2;
    int nt;
    const int me = (int)i;
    const int cl = emia_nb_closest(me, nn, crops, meta, crop_off, bbox, class_idx, cell_off, ent, g, &D2, &nt,
                                   [&](int k) { if (k > me) emia_nb_unite(parent, me, k); });
    double* f = nbf + EMIA_NB_F * i;
    int32_t* o = nbi + EMIA_NB_I * i;
    f[2] = sqrt(d2) * um_pix;
    f[3] = sqrt((double)D2) * um_pix;
    o[1] = nn; o[2] = cl; o[3] = nt;
}

// agglomerate = the root (lowest member) of the instance's component; sizes by a histogram of roots in the roots' size fields, then
// copied to every member
__global__ void __launch_bounds__(EMIA_NB_THREADS) k_nb_roots(int64_t n, int32_t* parent, int32_t* __restrict__ nbi) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !nbi[EMIA_NB_I * i]) return;
    const int r = emia_nb_find(parent, (int)i);
    nbi[EMIA_NB_I * i + 4] = r;
    atomicAdd(nbi + EMIA_NB_I * (int64_t)r + 5, 1);
}
__global__ void __launch_bounds__(EMIA_NB_THREADS) k_nb_sizes(int64_t n, int32_t* nbi) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !nbi[EMIA_NB_I * i]) return;
    const int r = nbi[EMIA_NB_I * i + 4];
    if (r != i) nbi[EMIA_NB_I * i + 5] = nbi[EMIA_NB_I * (int64_t)r + 5];
}

extern "C" int emia_neighbour_plan(const double* records, const int64_t* inst_cont_off, const int32_t* bbox, const int64_t* moments01,
                                   const int32_t* class_idx, int64_t n, int32_t n_class, int32_t H, int32_t W, int32_t cell_size,
                                   double* nbf, int32_t* nbi, int64_t* cell_cnt, void* stream) {
    if (n < 0 || n > INT32_MAX || n_class < 1 || H <= 0 || W <= 0 || cell_size <= 0)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_neighbour_plan: %s", "bad size");
    const EmiaNbGrid g{cell_size, (W + cell_size - 1) / cell_size, (H + cell_size - 1) / cell_size};
    const int64_t ncells = (int64_t)n_class * g.gx * g.gy;
    if (!cell_cnt) return emia_fail(EMIA_ERR_BAD_ARG, "emia_neighbour_plan: %s", "null pointer");
    if (cudaMemsetAsync(cell_cnt, 0, (ncells + 1) * sizeof(int64_t), (cudaStream_t)stream) != cudaSuccess)
        return emia_check_launch("emia_neighbour_plan memset: %s");
    if (n == 0) return EMIA_OK;
    if (!records || !inst_cont_off || !bbox || !moments01 || !class_idx || !nbf || !nbi)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_neighbour_plan: %s", "null pointer");
    k_nb_plan<<<(unsigned)((n + EMIA_NB_THREADS - 1) / EMIA_NB_THREADS), EMIA_NB_THREADS, 0, (cudaStream_t)stream>>>(
        records, inst_cont_off, bbox, moments01, class_idx, n, g, nbf, nbi, cell_cnt);
    return emia_check_launch("emia_neighbour_plan launch: %s");
}

extern "C" int emia_neighbour_search(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, const int32_t* bbox,
                                     const int32_t* class_idx, int64_t n, int32_t n_class, int32_t H, int32_t W, int32_t cell_size,
                                     const int64_t* cell_off, int32_t* ent, double um_pix, double* nbf, int32_t* nbi, int32_t* work,
                                     void* stream) {
    if (n < 0 || n > INT32_MAX || n_class < 1 || H <= 0 || W <= 0 || cell_size <= 0)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_neighbour_search: %s", "bad size");
    if (n == 0) return EMIA_OK;
    if (!crops || !meta || !crop_off || !bbox || !class_idx || !cell_off || !ent || !nbf || !nbi || !work)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_neighbour_search: %s", "null pointer");
    const EmiaNbGrid g{cell_size, (W + cell_size - 1) / cell_size, (H + cell_size - 1) / cell_size};
    const int64_t ncells = (int64_t)n_class * g.gx * g.gy;
    int32_t* parent = work;
    int32_t* cursor = work + n;
    cudaStream_t st = (cudaStream_t)stream;
    if (cudaMemsetAsync(cursor, 0, ncells * sizeof(int32_t), st) != cudaSuccess) return emia_check_launch("emia_neighbour_search memset: %s");
    const unsigned grid = (unsigned)((n + EMIA_NB_THREADS - 1) / EMIA_NB_THREADS);
    k_nb_scatter<<<grid, EMIA_NB_THREADS, 0, st>>>(bbox, class_idx, nbi, n, g, cell_off, cursor, ent, parent);
    k_nb_search<<<grid, EMIA_NB_THREADS, 0, st>>>(crops, (const int32_t*)meta, crop_off, bbox, class_idx, n, g, cell_off, ent, um_pix,
                                                   nbf, nbi, parent);
    k_nb_roots<<<grid, EMIA_NB_THREADS, 0, st>>>(n, parent, nbi);
    k_nb_sizes<<<grid, EMIA_NB_THREADS, 0, st>>>(n, nbi);
    return emia_check_launch("emia_neighbour_search launch: %s");
}

// ---- neighbours_results.csv: one row per listed instance -----------------------------------------------------------------------
// Lane f writes field f: 0 Instance_ID, 1 Class,Class_Name (strs[3 + class_idx]), 2 / 3 the centroid, 4 / 5 the nearest neighbour's
// Instance_ID and distance, 6 / 7 the closest neighbour's and the edge distance (all four empty without a candidate), 8 touching,
// 9 the agglomerate's Instance_ID, 10 its size, 11 "Detected scale bar,File name" (strs[2]) and the line end.  An Instance_ID is
// strs[0] + (index + 1) + strs[1].
#define EMIA_CSV_NB_LAST 11
template <bool kWrite>
__global__ void __launch_bounds__(EMIA_CSV_THREADS) k_csv_neighbour(const double* __restrict__ nbf, const int32_t* __restrict__ nbi, int64_t n,
                                                                    const int32_t* __restrict__ class_idx, const uint8_t* __restrict__ strs,
                                                                    const int64_t* __restrict__ str_off, int64_t* __restrict__ row_len,
                                                                    const int64_t* __restrict__ row_off, uint8_t* __restrict__ text) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= n) return;
    const int32_t* o = nbi + EMIA_NB_I * i;
    if (!o[0]) {                                    // not listed: no row
        if (!kWrite && lane == 0) row_len[i] = 0;
        return;
    }
    const double* f = nbf + EMIA_NB_F * i;
    uint8_t num[EMIA_TEXT_NUM_MAX];
    int nlen = 0;
    int s0 = -1, s1 = -1;                           // strings before / after the number
    int64_t id = -1;                                // an Instance_ID field: strs[0] + id + 1 + strs[1]
    if (lane == 0) id = i;
    else if (lane == 1) s0 = 3 + class_idx[i];
    else if (lane == 2 || lane == 3) nlen = emia_format_f64(num, f[lane - 2]);
    else if (lane == 4 && o[1] >= 0) id = o[1];
    else if (lane == 5 && o[1] >= 0) nlen = emia_format_f64(num, f[2]);
    else if (lane == 6 && o[2] >= 0) id = o[2];
    else if (lane == 7 && o[2] >= 0) nlen = emia_format_f64(num, f[3]);
    else if (lane == 8) nlen = emia_write_i64(num, o[3]);
    else if (lane == 9) id = o[4];
    else if (lane == 10) nlen = emia_write_i64(num, o[5]);
    else if (lane == EMIA_CSV_NB_LAST) s0 = 2;
    if (id >= 0) { s0 = 0; s1 = 1; nlen = emia_write_i64(num, id + 1); }
    const int64_t a0 = s0 >= 0 ? str_off[s0] : 0, l0 = s0 >= 0 ? str_off[s0 + 1] - a0 : 0;
    const int64_t a1 = s1 >= 0 ? str_off[s1] : 0, l1 = s1 >= 0 ? str_off[s1 + 1] - a1 : 0;
    const int term = lane < EMIA_CSV_NB_LAST ? 1 : lane == EMIA_CSV_NB_LAST ? 2 : 0;
    const int64_t len = l0 + nlen + l1 + term;
    int64_t inc = len;
    for (int d = 1; d < 32; d <<= 1) {
        const int64_t v = __shfl_up_sync(FULL, inc, d);
        if (lane >= d) inc += v;
    }
    if (!kWrite) {
        if (lane == 31) row_len[i] = inc;
        return;
    }
    uint8_t* p = text + row_off[i] + inc - len;
    for (int64_t j = 0; j < l0; ++j) *p++ = strs[a0 + j];
    for (int j = 0; j < nlen; ++j) *p++ = num[j];
    for (int64_t j = 0; j < l1; ++j) *p++ = strs[a1 + j];
    if (term == 1) *p = ',';
    else if (term == 2) { p[0] = '\r'; p[1] = '\n'; }
}

static int emia_csv_neighbour_launch(const char* what, bool write, const double* nbf, const int32_t* nbi, int64_t n,
                                     const int32_t* class_idx, const uint8_t* strs, const int64_t* str_off, int n_str, int64_t* row_len,
                                     const int64_t* row_off, uint8_t* text, void* stream) {
    if (n < 0 || n_str < 3) return emia_fail(EMIA_ERR_BAD_ARG, "%s: bad size", what);
    if (n == 0) return EMIA_OK;
    if (!nbf || !nbi || !class_idx || !strs || !str_off || (write ? (!row_off || !text) : !row_len))
        return emia_fail(EMIA_ERR_BAD_ARG, "%s: null pointer", what);
    const unsigned grid = (unsigned)((n * 32 + EMIA_CSV_THREADS - 1) / EMIA_CSV_THREADS);
    if (write)
        k_csv_neighbour<true><<<grid, EMIA_CSV_THREADS, 0, (cudaStream_t)stream>>>(nbf, nbi, n, class_idx, strs, str_off, nullptr, row_off,
                                                                                   text);
    else
        k_csv_neighbour<false><<<grid, EMIA_CSV_THREADS, 0, (cudaStream_t)stream>>>(nbf, nbi, n, class_idx, strs, str_off, row_len, nullptr,
                                                                                    nullptr);
    return emia_check_launch(write ? "emia_csv_neighbour_write launch: %s" : "emia_csv_neighbour_count launch: %s");
}

extern "C" int emia_csv_neighbour_count(const double* nbf, const int32_t* nbi, int64_t n, const int32_t* class_idx, const uint8_t* strs,
                                        const int64_t* str_off, int n_str, int64_t* row_len, void* stream) {
    return emia_csv_neighbour_launch("emia_csv_neighbour_count", false, nbf, nbi, n, class_idx, strs, str_off, n_str, row_len, nullptr,
                                     nullptr, stream);
}
extern "C" int emia_csv_neighbour_write(const double* nbf, const int32_t* nbi, int64_t n, const int32_t* class_idx, const uint8_t* strs,
                                        const int64_t* str_off, int n_str, const int64_t* row_off, uint8_t* text, void* stream) {
    return emia_csv_neighbour_launch("emia_csv_neighbour_write", true, nbf, nbi, n, class_idx, strs, str_off, n_str, nullptr, row_off,
                                     text, stream);
}
