// emia_cocoeval_kernels.cuh — COCO `segm` evaluation on the device (part of emia_kernels.cu; rules: core/emia_cocoeval.cuh,
// definition: oracle/cocoeval.py).
//
// Layout (the host builds it, engine.coco_evaluate): the evaluated detections ("DT list", n_dt) and GTs ("GT list") are sorted by
// (category, image, file order), so a category and a (category, image) "segment" are contiguous ranges of each list.  Stages:
//   order       stable LSD radix sorts of the DT list (8-bit digits, one CTA per 256-element tile: tile histograms ->
//               emia_exclusive_scan_i64 -> stable scatter with __match_any_sync ranks): by score descending (64-bit key), then that
//               sequence by category (corder: accumulate's order, score desc then image then file order) and by segment (morder:
//               evaluateImg's order within each segment, "match order"); rank = place in the segment.  O(n) per pass;
//   pairs       per frame size: GT boxes binned in a grid keyed by (segment, cell) (count -> scan -> scatter), each kept detection
//               (rank < maxDets[-1]) walks the cells its box covers and takes a GT whose box meets its own in the cell holding the
//               top-left corner of the two boxes' intersection, so a pair is seen once; count -> scan (over all frame sizes, in
//               match order) -> fill, one warp per detection: the intersection popcount (emia_crop_inter_warp), the IoU and the
//               GT's flags (crowd, id 0, _ignore per area range);
//   match       one warp per (segment, area range), lane t = IoU threshold t, a matched-GT bitmap per lane; streams the segment's
//               pairs (which are in rank order) 32 at a time; per detection and area range a word of tp bits (0..9) and fp bits
//               (10..19), i.e. dtm != 0 and not dtIg / dtm == 0 and not dtIg;
//   accumulate  one CTA per (category, area range, maxDet, threshold): block scans of the included detections' tp / fp, rc and pr
//               in numpy's operation order; q[r] = the largest pr of the detections with rc >= recThrs[r] (what the reverse
//               running maximum and searchsorted give), gathered in 101 shared-memory maxima: no per-detection scratch.
#pragma once

#define EMIA_CE_THREADS 128
#define EMIA_CE_ACC_THREADS 256
#define EMIA_CE_PARAMS (EMIA_CE_T + EMIA_CE_R + 2 * EMIA_CE_A + 1)

struct EmiaCeParams {
    double thr[EMIA_CE_T];          // min(iouThrs[t], 1 - 1e-10), numpy's values
    double rec[EMIA_CE_R];          // recThrs
    double lo[EMIA_CE_A], hi[EMIA_CE_A];
    double eps;                     // np.spacing(1)
    int max_det[EMIA_CE_M];
};

static EmiaCeParams emia_ce_params(const double* p, const int32_t* max_dets) {
    EmiaCeParams P;
    for (int t = 0; t < EMIA_CE_T; ++t) P.thr[t] = p[t];
    for (int r = 0; r < EMIA_CE_R; ++r) P.rec[r] = p[EMIA_CE_T + r];
    for (int a = 0; a < EMIA_CE_A; ++a) {
        P.lo[a] = p[EMIA_CE_T + EMIA_CE_R + a];
        P.hi[a] = p[EMIA_CE_T + EMIA_CE_R + EMIA_CE_A + a];
    }
    P.eps = p[EMIA_CE_PARAMS - 1];
    for (int m = 0; m < EMIA_CE_M; ++m) P.max_det[m] = max_dets ? max_dets[m] : 0;
    return P;
}

// ---- order: stable radix sorts of the DT list ------------------------------------------------------------------------------------
#define EMIA_CE_SORT_TILE 256
#define EMIA_CE_SORT_BINS 256

// keys: score descending as an unsigned 64-bit key (-0.0 and 0.0 tie, as numpy's comparison has them), category, segment;
// idx = 0 .. n - 1
__global__ void __launch_bounds__(EMIA_CE_THREADS) k_ce_keys(const double* __restrict__ score, const int32_t* __restrict__ cat,
                                                             const int32_t* __restrict__ seg, int64_t n, uint64_t* __restrict__ skey,
                                                             uint64_t* __restrict__ ckey, uint64_t* __restrict__ gkey,
                                                             int32_t* __restrict__ idx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double v = score[i];
    uint64_t u = (uint64_t)__double_as_longlong(v == 0.0 ? 0.0 : v);
    u = (u >> 63) ? ~u : (u | 0x8000000000000000ull);        // ascending order of the doubles
    skey[i] = ~u;                                              // descending
    ckey[i] = (uint64_t)cat[i];
    gkey[i] = (uint64_t)seg[i];
    idx[i] = (int32_t)i;
}

// digit of element in[i] at `shift`, or EMIA_CE_SORT_BINS past the end
__device__ __forceinline__ int emia_ce_digit(const uint64_t* key, const int32_t* in, int64_t n, int64_t i, int shift) {
    return i < n ? (int)((key[in[i]] >> shift) & (EMIA_CE_SORT_BINS - 1)) : EMIA_CE_SORT_BINS;
}

// counts[d * n_tiles + tile] = elements of the tile with digit d (bin-major: its exclusive scan is the stable scatter base)
__global__ void __launch_bounds__(EMIA_CE_SORT_TILE) k_ce_sort_hist(const uint64_t* __restrict__ key, const int32_t* __restrict__ in,
                                                                    int64_t n, int shift, int64_t* __restrict__ counts) {
    __shared__ int hist[EMIA_CE_SORT_BINS];
    hist[threadIdx.x] = 0;
    __syncthreads();
    const int d = emia_ce_digit(key, in, n, (int64_t)blockIdx.x * EMIA_CE_SORT_TILE + threadIdx.x, shift);
    if (d < EMIA_CE_SORT_BINS) atomicAdd(&hist[d], 1);
    __syncthreads();
    counts[(int64_t)threadIdx.x * gridDim.x + blockIdx.x] = hist[threadIdx.x];
}

// out[base(d, tile) + the element's rank among the tile's elements of digit d, in tile order] = in[i]
__global__ void __launch_bounds__(EMIA_CE_SORT_TILE) k_ce_sort_scatter(const uint64_t* __restrict__ key, const int32_t* __restrict__ in,
                                                                       int64_t n, int shift, const int64_t* __restrict__ base,
                                                                       int32_t* __restrict__ out) {
    __shared__ int wcnt[EMIA_CE_SORT_TILE / 32][EMIA_CE_SORT_BINS + 1];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int k = threadIdx.x; k < (EMIA_CE_SORT_TILE / 32) * (EMIA_CE_SORT_BINS + 1); k += blockDim.x) (&wcnt[0][0])[k] = 0;
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * EMIA_CE_SORT_TILE + threadIdx.x;
    const int d = emia_ce_digit(key, in, n, i, shift);
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    if (lane == __ffs(peers) - 1) wcnt[w][d] = __popc(peers);
    __syncthreads();
    if (d == EMIA_CE_SORT_BINS) return;
    int r = __popc(peers & ((1u << lane) - 1u));
    for (int k = 0; k < w; ++k) r += wcnt[k][d];
    out[base[(int64_t)d * gridDim.x + blockIdx.x] + r] = in[i];
}

// rank[i] = place of DT i in its segment (morder lists the segments in rank order)
__global__ void __launch_bounds__(EMIA_CE_THREADS) k_ce_rank(const int32_t* __restrict__ morder, const int32_t* __restrict__ seg,
                                                             const int64_t* __restrict__ seg_off, int64_t n, int32_t* __restrict__ rank) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const int i = morder[p];
    rank[i] = (int32_t)(p - seg_off[seg[i]]);
}

// ---- pairs -----------------------------------------------------------------------------------------------------------------------
template <bool kScatter>
__global__ void __launch_bounds__(EMIA_CE_THREADS) k_ce_grid(const int32_t* __restrict__ bbox, const int32_t* __restrict__ gseg,
                                                             int64_t n, EmiaNbGrid g, int64_t* __restrict__ cell_cnt,
                                                             const int64_t* __restrict__ cell_off, int32_t* __restrict__ cursor,
                                                             int32_t* __restrict__ ent) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || gseg[i] < 0 || bbox[4 * i] < 0) return;
    const int32_t* b = bbox + 4 * i;
    const int64_t plane = (int64_t)gseg[i] * g.gx * g.gy;
    for (int y = b[0] / g.cs; y <= b[2] / g.cs; ++y)
        for (int x = b[1] / g.cs; x <= b[3] / g.cs; ++x) {
            const int64_t c = plane + (int64_t)y * g.gx + x;
            if (kScatter) ent[cell_off[c] + atomicAdd(cursor + c, 1)] = (int32_t)i;
            else atomicAdd((unsigned long long*)(cell_cnt + c), 1ull);
        }
}

// the match position of local detection j (its place in the pair CSR), or -1 when it is not evaluated or past maxDets[-1]
__device__ __forceinline__ int64_t emia_ce_dt_slot(int64_t j, const int32_t* dt_eval, const int32_t* rank, const int32_t* dt_seg,
                                                   const int64_t* seg_dt_off, int max_det) {
    const int e = dt_eval[j];
    if (e < 0) return -1;
    const int r = rank[e];
    return r < max_det ? seg_dt_off[dt_seg[e]] + r : -1;
}

// GT k of cell (cy, cx) is a pair of box b when the boxes meet and the top-left corner of their intersection lies in this cell
__device__ __forceinline__ bool emia_ce_pair_here(const int32_t* b, const int32_t* gb, int cy, int cx, int cs) {
    const int y0 = max(b[0], gb[0]), x0 = max(b[1], gb[1]);
    return gb[0] >= 0 && y0 <= min(b[2], gb[2]) && x0 <= min(b[3], gb[3]) && y0 / cs == cy && x0 / cs == cx;
}

__global__ void __launch_bounds__(EMIA_CE_THREADS) k_ce_pair_count(const int32_t* __restrict__ gt_bbox, const int32_t* __restrict__ dt_bbox,
                                                                   const int32_t* __restrict__ dt_eval, const int32_t* __restrict__ dt_gseg,
                                                                   int64_t n_dt, EmiaNbGrid g, const int64_t* __restrict__ cell_off,
                                                                   const int32_t* __restrict__ ent, const int32_t* __restrict__ rank,
                                                                   const int32_t* __restrict__ dt_seg, const int64_t* __restrict__ seg_dt_off,
                                                                   int max_det, int64_t* __restrict__ pair_cnt) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_dt) return;
    const int64_t slot = emia_ce_dt_slot(j, dt_eval, rank, dt_seg, seg_dt_off, max_det);
    if (slot < 0) return;
    const int32_t* b = dt_bbox + 4 * j;
    int cnt = 0;
    if (dt_gseg[j] >= 0 && b[0] >= 0) {
        const int64_t plane = (int64_t)dt_gseg[j] * g.gx * g.gy;
        for (int y = b[0] / g.cs; y <= b[2] / g.cs; ++y)
            for (int x = b[1] / g.cs; x <= b[3] / g.cs; ++x) {
                const int64_t c = plane + (int64_t)y * g.gx + x;
                const int64_t q1 = cell_off[c + 1];
                for (int64_t q = cell_off[c]; q < q1; ++q) cnt += emia_ce_pair_here(b, gt_bbox + 4 * ent[q], y, x, g.cs);
            }
    }
    pair_cnt[slot] = cnt;
}

struct EmiaCeSide {                  // one InstanceSet of the frame size
    const uint32_t* crops; const int32_t* meta; const int64_t* crop_off; const int32_t* bbox; const int32_t* area;
};

__global__ void __launch_bounds__(EMIA_CE_THREADS) k_ce_pair_fill(EmiaCeSide gt, const int32_t* __restrict__ gt_eval, EmiaCeSide dt,
                                                                  const int32_t* __restrict__ dt_eval, const int32_t* __restrict__ dt_gseg,
                                                                  int64_t n_dt, EmiaNbGrid g, const int64_t* __restrict__ cell_off,
                                                                  const int32_t* __restrict__ ent, const int32_t* __restrict__ rank,
                                                                  const int32_t* __restrict__ dt_seg, const int64_t* __restrict__ seg_dt_off,
                                                                  const double* __restrict__ gt_area_eval, const int32_t* __restrict__ gt_flags,
                                                                  EmiaCeParams P, const int64_t* __restrict__ pair_off,
                                                                  int32_t* __restrict__ pair_g, int32_t* __restrict__ pair_d,
                                                                  int32_t* __restrict__ pair_f, double* __restrict__ pair_iou) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int64_t j = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (j >= n_dt) return;
    const int64_t slot = emia_ce_dt_slot(j, dt_eval, rank, dt_seg, seg_dt_off, P.max_det[EMIA_CE_M - 1]);
    const int32_t* b = dt.bbox + 4 * j;
    if (slot < 0 || dt_gseg[j] < 0 || b[0] < 0) return;
    const int e = dt_eval[j];
    const int32_t* md = dt.meta + 8 * j;
    const EmiaCropRef rd{dt.crops + dt.crop_off[j], md[0], md[1], md[2], md[3]};
    int64_t p = pair_off[slot];
    const int64_t plane = (int64_t)dt_gseg[j] * g.gx * g.gy;
    for (int y = b[0] / g.cs; y <= b[2] / g.cs; ++y)
        for (int x = b[1] / g.cs; x <= b[3] / g.cs; ++x) {
            const int64_t c = plane + (int64_t)y * g.gx + x;
            for (int64_t q0 = cell_off[c]; q0 < cell_off[c + 1]; q0 += 32) {
                const int64_t q = q0 + lane;
                const int k = q < cell_off[c + 1] ? ent[q] : -1;
                unsigned hit = __ballot_sync(FULL, k >= 0 && emia_ce_pair_here(b, gt.bbox + 4 * k, y, x, g.cs));
                while (hit) {
                    const int src = __ffs(hit) - 1;
                    hit &= hit - 1;
                    const int kk = __shfl_sync(FULL, k, src);
                    const int32_t* mg = gt.meta + 8 * kk;
                    const EmiaCropRef rg{gt.crops + gt.crop_off[kk], mg[0], mg[1], mg[2], mg[3]};
                    const int inter = emia_crop_inter_warp(rd, rg, lane);
                    if (lane == 0) {
                        const int ge = gt_eval[kk];
                        const int f = gt_flags[ge];
                        const double ga = gt_area_eval[ge];
                        int ign = 0;
                        for (int a = 0; a < EMIA_CE_A; ++a) ign |= (int)emia_ce_ignore(ga, f & EMIA_CE_CROWD, P.lo[a], P.hi[a]) << a;
                        pair_g[p] = ge;
                        pair_d[p] = e;
                        pair_f[p] = f | ign << 4;
                        pair_iou[p] = emia_ce_iou(inter, dt.area[j], gt.area[kk], f & EMIA_CE_CROWD);
                    }
                    ++p;
                }
            }
        }
}

// ---- match -----------------------------------------------------------------------------------------------------------------------
// block = segment, warp = area range, lane t < EMIA_CE_T = IoU threshold t (the other lanes follow with a threshold no IoU reaches)
__global__ void __launch_bounds__(32 * EMIA_CE_A) k_ce_match(const int64_t* __restrict__ seg_dt_off, const int64_t* __restrict__ seg_gt_off,
                                                             const int64_t* __restrict__ wseg_off, int64_t n_words,
                                                             const int32_t* __restrict__ morder, const double* __restrict__ dt_area,
                                                             const int64_t* __restrict__ pair_off, const int32_t* __restrict__ pair_g,
                                                             const int32_t* __restrict__ pair_d, const int32_t* __restrict__ pair_f,
                                                             const double* __restrict__ pair_iou, int64_t n_dt, EmiaCeParams P,
                                                             uint32_t* matched, uint32_t* __restrict__ state) {
    const unsigned FULL = 0xffffffffu;
    const int s = blockIdx.x, a = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t d0 = seg_dt_off[s], dn = min(seg_dt_off[s + 1] - d0, (int64_t)P.max_det[EMIA_CE_M - 1]);
    const int64_t g0 = seg_gt_off[s];
    const double lo = P.lo[a], hi = P.hi[a];
    uint32_t* st = state + a * n_dt;
    for (int64_t q = lane; q < dn; q += 32) {                       // unmatched: a false positive unless outside the area range
        const int i = morder[d0 + q];
        st[i] = emia_ce_ignore(dt_area[i], false, lo, hi) ? 0u : 0x3ffu << 10;
    }
    __syncwarp();
    const double thr = lane < EMIA_CE_T ? P.thr[lane] : 2.0;
    uint32_t* bm = matched + (int64_t)(a * EMIA_CE_T + min(lane, EMIA_CE_T - 1)) * n_words + wseg_off[s];
    const int64_t p1 = pair_off[d0 + dn];
    int cur = -1, bg = -1, bf = 0;
    bool bign = false;
    double biou = 0.0;
    auto commit = [&]() {
        const bool out = emia_ce_ignore(dt_area[cur], false, lo, hi);
        bool tp = false, fp = !out;
        if (bg >= 0) {
            if (lane < EMIA_CE_T) bm[bg >> 5] |= 1u << (bg & 31);
            const bool id0 = bf & EMIA_CE_ID0;                      // dtm == 0: counted as no match
            tp = !id0 && !bign;
            fp = id0 && !(bign || out);
        }
        const unsigned tb = __ballot_sync(FULL, tp) & 0x3ffu, fb = __ballot_sync(FULL, fp) & 0x3ffu;
        if (lane == 0) st[cur] = tb | fb << 10;
    };
    for (int64_t base = pair_off[d0]; base < p1; base += 32) {
        const int64_t p = base + lane;
        int rd = -1, rg = 0, rf = 0;
        double ri = 0.0;
        if (p < p1) { rd = pair_d[p]; rg = (int)(pair_g[p] - g0); rf = pair_f[p]; ri = pair_iou[p]; }
        const int cnt = (int)min((int64_t)32, p1 - base);
        for (int r = 0; r < cnt; ++r) {
            const int d = __shfl_sync(FULL, rd, r);
            const int gp = __shfl_sync(FULL, rg, r);
            const int f = __shfl_sync(FULL, rf, r);
            const double iou = __shfl_sync(FULL, ri, r);
            if (d != cur) {
                if (cur >= 0) commit();
                cur = d;
                bg = -1;
            }
            const bool avail = (f & EMIA_CE_CROWD) || !((bm[gp >> 5] >> (gp & 31)) & 1u);
            emia_ce_consider(bg, bign, biou, gp, iou, (f >> (4 + a)) & 1, avail, thr);
            if (bg == gp) bf = f;
        }
    }
    if (cur >= 0) commit();
}

// ---- accumulate ------------------------------------------------------------------------------------------------------------------
// inclusive block scan of three counts (all threads call); *tot = the block totals
__device__ __forceinline__ int3 emia_ce_scan3(int3 v, int3* tot, int3* sm) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int d = 1; d < 32; d <<= 1) {
        const int x = __shfl_up_sync(0xffffffffu, v.x, d), y = __shfl_up_sync(0xffffffffu, v.y, d), z = __shfl_up_sync(0xffffffffu, v.z, d);
        if (lane >= d) { v.x += x; v.y += y; v.z += z; }
    }
    if (lane == 31) sm[w] = v;
    __syncthreads();
    int3 pre = make_int3(0, 0, 0), all = make_int3(0, 0, 0);
    for (int k = 0; k < nw; ++k) {
        if (k < w) { pre.x += sm[k].x; pre.y += sm[k].y; pre.z += sm[k].z; }
        all.x += sm[k].x; all.y += sm[k].y; all.z += sm[k].z;
    }
    __syncthreads();
    *tot = all;
    return make_int3(v.x + pre.x, v.y + pre.y, v.z + pre.z);
}

__global__ void __launch_bounds__(EMIA_CE_ACC_THREADS) k_ce_accumulate(const int32_t* __restrict__ corder, const int32_t* __restrict__ rank,
                                                                       const uint32_t* __restrict__ state, const int64_t* __restrict__ cat_dt_off,
                                                                       const int64_t* __restrict__ cat_gt_off, const double* __restrict__ gt_area,
                                                                       const int32_t* __restrict__ gt_flags, int64_t n_dt, int K,
                                                                       EmiaCeParams P, double* __restrict__ precision,
                                                                       double* __restrict__ recall) {
    __shared__ int3 sm3[EMIA_CE_ACC_THREADS / 32];
    __shared__ unsigned long long qmax[EMIA_CE_R];      // bit patterns of non-negative doubles order as integers
    __shared__ int s_npig;
    const int T = EMIA_CE_T, M = EMIA_CE_M, A = EMIA_CE_A, R = EMIA_CE_R;
    const int b = blockIdx.x, t = b % T, m = (b / T) % M, a = (b / (T * M)) % A, k = b / (T * M * A);
    if (threadIdx.x == 0) s_npig = 0;
    for (int r = threadIdx.x; r < R; r += blockDim.x) qmax[r] = 0ull;     // 0.0: the value past the end of the curve
    __syncthreads();
    int cnt = 0;
    for (int64_t g = cat_gt_off[k] + threadIdx.x; g < cat_gt_off[k + 1]; g += blockDim.x)
        cnt += !emia_ce_ignore(gt_area[g], gt_flags[g] & EMIA_CE_CROWD, P.lo[a], P.hi[a]);
    if (cnt) atomicAdd(&s_npig, cnt);
    __syncthreads();
    const int npig = s_npig;
    if (npig == 0) return;                                          // the entry stays -1
    const int md = P.max_det[m];
    const int64_t lo = cat_dt_off[k], hi = cat_dt_off[k + 1];
    int3 carry = make_int3(0, 0, 0);
    for (int64_t c = lo; c < hi; c += blockDim.x) {
        const int64_t j = c + threadIdx.x;
        const int i = j < hi ? corder[j] : -1;
        const bool inc = i >= 0 && rank[i] < md;
        const uint32_t w = inc ? state[a * n_dt + i] : 0u;
        int3 tot;
        const int3 sc = emia_ce_scan3(make_int3(inc, (w >> t) & 1u, (w >> (10 + t)) & 1u), &tot, sm3);
        if (inc) {
            const double tp = (double)(carry.y + sc.y), fp = (double)(carry.z + sc.z);
            const double rc = tp / (double)npig;
            const double pr = emia_ce_precision(tp, fp, P.eps);
            const int nr = emia_ce_rec_count(P.rec, R, rc);         // recall thresholds this point reaches
            if (nr > 0 && pr > 0.0) atomicMax(&qmax[nr - 1], (unsigned long long)__double_as_longlong(pr));
        }
        carry.x += tot.x; carry.y += tot.y; carry.z += tot.z;
    }
    __syncthreads();
    if (threadIdx.x == 0)                                           // rc[-1] = tp / npig of the whole sequence, 0 without detections
        recall[((int64_t)(t * K + k) * A + a) * M + m] = carry.x ? (double)carry.y / (double)npig : 0.0;
    if (threadIdx.x < 32) {                                         // q[r] = max over buckets >= r: a suffix max, one warp
        double run = 0.0;
        for (int r0 = ((R - 1) / 32) * 32; r0 >= 0; r0 -= 32) {
            const int r = r0 + 31 - (int)threadIdx.x;               // lane 0 holds the highest r of the chunk
            double v = r < R ? __longlong_as_double((long long)qmax[r]) : 0.0;
            for (int d = 1; d < 32; d <<= 1) {
                const double x = __shfl_up_sync(0xffffffffu, v, d);
                if ((int)threadIdx.x >= d) v = fmax(v, x);
            }
            v = fmax(v, run);
            if (r < R) precision[(((int64_t)(t * R + r) * K + k) * A + a) * M + m] = v;
            run = __shfl_sync(0xffffffffu, v, 31);
        }
    }
}

// ---- entry points ----------------------------------------------------------------------------------------------------------------
static unsigned emia_ce_grid_of(int64_t n, int per_block) { return (unsigned)((n + per_block - 1) / per_block); }

static size_t emia_ce_align(size_t b) { return (b + 255) & ~(size_t)255; }
static int64_t emia_ce_tiles(int64_t n) { return (n + EMIA_CE_SORT_TILE - 1) / EMIA_CE_SORT_TILE; }

extern "C" size_t emia_cocoeval_order_workspace_bytes(int64_t n_dt) {
    const int64_t n = n_dt > 0 ? n_dt : 1, nc = EMIA_CE_SORT_BINS * emia_ce_tiles(n);
    return 3 * emia_ce_align(n * sizeof(uint64_t)) + 3 * emia_ce_align(n * sizeof(int32_t)) + emia_ce_align((nc + 1) * sizeof(int64_t)) +
           emia_ce_align(emia_scan_workspace_bytes(nc));
}

// stable sort of in[0, n) by key (the low `bits` bits) into out; tmp: n ints (in, out and tmp distinct)
static int emia_ce_radix(const uint64_t* key, const int32_t* in, int32_t* out, int32_t* tmp, int64_t n, int bits, int64_t* counts,
                         void* scan_ws, size_t scan_bytes, cudaStream_t st) {
    const int passes = (bits + 7) / 8;
    if (passes == 0) {
        if (cudaMemcpyAsync(out, in, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
            return emia_check_launch("emia_cocoeval_order copy: %s");
        return EMIA_OK;
    }
    const int64_t tiles = emia_ce_tiles(n);
    const int32_t* src = in;
    for (int k = 0; k < passes; ++k) {
        int32_t* dst = ((passes - 1 - k) & 1) ? tmp : out;
        k_ce_sort_hist<<<(unsigned)tiles, EMIA_CE_SORT_TILE, 0, st>>>(key, src, n, 8 * k, counts);
        if (int rc = emia_exclusive_scan_i64(counts, EMIA_CE_SORT_BINS * tiles, scan_ws, scan_bytes, st)) return rc;
        k_ce_sort_scatter<<<(unsigned)tiles, EMIA_CE_SORT_TILE, 0, st>>>(key, src, n, 8 * k, counts, dst);
        src = dst;
    }
    return emia_check_launch("emia_cocoeval_order launch: %s");
}

static int emia_ce_bits(int64_t v) {                    // bits of the largest key value v
    int b = 0;
    while (v > 0) { ++b; v >>= 1; }
    return b;
}

extern "C" int emia_cocoeval_order(const double* score, const int32_t* cat, const int32_t* seg, const int64_t* seg_off, int64_t n,
                                   int32_t n_cat, int64_t n_seg, int32_t* rank, int32_t* corder, int32_t* morder, void* workspace,
                                   size_t workspace_bytes, void* stream) {
    if (n < 0 || n > INT32_MAX || n_cat < 1 || n_seg < 1) return emia_fail(EMIA_ERR_BAD_ARG, "emia_cocoeval_order: %s", "bad size");
    if (n == 0) return EMIA_OK;
    if (!score || !cat || !seg || !seg_off || !rank || !corder || !morder || !workspace)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_cocoeval_order: %s", "null pointer");
    if (workspace_bytes < emia_cocoeval_order_workspace_bytes(n))
        return emia_fail(EMIA_ERR_WORKSPACE, "emia_cocoeval_order: %s", "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t nc = EMIA_CE_SORT_BINS * emia_ce_tiles(n);
    unsigned char* w = (unsigned char*)workspace;
    uint64_t* skey = (uint64_t*)w; w += emia_ce_align(n * sizeof(uint64_t));
    uint64_t* ckey = (uint64_t*)w; w += emia_ce_align(n * sizeof(uint64_t));
    uint64_t* gkey = (uint64_t*)w; w += emia_ce_align(n * sizeof(uint64_t));
    int32_t* iota = (int32_t*)w; w += emia_ce_align(n * sizeof(int32_t));
    int32_t* byscore = (int32_t*)w; w += emia_ce_align(n * sizeof(int32_t));
    int32_t* tmp = (int32_t*)w; w += emia_ce_align(n * sizeof(int32_t));
    int64_t* counts = (int64_t*)w; w += emia_ce_align((nc + 1) * sizeof(int64_t));
    const size_t scan_bytes = emia_scan_workspace_bytes(nc);
    const unsigned grid = emia_ce_grid_of(n, EMIA_CE_THREADS);
    k_ce_keys<<<grid, EMIA_CE_THREADS, 0, st>>>(score, cat, seg, n, skey, ckey, gkey, iota);
    if (int rc = emia_check_launch("emia_cocoeval_order launch: %s")) return rc;
    // the DT list is in (category, image, file order): stable by score desc keeps (image, file order) among equal scores
    if (int rc = emia_ce_radix(skey, iota, byscore, tmp, n, 64, counts, w, scan_bytes, st)) return rc;
    if (int rc = emia_ce_radix(ckey, byscore, corder, tmp, n, emia_ce_bits(n_cat - 1), counts, w, scan_bytes, st)) return rc;
    if (int rc = emia_ce_radix(gkey, byscore, morder, tmp, n, emia_ce_bits(n_seg - 1), counts, w, scan_bytes, st)) return rc;
    k_ce_rank<<<grid, EMIA_CE_THREADS, 0, st>>>(morder, seg, seg_off, n, rank);
    return emia_check_launch("emia_cocoeval_order launch: %s");
}

static int emia_ce_grid_dims(const char* what, int32_t n_seg, int32_t H, int32_t W, int32_t cell_size, EmiaNbGrid* g) {
    if (n_seg < 1 || H <= 0 || W <= 0 || cell_size <= 0) return emia_fail(EMIA_ERR_BAD_ARG, "%s: bad size", what);
    *g = EmiaNbGrid{cell_size, (W + cell_size - 1) / cell_size, (H + cell_size - 1) / cell_size};
    return EMIA_OK;
}

extern "C" int emia_cocoeval_grid(const int32_t* gt_bbox, const int32_t* gt_gseg, int64_t n_gt, int32_t n_seg, int32_t H, int32_t W,
                                  int32_t cell_size, int64_t* cell_cnt, void* stream) {
    EmiaNbGrid g;
    if (n_gt < 0 || n_gt > INT32_MAX) return emia_fail(EMIA_ERR_BAD_ARG, "emia_cocoeval_grid: %s", "bad size");
    if (int rc = emia_ce_grid_dims("emia_cocoeval_grid", n_seg, H, W, cell_size, &g)) return rc;
    const int64_t ncells = (int64_t)n_seg * g.gx * g.gy;
    if (!cell_cnt || (n_gt && (!gt_bbox || !gt_gseg))) return emia_fail(EMIA_ERR_BAD_ARG, "emia_cocoeval_grid: %s", "null pointer");
    if (cudaMemsetAsync(cell_cnt, 0, (ncells + 1) * sizeof(int64_t), (cudaStream_t)stream) != cudaSuccess)
        return emia_check_launch("emia_cocoeval_grid memset: %s");
    if (n_gt == 0) return EMIA_OK;
    k_ce_grid<false><<<emia_ce_grid_of(n_gt, EMIA_CE_THREADS), EMIA_CE_THREADS, 0, (cudaStream_t)stream>>>(gt_bbox, gt_gseg, n_gt, g, cell_cnt,
                                                                                                          nullptr, nullptr, nullptr);
    return emia_check_launch("emia_cocoeval_grid launch: %s");
}

extern "C" int emia_cocoeval_pair_count(const int32_t* gt_bbox, const int32_t* gt_gseg, int64_t n_gt, const int32_t* dt_bbox,
                                        const int32_t* dt_eval, const int32_t* dt_gseg, int64_t n_dt, int32_t n_seg, int32_t H, int32_t W,
                                        int32_t cell_size, const int64_t* cell_off, int32_t* ent, int32_t* cursor, const int32_t* rank,
                                        const int32_t* dt_seg, const int64_t* seg_dt_off, int32_t max_det, int64_t* pair_cnt,
                                        void* stream) {
    EmiaNbGrid g;
    if (n_gt < 0 || n_gt > INT32_MAX || n_dt < 0 || n_dt > INT32_MAX || max_det < 1)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_cocoeval_pair_count: %s", "bad size");
    if (int rc = emia_ce_grid_dims("emia_cocoeval_pair_count", n_seg, H, W, cell_size, &g)) return rc;
    if (!cell_off || !cursor || (n_gt && (!gt_bbox || !gt_gseg || !ent)) ||
        (n_dt && (!dt_bbox || !dt_eval || !dt_gseg || !rank || !dt_seg || !seg_dt_off || !pair_cnt)))
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_cocoeval_pair_count: %s", "null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t ncells = (int64_t)n_seg * g.gx * g.gy;
    if (cudaMemsetAsync(cursor, 0, ncells * sizeof(int32_t), st) != cudaSuccess) return emia_check_launch("emia_cocoeval_pair_count memset: %s");
    if (n_gt)
        k_ce_grid<true><<<emia_ce_grid_of(n_gt, EMIA_CE_THREADS), EMIA_CE_THREADS, 0, st>>>(gt_bbox, gt_gseg, n_gt, g, nullptr, cell_off,
                                                                                           cursor, ent);
    if (n_dt)
        k_ce_pair_count<<<emia_ce_grid_of(n_dt, EMIA_CE_THREADS), EMIA_CE_THREADS, 0, st>>>(gt_bbox, dt_bbox, dt_eval, dt_gseg, n_dt, g,
                                                                                           cell_off, ent, rank, dt_seg, seg_dt_off,
                                                                                           max_det, pair_cnt);
    return emia_check_launch("emia_cocoeval_pair_count launch: %s");
}

extern "C" int emia_cocoeval_pair_fill(const uint32_t* gt_crops, const emia_inst_meta* gt_meta, const int64_t* gt_crop_off,
                                       const int32_t* gt_bbox, const int32_t* gt_area, const int32_t* gt_eval, const uint32_t* dt_crops,
                                       const emia_inst_meta* dt_meta, const int64_t* dt_crop_off, const int32_t* dt_bbox,
                                       const int32_t* dt_area, const int32_t* dt_eval, const int32_t* dt_gseg, int64_t n_dt,
                                       int32_t n_seg, int32_t H, int32_t W, int32_t cell_size, const int64_t* cell_off, const int32_t* ent,
                                       const int32_t* rank, const int32_t* dt_seg, const int64_t* seg_dt_off, const double* gt_area_eval,
                                       const int32_t* gt_flags, const double* params_host, const int32_t* max_dets_host,
                                       const int64_t* pair_off, int32_t* pair_g, int32_t* pair_d, int32_t* pair_f, double* pair_iou,
                                       void* stream) {
    EmiaNbGrid g;
    if (n_dt < 0 || n_dt > INT32_MAX) return emia_fail(EMIA_ERR_BAD_ARG, "emia_cocoeval_pair_fill: %s", "bad size");
    if (int rc = emia_ce_grid_dims("emia_cocoeval_pair_fill", n_seg, H, W, cell_size, &g)) return rc;
    if (n_dt == 0) return EMIA_OK;
    if (!dt_crops || !dt_meta || !dt_crop_off || !dt_bbox || !dt_area || !dt_eval || !dt_gseg || !cell_off || !rank || !dt_seg ||
        !seg_dt_off || !params_host || !max_dets_host || !pair_off || !gt_crops || !gt_meta || !gt_crop_off || !gt_bbox || !gt_area ||
        !gt_eval || !ent || !gt_area_eval || !gt_flags || !pair_g || !pair_d || !pair_f || !pair_iou)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_cocoeval_pair_fill: %s", "null pointer");
    const EmiaCeParams P = emia_ce_params(params_host, max_dets_host);
    const EmiaCeSide gs{gt_crops, (const int32_t*)gt_meta, gt_crop_off, gt_bbox, gt_area};
    const EmiaCeSide ds{dt_crops, (const int32_t*)dt_meta, dt_crop_off, dt_bbox, dt_area};
    k_ce_pair_fill<<<emia_ce_grid_of(n_dt * 32, EMIA_CE_THREADS), EMIA_CE_THREADS, 0, (cudaStream_t)stream>>>(
        gs, gt_eval, ds, dt_eval, dt_gseg, n_dt, g, cell_off, ent, rank, dt_seg, seg_dt_off, gt_area_eval, gt_flags, P, pair_off, pair_g,
        pair_d, pair_f, pair_iou);
    return emia_check_launch("emia_cocoeval_pair_fill launch: %s");
}

extern "C" int emia_cocoeval_match(const int64_t* seg_dt_off, const int64_t* seg_gt_off, const int64_t* wseg_off, int64_t n_seg,
                                   int64_t n_words, const int32_t* morder, const double* dt_area, const int64_t* pair_off,
                                   const int32_t* pair_g, const int32_t* pair_d, const int32_t* pair_f, const double* pair_iou,
                                   int64_t n_dt, const double* params_host, const int32_t* max_dets_host, uint32_t* matched,
                                   uint32_t* state, void* stream) {
    if (n_seg < 0 || n_seg > INT32_MAX || n_dt < 0 || n_dt > INT32_MAX || n_words < 0)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_cocoeval_match: %s", "bad size");
    if (n_seg == 0 || n_dt == 0) return EMIA_OK;
    if (!seg_dt_off || !seg_gt_off || !wseg_off || !morder || !dt_area || !pair_off || !params_host || !max_dets_host || !state ||
        (n_words && !matched))
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_cocoeval_match: %s", "null pointer");
    const EmiaCeParams P = emia_ce_params(params_host, max_dets_host);
    cudaStream_t st = (cudaStream_t)stream;
    if (n_words && cudaMemsetAsync(matched, 0, (size_t)n_words * EMIA_CE_A * EMIA_CE_T * sizeof(uint32_t), st) != cudaSuccess)
        return emia_check_launch("emia_cocoeval_match memset: %s");
    k_ce_match<<<(unsigned)n_seg, 32 * EMIA_CE_A, 0, st>>>(seg_dt_off, seg_gt_off, wseg_off, n_words, morder, dt_area, pair_off, pair_g,
                                                          pair_d, pair_f, pair_iou, n_dt, P, matched, state);
    return emia_check_launch("emia_cocoeval_match launch: %s");
}

extern "C" int emia_cocoeval_accumulate(const int32_t* corder, const int32_t* rank, const uint32_t* state, const int64_t* cat_dt_off,
                                        const int64_t* cat_gt_off, const double* gt_area, const int32_t* gt_flags, int64_t n_dt,
                                        int32_t n_cat, const double* params_host, const int32_t* max_dets_host, double* precision,
                                        double* recall, void* stream) {
    if (n_dt < 0 || n_dt > INT32_MAX || n_cat < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_cocoeval_accumulate: %s", "bad size");
    if (n_cat == 0) return EMIA_OK;
    if (!cat_dt_off || !cat_gt_off || !params_host || !max_dets_host || !precision || !recall || (n_dt && (!corder || !rank || !state)) ||
        !gt_area || !gt_flags)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_cocoeval_accumulate: %s", "null pointer");
    const EmiaCeParams P = emia_ce_params(params_host, max_dets_host);
    const unsigned grid = (unsigned)n_cat * EMIA_CE_A * EMIA_CE_M * EMIA_CE_T;
    k_ce_accumulate<<<grid, EMIA_CE_ACC_THREADS, 0, (cudaStream_t)stream>>>(corder, rank, state, cat_dt_off, cat_gt_off, gt_area, gt_flags,
                                                                            n_dt, n_cat, P, precision, recall);
    return emia_check_launch("emia_cocoeval_accumulate launch: %s");
}
