// emia_morpho_kernels.cuh — K5: external contours + morphometry (part of emia_kernels.cu).
// One thread per instance: border following is inherently sequential per component, so parallelism comes from
// the number of instances in flight (10^5..10^6 per launch); the crop (a few hundred bytes) stays in L1.
#pragma once

__device__ __forceinline__ EmiaBitView emia_make_view(const uint32_t* crops, const emia_inst_meta& m, int64_t off) {
    EmiaBitView v;
    v.bits = crops + off; v.pitch_words = m.cw; v.h = m.ch; v.wwords = m.cw;
    v.x_origin = m.wc0 * 32; v.y_origin = m.ry0;
    return v;
}

// ---- border following: one THREAD per instance ---------------------------------------------------------------------
#define EMIA_TRACE_THREADS 128

// diag[k] = sqrtf(2 k^2): the diagonal-run terms of cv2.arcLength (see emia_arc_length_closed), per CTA in shared memory
__device__ __forceinline__ void emia_fill_diag_table(float* diag) {
    for (int k = threadIdx.x; k < EMIA_DIAG_TABLE; k += blockDim.x) {
        const float f = (float)k;
        const float f2 = f * f;
        diag[k] = sqrtf(f2 + f2);
    }
    __syncthreads();
}

// clear the two mark planes of the instances [0, n): words [2 * crop_off[0], 2 * crop_off[n]) of `marks`, coalesced
__global__ void __launch_bounds__(256) k_clear_marks(uint32_t* __restrict__ marks, const int64_t* __restrict__ crop_off, int64_t n) {
    const int64_t lo = 2 * crop_off[0], hi = 2 * crop_off[n];
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t i = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    // head up to a 16-byte boundary, then 128-bit stores, then the tail
    const int64_t lo4 = (lo + 3) & ~(int64_t)3, hi4 = hi & ~(int64_t)3;
    if (lo4 >= hi4) { for (; i < hi; i += stride) marks[i] = 0u; return; }
    if (i < lo4) marks[i] = 0u;
    uint4* m4 = (uint4*)(marks + lo4);
    const int64_t n4 = (hi4 - lo4) >> 2;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n4; q += stride) m4[q] = make_uint4(0u, 0u, 0u, 0u);
    const int64_t t = hi4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < hi) marks[t] = 0u;
}
static void emia_launch_clear_marks(uint32_t* marks, const int64_t* crop_off, int64_t n, cudaStream_t st) {
    k_clear_marks<<<emia_num_sms() * 8, 256, 0, st>>>(marks, crop_off, n);
}

template <bool kStore>
__global__ void __launch_bounds__(EMIA_TRACE_THREADS) k_contour_trace(
    const uint32_t* __restrict__ crops, const emia_inst_meta* __restrict__ meta, const int64_t* __restrict__ crop_off, int64_t n,
    uint32_t* __restrict__ marks, int64_t* __restrict__ n_contours, int64_t* __restrict__ n_points,
    int64_t* __restrict__ scratch_bytes, const int64_t* __restrict__ cont_off, const int64_t* __restrict__ pt_off,
    uint32_t* __restrict__ pts, int32_t* __restrict__ cstart, double* __restrict__ perim0) {
    __shared__ float s_diag[EMIA_DIAG_TABLE];
    if (kStore) emia_fill_diag_table(s_diag);
    const int64_t i = (int64_t)blockIdx.x * EMIA_TRACE_THREADS + threadIdx.x;
    if (i >= n) return;
    const emia_inst_meta m = meta[i];
    const int words = m.ch * m.cw;
    if (words <= 0) {
        if (kStore) { cstart[cont_off[i] + i] = 0; if (perim0) perim0[i] = 0.0; }
        else { n_contours[i] = 0; n_points[i] = 0; scratch_bytes[i] = 0; }
        return;
    }
    const int64_t off = crop_off[i];
    const EmiaBitView v = emia_make_view(crops, m, off);
    uint32_t* mk = marks + 2 * off;
    uint32_t* ng = mk + words;
    EmiaContourOut o;
    if (kStore) {
        o.pts = pts + pt_off[i]; o.cap_pts = (int)(pt_off[i + 1] - pt_off[i]);
        o.cstart = cstart + cont_off[i] + i; o.cap_contours = (int)(cont_off[i + 1] - cont_off[i]); o.store = 1;
    } else {
        o.pts = nullptr; o.cap_pts = 0; o.cstart = nullptr; o.cap_contours = 0; o.store = 0;
    }
    o.track = 0; o.diag = nullptr;
    emia_find_external_contours(v, mk, ng, o, 1);
    if (!kStore) {
        n_contours[i] = o.n_contours;
        n_points[i] = o.n_pts;
        scratch_bytes[i] = (int64_t)emia_measure_item_scratch_bytes(o.n_pts, o.n_contours);
    } else if (perim0) {
        // arcLength of contours[0] in OpenCV order = the LAST discovered contour (deduplicate_masks_smart's compactness, Q10)
        const int nc = o.n_contours;
        perim0[i] = nc ? emia_arc_length_closed(o.pts + o.cstart[nc - 1], o.cstart[nc] - o.cstart[nc - 1], s_diag) : 0.0;
    }
}
#define EMIA_TRACE_SMEM_BYTES ((size_t)0)

// ---- convex hull: one WARP per single-contour work item ---------------------------------------------------------------
// The hull (Sklansky on the vertices sorted by (x, y, index)) was 75 % of the per-thread morphometry kernel: a chain of
// dependent, uncoalesced global loads (ncu source view, profiles/).  For the common case (one contour, <= EMIA_PRESORT_MAX
// vertices) a warp now sorts the keys with a bitonic network in shared memory, runs the four monotone chains on four
// lanes (keys and stacks in shared memory), one lane assembles the hull exactly as the serial code does, gathers the hull
// points into shared memory and runs the rotating calipers there; the calipers result (6 floats) is written where
// emia_measure_contour(prepared = 3) expects it in the item's scratch block.
// Work items: item `it` measures instance item_inst[it] (identity when item_inst == nullptr; < 0 = nothing to do); its records
// start at rec_off[it] (rec_off[it+1] - rec_off[it] = number of contours) and its scratch at scratch_off[it].
// inst_cont_off (per INSTANCE) locates the packed cstart layout and is only read when cstart_stride == 0.
#define EMIA_PRESORT_MAX 256
#ifndef EMIA_PRESORT_WARPS
#define EMIA_PRESORT_WARPS 4
#endif
// Packed path: the serial phases (four Sklansky chains, hull assembly) used 4 and 1 lanes of the warp and were 60 % of the
// kernel's issue slots.  A warp therefore takes EMIA_HULL_PACK work items: it pre-filters and sorts them one after the other
// (all lanes), parks each sorted key list (<= EMIA_HULL_FAST_MAX survivors, 32-bit compact keys) in a small shared-memory slot,
// and then runs the chains of ALL its items at once (lane = item * 4 + chain) and the assembly on one lane per item.
// Items with more survivors or a larger extent take the one-item-per-warp path afterwards (its buffers alias the slots).
#ifndef EMIA_HULL_PACK
#define EMIA_HULL_PACK 8
#endif
#define EMIA_HULL_FAST_MAX 64
struct EmiaHullSmem {
    uint64_t keys[EMIA_PRESORT_MAX];
    uint16_t stacks[4][EMIA_PRESORT_MAX + 4];
    int hull[EMIA_PRESORT_MAX];
    int tmp[EMIA_PRESORT_MAX];
};
struct EmiaHullSlot {
    uint32_t keys[EMIA_HULL_FAST_MAX];
    uint8_t stacks[4][EMIA_HULL_FAST_MAX + 4];
    uint8_t hull[EMIA_HULL_FAST_MAX + 8];
    uint8_t tmp[EMIA_HULL_FAST_MAX + 8];
    int cnt[4];
    int m, miny, maxy, len;
    long long scratch_off;
    const uint32_t* p;                                        // the contour's vertices
};
union EmiaHullWarpSmem {
    EmiaHullSmem one;                                         // one-item path
    struct {
        uint32_t staging[EMIA_PRESORT_MAX];                   // the first bytes of one.keys: pre-filter area of the current item (32-bit keys)
        EmiaHullSlot slot[EMIA_HULL_PACK];
    } packed;
};
__device__ __forceinline__ uint64_t emia_make_key(uint64_t, int x, int y, int ox, int oy, int t) { (void)ox; (void)oy; return EMIA_KEY(x, y, t); }
__device__ __forceinline__ uint32_t emia_make_key(uint32_t, int x, int y, int ox, int oy, int t) { return EMIA_KEY32(x - ox, y - oy, t); }

// The four extreme vertices of a contour (left, top, right, bottom; first in (x, y) resp. (y, x) order), warp-cooperative.
struct EmiaHullQuad { int qx[4], qy[4]; int ox, oy; bool compact; };
__device__ __forceinline__ EmiaHullQuad emia_hull_extremes(const uint32_t* __restrict__ p, int len, int lane) {
    // (x << 16 | y) for left / right, (y << 16 | x) for top / bottom
    uint32_t lx = 0xFFFFFFFFu, rx = 0u, ty = 0xFFFFFFFFu, by = 0u;
    for (int t = lane; t < len; t += 32) {
        const uint32_t q = p[t];
        const uint32_t xy = ((uint32_t)EMIA_PT_X(q) << 16) | (uint32_t)EMIA_PT_Y(q), yx = ((uint32_t)EMIA_PT_Y(q) << 16) | (uint32_t)EMIA_PT_X(q);
        lx = min(lx, xy); rx = max(rx, xy); ty = min(ty, yx); by = max(by, yx);
    }
    for (int o = 16; o > 0; o >>= 1) {
        lx = min(lx, __shfl_xor_sync(0xffffffffu, lx, o)); rx = max(rx, __shfl_xor_sync(0xffffffffu, rx, o));
        ty = min(ty, __shfl_xor_sync(0xffffffffu, ty, o)); by = max(by, __shfl_xor_sync(0xffffffffu, by, o));
    }
    EmiaHullQuad Q;
    Q.qx[0] = (int)(lx >> 16); Q.qx[1] = (int)(ty & 0xFFFF); Q.qx[2] = (int)(rx >> 16); Q.qx[3] = (int)(by & 0xFFFF);
    Q.qy[0] = (int)(lx & 0xFFFF); Q.qy[1] = (int)(ty >> 16); Q.qy[2] = (int)(rx & 0xFFFF); Q.qy[3] = (int)(by >> 16);
    Q.ox = (int)(lx >> 16); Q.oy = (int)(ty >> 16);
    Q.compact = ((int)(rx >> 16) - Q.ox) < 4096 && ((int)(by >> 16) - Q.oy) < 4096;             // len <= 256 holds for the callers
    return Q;
}

// Akl-Toussaint pre-filter: vertices strictly inside the quadrilateral of the four extreme vertices (left, top, right,
// bottom) cannot be hull vertices; dropping them (typically 50-70 % of a blob's contour) shrinks the sort and the chains.
// Extremes and all vertices ON the quadrilateral survive, so the sorted order of the survivors, the first min-/max-y
// entries and the chains' results are those of the full set; keys keep the ORIGINAL vertex index.  Returns the survivor count.
// I: arithmetic type of the cross products (int when the extent is below 4096 x 4096: |products| < 2^24; else long long).
template <typename K, typename I>
__device__ __forceinline__ int emia_hull_prefilter(K* k, const uint32_t* __restrict__ p, int len, int lane, const EmiaHullQuad& Q) {
    I ex[4], ey[4];
    int edges = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int f = (e + 1) & 3;
        ex[e] = (I)(Q.qx[f] - Q.qx[e]); ey[e] = (I)(Q.qy[f] - Q.qy[e]);
        edges += (ex[e] != 0 || ey[e] != 0);                            // coinciding extremes: the quadrilateral is a triangle
    }
    int run = 0;
    for (int t0 = 0; t0 < len; t0 += 32) {
        const int t = t0 + lane;
        bool keep = false;
        K key = (K)~(K)0;
        if (t < len) {
            const uint32_t q = p[t];
            const int x = EMIA_PT_X(q), y = EMIA_PT_Y(q);
            int pos = 0, neg = 0;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const I cr = ex[e] * (I)(y - Q.qy[e]) - ey[e] * (I)(x - Q.qx[e]);       // 0 for a degenerate edge
                pos += cr > 0; neg += cr < 0;
            }
            const bool inside = edges >= 3 && (pos == edges || neg == edges);
            keep = !inside;
            key = emia_make_key((K)0, x, y, Q.ox, Q.oy, t);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (keep) k[run + __popc(bal & ((1u << lane) - 1u))] = key;
        run += __popc(bal);
    }
    return run;
}

// Bitonic sort of up to 64 keys held two per lane (k0: element `lane`, k1: element `lane + 32`; unused elements all-ones) with
// shuffles — no shared memory, no barriers.  two = false: only k0 is sorted (<= 32 keys).
__device__ __forceinline__ void emia_hull_sort_regs(uint32_t& k0, uint32_t& k1, int lane, bool two) {
#pragma unroll
    for (int size = 2; size <= 64; size <<= 1) {
        if (size == 64 && !two) break;
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            if (stride == 32) {                     // partner in the same lane; size == 64: ascending everywhere
                const uint32_t lo = min(k0, k1), hi = max(k0, k1);
                k0 = lo; k1 = hi;
            } else {
                const bool lower = (lane & stride) == 0;
                const bool up0 = size == 64 ? true : (lane & size) == 0;                 // element lane
                const bool up1 = size == 64 ? true : size == 32 ? false : (lane & size) == 0;     // element lane + 32
                const uint32_t o0 = __shfl_xor_sync(0xffffffffu, k0, stride);
                k0 = (lower == up0) ? min(k0, o0) : max(k0, o0);
                if (two) {
                    const uint32_t o1 = __shfl_xor_sync(0xffffffffu, k1, stride);
                    k1 = (lower == up1) ? min(k1, o1) : max(k1, o1);
                }
            }
        }
    }
}

// Bitonic sort of k[0..m) (padded with all-ones keys to a power of two >= 32) by one warp, then the first index of the
// minimum / maximum y in sorted order (the serial scan keeps the first occurrence).
template <typename K>
__device__ __forceinline__ void emia_hull_sort(K* k, int m, int lane, int* miny_ind, int* maxy_ind) {
    int N = 32;
    while (N < m) N <<= 1;
    for (int t = m + lane; t < N; t += 32) k[t] = (K)~(K)0;
    __syncwarp();
    for (int size = 2; size <= N; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = lane; t < (N >> 1); t += 32) {
                const int lo = ((t & ~(stride - 1)) << 1) | (t & (stride - 1));      // stride is a power of two
                const int hi = lo + stride;
                const bool up = ((lo & size) == 0);
                const K a = k[lo], b = k[hi];
                if ((a > b) == up) { k[lo] = b; k[hi] = a; }
            }
            __syncwarp();
        }
    }
    int mn = 0x7fffffff, mx = 0x7fffffff;
    for (int t = lane; t < m; t += 32) {
        const int y = emia_ky(k[t]);
        mn = min(mn, (y << 9) | t);                   // y < 2^20, t < 2^9
        mx = min(mx, ((0xFFFFF - y) << 9) | t);
    }
    for (int o = 16; o > 0; o >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = min(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    *miny_ind = mn & 511; *maxy_ind = mx & 511;
}

// One item per warp (any extent, up to EMIA_PRESORT_MAX vertices), templated on the key type (uint32_t: extent < 4096 x 4096,
// coordinates relative to (ox, oy)): chains on four lanes, assembly on lane 0.
template <typename K>
__device__ __forceinline__ void emia_hull_warp(K* k, EmiaHullSmem& S, const uint32_t* __restrict__ p, int len, int lane,
                                               const EmiaHullQuad& Q, int* r) {
    const int m = Q.compact ? emia_hull_prefilter<K, int>(k, p, len, lane, Q) : emia_hull_prefilter<K, long long>(k, p, len, lane, Q);
    int miny_ind, maxy_ind;
    emia_hull_sort<K>(k, m, lane, &miny_ind, &maxy_ind);
    int nout = 0;
    const bool degenerate = (emia_kx(k[0]) == emia_kx(k[m - 1]) && emia_ky(k[0]) == emia_ky(k[m - 1]));
    if (degenerate) {
        if (lane == 0) S.hull[0] = 0;
        nout = 1;
    } else {
        int cnt = 0;
        if (lane < 4) {
            const int start = (lane & 1) ? m - 1 : 0;
            const int end = (lane < 2) ? maxy_ind : miny_ind;
            const int nsign = (lane < 2) ? -1 : 1;
            const int sign2 = (lane == 0 || lane == 3) ? 1 : -1;
            cnt = emia_sklansky(k, start, end, S.stacks[lane], nsign, sign2);
        }
        __syncwarp();
        const int tl = __shfl_sync(0xffffffffu, cnt, 0), tr = __shfl_sync(0xffffffffu, cnt, 1);
        const int bl = __shfl_sync(0xffffffffu, cnt, 2), br = __shfl_sync(0xffffffffu, cnt, 3);
        if (lane == 0) {
            const int stop_idx = emia_hull_emit_upper(k, 0, S.stacks[0], tl, S.stacks[1], tr, S.hull, &nout);
            emia_hull_emit_lower(k, 0, S.stacks[2], bl, S.stacks[3], br, stop_idx, S.hull, &nout);
            emia_hull_cyclic_shift(S.hull, nout, S.tmp);
        }
        nout = __shfl_sync(0xffffffffu, nout, 0);
    }
    __syncwarp();
    // hull points (packed) over the shift buffer, which is dead; calipers on lane 0; result where
    // emia_measure_contour(prepared = 3) expects it
    uint32_t* hq = (uint32_t*)S.tmp;
    for (int t = lane; t < nout; t += 32) hq[t] = p[S.hull[t]];
    __syncwarp();
    if (lane == 0) {
        r[0] = nout;
        if (nout > 2) {
            float out[6];
            emia_rotating_calipers(hq, nout, out);
#pragma unroll
            for (int t = 0; t < 6; ++t) ((float*)(r + 1))[t] = out[t];
        } else {
            r[1] = (int)hq[0];
            if (nout > 1) r[2] = (int)hq[1];
        }
    }
    __syncwarp();
}

// Locates work item `it`: number of contours (0 = nothing to do), the instance's cstart entries and vertex list.
__device__ __forceinline__ int emia_hull_item(int64_t it, int64_t n, const int32_t* __restrict__ item_inst, const int64_t* __restrict__ rec_off,
                                              const int64_t* __restrict__ inst_cont_off, const int64_t* __restrict__ pt_off,
                                              const int32_t* __restrict__ cstart, int cstart_stride, const uint32_t* __restrict__ pts,
                                              const int32_t** cs_out, const uint32_t** p) {
    if (it >= n || it < 0) return 0;
    const int nc = (int)(rec_off[it + 1] - rec_off[it]);
    if (nc < 1) return 0;
    const int64_t i = item_inst ? (int64_t)item_inst[it] : it;
    if (i < 0) return 0;
    *cs_out = cstart_stride > 0 ? cstart + (size_t)i * cstart_stride : cstart + inst_cont_off[i] + i;
    *p = pts + pt_off[i];
    return nc;
}

#ifndef EMIA_HULL_MIN_CTAS
#define EMIA_HULL_MIN_CTAS 8
#endif
__global__ void __launch_bounds__(EMIA_PRESORT_WARPS * 32, EMIA_HULL_MIN_CTAS) k_contour_hull(int64_t n, const int32_t* __restrict__ item_inst,
                                                                         const int64_t* __restrict__ rec_off,
                                                                         const int64_t* __restrict__ inst_cont_off,
                                                                         const int64_t* __restrict__ pt_off,
                                                                         const int32_t* __restrict__ cstart, int cstart_stride,
                                                                         const int64_t* __restrict__ scratch_off,
                                                                         const uint32_t* __restrict__ pts, uint8_t* __restrict__ scratch,
                                                                         const int32_t* __restrict__ abort_flag,
                                                                         const int32_t* __restrict__ order) {
    if (abort_flag && *abort_flag) return;
    __shared__ EmiaHullWarpSmem s_all[EMIA_PRESORT_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t it0 = ((int64_t)blockIdx.x * EMIA_PRESORT_WARPS + warp) * EMIA_HULL_PACK;
    if (it0 >= n) return;
    EmiaHullWarpSmem& W = s_all[warp];
    uint32_t* stage = (uint32_t*)W.packed.staging;
    unsigned fast = 0u, slow = 0u;                    // warp-uniform item masks
    // phase 0: lane j < PACK looks item j up (a chain of four dependent global loads: list entry -> contour table -> vertex
    // offset) and touches its vertices, so that the warp pays that latency once and not once per item
    int my_nc = 0, my_len = 0;
    const uint32_t* my_p = nullptr;
    long long my_sc = 0;
    // the work item of pack position j: list slot it0 + j, or — with a length-sorted order — slot order[it0 + j]
    long long my_slot = -1;
    if (lane < EMIA_HULL_PACK && it0 + lane < n) my_slot = order ? (long long)order[it0 + lane] : (long long)(it0 + lane);
    if (lane < EMIA_HULL_PACK) {
        const int32_t* cs;
        my_nc = emia_hull_item(my_slot, n, item_inst, rec_off, inst_cont_off, pt_off, cstart, cstart_stride, pts, &cs, &my_p);
        if (my_nc) {
            my_len = cs[1] - cs[0];
            my_p += cs[0];
            my_sc = (long long)scratch_off[my_slot];
            for (int t = 0; t < my_len && t < EMIA_PRESORT_MAX; t += 32) asm volatile("prefetch.global.L1 [%0];" ::"l"(my_p + t));
        }
    }
    // phase 1: pre-filter + sort, one item after the other, all lanes
    for (int j = 0; j < EMIA_HULL_PACK; ++j) {
        const int nc = __shfl_sync(0xffffffffu, my_nc, j);
        if (nc == 0) continue;
        const int len = __shfl_sync(0xffffffffu, my_len, j);
        const uint32_t* p = (const uint32_t*)__shfl_sync(0xffffffffu, (unsigned long long)my_p, j);
        const long long sc_off = __shfl_sync(0xffffffffu, my_sc, j);
        if (nc > 1) { slow |= 1u << j; continue; }                 // several contours: one after the other in phase 5
        if (len > EMIA_PRESORT_MAX || len < 1) continue;           // k_contour_measure runs the serial hull itself
        const EmiaHullQuad Q = emia_hull_extremes(p, len, lane);
        if (!Q.compact) { slow |= 1u << j; continue; }
        const int m = emia_hull_prefilter<uint32_t, int>(stage, p, len, lane, Q);
        __syncwarp();
        if (m > EMIA_HULL_FAST_MAX) { slow |= 1u << j; continue; }
        // sort in registers, then the first index of the minimum / maximum y in sorted order
        uint32_t k0 = lane < m ? stage[lane] : 0xFFFFFFFFu, k1 = lane + 32 < m ? stage[lane + 32] : 0xFFFFFFFFu;
        __syncwarp();                                  // the next item's pre-filter overwrites the staging area
        emia_hull_sort_regs(k0, k1, lane, m > 32);
        int mn = 0x7fffffff, mx = 0x7fffffff;
        if (lane < m) { const int y = emia_ky(k0); mn = (y << 9) | lane; mx = ((0xFFFFF - y) << 9) | lane; }
        if (lane + 32 < m) { const int y = emia_ky(k1); mn = min(mn, (y << 9) | (lane + 32)); mx = min(mx, ((0xFFFFF - y) << 9) | (lane + 32)); }
        for (int o = 16; o > 0; o >>= 1) {
            mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            mx = min(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        }
        EmiaHullSlot& S = W.packed.slot[j];
        S.keys[lane] = k0;
        if (m > 32) S.keys[lane + 32] = k1;
        if (lane == 0) { S.m = m; S.miny = mn & 511; S.maxy = mx & 511; S.len = len; S.scratch_off = sc_off; S.p = p; }
        fast |= 1u << j;
        __syncwarp();
    }
    // phase 2: the chains of every parked item at once.  Lane = item * LPI + sub; with two lanes per item one lane runs the two
    // upper chains and the other the two lower ones — each pair covers the whole sorted array once, so the lanes of an item
    // are balanced by construction.
    {
        constexpr int LPI = 32 / EMIA_HULL_PACK, CPL = 4 / LPI;      // lanes per item, chains per lane
        const int j = lane / LPI, sub = lane % LPI;
        EmiaHullSlot& S = W.packed.slot[j];
        const bool mine = (fast >> j) & 1u;
        bool degenerate = false;
        if (mine) {
            const int m = S.m;
            degenerate = (emia_kx(S.keys[0]) == emia_kx(S.keys[m - 1]) && emia_ky(S.keys[0]) == emia_ky(S.keys[m - 1]));
            if (!degenerate) {
#pragma unroll
                for (int cc = 0; cc < CPL; ++cc) {
                    const int c = sub * CPL + cc;
                    const int start = (c & 1) ? m - 1 : 0;
                    const int end = (c < 2) ? S.maxy : S.miny;
                    const int nsign = (c < 2) ? -1 : 1;
                    const int sign2 = (c == 0 || c == 3) ? 1 : -1;
                    S.cnt[c] = emia_sklansky(S.keys, start, end, S.stacks[c], nsign, sign2);
                }
            }
        }
        __syncwarp();
        // phase 3: assembly, one lane per item
        int nout = 0;
        if (mine && sub == 0) {
            if (degenerate) { S.hull[0] = 0; nout = 1; }
            else {
                const int stop_idx = emia_hull_emit_upper(S.keys, 0, S.stacks[0], S.cnt[0], S.stacks[1], S.cnt[1], S.hull, &nout);
                emia_hull_emit_lower(S.keys, 0, S.stacks[2], S.cnt[2], S.stacks[3], S.cnt[3], stop_idx, S.hull, &nout);
                emia_hull_cyclic_shift(S.hull, nout, S.tmp);
            }
        }
        nout = __shfl_sync(0xffffffffu, nout, lane - sub);
        __syncwarp();
        // phase 4: the hull points (original vertices, packed) into shared memory — over the chain stacks, which are dead — and
        // the rotating calipers on them, one lane per item; the result goes to the item's scratch block where
        // emia_measure_contour(prepared = 3) expects it (emia_measure_rect_off)
        uint32_t* hq = (uint32_t*)&S.stacks[0][0];
        if (mine) for (int t = sub; t < nout; t += LPI) hq[t] = S.p[S.hull[t]];
        __syncwarp();
        if (mine && sub == 0) {
            int* r = (int*)(scratch + S.scratch_off + emia_measure_rect_off(S.len));
            r[0] = nout;
            if (nout > 2) {
                float out[6];
                emia_rotating_calipers(hq, nout, out);
#pragma unroll
                for (int t = 0; t < 6; ++t) ((float*)(r + 1))[t] = out[t];
            } else {
                r[1] = (int)hq[0];
                if (nout > 1) r[2] = (int)hq[1];
            }
        }
        __syncwarp();
    }
    // phase 5: the rare large or multi-contour items, one contour at a time (the buffers alias the slots, which are dead now);
    // contour k of an item owns the k-th sub-block of the item's scratch (emia_measure_sub_bytes)
    for (int j = 0; j < EMIA_HULL_PACK; ++j) {
        if (!((slow >> j) & 1u)) continue;
        const uint32_t* p0; const int32_t* cs;
        const long long slot = __shfl_sync(0xffffffffu, my_slot, j);
        const int nc = emia_hull_item(slot, n, item_inst, rec_off, inst_cont_off, pt_off, cstart, cstart_stride, pts, &cs, &p0);
        uint8_t* sc = scratch + scratch_off[slot];
        for (int k = 0; k < nc; ++k) {
            const int len = cs[k + 1] - cs[k];
            if (len >= 1 && len <= EMIA_PRESORT_MAX) {
                const uint32_t* p = p0 + cs[k];
                const EmiaHullQuad Q = emia_hull_extremes(p, len, lane);
                int* r = (int*)(sc + emia_measure_rect_off(len));
                if (Q.compact) emia_hull_warp<uint32_t>((uint32_t*)W.one.keys, W.one, p, len, lane, Q, r);
                else emia_hull_warp<uint64_t>(W.one.keys, W.one, p, len, lane, Q, r);
            }
            sc += emia_measure_sub_bytes(len);
        }
    }
}
#define EMIA_HULL_GRID(n) ((unsigned)(((n) + EMIA_PRESORT_WARPS * EMIA_HULL_PACK - 1) / (EMIA_PRESORT_WARPS * EMIA_HULL_PACK)))

// ---- morphometry: one THREAD per instance over the stored vertex lists ---------------------------------------------
#ifndef EMIA_MEASURE_THREADS
#define EMIA_MEASURE_THREADS 128
#endif
#ifndef EMIA_MEASURE_MIN_CTAS
#define EMIA_MEASURE_MIN_CTAS 4
#endif
#define EMIA_MEASURE_GRID(n) ((unsigned)(((n) + EMIA_MEASURE_THREADS - 1) / EMIA_MEASURE_THREADS))
__global__ void __launch_bounds__(EMIA_MEASURE_THREADS, EMIA_MEASURE_MIN_CTAS) k_contour_measure(int64_t n, const int32_t* __restrict__ item_inst,
                                                         const int64_t* __restrict__ rec_off, const int64_t* __restrict__ inst_cont_off,
                                                         const int64_t* __restrict__ pt_off,
                                                         const int64_t* __restrict__ scratch_off, double um_pix, double min_area,
                                                         const uint32_t* __restrict__ pts, const int32_t* __restrict__ cstart,
                                                         int cstart_stride, int presort_max, double* __restrict__ records,
                                                         int32_t* __restrict__ rec_inst, double* __restrict__ perim0,
                                                         uint8_t* __restrict__ scratch, const int32_t* __restrict__ abort_flag,
                                                         const int32_t* __restrict__ order) {
    if (abort_flag && *abort_flag) return;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    // with a length-sorted order the 32 contours of a warp have similar vertex counts: the per-vertex loops (ellipse fit, area,
    // perimeter: 75 % of this kernel's instructions) ran with 15.7 of 32 lanes active in list order (ncu source view)
    const int64_t it = order ? (int64_t)order[t] : t;
    if (it < 0 || it >= n) return;
    const int64_t i = item_inst ? (int64_t)item_inst[it] : it;
    if (i < 0) return;
    const int64_t c0 = rec_off[it];
    const int nc = (int)(rec_off[it + 1] - c0);
    if (nc == 0) { if (perim0) perim0[i] = 0.0; return; }
    const int32_t* cs = cstart_stride > 0 ? cstart + (size_t)i * cstart_stride : cstart + inst_cont_off[i] + i;
    const uint32_t* p = pts + pt_off[i];
    uint8_t* sc0 = scratch + scratch_off[it];
    size_t sub_end = 0;                                // sub-blocks are laid out in discovery order, measured in reverse
    for (int k = 0; k < nc; ++k) sub_end += emia_measure_sub_bytes(cs[k + 1] - cs[k]);
    for (int j = 0; j < nc; ++j) {
        const int k = nc - 1 - j;                     // OpenCV returns contours in reverse discovery order
        const uint32_t* cp = p + cs[k];
        const int len = cs[k + 1] - cs[k];
        sub_end -= emia_measure_sub_bytes(len);
        double* rec = records + (size_t)(c0 + j) * EMIA_REC_FIELDS;
        // the reference skips a contour below the area gate BEFORE measuring it (src/functions/inference.py:1176-1190): such a
        // record carries area, perimeter and vertex count only (specks are also where fitEllipse is ill-conditioned and slow)
        const double area = emia_contour_area(cp, len);
        if (area < min_area) {
            for (int f = 0; f < EMIA_REC_FIELDS; ++f) rec[f] = 0.0;
            rec[EMIA_REC_AREA] = area;
            rec[EMIA_REC_PERIMETER] = emia_arc_length_closed(cp, len);
            rec[EMIA_F_NVERT] = (double)len;
        } else {
            emia_measure_contour(cp, len, um_pix, sc0 + sub_end, rec, (len >= 1 && len <= presort_max) ? 3 : 0);
            rec[EMIA_REC_MEASURED] = 1.0;
        }
        rec_inst[c0 + j] = (int32_t)i;
        if (j == 0 && perim0) perim0[i] = rec[EMIA_REC_PERIMETER];
    }
}

extern "C" int emia_contour_count(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, int64_t n,
                                  uint32_t* marks, int64_t* n_contours, int64_t* n_points, int64_t* scratch_bytes,
                                  void* stream) {
    if (n < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_count: %s", "bad n");
    if (n == 0) return EMIA_OK;
    if (!crops || !meta || !crop_off || !marks || !n_contours || !n_points || !scratch_bytes)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_count: %s", "null pointer");
    const unsigned grid = (unsigned)((n + EMIA_TRACE_THREADS - 1) / EMIA_TRACE_THREADS);
    emia_launch_clear_marks(marks, crop_off, n, (cudaStream_t)stream);
    k_contour_trace<false><<<grid, EMIA_TRACE_THREADS, EMIA_TRACE_SMEM_BYTES, (cudaStream_t)stream>>>(crops, meta, crop_off, n, marks, n_contours, n_points,
                                                                                  scratch_bytes, nullptr, nullptr, nullptr, nullptr, nullptr);
    return emia_check_launch("emia_contour_count launch: %s");
}

extern "C" int emia_contour_measure(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, int64_t n,
                                    uint32_t* marks, const int64_t* cont_off, const int64_t* pt_off,
                                    const int64_t* scratch_off, double um_pix, double min_area, uint32_t* pts,
                                    int32_t* cstart, double* records, int32_t* rec_inst, double* perim0,
                                    uint8_t* scratch, void* stream) {
    if (n < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_measure: %s", "bad n");
    if (n == 0) return EMIA_OK;
    if (!crops || !meta || !crop_off || !marks || !cont_off || !pt_off || !scratch_off || !pts || !cstart || !records ||
        !rec_inst || !perim0 || !scratch)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_measure: %s", "null pointer");
    const unsigned gridt = (unsigned)((n + EMIA_TRACE_THREADS - 1) / EMIA_TRACE_THREADS);
    emia_launch_clear_marks(marks, crop_off, n, (cudaStream_t)stream);
    k_contour_trace<true><<<gridt, EMIA_TRACE_THREADS, EMIA_TRACE_SMEM_BYTES, (cudaStream_t)stream>>>(crops, meta, crop_off, n, marks, nullptr, nullptr, nullptr,
                                                                                  cont_off, pt_off, pts, cstart, nullptr);
    const unsigned grid = EMIA_MEASURE_GRID(n);
    k_contour_hull<<<EMIA_HULL_GRID(n), EMIA_PRESORT_WARPS * 32, 0, (cudaStream_t)stream>>>(
        n, nullptr, cont_off, cont_off, pt_off, cstart, 0, scratch_off, pts, scratch, nullptr, nullptr);
    k_contour_measure<<<grid, EMIA_MEASURE_THREADS, 0, (cudaStream_t)stream>>>(n, nullptr, cont_off, cont_off, pt_off, scratch_off, um_pix, min_area, pts, cstart, 0,
                                                              EMIA_PRESORT_MAX, records, rec_inst, perim0, scratch, nullptr, nullptr);
    return emia_check_launch("emia_contour_measure launch: %s");
}


// pass 2 of the exact path without the measurement: store the vertex lists (+ perim0)
extern "C" int emia_contour_store(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, int64_t n,
                                  uint32_t* marks, const int64_t* cont_off, const int64_t* pt_off, uint32_t* pts, int32_t* cstart,
                                  double* perim0, void* stream) {
    if (n < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_store: %s", "bad n");
    if (n == 0) return EMIA_OK;
    if (!crops || !meta || !crop_off || !marks || !cont_off || !pt_off || !pts || !cstart)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_store: %s", "null pointer");
    const unsigned gridt = (unsigned)((n + EMIA_TRACE_THREADS - 1) / EMIA_TRACE_THREADS);
    emia_launch_clear_marks(marks, crop_off, n, (cudaStream_t)stream);
    k_contour_trace<true><<<gridt, EMIA_TRACE_THREADS, EMIA_TRACE_SMEM_BYTES, (cudaStream_t)stream>>>(crops, meta, crop_off, n, marks, nullptr, nullptr, nullptr,
                                                                                  cont_off, pt_off, pts, cstart, perim0);
    return emia_check_launch("emia_contour_store launch: %s");
}

// ---- single-pass variant: vertices go to per-instance slabs of bounded capacity -------------------------------------
// cap_pts(i) = 4 * (ch + 32 * cw) + 32 (a blob's border is about 2 * (h + w) pixels); cstart slab of capc + 1 entries.
// Instances that exceed either capacity raise *overflow; the caller then re-runs the exact two-pass path.
__global__ void k_trace_caps(const emia_inst_meta* __restrict__ meta, int64_t n, int64_t* __restrict__ cap) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const emia_inst_meta m = meta[i];
    cap[i] = (m.ch > 0 && m.cw > 0) ? (int64_t)(4 * (m.ch + 32 * m.cw) + 32) : 0;
}

// Seed of every crop for k_contour_trace_slab (emia_trace_seed, one warp per instance, coalesced over the crop words): the first
// foreground pixel in raster order and the number of border-start candidates, written to seed[i].
__global__ void __launch_bounds__(256) k_trace_seed(const uint32_t* __restrict__ crops, const emia_inst_meta* __restrict__ meta,
                                                    const int64_t* __restrict__ crop_off, int64_t n, int64_t* __restrict__ seed,
                                                    const int32_t* __restrict__ abort_flag) {
    if (abort_flag && *abort_flag) return;
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += warps) {
        const emia_inst_meta m = meta[i];
        const int cw = m.cw, words = m.ch * m.cw;
        if (words <= 0 || !EMIA_SEED_FITS(m.ch, m.cw)) {
            if (lane == 0) seed[i] = words <= 0 ? EMIA_SEED_EMPTY : EMIA_SEED_CLASSIC;
            continue;
        }
        const uint32_t* bits = crops + crop_off[i];
        unsigned first = 0xFFFFFFFFu, ncand = 0u;
        // word j of the crop is column c = j % cw of its row; 32 % cw < cw steps c from one word of this lane to the next
        const int step = 32 % cw;
        int c = lane % cw;
        for (int j = lane; j < words; j += 32) {
            const uint32_t F = bits[j];
            const uint32_t left = (F << 1) | (c > 0 ? (bits[j - 1] >> 31) : 0u);
            ncand += __popc(F & ~left);
            if (F != 0u && first == 0xFFFFFFFFu) first = (unsigned)j;
            c += step;
            if (c >= cw) c -= cw;
        }
        first = __reduce_min_sync(0xFFFFFFFFu, first);
        ncand = __reduce_add_sync(0xFFFFFFFFu, ncand);
        if (lane == 0) {
            if (first == 0xFFFFFFFFu) seed[i] = EMIA_SEED_EMPTY;
            else {
                const int y = (int)first / cw;
                seed[i] = EMIA_SEED_PACK(((int)first - y * cw) * 32 + __ffs(bits[first]) - 1, y, ncand);
            }
        }
    }
}

// Lanes are PERSISTENT inside a CTA-owned chunk of instances: a lane that finishes its instance takes the next one from a
// shared-memory counter INSIDE the same flat loop (phase "next"), so the warp keeps executing one instruction stream with
// most lanes busy — border lengths differ 4x between instances and one-instance-per-thread left 8 of 32 lanes active (ncu).
#define EMIA_TRACE_CHUNK 1024          // instances per CTA (upper bound; smaller inputs use smaller chunks to fill the GPU)
#ifndef EMIA_TRACE_MIN_CTAS
#define EMIA_TRACE_MIN_CTAS 8
#endif
__global__ void __launch_bounds__(EMIA_TRACE_THREADS, EMIA_TRACE_MIN_CTAS) k_contour_trace_slab(
    const uint32_t* __restrict__ crops, const emia_inst_meta* __restrict__ meta, const int64_t* __restrict__ crop_off, int64_t n,
    uint32_t* __restrict__ marks, const int64_t* __restrict__ pt_cap_off, int capc, uint32_t* __restrict__ pts,
    int32_t* __restrict__ cstart_slab, int64_t* __restrict__ n_contours, int64_t* __restrict__ scratch_bytes,
    int32_t* __restrict__ overflow, double* __restrict__ perim0, int chunk, const int32_t* __restrict__ abort_flag) {
    if (abort_flag && *abort_flag) return;      // a caller-side capacity guard tripped: write nothing
    __shared__ float s_diag[EMIA_DIAG_TABLE];
    __shared__ int s_next;
    emia_fill_diag_table(s_diag);
    const int64_t lo = (int64_t)blockIdx.x * chunk;
    const int64_t hi = (lo + chunk < n) ? lo + chunk : n;
    if (threadIdx.x == 0) s_next = EMIA_TRACE_THREADS;
    __syncthreads();
    EmiaTraceState T;
    int64_t i = -1;
    int32_t* cs = nullptr;
    int phase = EMIA_TRACE_DONE;
    int first = 1;
    for (;;) {
        if (phase == EMIA_TRACE_DONE) {
            if (i >= 0) {
                // epilogue of instance i
                if (T.o.overflow) { atomicAdd(overflow, 1); n_contours[i] = 0; scratch_bytes[i] = 0; }
                else {
                    const int nc = T.o.n_contours;
                    n_contours[i] = nc;
                    scratch_bytes[i] = (int64_t)emia_measure_item_scratch_bytes(T.o.n_pts, nc);
                    // arcLength of contours[0] in OpenCV order = the LAST discovered contour (deduplicate_masks_smart, Q10),
                    // accumulated while the border was followed
                    if (perim0 && nc) perim0[i] = T.o.perim_last;
                }
            }
            // next instance of this CTA's chunk
            const int k = first ? (int)threadIdx.x : atomicAdd(&s_next, 1);
            first = 0;
            i = lo + k;
            if (i >= hi) break;
            const emia_inst_meta m = meta[i];
            cs = cstart_slab + (size_t)i * (capc + 1);
            if (perim0) perim0[i] = 0.0;
            if (m.ch * m.cw <= 0) { cs[0] = 0; n_contours[i] = 0; scratch_bytes[i] = 0; i = -1; continue; }
            const int64_t off = crop_off[i];
            T.v = emia_make_view(crops, m, off);
            T.o.pts = pts + pt_cap_off[i]; T.o.cap_pts = (int)(pt_cap_off[i + 1] - pt_cap_off[i]);
            T.o.cstart = cs; T.o.cap_contours = capc; T.o.store = 1;
            T.o.track = perim0 != nullptr; T.o.diag = s_diag;
            phase = emia_trace_begin_seeded(T, n_contours[i]);   // the seed k_trace_seed left in n_contours[i]
        } else if (phase == EMIA_TRACE_SCAN) {
            if (!T.mk) {
                // the seeded contour is closed: it was the only one, or the crop is traced again with marks
                if (T.wleft == 0) { phase = EMIA_TRACE_DONE; continue; }
                uint32_t* mk = marks + 2 * crop_off[i];
                emia_trace_restart(T, mk, mk + T.v.h * T.v.wwords);
            }
            phase = emia_trace_scan_step(T);
        } else if (phase == EMIA_TRACE_START) {
            phase = emia_trace_start(T);
        } else {
            phase = emia_trace_follow_step(T);
        }
    }
}

extern "C" int emia_contour_trace_plan(const emia_inst_meta* meta, int64_t n, int64_t* pt_cap, void* stream) {
    if (n < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_trace_plan: %s", "bad n");
    if (n == 0) return EMIA_OK;
    if (!meta || !pt_cap) return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_trace_plan: %s", "null pointer");
    k_trace_caps<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(meta, n, pt_cap);
    return emia_check_launch("emia_contour_trace_plan launch: %s");
}

extern "C" int emia_contour_trace_slab(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off, int64_t n,
                                       uint32_t* marks, const int64_t* pt_cap_off, int32_t cap_contours, uint32_t* pts,
                                       int32_t* cstart_slab, int64_t* n_contours, int64_t* scratch_bytes, int32_t* overflow,
                                       double* perim0, const int32_t* abort_flag, void* stream) {
    if (n < 0 || cap_contours < 1) return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_trace_slab: %s", "bad argument");
    if (n == 0) return EMIA_OK;
    if (!crops || !meta || !crop_off || !marks || !pt_cap_off || !pts || !cstart_slab || !n_contours || !scratch_bytes || !overflow)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_trace_slab: %s", "null pointer");
    // chunk: enough CTAs to fill every SM 8 times over, at least one instance per lane and at most EMIA_TRACE_CHUNK per CTA
    int64_t chunk = (n + (int64_t)emia_num_sms() * 8 - 1) / ((int64_t)emia_num_sms() * 8);
    chunk = (chunk + EMIA_TRACE_THREADS - 1) / EMIA_TRACE_THREADS * EMIA_TRACE_THREADS;
    if (chunk < EMIA_TRACE_THREADS) chunk = EMIA_TRACE_THREADS;
    if (chunk > EMIA_TRACE_CHUNK) chunk = EMIA_TRACE_CHUNK;
    const unsigned grid = (unsigned)((n + chunk - 1) / chunk);
    k_trace_seed<<<emia_num_sms() * 8, 256, 0, (cudaStream_t)stream>>>(crops, meta, crop_off, n, n_contours, abort_flag);
    k_contour_trace_slab<<<grid, EMIA_TRACE_THREADS, 0, (cudaStream_t)stream>>>(crops, meta, crop_off, n, marks, pt_cap_off, cap_contours, pts,
                                                                             cstart_slab, n_contours, scratch_bytes, overflow, perim0, (int)chunk, abort_flag);
    return emia_check_launch("emia_contour_trace_slab launch: %s");
}

extern "C" int emia_contour_measure_stored(const emia_inst_meta* meta, int64_t n, const int64_t* cont_off, const int64_t* pt_off,
                                           const int32_t* cstart, int32_t cstart_stride, const int64_t* scratch_off, double um_pix,
                                           double min_area, const uint32_t* pts, double* records, int32_t* rec_inst, double* perim0,
                                           uint8_t* scratch, void* stream) {
    if (n < 0 || cstart_stride < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_measure_stored: %s", "bad argument");
    if (n == 0) return EMIA_OK;
    if (!meta || !cont_off || !pt_off || !cstart || !scratch_off || !pts || !records || !rec_inst || !perim0 || !scratch)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_measure_stored: %s", "null pointer");
    k_contour_hull<<<EMIA_HULL_GRID(n), EMIA_PRESORT_WARPS * 32, 0, (cudaStream_t)stream>>>(
        n, nullptr, cont_off, cont_off, pt_off, cstart, cstart_stride, scratch_off, pts, (uint8_t*)scratch, nullptr, nullptr);
    k_contour_measure<<<EMIA_MEASURE_GRID(n), EMIA_MEASURE_THREADS, 0, (cudaStream_t)stream>>>(n, nullptr, cont_off, cont_off, pt_off, scratch_off, um_pix, min_area, pts,
                                                                                  cstart, cstart_stride, EMIA_PRESORT_MAX, records, rec_inst, perim0, scratch, nullptr, nullptr);
    return emia_check_launch("emia_contour_measure_stored launch: %s");
}

// ---- measure only the members of G lists (the reference measures what survived de-dup + spatial constraints) ---------
// emia_list_measure_plan: per list slot, the number of records and scratch bytes (0 for dead slots) and the instance id (-1 dead);
// the caller scans rec_cnt / scr_cnt (L + 1 entries each) and sizes `records` / `scratch` from the totals.
__global__ void k_list_measure_plan(const int32_t* __restrict__ cap_off, int G, const int32_t* __restrict__ in_len,
                                    const int32_t* __restrict__ in_idx, int L, const int64_t* __restrict__ n_contours,
                                    const int64_t* __restrict__ scratch_bytes, int32_t* __restrict__ item_inst,
                                    int64_t* __restrict__ rec_cnt, int64_t* __restrict__ scr_cnt) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= L) return;
    int lo = 0, hi = G;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (cap_off[mid] <= s) lo = mid; else hi = mid; }
    int inst = -1;
    int64_t rc = 0, sc = 0;
    if (s - cap_off[lo] < in_len[lo]) {
        inst = in_idx[s];
        rc = n_contours[inst]; sc = scratch_bytes[inst];
    }
    item_inst[s] = inst; rec_cnt[s] = rc; scr_cnt[s] = sc;
}

extern "C" int emia_list_measure_plan(const int32_t* cap_off, int32_t G, int32_t total_cap, const int32_t* in_len,
                                      const int32_t* in_idx, const int64_t* n_contours, const int64_t* scratch_bytes,
                                      int32_t* item_inst, int64_t* rec_cnt, int64_t* scr_cnt, void* stream) {
    if (G < 0 || total_cap < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_list_measure_plan: %s", "bad argument");
    if (G == 0 || total_cap == 0) return EMIA_OK;
    if (!cap_off || !in_len || !in_idx || !n_contours || !scratch_bytes || !item_inst || !rec_cnt || !scr_cnt)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_list_measure_plan: %s", "null pointer");
    k_list_measure_plan<<<(unsigned)((total_cap + 255) / 256), 256, 0, (cudaStream_t)stream>>>(cap_off, G, in_len, in_idx, total_cap, n_contours,
                                                                                            scratch_bytes, item_inst, rec_cnt, scr_cnt);
    return emia_check_launch("emia_list_measure_plan launch: %s");
}

// ---- work order of the list morphometry: slots sorted by vertex count, longest first (counting sort over 64 length classes) ----
// A warp of k_contour_measure is as slow as its longest contour and k_contour_hull balances the chains of the 8 items of a warp, so
// both run over `order` instead of the list order; dead slots go last.  Records / scratch are addressed per SLOT: the results do
// not depend on the order (the position of a slot inside its length class is whatever the atomics give).
#define EMIA_ORDER_BINS 64
__device__ __forceinline__ int emia_order_key(int64_t s, const int32_t* __restrict__ item_inst, const int64_t* __restrict__ rec_off,
                                              const int64_t* __restrict__ inst_cont_off, const int32_t* __restrict__ cstart, int cstart_stride) {
    const int64_t i = item_inst ? (int64_t)item_inst[s] : s;
    if (i < 0) return EMIA_ORDER_BINS - 1;
    const int nc = (int)(rec_off[s + 1] - rec_off[s]);
    if (nc < 1) return EMIA_ORDER_BINS - 1;
    const int32_t* cs = cstart_stride > 0 ? cstart + (size_t)i * cstart_stride : cstart + inst_cont_off[i] + i;
    const int v = cs[nc] - cs[0];
    return (EMIA_ORDER_BINS - 2) - min(max(v, 0) >> 3, EMIA_ORDER_BINS - 2);
}
__global__ void __launch_bounds__(256) k_measure_order_hist(int64_t n, const int32_t* __restrict__ item_inst, const int64_t* __restrict__ rec_off,
                                                            const int64_t* __restrict__ inst_cont_off, const int32_t* __restrict__ cstart,
                                                            int cstart_stride, int32_t* __restrict__ bins) {
    __shared__ int h[EMIA_ORDER_BINS];
    if (threadIdx.x < EMIA_ORDER_BINS) h[threadIdx.x] = 0;
    __syncthreads();
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n) atomicAdd(&h[emia_order_key(s, item_inst, rec_off, inst_cont_off, cstart, cstart_stride)], 1);
    __syncthreads();
    if (threadIdx.x < EMIA_ORDER_BINS && h[threadIdx.x]) atomicAdd(&bins[threadIdx.x], h[threadIdx.x]);
}
__global__ void __launch_bounds__(256) k_measure_order_scatter(int64_t n, const int32_t* __restrict__ item_inst, const int64_t* __restrict__ rec_off,
                                                               const int64_t* __restrict__ inst_cont_off, const int32_t* __restrict__ cstart,
                                                               int cstart_stride, int32_t* __restrict__ bins, int32_t* __restrict__ order) {
    __shared__ int h[EMIA_ORDER_BINS], base[EMIA_ORDER_BINS];
    const int tid = threadIdx.x;
    if (tid < EMIA_ORDER_BINS) h[tid] = 0;
    if (tid < 32) {               // exclusive scan of the 64 class totals (two per lane)
        const int a = bins[2 * tid], b = bins[2 * tid + 1];
        int inc = a + b;
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, inc, o); if (tid >= o) inc += v; }
        base[2 * tid] = inc - a - b;
        base[2 * tid + 1] = inc - b;
    }
    __syncthreads();
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + tid;
    int key = -1, rank = 0;
    if (s < n) { key = emia_order_key(s, item_inst, rec_off, inst_cont_off, cstart, cstart_stride); rank = atomicAdd(&h[key], 1); }
    __syncthreads();
    if (tid < EMIA_ORDER_BINS && h[tid]) base[tid] += atomicAdd(&bins[EMIA_ORDER_BINS + tid], h[tid]);
    __syncthreads();
    if (key >= 0) order[base[key] + rank] = (int32_t)s;
}

extern "C" int emia_list_measure_order(int64_t n_items, const int32_t* item_inst, const int64_t* rec_off, const int64_t* inst_cont_off,
                                       const int32_t* cstart, int32_t cstart_stride, int32_t* order, int32_t* bins, void* stream) {
    if (n_items < 0 || n_items > 0x7fffffff || cstart_stride < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_list_measure_order: %s", "bad argument");
    if (n_items == 0) return EMIA_OK;
    if (!rec_off || !cstart || !order || !bins || (cstart_stride == 0 && !inst_cont_off))
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_list_measure_order: %s", "null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (cudaMemsetAsync(bins, 0, 2 * EMIA_ORDER_BINS * sizeof(int32_t), st) != cudaSuccess)
        return emia_fail(EMIA_ERR_LAUNCH, "emia_list_measure_order: %s", "memset failed");
    const unsigned grid = (unsigned)((n_items + 255) / 256);
    k_measure_order_hist<<<grid, 256, 0, st>>>(n_items, item_inst, rec_off, inst_cont_off, cstart, cstart_stride, bins);
    k_measure_order_scatter<<<grid, 256, 0, st>>>(n_items, item_inst, rec_off, inst_cont_off, cstart, cstart_stride, bins, order);
    return emia_check_launch("emia_list_measure_order launch: %s");
}

extern "C" int emia_contour_measure_list(int64_t n_items, const int32_t* item_inst, const int64_t* rec_off, const int64_t* scr_off,
                                         const int64_t* inst_cont_off, const int64_t* pt_off, const int32_t* cstart,
                                         int32_t cstart_stride, double um_pix, double min_area, const uint32_t* pts, double* records,
                                         int32_t* rec_inst, uint8_t* scratch, const int32_t* abort_flag, const int32_t* order, void* stream) {
    if (n_items < 0 || cstart_stride < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_measure_list: %s", "bad argument");
    if (n_items == 0) return EMIA_OK;
    if (!item_inst || !rec_off || !scr_off || !pt_off || !cstart || !pts || !records || !rec_inst || !scratch ||
        (cstart_stride == 0 && !inst_cont_off))
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_measure_list: %s", "null pointer");
    k_contour_hull<<<EMIA_HULL_GRID(n_items), EMIA_PRESORT_WARPS * 32, 0, (cudaStream_t)stream>>>(
        n_items, item_inst, rec_off, inst_cont_off, pt_off, cstart, cstart_stride, scr_off, pts, scratch, abort_flag, order);
    k_contour_measure<<<EMIA_MEASURE_GRID(n_items), EMIA_MEASURE_THREADS, 0, (cudaStream_t)stream>>>(n_items, item_inst, rec_off, inst_cont_off, pt_off, scr_off,
                                                                                        um_pix, min_area, pts, cstart, cstart_stride,
                                                                                        EMIA_PRESORT_MAX, records, rec_inst, nullptr, scratch, abort_flag, order);
    return emia_check_launch("emia_contour_measure_list launch: %s");
}

// ---- shape descriptors of the records of emia_contour_measure_list: one THREAD per list slot, as k_contour_measure ------------
// Contour k of a slot reuses the k-th sub-block of the slot's scratch (dead once the records are written); rows of records below
// the area gate are NaN.
__global__ void __launch_bounds__(EMIA_MEASURE_THREADS) k_contour_shape(int64_t n, const int32_t* __restrict__ item_inst,
                                                                        const int64_t* __restrict__ rec_off,
                                                                        const int64_t* __restrict__ inst_cont_off,
                                                                        const int64_t* __restrict__ pt_off,
                                                                        const int64_t* __restrict__ scratch_off, double um_pix,
                                                                        const uint32_t* __restrict__ pts, const int32_t* __restrict__ cstart,
                                                                        int cstart_stride, const double* __restrict__ records,
                                                                        uint8_t* __restrict__ scratch, const int32_t* __restrict__ order,
                                                                        double* __restrict__ shape) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int64_t it = order ? (int64_t)order[t] : t;
    if (it < 0 || it >= n) return;
    const int64_t i = item_inst ? (int64_t)item_inst[it] : it;
    if (i < 0) return;
    const int64_t c0 = rec_off[it];
    const int nc = (int)(rec_off[it + 1] - c0);
    if (nc == 0) return;
    const int32_t* cs = cstart_stride > 0 ? cstart + (size_t)i * cstart_stride : cstart + inst_cont_off[i] + i;
    const uint32_t* p = pts + pt_off[i];
    uint8_t* sc0 = scratch + scratch_off[it];
    size_t sub_end = 0;
    for (int k = 0; k < nc; ++k) sub_end += emia_measure_sub_bytes(cs[k + 1] - cs[k]);
    for (int j = 0; j < nc; ++j) {
        const int k = nc - 1 - j;                     // records are in OpenCV order: reverse discovery order
        const int len = cs[k + 1] - cs[k];
        sub_end -= emia_measure_sub_bytes(len);
        double* out = shape + (size_t)(c0 + j) * EMIA_S_COUNT;
        if (records[(size_t)(c0 + j) * EMIA_REC_FIELDS + EMIA_REC_MEASURED] != 1.0) {
            for (int f = 0; f < EMIA_S_COUNT; ++f) out[f] = __longlong_as_double(0x7ff8000000000000ll);
        } else {
            emia_shape_contour(p + cs[k], len, um_pix, sc0 + sub_end, out);
        }
    }
}

extern "C" int emia_contour_shape_list(int64_t n_items, const int32_t* item_inst, const int64_t* rec_off, const int64_t* scr_off,
                                       const int64_t* inst_cont_off, const int64_t* pt_off, const int32_t* cstart, int32_t cstart_stride,
                                       double um_pix, const uint32_t* pts, const double* records, uint8_t* scratch, const int32_t* order,
                                       double* shape, void* stream) {
    if (n_items < 0 || cstart_stride < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_shape_list: %s", "bad argument");
    if (n_items == 0) return EMIA_OK;
    if (!item_inst || !rec_off || !scr_off || !pt_off || !cstart || !pts || !records || !scratch || !shape ||
        (cstart_stride == 0 && !inst_cont_off))
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_contour_shape_list: %s", "null pointer");
    k_contour_shape<<<EMIA_MEASURE_GRID(n_items), EMIA_MEASURE_THREADS, 0, (cudaStream_t)stream>>>(
        n_items, item_inst, rec_off, inst_cont_off, pt_off, scr_off, um_pix, pts, cstart, cstart_stride, records, scratch, order, shape);
    return emia_check_launch("emia_contour_shape_list launch: %s");
}
