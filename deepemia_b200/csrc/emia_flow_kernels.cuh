// emia_flow_kernels.cuh — list / unit plumbing of the batched flows (part of emia_kernels.cu).
//
// The reference runs its flows one predictor call at a time, in Python, with a host round trip after every step
// (run_class_specific_inference src/functions/inference.py:1353-1461, tile_based_inference_pipeline :2299-2485,
// run_ensemble_inference :1464-1598, run_adaptive_multiscale_inference :1833-1984).  Here the head outputs of ALL units
// (tiles, images, scales, models) of a batch sit in flat arrays; every step is one launch over all of them, and what the
// reference does with Python lists (boolean indexing, list.extend, `+`) is done by these kernels on (len, idx) lists:
//   emia_group_filter_heads  : `cls == target & score >= thr` (+ Boxes.nonempty() of detector_postprocess, + the
//                              `ori_score.all() < 0.5` early exit of postprocess_masks)
//   emia_group_mark_members  : `len(processed_masks) > 2` gate of process_masks_parallel (:1443)
//   emia_group_flatten       : `full_image_masks + all_tile_masks` (:2452-2454), `all_masks.extend(...)` (:1563, :1958)
//   emia_unit_broadcast_i32  : per-unit constants (tile x / y offsets :2411-2414) expanded to instances
//   emia_scale_f32           : `score * weight` of the ensemble (:1553)
//   emia_gather_*            : boolean / fancy indexing of instance arrays (replaces per-mask Python list handling)
//   emia_capacity_guard      : sync-free execution — variable-size outputs go into caller-sized arenas; a total that exceeds
//                              its arena raises the abort flag AND empties the instance geometry, so that no later kernel
//                              touches memory outside the arenas; the host looks at the flag once, with the results.
#pragma once

// ---- capacity guards ---------------------------------------------------------------------------------------------------
__global__ void k_capacity_guard(const int64_t* __restrict__ total, int64_t capacity, int32_t* __restrict__ abort_flag,
                                 emia_inst_meta* __restrict__ poison_meta, int64_t poison_n) {
    const bool over = (*total > capacity) || (*abort_flag != 0);
    if (!over) return;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < poison_n; i += (int64_t)gridDim.x * blockDim.x) {
        emia_inst_meta m = poison_meta[i];
        m.ch = 0; m.cw = 0; m.rx1 = m.rx0;
        poison_meta[i] = m;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *abort_flag = 1;
}
extern "C" int emia_capacity_guard(const int64_t* total, int64_t capacity, int32_t* abort_flag, emia_inst_meta* poison_meta,
                                   int64_t poison_n, void* stream) {
    if (!total || !abort_flag || capacity < 0 || poison_n < 0 || (poison_n > 0 && !poison_meta))
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_capacity_guard: %s", "bad argument");
    int64_t blocks = (poison_n + 255) / 256;
    if (blocks < 1) blocks = 1;
    if (blocks > 1024) blocks = 1024;
    // the flag is read by every thread before any thread of the grid may set it only when `over` already holds for all of them
    k_capacity_guard<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(total, capacity, abort_flag, poison_meta, poison_n);
    return emia_check_launch("emia_capacity_guard launch: %s");
}

// ---- list filters ---------------------------------------------------------------------------------------------------------
// one warp per group; members that pass, in list order.  target_class < 0: any class.  zero_score_empties != 0: a list that
// still holds a member with score == 0 becomes empty (postprocess_masks: `if ... ori_score.all() < 0.5: return []`,
// src/utils/mask_utils.py:59 — `.all()` is False as soon as one score is exactly 0).
__global__ void k_group_filter_heads(const int32_t* __restrict__ cap_off, int G, const int32_t* __restrict__ in_len,
                                     const int32_t* __restrict__ in_idx, const emia_inst_meta* __restrict__ meta,
                                     const int32_t* __restrict__ classes, const float* __restrict__ scores, int target_class,
                                     float min_score, int zero_score_empties, int32_t* __restrict__ out_len,
                                     int32_t* __restrict__ out_idx) {
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= G) return;
    const int base = cap_off[g], len = in_len[g];
    int run = 0, zero = 0;
    for (int k0 = 0; k0 < len; k0 += 32) {
        const int k = k0 + lane;
        int inst = 0, keep = 0;
        if (k < len) {
            inst = in_idx[base + k];
            const float sc = scores[inst];
            keep = meta[inst].valid != 0 && (target_class < 0 || classes[inst] == target_class) && sc >= min_score;
            if (keep && sc == 0.0f) zero = 1;
        }
        const unsigned b = __ballot_sync(0xffffffffu, keep);
        if (keep) out_idx[base + run + __popc(b & ((1u << lane) - 1u))] = inst;
        run += __popc(b);
    }
    zero = __any_sync(0xffffffffu, zero);
    if (lane == 0) out_len[g] = (zero_score_empties && zero) ? 0 : run;
}
extern "C" int emia_group_filter_heads(const int32_t* cap_off, int32_t G, const int32_t* in_len, const int32_t* in_idx,
                                       const emia_inst_meta* meta, const int32_t* classes, const float* scores, int32_t target_class,
                                       float min_score, int32_t zero_score_empties, int32_t* out_len, int32_t* out_idx, void* stream) {
    if (G < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_group_filter_heads: %s", "bad G");
    if (G == 0) return EMIA_OK;
    if (!cap_off || !in_len || !in_idx || !meta || !classes || !scores || !out_len || !out_idx)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_group_filter_heads: %s", "null pointer");
    k_group_filter_heads<<<(unsigned)(((size_t)G * 32 + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        cap_off, G, in_len, in_idx, meta, classes, scores, target_class, min_score, zero_score_empties, out_len, out_idx);
    return emia_check_launch("emia_group_filter_heads launch: %s");
}

// flag[inst] = value for the members of lists longer than min_len (n_inst entries; cleared first unless keep != 0)
__global__ void k_group_mark_members(const int32_t* __restrict__ cap_off, int G, int L, const int32_t* __restrict__ in_len,
                                     const int32_t* __restrict__ in_idx, int min_len, int value, int32_t* __restrict__ flag) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= L) return;
    const int g = emia_find_group(cap_off, G, s);
    const int len = in_len[g];
    if (s - cap_off[g] < len && len > min_len) flag[in_idx[s]] = value;
}
extern "C" int emia_group_mark_members(const int32_t* cap_off, int32_t G, int32_t total_cap, const int32_t* in_len,
                                       const int32_t* in_idx, int32_t min_len, int32_t value, int32_t keep, int32_t* flag, int64_t n_inst,
                                       void* stream) {
    if (G < 0 || total_cap < 0 || n_inst < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_group_mark_members: %s", "bad argument");
    if (n_inst == 0) return EMIA_OK;
    if (!flag) return emia_fail(EMIA_ERR_BAD_ARG, "emia_group_mark_members: %s", "null pointer");
    if (!keep) cudaMemsetAsync(flag, 0, (size_t)n_inst * 4, (cudaStream_t)stream);
    if (G == 0 || total_cap == 0) return EMIA_OK;
    if (!cap_off || !in_len || !in_idx) return emia_fail(EMIA_ERR_BAD_ARG, "emia_group_mark_members: %s", "null pointer");
    k_group_mark_members<<<(unsigned)((total_cap + 127) / 128), 128, 0, (cudaStream_t)stream>>>(cap_off, G, total_cap, in_len, in_idx,
                                                                                              min_len, value, flag);
    return emia_check_launch("emia_group_mark_members launch: %s");
}

// output list s = the members of the groups grp_list[seg_start[s] .. seg_start[s+1]) one after the other (that order, list
// order inside a group); its slots start at out_cap_off[s].  id_add[g] (optional, indexed by group) is added to every member id
// of group g (instances that were re-numbered when their sets were combined).  One CTA per output list.
__global__ void __launch_bounds__(1024) k_group_flatten(const int32_t* __restrict__ cap_off, const int32_t* __restrict__ in_len,
                                                       const int32_t* __restrict__ in_idx, const int32_t* __restrict__ grp_list,
                                                       const int32_t* __restrict__ seg_start, const int32_t* __restrict__ id_add,
                                                       const int32_t* __restrict__ out_cap_off, int32_t* __restrict__ out_len,
                                                       int32_t* __restrict__ out_idx) {
    __shared__ int s_off[1024];
    __shared__ int s_wsum[32];
    __shared__ int s_run;
    const int sgm = blockIdx.x;
    const int ga = seg_start[sgm], gb = seg_start[sgm + 1];
    const int obase = out_cap_off[sgm];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_run = 0;
    __syncthreads();
    for (int g0 = ga; g0 < gb; g0 += 1024) {
        const int gi = g0 + tid;
        const int len = (gi < gb) ? in_len[grp_list[gi]] : 0;
        int inc = len;
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        if (lane == 31) s_wsum[warp] = inc;
        __syncthreads();
        int wbase = s_run;
        for (int w = 0; w < warp; ++w) wbase += s_wsum[w];
        s_off[tid] = wbase + inc - len;
        __syncthreads();
        const int cnt = min(1024, gb - g0);
        for (int j = warp; j < cnt; j += 32) {
            const int gj = grp_list[g0 + j];
            const int lj = in_len[gj], src = cap_off[gj], dst = obase + s_off[j];
            const int add = id_add ? id_add[gj] : 0;
            for (int k = lane; k < lj; k += 32) out_idx[dst + k] = in_idx[src + k] + add;
        }
        __syncthreads();
        if (tid == 0) { int t = 0; for (int w = 0; w < 32; ++w) t += s_wsum[w]; s_run += t; }
        __syncthreads();
    }
    if (tid == 0) out_len[sgm] = s_run;
}
extern "C" int emia_group_flatten(const int32_t* cap_off, int32_t G, const int32_t* in_len, const int32_t* in_idx,
                                  const int32_t* grp_list, const int32_t* seg_start, int32_t S, const int32_t* id_add,
                                  const int32_t* out_cap_off, int32_t* out_len, int32_t* out_idx, void* stream) {
    if (G < 0 || S < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_group_flatten: %s", "bad argument");
    if (S == 0) return EMIA_OK;
    if (!cap_off || !in_len || !in_idx || !grp_list || !seg_start || !out_cap_off || !out_len || !out_idx)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_group_flatten: %s", "null pointer");
    k_group_flatten<<<(unsigned)S, 1024, 0, (cudaStream_t)stream>>>(cap_off, in_len, in_idx, grp_list, seg_start, id_add, out_cap_off, out_len,
                                                                   out_idx);
    return emia_check_launch("emia_group_flatten launch: %s");
}

// ---- per-unit constants -> per-instance arrays -----------------------------------------------------------------------------
// out[i * k + c] = vals[u * k + c] for the unit u with unit_off[u] <= i < unit_off[u + 1]
__global__ void k_unit_broadcast_i32(const int32_t* __restrict__ unit_off, int U, int64_t n, const int32_t* __restrict__ vals, int k,
                                     int32_t* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int lo = 0, hi = U;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (unit_off[mid] <= i) lo = mid; else hi = mid; }
    for (int c = 0; c < k; ++c) out[i * k + c] = vals[lo * k + c];
}
extern "C" int emia_unit_broadcast_i32(const int32_t* unit_off, int32_t U, int64_t n, const int32_t* vals, int32_t k, int32_t* out,
                                       void* stream) {
    if (U < 0 || n < 0 || k < 1 || k > 16) return emia_fail(EMIA_ERR_BAD_ARG, "emia_unit_broadcast_i32: %s", "bad argument");
    if (n == 0 || U == 0) return EMIA_OK;
    if (!unit_off || !vals || !out) return emia_fail(EMIA_ERR_BAD_ARG, "emia_unit_broadcast_i32: %s", "null pointer");
    k_unit_broadcast_i32<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(unit_off, U, n, vals, k, out);
    return emia_check_launch("emia_unit_broadcast_i32 launch: %s");
}

// out[i] = in[i] * w, one float32 rounding (numpy: np.float32 * python float -> float32 product with the weight rounded to float32)
__global__ void k_scale_f32(const float* __restrict__ in, float w, int64_t n, float* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __fmul_rn(in[i], w);
}
extern "C" int emia_scale_f32(const float* in, float w, int64_t n, float* out, void* stream) {
    if (n < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_scale_f32: %s", "bad n");
    if (n == 0) return EMIA_OK;
    if (!in || !out) return emia_fail(EMIA_ERR_BAD_ARG, "emia_scale_f32: %s", "null pointer");
    k_scale_f32<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(in, w, n, out);
    return emia_check_launch("emia_scale_f32 launch: %s");
}

// ---- gathers: new instance arrays from selected instances of an existing set -----------------------------------------------------
__global__ void k_gather_plan(const emia_inst_meta* __restrict__ src_meta, const int32_t* __restrict__ idx, int64_t k,
                              emia_inst_meta* __restrict__ dst_meta, int64_t* __restrict__ dst_words) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) return;
    const emia_inst_meta m = src_meta[idx ? idx[j] : j];
    dst_meta[j] = m;
    dst_words[j] = (int64_t)m.ch * m.cw;
}
extern "C" int emia_gather_plan(const emia_inst_meta* src_meta, const int32_t* idx, int64_t k, emia_inst_meta* dst_meta,
                                int64_t* dst_crop_words, void* stream) {
    if (k < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_gather_plan: %s", "bad k");
    if (k == 0) return EMIA_OK;
    if (!src_meta || !dst_meta || !dst_crop_words) return emia_fail(EMIA_ERR_BAD_ARG, "emia_gather_plan: %s", "null pointer");
    k_gather_plan<<<(unsigned)((k + 255) / 256), 256, 0, (cudaStream_t)stream>>>(src_meta, idx, k, dst_meta, dst_crop_words);
    return emia_check_launch("emia_gather_plan launch: %s");
}
// one warp per gathered instance: crop words + bbox + area
__global__ void __launch_bounds__(128) k_gather_crops(const uint32_t* __restrict__ src_crops, const int64_t* __restrict__ src_crop_off,
                                                      const int32_t* __restrict__ src_bbox, const int32_t* __restrict__ src_area,
                                                      const int32_t* __restrict__ idx, int64_t k, const emia_inst_meta* __restrict__ dst_meta,
                                                      const int64_t* __restrict__ dst_crop_off, uint32_t* __restrict__ dst_crops,
                                                      int32_t* __restrict__ dst_bbox, int32_t* __restrict__ dst_area) {
    const int lane = threadIdx.x & 31;
    const int64_t j = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (j >= k) return;
    const int64_t i = idx ? idx[j] : j;
    const emia_inst_meta m = dst_meta[j];
    const uint32_t* s = src_crops + src_crop_off[i];
    uint32_t* d = dst_crops + dst_crop_off[j];
    const int nw = m.ch * m.cw;
    for (int t = lane; t < nw; t += 32) d[t] = s[t];
    if (lane == 0) {
        ((int4*)dst_bbox)[j] = ((const int4*)src_bbox)[i];
        dst_area[j] = src_area[i];
    }
}
extern "C" int emia_gather_crops(const uint32_t* src_crops, const int64_t* src_crop_off, const int32_t* src_bbox,
                                 const int32_t* src_area, const int32_t* idx, int64_t k, const emia_inst_meta* dst_meta,
                                 const int64_t* dst_crop_off, uint32_t* dst_crops, int32_t* dst_bbox, int32_t* dst_area, void* stream) {
    if (k < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_gather_crops: %s", "bad k");
    if (k == 0) return EMIA_OK;
    if (!src_crops || !src_crop_off || !src_bbox || !src_area || !dst_meta || !dst_crop_off || !dst_crops || !dst_bbox || !dst_area)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_gather_crops: %s", "null pointer");
    k_gather_crops<<<(unsigned)((k * 32 + 127) / 128), 128, 0, (cudaStream_t)stream>>>(src_crops, src_crop_off, src_bbox, src_area, idx, k,
                                                                                    dst_meta, dst_crop_off, dst_crops, dst_bbox, dst_area);
    return emia_check_launch("emia_gather_crops launch: %s");
}
// 32-bit payloads (scores as raw bits, classes, flags): dst[j] = src[idx[j]]
__global__ void k_gather_b32(const uint32_t* __restrict__ src, const int32_t* __restrict__ idx, int64_t k, uint32_t* __restrict__ dst) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < k) dst[j] = src[idx[j]];
}
extern "C" int emia_gather_b32(const void* src, const int32_t* idx, int64_t k, void* dst, void* stream) {
    if (k < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_gather_b32: %s", "bad k");
    if (k == 0) return EMIA_OK;
    if (!src || !idx || !dst) return emia_fail(EMIA_ERR_BAD_ARG, "emia_gather_b32: %s", "null pointer");
    k_gather_b32<<<(unsigned)((k + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const uint32_t*)src, idx, k, (uint32_t*)dst);
    return emia_check_launch("emia_gather_b32 launch: %s");
}
