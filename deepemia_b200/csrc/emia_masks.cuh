// emia_masks.cuh — byte-mask import/export kernels (part of emia_kernels.cu).
#pragma once

// one CTA per mask: bbox + area of an H x W byte mask
__global__ void __launch_bounds__(256) k_mask_bbox(const uint8_t* __restrict__ masks, int64_t n, int H, int W,
                                                   emia_inst_meta* __restrict__ meta, int64_t* __restrict__ crop_words,
                                                   int32_t* __restrict__ bbox, int32_t* __restrict__ area) {
    __shared__ int s_red[5];
    for (int64_t inst = blockIdx.x; inst < n; inst += gridDim.x) {
        if (threadIdx.x < 5) s_red[threadIdx.x] = (threadIdx.x == 0) ? 0 : ((threadIdx.x <= 2) ? 0x7fffffff : -1);
        __syncthreads();
        const uint8_t* m = masks + (size_t)inst * H * W;
        int a = 0, ymin = 0x7fffffff, xmin = 0x7fffffff, ymax = -1, xmax = -1;
        const int64_t total = (int64_t)H * W;
        for (int64_t k = threadIdx.x; k < total; k += blockDim.x) {
            if (m[k]) {
                const int y = (int)(k / W), x = (int)(k - (int64_t)y * W);
                ++a;
                ymin = min(ymin, y); ymax = max(ymax, y); xmin = min(xmin, x); xmax = max(xmax, x);
            }
        }
        if (a) {
            atomicAdd(&s_red[0], a);
            atomicMin(&s_red[1], ymin); atomicMin(&s_red[2], xmin);
            atomicMax(&s_red[3], ymax); atomicMax(&s_red[4], xmax);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            const int ar = s_red[0];
            area[inst] = ar;
            ((int4*)bbox)[inst] = ar > 0 ? make_int4(s_red[1], s_red[2], s_red[3], s_red[4]) : make_int4(-1, -1, -1, -1);
            const emia_inst_meta mt = emia_meta_from_bbox(ar, s_red[1], s_red[2], s_red[3], s_red[4]);
            meta[inst] = mt;
            crop_words[inst] = (int64_t)mt.ch * mt.cw;
        }
        __syncthreads();
    }
}

// one CTA per mask, one warp per (row, word) of the crop
__global__ void __launch_bounds__(256) k_mask_pack(const uint8_t* __restrict__ masks, int64_t n, int H, int W,
                                                   const emia_inst_meta* __restrict__ meta, const int64_t* __restrict__ crop_off,
                                                   uint32_t* __restrict__ crops) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (int64_t inst = blockIdx.x; inst < n; inst += gridDim.x) {
        const emia_inst_meta m = meta[inst];
        const uint8_t* src = masks + (size_t)inst * H * W;
        uint32_t* crop = crops + crop_off[inst];
        const int items = m.ch * m.cw;
        for (int it = warp; it < items; it += nwarps) {
            const int r = it / m.cw, c = it - r * m.cw;
            const int x = (m.wc0 + c) * 32 + lane, y = m.ry0 + r;
            const bool bit = (x < W) && src[(size_t)y * W + x] != 0;
            const uint32_t word = __ballot_sync(0xffffffffu, bit);
            if (lane == 0) crop[it] = word;
        }
    }
}

// one CTA per output mask (full H x W frame of 0/1 bytes)
__global__ void __launch_bounds__(256) k_mask_unpack(const uint32_t* __restrict__ crops, const emia_inst_meta* __restrict__ meta,
                                                     const int64_t* __restrict__ crop_off, const int32_t* __restrict__ idx,
                                                     int64_t n_idx, int H, int W, uint8_t* __restrict__ out) {
    for (int64_t k = blockIdx.x; k < n_idx; k += gridDim.x) {
        const int inst = idx ? idx[k] : (int)k;
        const emia_inst_meta m = meta[inst];
        const uint32_t* crop = crops + crop_off[inst];
        uint8_t* dst = out + (size_t)k * H * W;
        const int64_t total = (int64_t)H * W;
        for (int64_t p = threadIdx.x; p < total; p += blockDim.x) {
            const int y = (int)(p / W), x = (int)(p - (int64_t)y * W);
            uint8_t v = 0;
            const int r = y - m.ry0, c = (x >> 5) - m.wc0;
            if (r >= 0 && r < m.ch && c >= 0 && c < m.cw) v = (crop[(size_t)r * m.cw + c] >> (x & 31)) & 1u;
            dst[p] = v;
        }
    }
}

extern "C" int emia_mask_bbox(const uint8_t* masks, int64_t n, int H, int W, emia_inst_meta* meta, int64_t* crop_words,
                              int32_t* bbox, int32_t* area, void* stream) {
    if (n < 0 || H <= 0 || W <= 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_mask_bbox: %s", "bad shape");
    if (n == 0) return EMIA_OK;
    if (!masks || !meta || !crop_words || !bbox || !area) return emia_fail(EMIA_ERR_BAD_ARG, "emia_mask_bbox: %s", "null pointer");
    const unsigned grid = (unsigned)(n < 65535 ? n : 65535);
    k_mask_bbox<<<grid, 256, 0, (cudaStream_t)stream>>>(masks, n, H, W, meta, crop_words, bbox, area);
    return emia_check_launch("emia_mask_bbox launch: %s");
}
extern "C" int emia_mask_pack(const uint8_t* masks, int64_t n, int H, int W, const emia_inst_meta* meta,
                              const int64_t* crop_off, uint32_t* crops, void* stream) {
    if (n < 0 || H <= 0 || W <= 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_mask_pack: %s", "bad shape");
    if (n == 0) return EMIA_OK;
    if (!masks || !meta || !crop_off || !crops) return emia_fail(EMIA_ERR_BAD_ARG, "emia_mask_pack: %s", "null pointer");
    const unsigned grid = (unsigned)(n < 65535 ? n : 65535);
    k_mask_pack<<<grid, 256, 0, (cudaStream_t)stream>>>(masks, n, H, W, meta, crop_off, crops);
    return emia_check_launch("emia_mask_pack launch: %s");
}
extern "C" int emia_mask_unpack(const uint32_t* crops, const emia_inst_meta* meta, const int64_t* crop_off,
                                const int32_t* idx, int64_t n_idx, int H, int W, uint8_t* masks_out, void* stream) {
    if (n_idx < 0 || H <= 0 || W <= 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_mask_unpack: %s", "bad shape");
    if (n_idx == 0) return EMIA_OK;
    if (!crops || !meta || !crop_off || !masks_out) return emia_fail(EMIA_ERR_BAD_ARG, "emia_mask_unpack: %s", "null pointer");
    const unsigned grid = (unsigned)(n_idx < 65535 ? n_idx : 65535);
    k_mask_unpack<<<grid, 256, 0, (cudaStream_t)stream>>>(crops, meta, crop_off, idx, n_idx, H, W, masks_out);
    return emia_check_launch("emia_mask_unpack launch: %s");
}
