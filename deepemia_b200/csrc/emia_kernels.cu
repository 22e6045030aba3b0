// emia_kernels.cu — sm_100a kernels + C ABI (include/emia.h) of the deepEMIA post-head hot path.
// Build: nvcc -O3 -lineinfo -fmad=false -gencode arch=compute_100a,code=sm_100a -shared -Xcompiler -fPIC
// (-fmad=false: no implicit FMA contraction; see core/emia_common.cuh).
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <type_traits>
#include "../../include/emia.h"
#include "core/emia_common.cuh"
#include "core/emia_contour.cuh"
#include "core/emia_hull.cuh"
#include "core/emia_ellipse.cuh"
#include "core/emia_measure.cuh"
#include "core/emia_paste.cuh"
#include "core/emia_nms.cuh"
#include "core/emia_moments.cuh"
#include "core/emia_rle.cuh"
#include "core/emia_text.cuh"
#include "core/emia_shape.cuh"
#include "core/emia_neighbour.cuh"
#include "core/emia_coco.cuh"
#include "core/emia_cocoeval.cuh"

static thread_local char g_err[512] = "";
static int emia_fail(int code, const char* fmt, const char* detail) {
    snprintf(g_err, sizeof(g_err), fmt, detail);
    return code;
}
static int emia_check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return emia_fail(EMIA_ERR_LAUNCH, what, cudaGetErrorString(e));
    return EMIA_OK;
}
// Opt-in dynamic shared memory of a kernel: the limit is only ever RAISED.  A per-call cudaFuncSetAttribute(..., exactly what this
// launch needs) lowers it again after a larger launch — harmless for plain launches and for graph replays (the node keeps its own
// attributes), but a tool that re-launches captured kernel nodes one by one (ncu) then sees a launch above the function's current
// limit ("LaunchFailed" on the first graph replay of a 2048-tile step whose second captured shard was smaller).
#include <mutex>
static void emia_need_dyn_smem(const void* fn, size_t bytes) {
    static std::mutex mu;
    static const void* fns[64];
    static size_t cur[64];
    static int devs[64];
    static int nfn = 0;
    if (bytes <= 48 * 1024) return;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> g(mu);
    for (int i = 0; i < nfn; ++i)
        if (fns[i] == fn && devs[i] == dev) {
            if (bytes > cur[i]) { cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes); cur[i] = bytes; }
            return;
        }
    if (nfn < 64) { fns[nfn] = fn; cur[nfn] = bytes; devs[nfn] = dev; ++nfn; }
    cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}
static int emia_num_sms() {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    return sms;
}

extern "C" int emia_version(void) { return 100; }
extern "C" const char* emia_last_error(void) { return g_err; }

// =================================================================================================
// exclusive scan (int64): reduce-then-scan over 4096-element tiles.  Up to 1024 tiles (4 M elements) take three
// launches (tile sums -> scan of the sums in one CTA -> per-tile scan + offset) with the tile sums in a caller workspace
// (emia_scan_workspace_bytes); larger inputs, or no workspace, fall back to a single CTA that walks the array.
// =================================================================================================
#define EMIA_SCAN_THREADS 512
#define EMIA_SCAN_ITEMS 8
#define EMIA_SCAN_TILE (EMIA_SCAN_THREADS * EMIA_SCAN_ITEMS)
#define EMIA_SCAN_MAX_TILES 1024

__device__ __forceinline__ int64_t emia_block_exclusive_scan(int64_t v, int64_t* s_warp, int64_t* total) {
    // exclusive scan of one value per thread across the CTA (EMIA_SCAN_THREADS threads)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t inc = v;
    for (int off = 1; off < 32; off <<= 1) {
        const int64_t t = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int64_t w = (lane < EMIA_SCAN_THREADS / 32) ? s_warp[lane] : 0;
        for (int off = 1; off < 32; off <<= 1) {
            const int64_t t = __shfl_up_sync(0xffffffffu, w, off);
            if (lane >= off) w += t;
        }
        if (lane < EMIA_SCAN_THREADS / 32) s_warp[lane] = w;
    }
    __syncthreads();
    const int64_t base = warp ? s_warp[warp - 1] : 0;
    *total = s_warp[EMIA_SCAN_THREADS / 32 - 1];
    __syncthreads();
    return base + inc - v;
}

__global__ void __launch_bounds__(EMIA_SCAN_THREADS) k_scan_tile_sums(const int64_t* __restrict__ data, int64_t n, int64_t* __restrict__ sums) {
    __shared__ int64_t s_warp[EMIA_SCAN_THREADS / 32];
    const int64_t base = (int64_t)blockIdx.x * EMIA_SCAN_TILE;
    int64_t v = 0;
    for (int k = 0; k < EMIA_SCAN_ITEMS; ++k) {
        const int64_t i = base + (int64_t)k * EMIA_SCAN_THREADS + threadIdx.x;
        if (i < n) v += data[i];
    }
    int64_t total;
    emia_block_exclusive_scan(v, s_warp, &total);
    if (threadIdx.x == 0) sums[blockIdx.x] = total;
}
__global__ void __launch_bounds__(EMIA_SCAN_THREADS) k_scan_sums(int64_t* __restrict__ sums, int ntiles, int64_t* __restrict__ total_out) {
    __shared__ int64_t s_warp[EMIA_SCAN_THREADS / 32];
    // ntiles <= 1024 = 2 per thread
    const int i0 = threadIdx.x * 2, i1 = i0 + 1;
    const int64_t a = i0 < ntiles ? sums[i0] : 0, b = i1 < ntiles ? sums[i1] : 0;
    int64_t total;
    const int64_t ex = emia_block_exclusive_scan(a + b, s_warp, &total);
    if (i0 < ntiles) sums[i0] = ex;
    if (i1 < ntiles) sums[i1] = ex + a;
    if (threadIdx.x == 0) *total_out = total;
}
__global__ void __launch_bounds__(EMIA_SCAN_THREADS) k_scan_apply(int64_t* __restrict__ data, int64_t n, const int64_t* __restrict__ sums) {
    __shared__ int64_t s_warp[EMIA_SCAN_THREADS / 32];
    const int64_t base = (int64_t)blockIdx.x * EMIA_SCAN_TILE + (int64_t)threadIdx.x * EMIA_SCAN_ITEMS;
    int64_t v[EMIA_SCAN_ITEMS];
    int64_t t = 0;
    for (int k = 0; k < EMIA_SCAN_ITEMS; ++k) { v[k] = (base + k < n) ? data[base + k] : 0; t += v[k]; }
    int64_t total;
    int64_t run = emia_block_exclusive_scan(t, s_warp, &total) + sums[blockIdx.x];
    for (int k = 0; k < EMIA_SCAN_ITEMS; ++k) {
        if (base + k < n) data[base + k] = run;
        run += v[k];
    }
}
__global__ void __launch_bounds__(1024) k_exclusive_scan_i64_serial(int64_t* data, int64_t n) {
    __shared__ int64_t part[1024];
    const int t = threadIdx.x;
    const int64_t chunk = (n + 1023) / 1024;
    const int64_t lo = (int64_t)t * chunk;
    const int64_t hi = lo + chunk < n ? lo + chunk : n;
    int64_t s = 0;
    for (int64_t i = lo; i < hi; ++i) s += data[i];
    part[t] = s;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {
        int64_t v = (t >= off) ? part[t - off] : 0;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    int64_t run = (t == 0) ? 0 : part[t - 1];
    for (int64_t i = lo; i < hi; ++i) {
        const int64_t v = data[i];
        data[i] = run;
        run += v;
    }
    if (t == 1023) data[n] = part[1023];
}

// n <= 32 K: one CTA, one launch (1024 threads x 32 items, warp shuffles + one shared-memory pass)
#define EMIA_SCAN_SMALL_MAX 32768
__global__ void __launch_bounds__(1024) k_exclusive_scan_small(int64_t* __restrict__ data, int n) {
    __shared__ int64_t s_warp[32];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int per = (n + 1023) / 1024;                       // <= 32 consecutive items per thread
    const int lo = t * per, hi = min(n, lo + per);
    int64_t sum = 0;
    for (int i = lo; i < hi; ++i) sum += data[i];
    int64_t inc = sum;
    for (int off = 1; off < 32; off <<= 1) { const int64_t v = __shfl_up_sync(0xffffffffu, inc, off); if (lane >= off) inc += v; }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int64_t w = s_warp[lane];
        for (int off = 1; off < 32; off <<= 1) { const int64_t v = __shfl_up_sync(0xffffffffu, w, off); if (lane >= off) w += v; }
        s_warp[lane] = w;
    }
    __syncthreads();
    int64_t run = (warp ? s_warp[warp - 1] : 0) + inc - sum;
    for (int i = lo; i < hi; ++i) { const int64_t v = data[i]; data[i] = run; run += v; }
    if (t == 1023) data[n] = s_warp[31];
}

extern "C" size_t emia_scan_workspace_bytes(int64_t n) {
    (void)n;
    return (size_t)EMIA_SCAN_MAX_TILES * sizeof(int64_t);
}

extern "C" int emia_exclusive_scan_i64(int64_t* data, int64_t n, void* workspace, size_t workspace_bytes, void* stream) {
    if (!data || n < 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_exclusive_scan_i64: %s", "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (n <= EMIA_SCAN_SMALL_MAX) {
        k_exclusive_scan_small<<<1, 1024, 0, st>>>(data, (int)n);
        return emia_check_launch("emia_exclusive_scan_i64 launch: %s");
    }
    const int64_t ntiles = (n + EMIA_SCAN_TILE - 1) / EMIA_SCAN_TILE;
    if (ntiles == 0 || ntiles > EMIA_SCAN_MAX_TILES || !workspace || workspace_bytes < (size_t)ntiles * sizeof(int64_t)) {
        k_exclusive_scan_i64_serial<<<1, 1024, 0, st>>>(data, n);
        return emia_check_launch("emia_exclusive_scan_i64 launch: %s");
    }
    int64_t* sums = (int64_t*)workspace;
    k_scan_tile_sums<<<(unsigned)ntiles, EMIA_SCAN_THREADS, 0, st>>>(data, n, sums);
    k_scan_sums<<<1, EMIA_SCAN_THREADS, 0, st>>>(sums, (int)ntiles, data + n);
    k_scan_apply<<<(unsigned)ntiles, EMIA_SCAN_THREADS, 0, st>>>(data, n, sums);
    return emia_check_launch("emia_exclusive_scan_i64 launch: %s");
}

// =================================================================================================
// K1 — paste + threshold + bit-pack
// =================================================================================================
__global__ void k_paste_plan(const float4* __restrict__ boxes, int64_t n, float sx, float sy, int H, int W,
                             emia_inst_meta* __restrict__ meta, int64_t* __restrict__ crop_words) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 b = boxes[i];
    const EmiaPasteBox pb = emia_paste_prepare(b.x, b.y, b.z, b.w, sx, sy, W, H);
    emia_inst_meta m;
    m.valid = pb.valid && pb.rx1 > pb.rx0 && pb.ry1 > pb.ry0;
    if (m.valid) {
        m.ry0 = pb.ry0; m.ch = pb.ry1 - pb.ry0;
        m.rx0 = pb.rx0; m.rx1 = pb.rx1;
        m.wc0 = pb.rx0 >> 5;
        m.cw = ((pb.rx1 - 1) >> 5) - m.wc0 + 1;
    } else {
        m.ry0 = m.ch = m.rx0 = m.rx1 = m.wc0 = m.cw = 0;
    }
    m.valid = pb.valid;
    m.reserved = 0;
    meta[i] = m;
    crop_words[i] = (int64_t)m.ch * m.cw;
}

extern "C" int emia_paste_plan(const float* boxes, int64_t n, float scale_x, float scale_y, int H, int W,
                               emia_inst_meta* meta, int64_t* crop_words, void* stream) {
    if (n < 0 || H <= 0 || W <= 0 || (n > 0 && (!boxes || !meta || !crop_words)))
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_paste_plan: %s", "bad argument");
    if (n == 0) return EMIA_OK;
    const int threads = 256;
    const unsigned blocks = (unsigned)((n + threads - 1) / threads);
    k_paste_plan<<<blocks, threads, 0, (cudaStream_t)stream>>>((const float4*)boxes, n, scale_x, scale_y, H, W, meta, crop_words);
    return emia_check_launch("emia_paste_plan launch: %s");
}

#define EMIA_PASTE_THREADS 256
#define EMIA_PASTE_TILE_WORDS 2048   // shared staging tile (words) for one band of crop rows

__device__ __forceinline__ void emia_st_stream_u4(uint4* p, uint4 v) {
    asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// One CTA per instance (grid-stride).  Frame = H rows x pitch_words words (pitch_words % 4 == 0).
//  phase 0: stage the 28x28 probabilities and the per-column sampling taps in shared memory
//  phase 1: zero-fill every 16-byte chunk of the frame that lies outside the crop's rows/chunk-columns
//  phase 2: band by band: one warp per (row, word): 32 lanes sample 32 pixels, ballot -> word in shared memory;
//           then the band is written out: crop words (coalesced) and the frame chunks (128-bit stores)
template <bool kFrames>
__global__ void __launch_bounds__(EMIA_PASTE_THREADS) k_paste(
    const float* __restrict__ probs, const float4* __restrict__ boxes, const emia_inst_meta* __restrict__ meta,
    const int64_t* __restrict__ crop_off, int64_t n, float sx, float sy, int H, int W, uint32_t* __restrict__ frames,
    int64_t frame_slots, int pitch_words, uint32_t* __restrict__ crops, int32_t* __restrict__ bbox,
    int32_t* __restrict__ area, int max_cols, const int32_t* __restrict__ abort_flag) {
    if (abort_flag && *abort_flag) return;      // a caller-side capacity guard tripped: write nothing
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* s_prob = (float*)smem_raw;                                  // 784
    uint32_t* s_tile = (uint32_t*)(s_prob + EMIA_MASK_SIDE * EMIA_MASK_SIDE);   // EMIA_PASTE_TILE_WORDS
    int* s_ci0 = (int*)(s_tile + EMIA_PASTE_TILE_WORDS);               // max_cols
    float* s_cw1 = (float*)(s_ci0 + max_cols);                         // max_cols
    float* s_cw0 = s_cw1 + max_cols;                                   // max_cols
    __shared__ int s_red[5];   // area, ymin, xmin, ymax, xmax

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int nwarps = EMIA_PASTE_THREADS / 32;
    const int chunks_per_row = pitch_words >> 2;

    for (int64_t inst = blockIdx.x; inst < n; inst += gridDim.x) {
        const emia_inst_meta m = meta[inst];
        const float4 bx = boxes[inst];
        const EmiaPasteBox pb = emia_paste_prepare(bx.x, bx.y, bx.z, bx.w, sx, sy, W, H);
        const bool live = m.valid && m.ch > 0 && m.cw > 0;
        if (tid < 5) s_red[tid] = (tid == 0) ? 0 : ((tid == 1 || tid == 2) ? 0x7fffffff : -1);
        if (live) {
            const float* p = probs + inst * (EMIA_MASK_SIDE * EMIA_MASK_SIDE);
            for (int k = tid; k < EMIA_MASK_SIDE * EMIA_MASK_SIDE; k += EMIA_PASTE_THREADS) s_prob[k] = p[k];
            const int ncols = m.cw * 32;
            for (int k = tid; k < ncols; k += EMIA_PASTE_THREADS) {
                const int x = m.wc0 * 32 + k;
                const EmiaAxisTap a = emia_paste_axis(x, pb.x0, pb.x1);
                s_ci0[k] = a.i0; s_cw1[k] = a.w1; s_cw0[k] = a.w0;
            }
        }
        // chunk-column range of the crop inside a frame row
        const int cc0 = live ? (m.wc0 >> 2) : 0;
        const int cc1 = live ? ((m.wc0 + m.cw - 1) >> 2) : -1;   // inclusive
        uint4* frame = nullptr;
        if (kFrames) {
            frame = (uint4*)(frames + (size_t)(inst % frame_slots) * (size_t)H * (size_t)pitch_words);
            // ---- phase 1: zero-fill outside the crop window
            const uint4 z = make_uint4(0u, 0u, 0u, 0u);
            const int total = H * chunks_per_row;
            if (!live) {
                for (int q = tid; q < total; q += EMIA_PASTE_THREADS) emia_st_stream_u4(frame + q, z);
            } else {
                const int top = m.ry0 * chunks_per_row;                    // chunks above the crop rows
                const int bot0 = (m.ry0 + m.ch) * chunks_per_row;          // first chunk below
                for (int q = tid; q < top; q += EMIA_PASTE_THREADS) emia_st_stream_u4(frame + q, z);
                for (int q = bot0 + tid; q < total; q += EMIA_PASTE_THREADS) emia_st_stream_u4(frame + q, z);
                // rows of the crop: chunks left and right of [cc0, cc1]
                const int side = chunks_per_row - (cc1 - cc0 + 1);
                if (side > 0) {
                    const int items = m.ch * side;
                    for (int q = tid; q < items; q += EMIA_PASTE_THREADS) {
                        const int r = q / side;
                        int c = q - r * side;
                        if (c >= cc0) c += (cc1 - cc0 + 1);
                        emia_st_stream_u4(frame + (size_t)(m.ry0 + r) * chunks_per_row + c, z);
                    }
                }
            }
        }
        __syncthreads();
        if (live) {
            // ---- phase 2: bands of rows
            const int span_chunks = cc1 - cc0 + 1;
            const int span_words = span_chunks * 4;           // staged row width (chunk aligned)
            const int woff = m.wc0 - cc0 * 4;                 // crop word 0 sits at this word of the staged row
            const int rows_per_band = emia_max(1, EMIA_PASTE_TILE_WORDS / span_words);
            uint32_t* crop = crops + crop_off[inst];
            int l_area = 0, l_ymin = 0x7fffffff, l_xmin = 0x7fffffff, l_ymax = -1, l_xmax = -1;
            for (int r0 = 0; r0 < m.ch; r0 += rows_per_band) {
                const int nr = emia_min(rows_per_band, m.ch - r0);
                // clear the padding words of the staged band
                for (int k = tid; k < nr * span_words; k += EMIA_PASTE_THREADS) s_tile[k] = 0u;
                __syncthreads();
                const int items = nr * m.cw;
                for (int it = warp; it < items; it += nwarps) {
                    const int r = it / m.cw;
                    const int c = it - r * m.cw;
                    const int y = m.ry0 + r0 + r;
                    const EmiaAxisTap ay = emia_paste_axis(y, pb.y0, pb.y1);
                    const int k = c * 32 + lane;
                    const int x = m.wc0 * 32 + k;
                    bool bit = false;
                    if (x >= m.rx0 && x < m.rx1) {
                        EmiaAxisTap ax;
                        ax.i0 = s_ci0[k]; ax.w1 = s_cw1[k]; ax.w0 = s_cw0[k];
                        bit = emia_paste_sample(s_prob, ax, ay) >= 0.5f;
                    }
                    const uint32_t word = __ballot_sync(0xffffffffu, bit);
                    if (lane == 0) {
                        s_tile[r * span_words + woff + c] = word;
                        if (word) {
                            l_area += __popc(word);
                            l_ymin = min(l_ymin, y); l_ymax = max(l_ymax, y);
                            l_xmin = min(l_xmin, (m.wc0 + c) * 32 + (__ffs((int)word) - 1));
                            l_xmax = max(l_xmax, (m.wc0 + c) * 32 + (31 - __clz((int)word)));
                        }
                    }
                }
                __syncthreads();
                // write the band: crop words
                for (int k = tid; k < nr * m.cw; k += EMIA_PASTE_THREADS) {
                    const int r = k / m.cw;
                    const int c = k - r * m.cw;
                    crop[(size_t)(r0 + r) * m.cw + c] = s_tile[r * span_words + woff + c];
                }
                if (kFrames) {
                    const uint4* s4 = (const uint4*)s_tile;
                    for (int k = tid; k < nr * span_chunks; k += EMIA_PASTE_THREADS) {
                        const int r = k / span_chunks;
                        const int c = k - r * span_chunks;
                        emia_st_stream_u4(frame + (size_t)(m.ry0 + r0 + r) * chunks_per_row + cc0 + c, s4[r * span_chunks + c]);
                    }
                }
                __syncthreads();
            }
            if (lane == 0 && l_area) {
                atomicAdd(&s_red[0], l_area);
                atomicMin(&s_red[1], l_ymin); atomicMin(&s_red[2], l_xmin);
                atomicMax(&s_red[3], l_ymax); atomicMax(&s_red[4], l_xmax);
            }
            __syncthreads();
        }
        if (tid == 0) {
            const int a = live ? s_red[0] : 0;
            area[inst] = a;
            int4 bb;
            if (a > 0) bb = make_int4(s_red[1], s_red[2], s_red[3], s_red[4]);
            else bb = make_int4(-1, -1, -1, -1);
            ((int4*)bbox)[inst] = bb;
        }
        __syncthreads();
    }
}

// ---- variant 1: the frame is produced by bulk shared->global copies (cp.async.bulk, the TMA engine) ------------
// A CTA keeps a zeroed 16 KB buffer in shared memory; every 16 KB piece of the frame that does not touch the
// crop rows is one bulk copy from it (one instruction instead of 1024 STG.128); the pieces that do touch crop
// rows are composed in a second shared buffer first.  Crops/bbox/area are produced exactly as in variant 0.
#define EMIA_BULK_BYTES 16384
__device__ __forceinline__ void emia_bulk_s2g(void* gdst, const void* ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst),
                 "r"((uint32_t)__cvta_generic_to_shared(ssrc)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void emia_bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void emia_bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void emia_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__global__ void __launch_bounds__(EMIA_PASTE_THREADS) k_paste_bulk(
    const float* __restrict__ probs, const float4* __restrict__ boxes, const emia_inst_meta* __restrict__ meta,
    const int64_t* __restrict__ crop_off, int64_t n, float sx, float sy, int H, int W, uint32_t* __restrict__ frames,
    int64_t frame_slots, int pitch_words, uint32_t* __restrict__ crops, int32_t* __restrict__ bbox,
    int32_t* __restrict__ area, int max_cols, const int32_t* __restrict__ abort_flag) {
    if (abort_flag && *abort_flag) return;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint32_t* s_zero = (uint32_t*)smem_raw;                              // EMIA_BULK_BYTES
    uint32_t* s_band = s_zero + EMIA_BULK_BYTES / 4;                     // EMIA_BULK_BYTES
    float* s_prob = (float*)(s_band + EMIA_BULK_BYTES / 4);              // 784
    int* s_ci0 = (int*)(s_prob + EMIA_MASK_SIDE * EMIA_MASK_SIDE);
    float* s_cw1 = (float*)(s_ci0 + max_cols);
    float* s_cw0 = s_cw1 + max_cols;
    __shared__ int s_red[5];

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int nwarps = EMIA_PASTE_THREADS / 32;
    const int row_bytes = pitch_words * 4;
    const int rows_per_piece = EMIA_BULK_BYTES / row_bytes;             // >= 1 (checked on the host)
    const int piece_rows_bytes = rows_per_piece * row_bytes;

    for (int k = tid; k < EMIA_BULK_BYTES / 4; k += EMIA_PASTE_THREADS) s_zero[k] = 0u;
    emia_fence_async_smem();
    __syncthreads();

    for (int64_t inst = blockIdx.x; inst < n; inst += gridDim.x) {
        const emia_inst_meta m = meta[inst];
        const float4 bx = boxes[inst];
        const EmiaPasteBox pb = emia_paste_prepare(bx.x, bx.y, bx.z, bx.w, sx, sy, W, H);
        const bool live = m.valid && m.ch > 0 && m.cw > 0;
        if (tid < 5) s_red[tid] = (tid == 0) ? 0 : ((tid == 1 || tid == 2) ? 0x7fffffff : -1);
        if (live) {
            const float* p = probs + inst * (EMIA_MASK_SIDE * EMIA_MASK_SIDE);
            for (int k = tid; k < EMIA_MASK_SIDE * EMIA_MASK_SIDE; k += EMIA_PASTE_THREADS) s_prob[k] = p[k];
            const int ncols = m.cw * 32;
            for (int k = tid; k < ncols; k += EMIA_PASTE_THREADS) {
                const int x = m.wc0 * 32 + k;
                const EmiaAxisTap a = emia_paste_axis(x, pb.x0, pb.x1);
                s_ci0[k] = a.i0; s_cw1[k] = a.w1; s_cw0[k] = a.w0;
            }
        }
        unsigned char* frame = (unsigned char*)(frames + (size_t)(inst % frame_slots) * (size_t)H * (size_t)pitch_words);
        const int crop_r0 = live ? m.ry0 : H, crop_r1 = live ? m.ry0 + m.ch : H;   // crop rows [r0, r1)
        // pieces entirely outside the crop rows: straight from the zero buffer (issued by one thread)
        if (tid == 0) {
            for (int r = 0; r < H; r += rows_per_piece) {
                const int re = emia_min(r + rows_per_piece, H);
                if (re <= crop_r0 || r >= crop_r1)
                    emia_bulk_s2g(frame + (size_t)r * row_bytes, s_zero, (uint32_t)((re - r) * row_bytes));
            }
            emia_bulk_commit();
        }
        __syncthreads();
        int l_area = 0, l_ymin = 0x7fffffff, l_xmin = 0x7fffffff, l_ymax = -1, l_xmax = -1;
        if (live) {
            uint32_t* crop = crops + crop_off[inst];
            const int p0 = (crop_r0 / rows_per_piece) * rows_per_piece;
            for (int r = p0; r < crop_r1; r += rows_per_piece) {
                const int re = emia_min(r + rows_per_piece, H);
                const int nr = re - r;
                // the previous bulk read of s_band must have completed before it is overwritten
                if (tid == 0) emia_bulk_wait_read_all();
                __syncthreads();
                for (int k = tid; k < nr * pitch_words; k += EMIA_PASTE_THREADS) s_band[k] = 0u;
                __syncthreads();
                const int ya = emia_max(r, crop_r0), yb = emia_min(re, crop_r1);
                const int items = (yb - ya) * m.cw;
                for (int it = warp; it < items; it += nwarps) {
                    const int rr = it / m.cw;
                    const int c = it - rr * m.cw;
                    const int y = ya + rr;
                    const EmiaAxisTap ay = emia_paste_axis(y, pb.y0, pb.y1);
                    const int k = c * 32 + lane;
                    const int x = m.wc0 * 32 + k;
                    bool bit = false;
                    if (x >= m.rx0 && x < m.rx1) {
                        EmiaAxisTap ax;
                        ax.i0 = s_ci0[k]; ax.w1 = s_cw1[k]; ax.w0 = s_cw0[k];
                        bit = emia_paste_sample(s_prob, ax, ay) >= 0.5f;
                    }
                    const uint32_t word = __ballot_sync(0xffffffffu, bit);
                    if (lane == 0) {
                        s_band[(y - r) * pitch_words + m.wc0 + c] = word;
                        crop[(size_t)(y - crop_r0) * m.cw + c] = word;
                        if (word) {
                            l_area += __popc(word);
                            l_ymin = min(l_ymin, y); l_ymax = max(l_ymax, y);
                            l_xmin = min(l_xmin, (m.wc0 + c) * 32 + (__ffs((int)word) - 1));
                            l_xmax = max(l_xmax, (m.wc0 + c) * 32 + (31 - __clz((int)word)));
                        }
                    }
                }
                emia_fence_async_smem();
                __syncthreads();
                if (tid == 0) {
                    emia_bulk_s2g(frame + (size_t)r * row_bytes, s_band, (uint32_t)(nr * row_bytes));
                    emia_bulk_commit();
                }
            }
            if (lane == 0 && l_area) {
                atomicAdd(&s_red[0], l_area);
                atomicMin(&s_red[1], l_ymin); atomicMin(&s_red[2], l_xmin);
                atomicMax(&s_red[3], l_ymax); atomicMax(&s_red[4], l_xmax);
            }
            __syncthreads();
        }
        if (tid == 0) {
            const int a = live ? s_red[0] : 0;
            area[inst] = a;
            ((int4*)bbox)[inst] = a > 0 ? make_int4(s_red[1], s_red[2], s_red[3], s_red[4]) : make_int4(-1, -1, -1, -1);
            emia_bulk_wait_read_all();   // s_band / s_zero reads done before the next instance touches s_band
        }
        __syncthreads();
        (void)piece_rows_bytes;
    }
    // all bulk writes must be complete before the CTA (and its shared memory) goes away
    if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---- variant 2 (default): latency-hiding order + 256-bit stores + oversubscribed grid -------------------------------
// ncu on variant 0 (profiles/): 23 % of the stall samples sit on the global->shared copy of the 28x28 probabilities at
// the top of every instance (a DRAM read queued behind the kernel's own write stream) and 11 % of the instructions are
// the integer division of the (row, word) work split; a write-bandwidth probe (scripts/wbw_probe.cu) shows 256-bit
// stores from a grid 4-8x larger than the resident CTA count reach 7.0-7.2 TB/s where a persistent 128-bit grid stops
// at 6.1-6.3.  Hence:
//   1. cp.async (LDGSTS) the probabilities into a zero-padded 32 x 36 tile FIRST, then zero-fill the frame outside the
//      crop rows with st.global.v4.b64 while the copy is in flight, and only then wait for it;
//   2. per-column AND per-row sampling taps in shared memory, padded tile => no bounds tests, no per-pixel division;
//   3. grid = min(n, SMs x 32) CTAs of 256 threads, instance = blockIdx.x + k * gridDim.x.
// Needs 32-byte aligned frame rows (pitch_words % 8 == 0); other shapes use variant 0.
#define EMIA_P2_PAD_STRIDE 36                 // floats per padded tile row: data at columns 4..31, zeros elsewhere
#define EMIA_P2_PAD_ROWS 32                   // tile rows -2..29
#define EMIA_P2_BAND_ROWS 128                 // row taps staged per band
#define EMIA_P2_MAX_COLS 2112                 // W <= 2048 (+ one word of slack, multiple of 32)
#ifndef EMIA_P2_MIN_CTAS
#define EMIA_P2_MIN_CTAS 4
#endif

__device__ __forceinline__ void emia_st256_zero(void* p) {
    asm volatile("st.global.v4.b64 [%0], {%1, %1, %1, %1};" ::"l"(p), "l"(0ull) : "memory");
}
__device__ __forceinline__ void emia_st256(void* p, uint4 a, uint4 b) {
    asm volatile("st.global.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(p), "l"(((unsigned long long)a.y << 32) | a.x),
                 "l"(((unsigned long long)a.w << 32) | a.z), "l"(((unsigned long long)b.y << 32) | b.x),
                 "l"(((unsigned long long)b.w << 32) | b.z)
                 : "memory");
}
__device__ __forceinline__ void emia_cp_async16(void* sdst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(sdst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ int emia_clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

template <bool kHalf>
__global__ void __launch_bounds__(EMIA_PASTE_THREADS, EMIA_P2_MIN_CTAS) k_paste_v2(
    const void* __restrict__ probs_raw, const float4* __restrict__ boxes, const emia_inst_meta* __restrict__ meta,
    const int64_t* __restrict__ crop_off, int64_t n, float sx, float sy, int H, int W, uint32_t* __restrict__ frames,
    int64_t frame_slots, int pitch_words, uint32_t* __restrict__ crops, int32_t* __restrict__ bbox, int32_t* __restrict__ area,
    const int32_t* __restrict__ abort_flag) {
    if (abort_flag && *abort_flag) return;      // a caller-side capacity guard tripped: write nothing
    __shared__ __align__(16) float s_pp2[2][EMIA_P2_PAD_ROWS * EMIA_P2_PAD_STRIDE];   // padded probabilities, double-buffered
    __shared__ __align__(16) __half s_half2[2][kHalf ? EMIA_MASK_SIDE * EMIA_MASK_SIDE : 8];   // fp16 head outputs: staged, then widened
    const float* probs = (const float*)probs_raw;
    const __half* probs_h = (const __half*)probs_raw;
    __shared__ __align__(32) uint32_t s_tile[EMIA_PASTE_TILE_WORDS];              // one band of frame rows (chunk span)
    __shared__ int2 s_ctap[EMIA_P2_MAX_COLS];     // per column: (tile offset of tap i0, bits of w1); columns outside [rx0, rx1) read zeros
    __shared__ int2 s_rtap[EMIA_P2_BAND_ROWS];    // per row of the band: (tile offset of tap row, bits of w1)
    __shared__ int s_red[5];   // area, ymin, xmin, ymax, xmax

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int nwarps = EMIA_PASTE_THREADS / 32;
    const int cpr = pitch_words >> 3;               // 32-byte chunks per frame row
    for (int k = tid; k < 2 * EMIA_P2_PAD_ROWS * EMIA_P2_PAD_STRIDE; k += EMIA_PASTE_THREADS) (&s_pp2[0][0])[k] = 0.f;
    __syncthreads();
    // copy of the probabilities of instance `q` into buffer b (28 rows x 7 chunks of 16 bytes -> padded tile rows 2..29, columns
    // 4..31; fp16: 98 chunks staged and widened after the wait).  Always commits a group, so the group count is uniform.
    auto issue = [&](int64_t q, bool q_live, int b) {
        if (q_live) {
            if (kHalf) {
                if (tid < (EMIA_MASK_SIDE * EMIA_MASK_SIDE) / 8)
                    emia_cp_async16(&s_half2[b][tid * 8], probs_h + q * (EMIA_MASK_SIDE * EMIA_MASK_SIDE) + tid * 8);
            } else if (tid < EMIA_MASK_SIDE * 7) {
                const int r = tid / 7, c7 = tid - r * 7;
                emia_cp_async16(&s_pp2[b][(r + 2) * EMIA_P2_PAD_STRIDE + 4 + c7 * 4],
                                probs + q * (EMIA_MASK_SIDE * EMIA_MASK_SIDE) + r * EMIA_MASK_SIDE + c7 * 4);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // software pipeline over the CTA's instances: the meta / box / probabilities of instance k + 1 are fetched while instance k
    // is processed (ncu: 16 % of the stall samples sat on these dependent DRAM reads at the top of every instance)
    emia_inst_meta m_next;
    float4 bx_next = make_float4(0.f, 0.f, 0.f, 0.f);
    m_next.valid = 0; m_next.ch = m_next.cw = 0;
    if ((int64_t)blockIdx.x < n) { m_next = meta[blockIdx.x]; bx_next = boxes[blockIdx.x]; }
    issue(blockIdx.x, (int64_t)blockIdx.x < n && m_next.valid && m_next.ch > 0 && m_next.cw > 0, 0);
    int buf = 0;

    for (int64_t inst = blockIdx.x; inst < n; inst += gridDim.x) {
        const emia_inst_meta m = m_next;
        const float4 bx = bx_next;
        float* s_pp = s_pp2[buf];
        const __half* s_half = s_half2[buf];
        const EmiaPasteBox pb = emia_paste_prepare(bx.x, bx.y, bx.z, bx.w, sx, sy, W, H);
        const bool live = m.valid && m.ch > 0 && m.cw > 0;
        if (tid < 5) s_red[tid] = (tid == 0) ? 0 : ((tid == 1 || tid == 2) ? 0x7fffffff : -1);
        // ---- 1. zero-fill the frame outside the crop's rows / chunk span
        const int cc0 = live ? (m.wc0 >> 3) : 0;
        const int cc1 = live ? ((m.wc0 + m.cw - 1) >> 3) : -1;   // inclusive
        unsigned char* frame = nullptr;
        if (frames) {
            frame = (unsigned char*)(frames + (size_t)(inst % frame_slots) * (size_t)H * (size_t)pitch_words);
            const int total = H * cpr;
            const int top = live ? m.ry0 * cpr : total;
            const int bot0 = live ? (m.ry0 + m.ch) * cpr : total;
            for (int q = tid; q < top; q += EMIA_PASTE_THREADS) emia_st256_zero(frame + (size_t)q * 32);
            for (int q = bot0 + tid; q < total; q += EMIA_PASTE_THREADS) emia_st256_zero(frame + (size_t)q * 32);
            if (live && cc1 - cc0 + 1 < cpr) {
                for (int r = tid; r < m.ch; r += EMIA_PASTE_THREADS) {
                    unsigned char* row = frame + (size_t)(m.ry0 + r) * cpr * 32;
                    for (int c = 0; c < cc0; ++c) emia_st256_zero(row + c * 32);
                    for (int c = cc1 + 1; c < cpr; ++c) emia_st256_zero(row + c * 32);
                }
            }
        }
        // ---- 2. fetch the next instance (its copy lands while this one is sampled)
        {
            const int64_t nx = inst + gridDim.x;
            bool nlive = false;
            if (nx < n) { m_next = meta[nx]; bx_next = boxes[nx]; nlive = m_next.valid && m_next.ch > 0 && m_next.cw > 0; }
            issue(nx, nlive, buf ^ 1);
        }
        if (live) {
            // ---- 3. column taps (independent of the probabilities)
            const int ncols = m.cw * 32;
            for (int k = tid; k < ncols; k += EMIA_PASTE_THREADS) {
                const int x = m.wc0 * 32 + k;
                const EmiaAxisTap a = emia_paste_axis(x, pb.x0, pb.x1);
                // a column outside the sampling region reads the zero padding (taps -2, -1): its bits come out 0
                const int i0 = (x >= m.rx0 && x < m.rx1) ? emia_clampi(a.i0, -2, EMIA_MASK_SIDE) : -2;
                s_ctap[k] = make_int2(i0 + 4, __float_as_int(a.w1));
            }
        }
        asm volatile("cp.async.wait_group 1;" ::: "memory");       // everything but the prefetch just issued has landed
        __syncthreads();
        if (kHalf) {
            if (live)
                for (int k = tid; k < EMIA_MASK_SIDE * EMIA_MASK_SIDE; k += EMIA_PASTE_THREADS) {
                    const int r = k / EMIA_MASK_SIDE, c = k - r * EMIA_MASK_SIDE;
                    s_pp[(r + 2) * EMIA_P2_PAD_STRIDE + 4 + c] = __half2float(s_half[k]);
                }
            __syncthreads();
        }
        if (live) {
            const int span_chunks = cc1 - cc0 + 1;
            const int span_words = span_chunks * 8;             // staged row width (32-byte chunk aligned)
            const int woff = m.wc0 - cc0 * 8;                   // crop word 0 sits at this word of the staged row
            const int rows_per_band = emia_min(EMIA_P2_BAND_ROWS, emia_max(1, EMIA_PASTE_TILE_WORDS / span_words));
            const int step_r = nwarps / m.cw, step_c = nwarps - step_r * m.cw;
            uint32_t* crop = crops + crop_off[inst];
            int l_area = 0, l_ymin = 0x7fffffff, l_xmin = 0x7fffffff, l_ymax = -1, l_xmax = -1;
            for (int r0 = 0; r0 < m.ch; r0 += rows_per_band) {
                const int nr = emia_min(rows_per_band, m.ch - r0);
                for (int k = tid; k < nr * span_words; k += EMIA_PASTE_THREADS) s_tile[k] = 0u;
                for (int k = tid; k < nr; k += EMIA_PASTE_THREADS) {
                    const EmiaAxisTap a = emia_paste_axis(m.ry0 + r0 + k, pb.y0, pb.y1);
                    s_rtap[k] = make_int2((emia_clampi(a.i0, -2, EMIA_MASK_SIDE) + 2) * EMIA_P2_PAD_STRIDE, __float_as_int(a.w1));
                }
                __syncthreads();
                // one warp per (row, word): 32 lanes sample 32 pixels, ballot -> word
                int r = warp / m.cw, c = warp - r * m.cw;
                while (r < nr) {
                    const int2 ct = s_ctap[c * 32 + lane], rt = s_rtap[r];
                    const float xw1 = __int_as_float(ct.y), yw1 = __int_as_float(rt.y);
                    const float xw0 = 1.f - xw1, yw0 = 1.f - yw1;
                    const float* t = &s_pp[rt.x + ct.x];
                    const float nw = yw0 * xw0;
                    const float ne = yw0 * xw1;
                    const float sw = yw1 * xw0;
                    const float se = yw1 * xw1;
                    float acc = t[0] * nw;
                    acc = emia_fmaf(t[1], ne, acc);
                    acc = emia_fmaf(t[EMIA_P2_PAD_STRIDE], sw, acc);
                    acc = emia_fmaf(t[EMIA_P2_PAD_STRIDE + 1], se, acc);
                    const uint32_t word = __ballot_sync(0xffffffffu, acc >= 0.5f);
                    if (lane == 0) s_tile[r * span_words + woff + c] = word;
                    r += step_r; c += step_c;
                    if (c >= m.cw) { c -= m.cw; ++r; }
                }
                __syncthreads();
                // write the band: crop words (+ bbox / area from the same words), then the frame chunk span (256-bit stores)
                {
                    int rr = tid / m.cw, cc = tid - rr * m.cw;
                    const int sr = EMIA_PASTE_THREADS / m.cw, scw = EMIA_PASTE_THREADS - sr * m.cw;
                    while (rr < nr) {
                        const uint32_t word = s_tile[rr * span_words + woff + cc];
                        crop[(size_t)(r0 + rr) * m.cw + cc] = word;
                        if (word) {
                            const int y = m.ry0 + r0 + rr;
                            l_area += __popc(word);
                            l_ymin = min(l_ymin, y); l_ymax = max(l_ymax, y);
                            l_xmin = min(l_xmin, (m.wc0 + cc) * 32 + (__ffs((int)word) - 1));
                            l_xmax = max(l_xmax, (m.wc0 + cc) * 32 + (31 - __clz((int)word)));
                        }
                        rr += sr; cc += scw;
                        if (cc >= m.cw) { cc -= m.cw; ++rr; }
                    }
                }
                if (frames) {
                    const uint4* s4 = (const uint4*)s_tile;
                    int rr = tid / span_chunks, cc = tid - rr * span_chunks;
                    const int sr = EMIA_PASTE_THREADS / span_chunks, sc = EMIA_PASTE_THREADS - sr * span_chunks;
                    while (rr < nr) {
                        const int si = (rr * span_chunks + cc) * 2;
                        emia_st256(frame + ((size_t)(m.ry0 + r0 + rr) * cpr + cc0 + cc) * 32, s4[si], s4[si + 1]);
                        rr += sr; cc += sc;
                        if (cc >= span_chunks) { cc -= span_chunks; ++rr; }
                    }
                }
                __syncthreads();
            }
            for (int o = 16; o > 0; o >>= 1) {
                l_area += __shfl_xor_sync(0xffffffffu, l_area, o);
                l_ymin = min(l_ymin, __shfl_xor_sync(0xffffffffu, l_ymin, o)); l_xmin = min(l_xmin, __shfl_xor_sync(0xffffffffu, l_xmin, o));
                l_ymax = max(l_ymax, __shfl_xor_sync(0xffffffffu, l_ymax, o)); l_xmax = max(l_xmax, __shfl_xor_sync(0xffffffffu, l_xmax, o));
            }
            if (lane == 0 && l_area) {
                atomicAdd(&s_red[0], l_area);
                atomicMin(&s_red[1], l_ymin); atomicMin(&s_red[2], l_xmin);
                atomicMax(&s_red[3], l_ymax); atomicMax(&s_red[4], l_xmax);
            }
            __syncthreads();
        }
        if (tid == 0) {
            const int a = live ? s_red[0] : 0;
            area[inst] = a;
            ((int4*)bbox)[inst] = a > 0 ? make_int4(s_red[1], s_red[2], s_red[3], s_red[4]) : make_int4(-1, -1, -1, -1);
        }
        __syncthreads();
        buf ^= 1;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

extern "C" int emia_paste_threshold_bitpack(const float* probs, const float* boxes, const emia_inst_meta* meta,
                                            const int64_t* crop_off, int64_t n, float scale_x, float scale_y, int H,
                                            int W, uint32_t* frames, int64_t frame_slots, int pitch_words,
                                            uint32_t* crops, int32_t* bbox, int32_t* area, int variant_and_grid,
                                            const int32_t* abort_flag, void* stream) {
    // bits 0-7: variant; bits 8-15: resident CTAs per SM (0 = default) — a smaller grid leaves SM room for other streams
    const int variant = variant_and_grid & 0xff;
    const int ctas_req = (variant_and_grid >> 8) & 0xff;
    const bool probs_f16 = (variant_and_grid >> 16) & 1;      // EMIA_PASTE_PROBS_F16
    if (n < 0 || H <= 0 || W <= 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_paste_threshold_bitpack: %s", "bad shape");
    if (n == 0) return EMIA_OK;
    if (!probs || !boxes || !meta || !crop_off || !crops || !bbox || !area)
        return emia_fail(EMIA_ERR_BAD_ARG, "emia_paste_threshold_bitpack: %s", "null pointer");
    if (frames) {
        if (pitch_words * 32 < W || (pitch_words & 3) || frame_slots <= 0)
            return emia_fail(EMIA_ERR_BAD_ARG, "emia_paste_threshold_bitpack: %s", "pitch_words must be a multiple of 4 covering W; frame_slots > 0");
        if (((uintptr_t)frames & 15) != 0) return emia_fail(EMIA_ERR_BAD_ARG, "emia_paste_threshold_bitpack: %s", "frames must be 16-byte aligned");
    }
    const int max_cols = ((W + 31) / 32 + 1) * 32;
    cudaStream_t st = (cudaStream_t)stream;
    const int sms = emia_num_sms();
    if (variant == 2 && max_cols <= EMIA_P2_MAX_COLS && ((uintptr_t)probs & 15) == 0 &&
        (!frames || ((pitch_words & 7) == 0 && ((uintptr_t)frames & 31) == 0))) {
        const int64_t per_sm = ctas_req ? ctas_req : 32;
        const unsigned grid = (unsigned)(n < (int64_t)sms * per_sm ? n : (int64_t)sms * per_sm);
        if (probs_f16)
            k_paste_v2<true><<<grid, EMIA_PASTE_THREADS, 0, st>>>(probs, (const float4*)boxes, meta, crop_off, n, scale_x, scale_y, H, W, frames,
                                                                  frames ? frame_slots : 1, pitch_words, crops, bbox, area, abort_flag);
        else
            k_paste_v2<false><<<grid, EMIA_PASTE_THREADS, 0, st>>>(probs, (const float4*)boxes, meta, crop_off, n, scale_x, scale_y, H, W, frames,
                                                                   frames ? frame_slots : 1, pitch_words, crops, bbox, area, abort_flag);
        return emia_check_launch("emia_paste_threshold_bitpack (v2) launch: %s");
    }
    if (probs_f16) return emia_fail(EMIA_ERR_UNSUPPORTED, "emia_paste_threshold_bitpack: %s", "fp16 probabilities need variant 2 (W <= 2048, 32-byte frame rows)");
    if (variant == 1 && frames) {
        if (pitch_words * 4 > EMIA_BULK_BYTES) return emia_fail(EMIA_ERR_UNSUPPORTED, "emia_paste_threshold_bitpack: %s", "variant 1 needs a frame row <= 16 KB");
        const size_t smem = 2 * EMIA_BULK_BYTES + EMIA_MASK_SIDE * EMIA_MASK_SIDE * 4 + (size_t)max_cols * 12;
        emia_need_dyn_smem((const void*)k_paste_bulk, smem);
        const int64_t per_sm = ctas_req ? ctas_req : 4;
        const unsigned grid = (unsigned)(n < (int64_t)sms * per_sm ? n : (int64_t)sms * per_sm);
        k_paste_bulk<<<grid, EMIA_PASTE_THREADS, smem, st>>>(probs, (const float4*)boxes, meta, crop_off, n, scale_x, scale_y, H, W,
                                                             frames, frame_slots, pitch_words, crops, bbox, area, max_cols, abort_flag);
        return emia_check_launch("emia_paste_threshold_bitpack (bulk) launch: %s");
    }
    const size_t smem = EMIA_MASK_SIDE * EMIA_MASK_SIDE * 4 + EMIA_PASTE_TILE_WORDS * 4 + (size_t)max_cols * 12;
    const int64_t per_sm = ctas_req ? ctas_req : 8;
    const unsigned grid = (unsigned)(n < (int64_t)sms * per_sm ? n : (int64_t)sms * per_sm);
    if (frames) {
        emia_need_dyn_smem((const void*)k_paste<true>, smem);
        k_paste<true><<<grid, EMIA_PASTE_THREADS, smem, st>>>(probs, (const float4*)boxes, meta, crop_off, n, scale_x, scale_y, H, W,
                                                              frames, frame_slots, pitch_words, crops, bbox, area, max_cols, abort_flag);
    } else {
        emia_need_dyn_smem((const void*)k_paste<false>, smem);
        k_paste<false><<<grid, EMIA_PASTE_THREADS, smem, st>>>(probs, (const float4*)boxes, meta, crop_off, n, scale_x, scale_y, H, W,
                                                               nullptr, 1, pitch_words, crops, bbox, area, max_cols, abort_flag);
    }
    return emia_check_launch("emia_paste_threshold_bitpack launch: %s");
}

#include "emia_masks.cuh"
#include "emia_morpho_kernels.cuh"
#include "emia_group_kernels.cuh"
#include "emia_morph_kernels.cuh"
#include "emia_tile_kernels.cuh"
#include "emia_rle_kernels.cuh"
#include "emia_text_kernels.cuh"
#include "emia_coco_kernels.cuh"
#include "emia_cocoeval_kernels.cuh"
#include "emia_neighbour_kernels.cuh"
#include "emia_flow_kernels.cuh"
#include "emia_scalebar_kernels.cuh"
