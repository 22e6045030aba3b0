// hostsim_trace.cpp — g++ build of the seeded border trace (deepemia_b200/csrc/core/emia_contour.cuh) for
// tests/test_hostsim_trace.py and tests/test_gpu_trace_seed.py.
// TEST INFRASTRUCTURE ONLY: the CPU-only CI checks the seeded trace k_contour_trace_slab runs against the classic driver with the
// same source the sm_100a kernels execute.  Nothing in deepemia_b200/ loads this.
#include <vector>
#include <cstring>
#include "../../deepemia_b200/csrc/core/emia_common.cuh"
#include "../../deepemia_b200/csrc/core/emia_contour.cuh"

static void pack_bits(const uint8_t* mask, int H, int W, std::vector<uint32_t>& bits, int& ww) {
    ww = (W + 31) / 32;
    bits.assign((size_t)H * ww, 0u);
    for (int y = 0; y < H; ++y)
        for (int x = 0; x < W; ++x)
            if (mask[(size_t)y * W + x]) bits[(size_t)y * ww + (x >> 5)] |= 1u << (x & 31);
}

extern "C" {

// Seeded trace (emia_find_external_contours_seeded, what k_contour_trace_slab runs) against the classic driver on n masks
// of H x W bytes, or, when masks == nullptr, on all 2^(H*W) masks of that size.  The crop is placed at a non-zero frame origin
// and the seeded run starts with garbage in its mark planes.  stats[0] += masks whose seeded contour was the only one,
// stats[1] += masks with exactly one contour, stats[2] += seeded contours that were the only one although the classic trace
// found several (must stay 0).  Returns the index of the first mask whose results differ, or -1.
long long sim_trace_seeded_check(const uint8_t* masks, long long n, int H, int W, int cap_pts, int cap_c, long long* stats) {
    const int ww = (W + 31) / 32;
    std::vector<uint8_t> m((size_t)H * W);
    std::vector<uint32_t> bits, mk((size_t)H * ww), ng((size_t)H * ww), mk2((size_t)H * ww), ng2((size_t)H * ww);
    std::vector<uint32_t> pa(cap_pts + 1), pb(cap_pts + 1);
    std::vector<int> ca(cap_c + 2), cb(cap_c + 2);
    const long long total = masks ? n : (1LL << (H * W));
    for (long long k = 0; k < total; ++k) {
        const uint8_t* mask = masks ? masks + (size_t)k * H * W : m.data();
        if (!masks) for (int j = 0; j < H * W; ++j) m[j] = (uint8_t)((k >> j) & 1);
        int w2;
        pack_bits(mask, H, W, bits, w2);
        EmiaBitView v{bits.data(), ww, H, ww, 96, 7};
        EmiaContourOut a{}, b{};
        a.pts = pa.data(); a.cap_pts = cap_pts; a.cstart = ca.data(); a.cap_contours = cap_c; a.store = 1; a.track = 1;
        b = a; b.pts = pb.data(); b.cstart = cb.data();
        emia_find_external_contours(v, mk.data(), ng.data(), a);
        for (size_t j = 0; j < mk2.size(); ++j) { mk2[j] = 0x9E3779B9u * (uint32_t)(j + k); ng2[j] = ~mk2[j]; }
        int fast = 0;
        emia_find_external_contours_seeded(v, emia_trace_seed(v), mk2.data(), ng2.data(), b, &fast);
        if (a.overflow != b.overflow) return k;
        if (!a.overflow) {
            if (a.n_contours != b.n_contours || a.n_pts != b.n_pts) return k;
            if (std::memcmp(&a.perim_last, &b.perim_last, sizeof(double)) != 0) return k;
            if (std::memcmp(ca.data(), cb.data(), sizeof(int) * (a.n_contours + 1)) != 0) return k;
            if (std::memcmp(pa.data(), pb.data(), sizeof(uint32_t) * a.n_pts) != 0) return k;
            stats[1] += a.n_contours == 1;
        }
        stats[0] += fast;
        stats[2] += fast && !a.overflow && a.n_contours > 1;
    }
    return -1;
}
}  // extern "C"
