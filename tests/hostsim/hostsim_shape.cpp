// hostsim_shape.cpp — g++ build of the shape-descriptor core (deepemia_b200/csrc/core/emia_shape.cuh) for tests/test_hostsim_shape.py.
// TEST INFRASTRUCTURE ONLY: the CPU-only CI checks the core against oracle/shape.py and the convex hull against cv2.convexHull with
// the same source the sm_100a kernels execute.  Nothing in deepemia_b200/ loads this.
#include <vector>
#include "../../deepemia_b200/csrc/core/emia_shape.cuh"

extern "C" {

// contours k = 0..n-1 are pts[off[k]:off[k+1]] (packed x | y << 16); out[10 k ...] = their shape values
void sim_shape(const uint32_t* pts, const long long* off, long long n, double um_pix, double* out) {
    std::vector<uint64_t> scratch;
    for (long long k = 0; k < n; ++k) {
        const int len = (int)(off[k + 1] - off[k]);
        scratch.assign((28 * (size_t)len + 8 + 7) / 8, 0);
        emia_shape_contour(pts + off[k], len, um_pix, scratch.data(), out + 10 * k);
    }
}

// hull[hull_off[k] ...] = emia_convex_hull's point indices of contour k (counter-clockwise flag 0, as cv2.convexHull's default);
// hull_off[k + 1] - hull_off[k] = its size.  hull needs off[n] entries.
void sim_hulls(const uint32_t* pts, const long long* off, long long n, int* hull, long long* hull_off) {
    hull_off[0] = 0;
    for (long long k = 0; k < n; ++k) {
        const int len = (int)(off[k + 1] - off[k]);
        std::vector<uint64_t> keys(len + 1);
        std::vector<int> stack(len + 3), tmp(len + 1);
        const int nh = emia_convex_hull(pts + off[k], len, 0, keys.data(), stack.data(), hull + hull_off[k], tmp.data());
        hull_off[k + 1] = hull_off[k] + nh;
    }
}

}  // extern "C"
