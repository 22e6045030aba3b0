// hostsim_rle.cpp — g++ build of the RLE read-back core (deepemia_b200/csrc/core/emia_rle.cuh) for tests/test_hostsim_rle.py.
// TEST INFRASTRUCTURE ONLY: the CPU-only CI checks the number parser, the per-run checks and the canonical bbox geometry that the
// sm_100a kernels execute.  Nothing in deepemia_b200/ loads this.
#include <cstring>
#include "../../deepemia_b200/csrc/core/emia_rle.cuh"

extern "C" {

int sim_rle_parse_uint(const uint8_t* s, long long avail, long long* value) {
    int64_t v = 0;
    const int k = emia_rle_parse_uint(s, avail, &v);
    *value = v;
    return k;
}

// the decode plan of one instance, run by run in order as the kernel's lanes check them: status; meta[8], bbox[4], area
int sim_rle_plan(const long long* runs, long long nr, int H, int W, int* meta, int* bbox, long long* area) {
    const int64_t hw = (int64_t)H * W;
    int64_t a = 0;
    int ymin = 0x7fffffff, ymax = -1, xmin = 0x7fffffff, xmax = -1, code = EMIA_RLE_OK;
    for (int64_t k = 0; k < nr; ++k) {
        code = emia_rle_run_status(k ? runs[2 * k - 2] + runs[2 * k - 1] - 1 : 0, runs[2 * k], runs[2 * k + 1], hw);
        if (code) break;
        int y0, y1, x0, x1;
        emia_rle_run_extent(runs[2 * k], runs[2 * k + 1], H, &y0, &y1, &x0, &x1);
        a += runs[2 * k + 1];
        ymin = emia_min(ymin, y0); ymax = emia_max(ymax, y1); xmin = emia_min(xmin, x0); xmax = emia_max(xmax, x1);
    }
    if (code == EMIA_RLE_OK && a > INT32_MAX) code = EMIA_RLE_AREA;
    if (code != EMIA_RLE_OK) a = 0;
    const emia_inst_meta mt = emia_meta_from_bbox(a, ymin, xmin, ymax, xmax);
    memcpy(meta, &mt, sizeof(mt));
    const int bb[4] = {ymin, xmin, ymax, xmax};
    for (int k = 0; k < 4; ++k) bbox[k] = a ? bb[k] : -1;
    *area = a;
    return code;
}

}  // extern "C"
