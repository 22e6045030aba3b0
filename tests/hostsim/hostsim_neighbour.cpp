// hostsim_neighbour.cpp — g++ build of the neighbour core (deepemia_b200/csrc/core/emia_neighbour.cuh) for
// tests/test_hostsim_neighbours.py.  TEST INFRASTRUCTURE ONLY: the CPU-only CI checks the exact pair distance, the ring-search stop
// rule and the grid searches against oracle/neighbours.py with the same source the sm_100a kernels execute, run serially here.
// Nothing in deepemia_b200/ loads this.
#include <cmath>
#include <vector>
#include "../../deepemia_b200/csrc/core/emia_neighbour.cuh"

extern "C" {

// D2 of two crops (rows [ry0, ry0 + ch) x frame word columns [wc0, wc0 + cw), ch * cw words each), exact below `limit`
long long sim_pair_d2(const uint32_t* aw, int ary0, int awc0, int ach, int acw, const uint32_t* bw, int bry0, int bwc0, int bch, int bcw,
                      long long limit) {
    const EmiaNbCrop a{aw, ary0, awc0, ach, acw}, b{bw, bry0, bwc0, bch, bcw};
    return emia_nb_pair_d2(a, b, limit);
}

int sim_ring_done(int r, int cs, double best_d2) { return emia_nb_ring_done(r, cs, best_d2); }

// the device pass of emia_neighbour_plan + emia_neighbour_search, serially: listed[i] and the centroids cent[2 i ...] are given
// (the plan kernel derives them from the records and emia_moments01); nbf / nbi as in include/emia.h
void sim_neighbours(const uint32_t* crops, const int32_t* meta, const int64_t* crop_off, const int32_t* bbox, const int32_t* class_idx,
                    const uint8_t* listed, const double* cent, int n, int n_class, int H, int W, int cs, double um_pix, double* nbf,
                    int32_t* nbi) {
    const EmiaNbGrid g{cs, (W + cs - 1) / cs, (H + cs - 1) / cs};
    const int64_t ncells = (int64_t)n_class * g.gx * g.gy;
    std::vector<int64_t> cell_off(ncells + 1, 0);
    for (int i = 0; i < n; ++i) {
        double* f = nbf + EMIA_NB_F * i;
        int32_t* o = nbi + EMIA_NB_I * i;
        f[0] = listed[i] ? cent[2 * i] : NAN; f[1] = listed[i] ? cent[2 * i + 1] : NAN; f[2] = f[3] = NAN;
        o[0] = listed[i]; o[1] = o[2] = -1; o[3] = 0; o[4] = listed[i] ? i : -1; o[5] = 0;
        if (!listed[i]) continue;
        const int32_t* b = bbox + 4 * i;
        for (int y = b[0] / cs; y <= b[2] / cs; ++y)
            for (int x = b[1] / cs; x <= b[3] / cs; ++x) ++cell_off[((int64_t)class_idx[i] * g.gy + y) * g.gx + x];
    }
    int64_t acc = 0;
    for (int64_t c = 0; c <= ncells; ++c) { const int64_t v = cell_off[c]; cell_off[c] = acc; acc += v; }
    std::vector<int32_t> ent(acc > 0 ? acc : 1), cursor(ncells, 0), parent(n);
    for (int i = n - 1; i >= 0; --i) {                 // reverse order: the searches must not depend on the order inside a cell
        parent[i] = i;
        if (!listed[i]) continue;
        const int32_t* b = bbox + 4 * i;
        for (int y = b[0] / cs; y <= b[2] / cs; ++y)
            for (int x = b[1] / cs; x <= b[3] / cs; ++x) {
                const int64_t c = ((int64_t)class_idx[i] * g.gy + y) * g.gx + x;
                ent[cell_off[c] + cursor[c]++] = i;
            }
    }
    for (int i = 0; i < n; ++i) {
        if (!listed[i]) continue;
        double d2;
        const int nn = emia_nb_nearest(i, nbf, EMIA_NB_F, class_idx, cell_off.data(), ent.data(), g, &d2);
        if (nn < 0) continue;
        long long D2;
        int nt;
        int32_t* par = parent.data();
        const int cl = emia_nb_closest(i, nn, crops, meta, crop_off, bbox, class_idx, cell_off.data(), ent.data(), g, &D2, &nt,
                                       [&](int k) { if (k > i) emia_nb_unite(par, i, k); });
        nbf[EMIA_NB_F * i + 2] = std::sqrt(d2) * um_pix;
        nbf[EMIA_NB_F * i + 3] = std::sqrt((double)D2) * um_pix;
        nbi[EMIA_NB_I * i + 1] = nn; nbi[EMIA_NB_I * i + 2] = cl; nbi[EMIA_NB_I * i + 3] = nt;
    }
    for (int i = 0; i < n; ++i) {
        if (!listed[i]) continue;
        const int r = emia_nb_find(parent.data(), i);
        nbi[EMIA_NB_I * i + 4] = r;
        ++nbi[EMIA_NB_I * r + 5];
    }
    for (int i = 0; i < n; ++i)
        if (listed[i]) nbi[EMIA_NB_I * i + 5] = nbi[EMIA_NB_I * nbi[EMIA_NB_I * i + 4] + 5];
}

}  // extern "C"
