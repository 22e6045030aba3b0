// hostsim_cocoeval.cpp — g++ build of the COCO segm evaluation core (deepemia_b200/csrc/core/emia_cocoeval.cuh) for
// tests/test_hostsim_cocoeval.py.  TEST INFRASTRUCTURE ONLY: the CPU-only CI checks the match step, the IoU and the
// precision / recall lookup that the sm_100a kernels execute, driven the way k_ce_match and k_ce_accumulate drive them, against
// the dense loops of oracle/cocoeval.py.  Nothing in deepemia_b200/ loads this.
#include <cmath>
#include <vector>
#include "../../deepemia_b200/csrc/core/emia_cocoeval.cuh"

extern "C" {

double sim_ce_iou(long long inter, long long area_d, long long area_g, int crowd) { return emia_ce_iou(inter, area_d, area_g, crowd); }

// evaluateImg of one (image, category, area range): D detections in score order, G GTs in file order.  Detection d visits its
// candidates in the order cand[d * G ..] (a permutation of the GTs; IoU 0 entries included); ious [D, G].  m_out[t * D + d] = the
// file-order index of the matched GT or -1.
void sim_ce_match(int D, int G, const double* ious, const int* cand, const int* gt_ign, const int* gt_crowd, const double* thr, int T,
                  int* m_out) {
    std::vector<unsigned char> matched((size_t)T * G, 0);
    for (int t = 0; t < T; ++t)
        for (int d = 0; d < D; ++d) {
            int bg = -1;
            bool bign = false;
            double biou = 0.0;
            for (int c = 0; c < G; ++c) {
                const int g = cand[(size_t)d * G + c];
                const bool avail = gt_crowd[g] || !matched[(size_t)t * G + g];
                emia_ce_consider(bg, bign, biou, g, ious[(size_t)d * G + g], gt_ign[g] != 0, avail, thr[t]);
            }
            if (bg >= 0) matched[(size_t)t * G + bg] = 1;
            m_out[(size_t)t * D + d] = bg;
        }
}

// one precision / recall entry of accumulate for a sequence of n detections in score order: tp[i], fp[i] in {0, 1} (both 0: ignored)
// -> q[0 .. nr) and *recall, as k_ce_accumulate computes them: each point's precision goes to the bucket of the last recall
// threshold it reaches, q[r] = the largest bucket at or after r (0 when none)
void sim_ce_accumulate(int n, const int* tp, const int* fp, int npig, const double* rec_thrs, int nr, double eps, double* q,
                       double* recall) {
    std::vector<double> bucket(nr, 0.0);
    long long ctp = 0, cfp = 0;
    for (int i = 0; i < n; ++i) {
        ctp += tp[i];
        cfp += fp[i];
        const double rc = (double)ctp / (double)npig;
        const double pr = emia_ce_precision((double)ctp, (double)cfp, eps);
        const int k = emia_ce_rec_count(rec_thrs, nr, rc);
        if (k > 0) bucket[k - 1] = std::fmax(bucket[k - 1], pr);
    }
    *recall = n ? (double)ctp / (double)npig : 0.0;
    double run = 0.0;
    for (int r = nr - 1; r >= 0; --r) {
        run = std::fmax(run, bucket[r]);
        q[r] = run;
    }
}

}  // extern "C"
