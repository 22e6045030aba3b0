// emia_cocoeval.cuh — the rules of COCO `segm` evaluation (pycocotools COCOeval; definition in oracle/cocoeval.py) that the
// sm_100a kernels (emia_cocoeval_kernels.cuh) execute and tests/hostsim checks against the oracle's dense loops:
//   emia_ce_iou       maskApi.c rleIou of one pair from its intersection and the two popcounts;
//   emia_ce_ignore    _ignore of a GT for one area range;
//   emia_ce_consider  one candidate of the match step of one detection at one IoU threshold (evaluateImg);
//   emia_ce_rec_count the recall thresholds one point of the precision / recall curve reaches (accumulate's lookup).
#pragma once
#include "emia_common.cuh"

#define EMIA_CE_T 10                    // IoU thresholds .50:.05:.95
#define EMIA_CE_R 101                   // recall thresholds 0:.01:1
#define EMIA_CE_A 4                     // area ranges all, small, medium, large
#define EMIA_CE_M 3                     // maxDets
#define EMIA_CE_CROWD 1                 // GT flag bits
#define EMIA_CE_ID0 2                   // the GT's id is 0: its match counts as none (dtm == 0)

// inter / (area_d + area_g - inter), or inter / area_d for a crowd GT; 0 when inter == 0 (which covers empty masks)
EMIA_HD double emia_ce_iou(int64_t inter, int64_t area_d, int64_t area_g, bool crowd) {
    if (inter == 0) return 0.0;
    return (double)inter / (double)(crowd ? area_d : area_d + area_g - inter);
}

EMIA_HD bool emia_ce_ignore(double area, bool crowd, double lo, double hi) { return crowd || area < lo || area > hi; }

// The match of one detection at threshold thr: among the available GTs (not yet matched at thr, or crowd) with iou >= thr, the
// largest IoU among non-ignored GTs, ties to the later GT position g; only when there is none, the same among ignored GTs.  This is
// what evaluateImg's dense loop with its `break` computes, for candidates visited in any order.  best_g < 0: none yet.
EMIA_HD void emia_ce_consider(int& best_g, bool& best_ign, double& best_iou, int g, double iou, bool ign, bool avail, double thr) {
    if (!avail || !(iou >= thr)) return;
    if (best_g >= 0) {
        if (ign != best_ign) {
            if (ign) return;
        } else if (iou < best_iou || (iou == best_iou && g < best_g)) {
            return;
        }
    }
    best_g = g;
    best_ign = ign;
    best_iou = iou;
}

// the number of recall thresholds rec[0, n) (ascending) that recall rc reaches (rec[r] <= rc): a point of the curve is found by
// accumulate's searchsorted(rc, rec[r], "left") for exactly these r, so q[r] = the largest precision among points with count > r
EMIA_HD int emia_ce_rec_count(const double* rec, int n, double rc) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (rec[mid] <= rc) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// the precision of a prefix with tp true and fp false positives, in numpy's operation order: tp / ((fp + tp) + eps)
EMIA_HD double emia_ce_precision(double tp, double fp, double eps) { return tp / ((fp + tp) + eps); }
