// hostsim_coco.cpp — g++ build of the COCO counts-string core (deepemia_b200/csrc/core/emia_coco.cuh) for tests/test_hostsim_coco.py.
// TEST INFRASTRUCTURE ONLY: the CPU-only CI checks the delta lengths, the writer and the value decoder that the sm_100a kernels
// execute, and a sequential walk over a whole string with the kernels' rules (i > 2 delta coding, statuses in string order).
// Nothing in deepemia_b200/ loads this.
#include <climits>
#include "../../deepemia_b200/csrc/core/emia_coco.cuh"
#include "../../include/emia.h"

extern "C" {

int sim_coco_delta_len(long long x, int* chars) { return emia_coco_delta_len(x, chars); }
int sim_coco_put_delta(long long x, uint8_t* out) { return emia_coco_put_delta(out, x); }
long long sim_coco_value(const uint8_t* s, int k) { return emia_coco_value(s, k); }

// JSON text of the counts cnts[0, m) (k_coco_ann's code per count); returns its length.  out: NULL to count only
long long sim_coco_encode(const long long* cnts, long long m, uint8_t* out) {
    long long b = 0;
    for (long long i = 0; i < m; ++i) {
        const int64_t x = i > 2 ? cnts[i] - cnts[i - 2] : cnts[i];
        b += out ? emia_coco_put_delta(out + b, x) : emia_coco_delta_len(x, nullptr);
    }
    return b;
}

// the counts of the string s[0, len) into cnts (capacity len), *m = their number; returns the EMIA_COCO_* status that
// k_coco_counts reports for a frame of hw pixels
int sim_coco_decode(const uint8_t* s, long long len, long long hw, long long* cnts, long long* m) {
    long long nv = 0, start = 0, sum = 0;
    for (long long p = 0; p < len; ++p) {
        if (!emia_coco_char_ok(s[p])) { *m = nv; return EMIA_COCO_BAD_CHAR; }
        if (emia_coco_char_more(s[p])) continue;
        const int k = (int)(p - start + 1);
        if (k > EMIA_COCO_MAX_CHARS) { *m = nv; return EMIA_COCO_RANGE; }
        int64_t c = emia_coco_value(s + start, k);
        if (nv > 2) c += cnts[nv - 2];
        if (c < 0 || c > INT32_MAX) { *m = nv; return EMIA_COCO_RANGE; }
        cnts[nv++] = c;
        sum += c;
        start = p + 1;
    }
    *m = nv;
    if (start != len) return EMIA_COCO_OPEN_VALUE;
    return sum == hw ? EMIA_COCO_OK : EMIA_COCO_SUM;
}

// the JSON text of every delta xs[k] at out (out_off[n + 1] = byte offsets)
void sim_coco_put_many(const long long* xs, long long n, uint8_t* out, long long* out_off) {
    out_off[0] = 0;
    for (long long k = 0; k < n; ++k) out_off[k + 1] = out_off[k] + emia_coco_put_delta(out + out_off[k], xs[k]);
}

// sequence q = cnts[seq_off[q], seq_off[q + 1]): its string at out[out_off[q], out_off[q + 1]) (out NULL: offsets only)
void sim_coco_encode_many(const long long* cnts, const long long* seq_off, long long nseq, uint8_t* out, long long* out_off) {
    out_off[0] = 0;
    for (long long q = 0; q < nseq; ++q)
        out_off[q + 1] = out_off[q] + sim_coco_encode(cnts + seq_off[q], seq_off[q + 1] - seq_off[q], out ? out + out_off[q] : nullptr);
}

// string q = s[str_off[q], str_off[q + 1]) of a frame of hw[q] pixels: its counts at cnts[str_off[q] ..], m[q] of them, status[q]
void sim_coco_decode_many(const uint8_t* s, const long long* str_off, long long nseq, const long long* hw, long long* cnts,
                          long long* m, int* status) {
    for (long long q = 0; q < nseq; ++q)
        status[q] = sim_coco_decode(s + str_off[q], str_off[q + 1] - str_off[q], hw[q], cnts + str_off[q], m + q);
}

}  // extern "C"
