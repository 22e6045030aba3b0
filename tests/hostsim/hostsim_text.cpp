// hostsim_text.cpp — g++ build of the number formatting core (deepemia_b200/csrc/core/emia_text.cuh) for tests/test_hostsim_text.py.
// TEST INFRASTRUCTURE ONLY: the CPU-only CI checks the shortest digits against std::to_chars and the layouts against Python and
// numpy with the same source the sm_100a kernels execute.  Nothing in deepemia_b200/ loads this.
#include <charconv>
#include <cstring>
#include <random>
#include <thread>
#include <vector>
#include "../../deepemia_b200/csrc/core/emia_text.cuh"

namespace {

// (digits, decimal exponent of the first digit) of std::to_chars' shortest scientific form of a finite nonzero |v|
template <class T>
void ref_digits(T v, char* dig, int* x) {
    char buf[64];
    const auto r = std::to_chars(buf, buf + sizeof(buf), v < 0 ? -v : v, std::chars_format::scientific);
    *r.ptr = 0;
    int n = 0;
    const char* p = buf;
    for (; *p != 'e'; ++p)
        if (*p != '.') dig[n++] = *p;
    dig[n] = 0;
    *x = atoi(p + 1);
}

template <class T>
bool same_as_to_chars(T v) {
    const emia_decimal d = sizeof(T) == 8 ? emia_shortest_f64((double)v) : emia_shortest_f32((float)v);
    char want[32], got[32];
    int x;
    ref_digits(v, want, &x);
    const int n = emia_u64_digits(d.f);
    emia_put_u64((uint8_t*)got, d.f, n);
    got[n] = 0;
    return strcmp(got, want) == 0 && d.e + n - 1 == x;
}

struct Tally {
    long long checked = 0, bad = 0;
    uint64_t first_bad = 0;
};

template <class F>
Tally split(int threads, long long n, F&& body) {
    std::vector<Tally> part(threads);
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; ++t)
        pool.emplace_back([&, t] { body(t, n * t / threads, n * (t + 1) / threads, &part[t]); });
    for (auto& th : pool) th.join();
    Tally all;
    for (auto& p : part) {
        if (p.bad && !all.bad) all.first_bad = p.first_bad;
        all.checked += p.checked;
        all.bad += p.bad;
    }
    return all;
}

}  // namespace

extern "C" {

void sim_shortest_f64(double v, unsigned long long* f, int* e) { const emia_decimal d = emia_shortest_f64(v); *f = d.f; *e = d.e; }
void sim_shortest_f32(float v, unsigned long long* f, int* e) { const emia_decimal d = emia_shortest_f32(v); *f = d.f; *e = d.e; }

// out[k * EMIA_TEXT_NUM_MAX ...] = text of v[k], len[k] = its length; kind 0: repr(float), 1: str(np.float32), 2: str(int)
void sim_format(const double* v, const long long* iv, long long n, int kind, unsigned char* out, int* len) {
    for (long long k = 0; k < n; ++k) {
        uint8_t* o = out + k * EMIA_TEXT_NUM_MAX;
        len[k] = kind == 0 ? emia_format_f64(o, v[k]) : kind == 1 ? emia_format_f32(o, (float)v[k]) : emia_write_i64(o, iv[k]);
    }
}
int sim_i64_len(long long v) { return emia_i64_len(v); }

// float32 bit patterns [lo, hi) with step `step` (finite, nonzero ones) against std::to_chars, split over `threads` threads:
// number checked, number different, first different pattern
long long sim_check_f32(unsigned long long lo, unsigned long long hi, unsigned long long step, int threads, long long* bad,
                        unsigned long long* first_bad) {
    const long long n = (long long)((hi - lo + step - 1) / step);
    const Tally t = split(threads, n, [&](int, long long a, long long b, Tally* r) {
        for (long long i = a; i < b; ++i) {
            const uint32_t bits = (uint32_t)(lo + (unsigned long long)i * step);
            float v;
            memcpy(&v, &bits, 4);
            if (!std::isfinite(v) || v == 0.0f) continue;
            ++r->checked;
            if (!same_as_to_chars(v) && !r->bad++) r->first_bad = bits;
        }
    });
    *bad = t.bad;
    *first_bad = t.first_bad;
    return t.checked;
}

// n uniformly random binary64 bit patterns (finite, nonzero ones) of seed against std::to_chars, split over `threads` threads
long long sim_check_f64_random(unsigned long long seed, long long n, int threads, long long* bad, unsigned long long* first_bad) {
    const Tally t = split(threads, n, [&](int th, long long a, long long b, Tally* r) {
        std::mt19937_64 rng(seed * 1000003ull + (unsigned long long)th);
        for (long long i = a; i < b; ++i) {
            const uint64_t bits = rng();
            double v;
            memcpy(&v, &bits, 8);
            if (!std::isfinite(v) || v == 0.0) continue;
            ++r->checked;
            if (!same_as_to_chars(v) && !r->bad++) r->first_bad = bits;
        }
    });
    *bad = t.bad;
    *first_bad = t.first_bad;
    return t.checked;
}

// the given binary64 values against std::to_chars: index of the first different one, or -1
long long sim_check_f64_list(const double* v, long long n) {
    for (long long k = 0; k < n; ++k)
        if (std::isfinite(v[k]) && v[k] != 0.0 && !same_as_to_chars(v[k])) return k;
    return -1;
}

}  // extern "C"
