// CPU check of the fast tier's "%.4g" decision table (haf_grasping_b200/csrc/round4_table.hpp) against the formula the
// feature kernel used before it: for every one of the 2^32 float bit patterns of raw, the record lookup
//     b = exponent byte, s = |raw| >= thr[b], (mul, inv) = table[b][s]
// must give the same decimal exponent E, the same mul / inv bits and the same rounded value v as
//     E = floor(log10 2^k) by multiply-shift, + (|raw| >= 10^(E+1)), mul = 10^(3-E), inv = 10^(E-3) from power tables.
// usage: round4_table_check [n_threads]   -> prints "mismatches=<k> checked=<n>", exit status 1 on any mismatch
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>
#include "../haf_grasping_b200/csrc/round4_table.hpp"

static double pwd[96];
static float pwf[96];
static Round4Tab tab;
static std::atomic<long> mism{0}, checked{0};

static uint32_t fbits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
static uint64_t dbits(double d) { uint64_t u; memcpy(&u, &d, 8); return u; }

static void slice(uint64_t part, uint64_t nparts) {
    long bad = 0, n = 0;
    for (uint64_t i = part; i < (1ull << 32); i += nparts) {
        const uint32_t bits = (uint32_t)i;
        float raw; memcpy(&raw, &bits, 4);
        const float a = fabsf(raw);
        // the previous formula (kernels.cuh before the table)
        int E = ((std::max((int)(fbits(a) >> 23), 1) - 127) * 1233) >> 12;
        E += (a >= pwf[48 + E + 1]) ? 1 : 0;
        const double mul0 = pwd[48 + 3 - E];
        const float inv0 = pwf[48 + E - 3];
        const float v0 = copysignf((float)rint((double)a * mul0) * inv0, raw);
        // the record lookup (fast_tier_value)
        const uint32_t b = (bits >> 23) & 0xffu;
        const uint32_t s = (a >= tab.thr[b]) ? 1u : 0u;
        const int E1 = round4_e0((int)b) + (int)s;
        const double mul1 = tab.mul[b][s];
        const float inv1 = tab.inv[b][s];
        const float v1 = copysignf((float)rint((double)a * mul1) * inv1, raw);
        n++;
        if (E != E1 || dbits(mul0) != dbits(mul1) || fbits(inv0) != fbits(inv1) || fbits(v0) != fbits(v1)) {
            if (bad < 10) printf("MISMATCH raw=%a bits=%08x E %d/%d mul %a/%a inv %a/%a v %a/%a\n", raw, bits, E, E1, mul0, mul1,
                                 inv0, inv1, v0, v1);
            bad++;
        }
    }
    mism += bad;
    checked += n;
}

int main(int argc, char** argv) {
    for (int i = 0; i < 96; i++) { pwd[i] = pow(10.0, i - 48); pwf[i] = (float)pwd[i]; }
    make_round4_table(tab);
    const int nt = argc > 1 ? std::max(1, atoi(argv[1])) : 8;
    std::vector<std::thread> th;
    for (int t = 0; t < nt; t++) th.emplace_back(slice, (uint64_t)t, (uint64_t)nt);
    for (auto& t : th) t.join();
    printf("mismatches=%ld checked=%ld\n", mism.load(), checked.load());
    return mism.load() != 0 || checked.load() != (1l << 32);
}
