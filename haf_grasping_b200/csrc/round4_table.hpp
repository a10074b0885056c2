// "%.4g" decision table of the fast feature tier (kernels.cuh, fast_tier_value), built on the host and staged in shared
// memory by features_tc_kernel.  Plain C++ so that tests/round4_table_check.cpp checks this very table.
//
// The decimal exponent E of a float a = |raw| depends only on its biased binary exponent b (b = 0, subnormals and +-0,
// counts as b = 1) and on one comparison:
//     E0(b) = floor(log10 2^(b - 127)) = ((max(b, 1) - 127) * 1233) >> 12      (exact for every b in 1..254)
//     E     = E0(b) + (a >= thr[b]),  thr[b] = 10^(E0(b) + 1) rounded to float
// so the kernel reads thr[b], then the two scale factors of (b, side): a * 10^(3 - E) is rounded in double and the result
// scaled back by 10^(E - 3) in float.  b = 255 (inf / NaN) gets the entry the same formula gives it.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstddef>

struct Round4Tab {
    double mul[256][2];   // 10^(3 - E) for binade b and side s (E = E0(b) + s)
    float inv[256][2];    // 10^(E - 3) as float
    float thr[256];       // 10^(E0(b) + 1) as float: s = (a >= thr[b])
};
static_assert(sizeof(Round4Tab) == 256 * 2 * 8 + 256 * 2 * 4 + 256 * 4, "Round4Tab layout");
static_assert(sizeof(Round4Tab) % 16 == 0, "the tile behind the table must stay 16-byte aligned");

inline int round4_e0(int b) { return ((std::max(b, 1) - 127) * 1233) >> 12; }

inline void make_round4_table(Round4Tab& tab) {
    for (int b = 0; b < 256; b++) {
        const int e0 = round4_e0(b);
        tab.thr[b] = (float)pow(10.0, e0 + 1);
        for (int s = 0; s < 2; s++) {
            tab.mul[b][s] = pow(10.0, 3 - (e0 + s));
            tab.inv[b][s] = (float)pow(10.0, (e0 + s) - 3);
        }
    }
}
