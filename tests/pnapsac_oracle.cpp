/*
 * pnapsac_oracle.cpp - sequential Progressive NAPSAC sampler as DESIGN.md section 4.8 defines it: the reference the tests of
 * USAC_SAMPLER_PROGRESSIVE_NAPSAC compare against. TEST INFRASTRUCTURE ONLY, built by pnapsac_oracle.py into a temporary directory
 * together with the unmodified oracle sources (oracle/), whose Philox draws (orc_philox_unique) it uses. The reference tree has no
 * meaning to follow here: its progressive_sampler.hpp:149-172 never fills its sample.
 *
 * One stream, hypotheses 0 .. count-1 in order, with its own per-centre use counts u[] (all zero at hypothesis 0):
 *   h >= length: the uniform sampler's sample, orc_philox_unique(seed, h, 0, n, m);
 *   else centre p = orc_philox_unique(seed, h, 5, n, 1), t = ++u[p], s = min(k, min{s' >= m-1 : C(s', m-1) >= t}),
 *        sample = p, knn[p][j_1 .. j_{m-2}] with j = orc_philox_unique(seed, h, 6, s-1, m-2), then knn[p][s-1].
 */
#include <stdint.h>

#include <vector>

#include "../oracle/usac_oracle.h"

/* C(s, r) for the smallest s >= r with C(s, r) >= t, capped at k; the coefficients are built up from C(r, r) = 1 */
static int pnapsac_size(unsigned long long t, int r, int k) {
    int s = r;
    unsigned long long c = 1;
    while (s < k && c < t) {
        s++;
        c = c * (unsigned long long)s / (unsigned long long)(s - r);
    }
    return s;
}

/* out: count x m indices; knn: n x k, ascending distance */
extern "C" void pnapsac_table(uint64_t seed, int n, int m, const int* knn, int k, unsigned long long length, int count, int* out) {
    std::vector<unsigned> uses((size_t)n, 0u);
    for (int h = 0; h < count; h++) {
        int* smp = out + (size_t)h * m;
        if ((unsigned long long)h >= length) {
            orc_philox_unique(seed, (uint64_t)h, 0, n, m, smp);
            continue;
        }
        int p;
        orc_philox_unique(seed, (uint64_t)h, 5, n, 1, &p);
        const unsigned t = ++uses[(size_t)p];
        const int s = pnapsac_size(t, m - 1, k);
        const int* row = knn + (size_t)k * p;
        smp[0] = p;
        if (m > 2) {
            int j[8];
            orc_philox_unique(seed, (uint64_t)h, 6, s - 1, m - 2, j);
            for (int i = 0; i < m - 2; i++) smp[1 + i] = row[j[i]];
        }
        smp[m - 1] = row[s - 1];
    }
}
