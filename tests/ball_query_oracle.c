/*
 * tests/ball_query_oracle.c -- CPU restatement of ball query (pytorch3d ball_query, restated from memory; parity with
 * pytorch3d itself is unpinned).  TEST INFRASTRUCTURE ONLY, compiled by tests/ball_query_oracle.py.
 *
 *   - distance: the fp32 operation order of tests/knn_oracle.c: d = 0; for c: df = a[c]-b[c];
 *     mode 0: d = d + df*df, mode 1: d = fmaf(df, df, d)   (compile with -ffp-contract=off)
 *   - for a query i < len1: targets j = 0 .. len2-1 in ascending order, kept when d < radius2 (strict; NaN never kept);
 *     the first K kept fill slots 0.. with (d, j)
 *   - padding: the remaining slots and rows i >= len1 are dist 0, idx -1
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__x86_64__) && defined(__GNUC__)
#define PCL_CLONES __attribute__((target_clones("fma", "default")))
#else
#define PCL_CLONES
#endif

PCL_CLONES
static float sqdist(const float *a, const float *b, int D, int mode) {
    float d = 0.f;
    if (mode == 0) {
        for (int c = 0; c < D; c++) { const float df = a[c] - b[c]; d = d + df * df; }
    } else {
        for (int c = 0; c < D; c++) { const float df = a[c] - b[c]; d = fmaf(df, df, d); }
    }
    return d;
}

/* p1 (B,P1,D), p2 (B,P2,D) with element strides; len1/len2 nullable.  dists/idx (B,P1,K). */
int ball_query_oracle_forward(const float *p1, long b1, long r1, const int64_t *len1, const float *p2, long b2, long r2,
                              const int64_t *len2, int B, int P1, int P2, int D, int K, float radius2, int mode,
                              float *dists, int *idx) {
    if (B < 0 || P1 < 0 || P2 < 0 || D < 1 || K < 1) return -1;
    for (size_t e = 0; e < (size_t)B * P1 * K; e++) { dists[e] = 0.f; idx[e] = -1; }
    for (int n = 0; n < B; n++) {
        if ((len1 && (len1[n] < 0 || len1[n] > P1)) || (len2 && (len2[n] < 0 || len2[n] > P2))) return -2;
        const int l1 = len1 ? (int)len1[n] : P1, l2 = len2 ? (int)len2[n] : P2;
        for (int i = 0; i < l1; i++) {
            const float *a = p1 + n * b1 + i * r1;
            float *dr = dists + ((size_t)n * P1 + i) * K;
            int *ir = idx + ((size_t)n * P1 + i) * K;
            int c = 0;
            for (int j = 0; j < l2 && c < K; j++) {
                const float d = sqdist(a, p2 + n * b2 + j * r2, D, mode);
                if (d < radius2) { dr[c] = d; ir[c] = j; c++; }
            }
        }
    }
    return 0;
}
