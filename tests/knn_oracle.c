/*
 * tests/knn_oracle.c -- CPU restatement of K-nearest-neighbour search (pytorch3d knn_points / knn_points_backward,
 * norm=2; parity with pytorch3d itself is unpinned).  TEST INFRASTRUCTURE ONLY, compiled by tests/knn_oracle.py.
 *
 *   - distance: the fp32 operation order of knn1 in oracle/chamfer_oracle.c: d = 0; for c: df = a[c]-b[c];
 *     mode 0: d = d + df*df, mode 1: d = fmaf(df, df, d)   (compile with -ffp-contract=off)
 *   - ranking: the explicit key (distance, index), with every NaN distance ranked after +inf and reported as the NaN
 *     whose bits are 0x7fffffff; the K smallest keys of the first len2 targets, ascending
 *   - padding: slots k >= min(K, len2) and rows i >= len1 are dist 0, idx 0
 *   - backward: for i < len1, k < min(K, len2), j = idx: diff = (2*g) * (p1[i] - p2[j]) per channel,
 *     grad_p1[i] += diff, grad_p2[j] -= diff, sequentially in (n, i, k) order
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__x86_64__) && defined(__GNUC__)
#define PCL_CLONES __attribute__((target_clones("fma", "default")))
#else
#define PCL_CLONES
#endif

static uint64_t key_of(float d, int j) {
    uint32_t b;
    if (d != d) b = 0x7fffffffu;
    else memcpy(&b, &d, 4);
    return ((uint64_t)b << 32) | (uint32_t)j;
}

static float dist_of(uint64_t k) {
    const uint32_t b = (uint32_t)(k >> 32);
    float d;
    memcpy(&d, &b, 4);
    return d;
}

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

/* p1 (B,P1,D), p2 (B,P2,D) with element strides; len1/len2 nullable; list: K uint64 of scratch.  dists/idx (B,P1,K). */
int knn_oracle_forward(const float *p1, long b1, long r1, const int64_t *len1, const float *p2, long b2, long r2,
                       const int64_t *len2, int B, int P1, int P2, int D, int K, int mode, float *dists, int *idx,
                       uint64_t *list) {
    if (B < 0 || P1 < 0 || P2 < 0 || D < 1 || K < 1) return -1;
    memset(dists, 0, sizeof(float) * (size_t)B * P1 * K);
    memset(idx, 0, sizeof(int) * (size_t)B * P1 * K);
    for (int n = 0; n < B; n++) {
        if ((len1 && (len1[n] < 0 || len1[n] > P1)) || (len2 && (len2[n] < 0 || len2[n] > P2))) return -2;
        const int l1 = len1 ? (int)len1[n] : P1, l2 = len2 ? (int)len2[n] : P2;
        const int kv = K < l2 ? K : l2;
        for (int i = 0; i < l1; i++) {
            for (int k = 0; k < K; k++) list[k] = UINT64_MAX;
            const float *a = p1 + n * b1 + i * r1;
            for (int j = 0; j < l2; j++) {
                const uint64_t key = key_of(sqdist(a, p2 + n * b2 + j * r2, D, mode), j);
                if (!(key < list[K - 1])) continue;
                int p = K - 1;
                while (p > 0 && list[p - 1] > key) { list[p] = list[p - 1]; p--; }
                list[p] = key;
            }
            float *dr = dists + ((size_t)n * P1 + i) * K;
            int *ir = idx + ((size_t)n * P1 + i) * K;
            for (int k = 0; k < kv; k++) { dr[k] = dist_of(list[k]); ir[k] = (int)(uint32_t)list[k]; }
        }
    }
    return 0;
}

/* grad_dists (B,P1,K) dense; grad_p1 (B,P1,D), grad_p2 (B,P2,D) dense, overwritten. */
int knn_oracle_backward(const float *p1, long b1, long r1, const int64_t *len1, const float *p2, long b2, long r2,
                        const int64_t *len2, int B, int P1, int P2, int D, int K, const int *idx, const float *grad_dists,
                        float *grad_p1, float *grad_p2) {
    memset(grad_p1, 0, sizeof(float) * (size_t)B * P1 * D);
    memset(grad_p2, 0, sizeof(float) * (size_t)B * P2 * D);
    for (int n = 0; n < B; n++) {
        const int l1 = len1 ? (int)len1[n] : P1, l2 = len2 ? (int)len2[n] : P2;
        const int kv = K < l2 ? K : l2;
        for (int i = 0; i < l1; i++)
            for (int k = 0; k < kv; k++) {
                const size_t r = ((size_t)n * P1 + i) * K + k;
                const int j = idx[r];
                const float g2 = 2.0f * grad_dists[r];
                for (int c = 0; c < D; c++) {
                    const float diff = g2 * (p1[n * b1 + i * r1 + c] - p2[n * b2 + j * r2 + c]);
                    grad_p1[((size_t)n * P1 + i) * D + c] += diff;
                    grad_p2[((size_t)n * P2 + j) * D + c] -= diff;
                }
            }
    }
    return 0;
}
