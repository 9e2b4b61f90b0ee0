/* TEST INFRASTRUCTURE ONLY -- CPU restatement of b200pci_ball_query_p3d and b200pci_fps_p3d
 * (include/b200pci.h, P1 / P2) as plain sequential loops. Built by tests/p3d_oracle.py with
 * -ffp-contract=off, like the oracle: the only fused operations are the explicit fmaf calls of the
 * distance fma(dz,dz,fma(dy,dy,dx*dx)). The product never loads it.
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

static int clamp_len(const int64_t *len, int b, int P) {
    const int64_t v = len[b];
    return (int)(v < 0 ? 0 : (v > P ? P : v));
}

static float dist_xyz(const float *a, const float *b) {
    const float dx = a[0] - b[0], dy = a[1] - b[1], dz = a[2] - b[2];
    return fmaf(dz, dz, fmaf(dy, dy, dx * dx));
}

/* p1 [B,P1,3], p2 [B,P2,3] contiguous; lengths1 / lengths2 [B]; idx [B,P1,K], dists [B,P1,K]. */
void orc_ball_query_p3d(int B, int P1, int P2, int K, float radius, const float *p1, const float *p2,
                        const int64_t *lengths1, const int64_t *lengths2, int64_t *idx, float *dists) {
    const float r2 = radius * radius;
    for (int b = 0; b < B; ++b) {
        const int n1 = clamp_len(lengths1, b, P1), n2 = clamp_len(lengths2, b, P2);
        for (int i = 0; i < P1; ++i) {
            const size_t row = ((size_t)b * P1 + i) * K;
            int found = 0;
            if (i < n1)
                for (int j = 0; j < n2 && found < K; ++j) {
                    const float d2 = dist_xyz(p1 + ((size_t)b * P1 + i) * 3, p2 + ((size_t)b * P2 + j) * 3);
                    if (d2 < r2) {
                        idx[row + found] = j;
                        dists[row + found] = d2;
                        ++found;
                    }
                }
            for (int s = found; s < K; ++s) {
                idx[row + s] = -1;
                dists[row + s] = 0.f;
            }
        }
    }
}

/* points [B,P,3] contiguous; lengths, K, start [B]; idx [B,M]. mind: scratch of P floats. */
void orc_fps_p3d(int B, int P, int M, const float *points, const int64_t *lengths, const int64_t *K,
                 const int64_t *start, int64_t *idx, float *mind) {
    for (int b = 0; b < B; ++b) {
        const float *pts = points + (size_t)b * P * 3;
        const int n = clamp_len(lengths, b, P);
        const int64_t kb = K[b] < 0 ? 0 : (K[b] > M ? M : K[b]);
        const int m = (int)(kb < n ? kb : n);
        int64_t *out = idx + (size_t)b * M;
        for (int t = 0; t < M; ++t) out[t] = -1;
        if (m == 0) continue;
        int last = (int)(start[b] < 0 ? 0 : (start[b] >= n ? n - 1 : start[b]));
        out[0] = last;
        for (int j = 0; j < n; ++j) mind[j] = INFINITY;
        for (int t = 1; t < m; ++t) {
            int best = 0;
            float bestd = -1.f;
            for (int j = 0; j < n; ++j) {
                const float d = fminf(dist_xyz(pts + (size_t)j * 3, pts + (size_t)last * 3), mind[j]);
                mind[j] = d;
                if (d > bestd) { /* strict: the lowest index keeps a tie */
                    bestd = d;
                    best = j;
                }
            }
            last = best;
            out[t] = last;
        }
    }
}
