/* TEST INFRASTRUCTURE ONLY -- CPU restatement of the K-NN distance backward (b200pci_knn_backward,
 * include/b200pci.h), written as a plain sequential loop in the summation order of the deterministic
 * entry point. Built by tests/knn_grad_oracle.py with -ffp-contract=off, like the oracle: every
 * product and every sum is rounded on its own. The product never loads it.
 */
#include <stddef.h>
#include <stdint.h>

/* q [B,S,3], r [B,N,3], idx [B,S,K] (int64), grad_dist [B,S,K]; gq [B,S,3], gr [B,N,3] overwritten.
 * Slot (i, k) with j = idx[b,i,k] gives d_c = fl(fl(2 grad_dist) * fl(q_c - r_c)), added to gq[i]
 * (k ascending) and subtracted from gr[j] (flat slot t = i*K + k ascending); slots with k >= N or
 * j outside [0, N) give nothing. */
void orc_knn_backward(int B, int S, int N, int K, const float *q, const float *r, const int64_t *idx,
                      const float *grad_dist, float *gq, float *gr) {
    for (size_t t = 0; t < (size_t)B * S * 3; ++t) gq[t] = 0.f;
    for (size_t t = 0; t < (size_t)B * N * 3; ++t) gr[t] = 0.f;
    for (int b = 0; b < B; ++b)
        for (int i = 0; i < S; ++i)
            for (int k = 0; k < K && k < N; ++k) {
                const size_t s = ((size_t)b * S + i) * K + k;
                const int64_t j = idx[s];
                if (j < 0 || j >= N) continue;
                const float g2 = 2.f * grad_dist[s];
                const float *qi = q + ((size_t)b * S + i) * 3, *rj = r + ((size_t)b * N + j) * 3;
                float *gqi = gq + ((size_t)b * S + i) * 3, *grj = gr + ((size_t)b * N + j) * 3;
                for (int c = 0; c < 3; ++c) {
                    const float d = g2 * (qi[c] - rj[c]);
                    gqi[c] += d;
                    grj[c] -= d;
                }
            }
}
