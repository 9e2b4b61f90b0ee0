// Backward of b200pci_knn's distances, the per-query half shared by the atomic kernel (knn.cu) and
// the deterministic one (scatter.cu): one thread owns query (b, i) and walks its K slots in
// ascending k, so grad_q gets the same bits from both entry points (include/b200pci.h).
#pragma once

#include "common.cuh"

namespace b200pci {

struct KnnGradArgs {
    int S, N, K;
    const float *q;
    int64_t q_sb, q_sp, q_sc;
    const float *r;
    int64_t r_sb, r_sp, r_sc;
    const float *grad_dist;  // [B,S,K] contiguous
    float *grad_q;           // [B,S,3] contiguous, overwritten
};

// d(i,k)_c = fl(fl(2 grad_dist) * fl(q_c - r_c)); grad_q[b,i,c] = ((0 + d(i,0)_c) + d(i,1)_c) + ...
// `emit(j, dx, dy, dz)` receives each live slot's terms (the atomic kernel subtracts them from grad_r).
// A slot is dead when k >= N (the (inf, 0) padding of the DIRECT modes) or j is outside [0, N).
template <typename I, typename Emit>
__device__ __forceinline__ void knn_grad_query(const KnnGradArgs &a, int b, int i, const I *__restrict__ idx,
                                               Emit emit) {
    const float *qi = a.q + b * a.q_sb + i * a.q_sp;
    const float qx = __ldg(qi), qy = __ldg(qi + a.q_sc), qz = __ldg(qi + 2 * a.q_sc);
    const size_t row = ((size_t)b * a.S + i) * a.K;
    const int live = min(a.K, a.N);
    float ax = 0.f, ay = 0.f, az = 0.f;
    for (int k = 0; k < live; ++k) {
        const long long j = (long long)__ldg(idx + row + k);
        if (j < 0 || j >= a.N) continue;
        const float g2 = __fmul_rn(2.f, __ldg(a.grad_dist + row + k));
        const float *rj = a.r + b * a.r_sb + j * a.r_sp;
        const float dx = __fmul_rn(g2, __fsub_rn(qx, __ldg(rj)));
        const float dy = __fmul_rn(g2, __fsub_rn(qy, __ldg(rj + a.r_sc)));
        const float dz = __fmul_rn(g2, __fsub_rn(qz, __ldg(rj + 2 * a.r_sc)));
        ax = __fadd_rn(ax, dx);
        ay = __fadd_rn(ay, dy);
        az = __fadd_rn(az, dz);
        emit(j, dx, dy, dz);
    }
    float *gq = a.grad_q + ((size_t)b * a.S + i) * 3;
    gq[0] = ax;
    gq[1] = ay;
    gq[2] = az;
}

// Argument checks of both entry points. Returns non-zero for an error; with B200PCI_OK, *nothing
// says whether there is nothing to write (B = 0, or S = N = 0).
static inline int knn_grad_check(int B, int S, int N, int K, const float *q, const float *r, const void *idx,
                                 const float *grad_dist, const float *grad_q, const float *grad_r,
                                 const char *what, bool *nothing) {
    *nothing = false;
    B200PCI_CHECK_ARG(B >= 0 && S >= 0 && N >= 0 && K >= 0, "%s: negative size", what);
    if (B == 0 || (S == 0 && N == 0)) {
        *nothing = true;
        return B200PCI_OK;
    }
    B200PCI_CHECK_ARG(q && r && idx && grad_dist && grad_q && grad_r, "%s: null pointer", what);
    B200PCI_CHECK_ARG(B <= 65535, "%s: batch too large", what);
    B200PCI_CHECK_ARG((long long)S * K < (1LL << 31), "%s: 2^31 or more slots (S*K) per cloud", what);
    return B200PCI_OK;
}

}  // namespace b200pci
