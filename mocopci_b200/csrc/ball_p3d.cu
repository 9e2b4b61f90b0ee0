// Ball query in pytorch3d's form (pytorch3d.ops.ball_query; b200pci_ball_query_p3d).
//
// One warp per query; the 8 warps of a CTA take 8 consecutive queries of one cloud, so they stream
// the same refs through L1. The warp walks the refs j < lengths2[b] in ascending order, 128 per
// round (4 coalesced loads per lane issued before any test): each lane evaluates
// d2 = fma(dz,dz,fma(dy,dy,dx*dx)), d = p1 - p2 (pytorch3d's `dist2 += diff * diff` as nvcc
// contracts it), a ballot ranks the hits (d2 < radius^2, strict) in ref order and the lanes write
// them to consecutive slots. The warp stops at the end of the round in which it reached K hits;
// later hits of that round fail the slot bound. Then the lanes pad slots found..K-1 with (-1, 0)
// and, when asked, zero rows of nn. Queries i >= lengths1[b] get padding only. lengths are read
// here, on the device, and clamped to [0, P]: the call needs no host synchronisation.
#include "common.cuh"

namespace b200pci {

constexpr int BQ3_WARPS = 8;
constexpr int BQ3_ROUND = 4;  // 32-ref steps per round

struct Bq3Args {
    int P1, P2, K;
    float r2;
    const float *p1;
    long long p1_sb, p1_sp, p1_sc;
    const float *p2;
    long long p2_sb, p2_sp, p2_sc;
    const long long *len1, *len2;  // [B], nullable
    long long *idx;                // [B, P1, K]
    float *dists;                  // [B, P1, K]
    float *nn;                     // [B, P1, K, 3], nullable
};

static __device__ __forceinline__ int clamp_len(const long long *len, int b, int P) {
    if (len == nullptr) return P;
    const long long v = len[b];
    return (int)(v < 0 ? 0 : (v > P ? P : v));
}

static __global__ void __launch_bounds__(BQ3_WARPS * 32) ball_query_p3d_kernel(Bq3Args a) {
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * BQ3_WARPS + (threadIdx.x >> 5);
    const int b = blockIdx.y;
    if (i >= a.P1) return;  // whole warps
    const int n1 = clamp_len(a.len1, b, a.P1), n2 = clamp_len(a.len2, b, a.P2);
    const size_t row = ((size_t)b * a.P1 + i) * a.K;
    const int K = a.K;
    int found = 0;
    if (i < n1) {
        const float *q = a.p1 + b * a.p1_sb + i * a.p1_sp;
        const float qx = q[0], qy = q[a.p1_sc], qz = q[2 * a.p1_sc];
        const float *rb = a.p2 + b * a.p2_sb;
        for (int base = 0; base < n2 && found < K; base += 32 * BQ3_ROUND) {
            float rx[BQ3_ROUND], ry[BQ3_ROUND], rz[BQ3_ROUND];
#pragma unroll
            for (int u = 0; u < BQ3_ROUND; ++u) {
                const int j = base + 32 * u + lane;
                rx[u] = ry[u] = rz[u] = 0.f;
                if (j < n2) {
                    const float *r = rb + j * a.p2_sp;
                    rx[u] = __ldg(r);
                    ry[u] = __ldg(r + a.p2_sc);
                    rz[u] = __ldg(r + 2 * a.p2_sc);
                }
            }
#pragma unroll
            for (int u = 0; u < BQ3_ROUND; ++u) {
                const int j = base + 32 * u + lane;
                const float dx = __fsub_rn(qx, rx[u]), dy = __fsub_rn(qy, ry[u]), dz = __fsub_rn(qz, rz[u]);
                const float d2 = __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
                const bool hit = j < n2 && d2 < a.r2;
                const unsigned m = __ballot_sync(0xffffffffu, hit);
                const int pos = found + __popc(m & ((1u << lane) - 1u));
                if (hit && pos < K) {
                    a.idx[row + pos] = j;
                    a.dists[row + pos] = d2;
                    if (a.nn) {
                        float *o = a.nn + (row + pos) * 3;
                        o[0] = rx[u];
                        o[1] = ry[u];
                        o[2] = rz[u];
                    }
                }
                found += __popc(m);
            }
        }
        found = min(found, K);
    }
    for (int s = found + lane; s < K; s += 32) {
        a.idx[row + s] = -1;
        a.dists[row + s] = 0.f;
        if (a.nn) {
            float *o = a.nn + (row + s) * 3;
            o[0] = o[1] = o[2] = 0.f;
        }
    }
}

}  // namespace b200pci

using namespace b200pci;

extern "C" int b200pci_ball_query_p3d(int B, int P1, int P2, int K, float radius, const float *p1,
                                      int64_t p1_sb, int64_t p1_sp, int64_t p1_sc, const float *p2,
                                      int64_t p2_sb, int64_t p2_sp, int64_t p2_sc,
                                      const int64_t *lengths1, const int64_t *lengths2, int64_t *idx,
                                      float *dists, float *nn, void *stream) {
    B200PCI_CHECK_ARG(B >= 0 && P1 >= 0 && P2 >= 0, "ball_query_p3d: negative size");
    B200PCI_CHECK_ARG(K >= 1, "ball_query_p3d: K must be >= 1");
    B200PCI_CHECK_ARG(radius >= 0.f, "ball_query_p3d: radius must be >= 0 (and not NaN)");
    if (B == 0 || P1 == 0) return B200PCI_OK;
    B200PCI_CHECK_ARG(p1 && idx && dists && (p2 || P2 == 0), "ball_query_p3d: null pointer");
    B200PCI_CHECK_ARG(B <= 65535, "ball_query_p3d: batch too large");
    Bq3Args a;
    a.P1 = P1;
    a.P2 = P2;
    a.K = K;
    a.r2 = radius * radius;  // FP32, as pytorch3d's kernel squares its float radius
    a.p1 = p1;
    a.p1_sb = p1_sb;
    a.p1_sp = p1_sp;
    a.p1_sc = p1_sc;
    a.p2 = p2;
    a.p2_sb = p2_sb;
    a.p2_sp = p2_sp;
    a.p2_sc = p2_sc;
    a.len1 = reinterpret_cast<const long long *>(lengths1);
    a.len2 = reinterpret_cast<const long long *>(lengths2);
    a.idx = reinterpret_cast<long long *>(idx);
    a.dists = dists;
    a.nn = nn;
    dim3 grid((unsigned)((P1 + BQ3_WARPS - 1) / BQ3_WARPS), (unsigned)B);
    ball_query_p3d_kernel<<<grid, BQ3_WARPS * 32, 0, (cudaStream_t)stream>>>(a);
    B200PCI_LAUNCH_CHECK("ball_query_p3d_kernel");
    return B200PCI_OK;
}
