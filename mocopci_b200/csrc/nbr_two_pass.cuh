// The pending-list flavour of the two-pass path, used by ball_query (DESIGN.md "Neighbourhood
// searches"; KNN / three_nn / Chamfer use the scan + evaluate kernel of nbr_scan_tc.cuh):
//
//   scan   (nbr_scan)          the streaming filter with nothing else in the kernel: a warp owns
//                              4 x 32 queries and one split of the refs, and appends one
//                              (step << 8 | 8-group mask) entry per flagged 32-ref step to the
//                              query's pending list in global memory (predicated store, no branch).
//                              The lists keep the flagged steps in ascending ref order, which is
//                              what "the first nsample refs inside the radius" needs.
//   ball_select                one thread per query walks its lists in order, re-evaluates the
//                              flagged groups in the reference arithmetic and stops at nsample hits.
#pragma once
#include "nbr_engine.cuh"

namespace b200pci {

constexpr int SCAN_CAP = 96;  // pending entries per (query, split); a multiple of 4

// ---- pass 1: scan ----------------------------------------------------------------------------
template <int CW, int STAGES>
__device__ __forceinline__ void nbr_scan(const NbrParams &p) {
    constexpr int QT = NBR_QT;
    constexpr int G4 = NBR_TILE / 4;  // float4 per row per stage
    constexpr size_t warp_ring_bytes = (size_t)STAGES * 4 * NBR_TILE * sizeof(float);
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float *tiles = reinterpret_cast<float *>(smem + (size_t)warp * warp_ring_bytes);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + warp_ring_bytes * CW) + warp * STAGES;

    const int b = blockIdx.z, split = blockIdx.y;
    const size_t warp_linear =
        ((size_t)(blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * CW + warp;
    const int tile0 = split * p.tiles_per_split;
    const int ntiles = min(p.tiles_per_split, p.total_tiles - tile0);
    const float *ws = p.ws_ref + (size_t)b * 4 * p.Npad;
    constexpr uint32_t stage_bytes = 4 * NBR_TILE * sizeof(float);

    auto issue_tile = [&](int t) {  // lane 0 of the owning warp
        const int s = t % STAGES;
        mbar_arrive_expect_tx(&full[s], stage_bytes);
#pragma unroll
        for (int r = 0; r < 4; ++r)
            tma_load_1d(tiles + (size_t)(s * 4 + r) * NBR_TILE,
                        ws + (size_t)r * p.Npad + (size_t)(tile0 + t) * NBR_TILE,
                        NBR_TILE * sizeof(float), &full[s]);
    };
    if (lane == 0) {
        for (int s = 0; s < STAGES; ++s) mbar_init(&full[s], 1);
        mbar_fence_init();
        for (int t = 0; t < min(ntiles, STAGES); ++t) issue_tile(t);
    }
    __syncwarp();

    QueryRegs q[QT];
    float thr[QT];
    int cnt[QT];
    const int qi0 = (blockIdx.x * CW + warp) * (QT * 32) + lane;  // slot j: + 32 * j
    uint32_t *pend = p.pend + warp_linear * (size_t)(QT * SCAN_CAP * 32) + lane * 4;
#pragma unroll
    for (int j = 0; j < QT; ++j) {
        const int qi = qi0 + 32 * j;
        float x = 0.f, y = 0.f, z = 0.f, t0 = __int_as_float(0xff800000);  // -inf: never flagged
        if (qi < p.S) {
            const float *src = p.q + b * p.q_sb + qi * p.q_sp;
            x = src[p.q_ox];
            y = src[p.q_oy];
            z = src[2 * p.q_sc];
            t0 = p.tau_in ? p.tau_in[(size_t)b * p.S + qi] : p.tau_uniform;
        }
        q[j].set(x, y, z);
        thr[j] = q[j].threshold(t0);
        cnt[j] = 0;
    }

    constexpr int SPT = G4 / NBR_BLK;  // steps per tile
#pragma unroll 1
    for (int t = 0; t < ntiles; ++t) {
        const int s = t % STAGES;
        mbar_wait(&full[s], (t / STAGES) & 1);
        const float4 *sX = reinterpret_cast<const float4 *>(tiles + (size_t)(s * 4) * NBR_TILE);
        float4 X = sX[0], Y = sX[G4], Z = sX[2 * G4], W = sX[3 * G4];
        uint32_t ent = (uint32_t)((tile0 + t) * SPT) << 8;
#pragma unroll 1
        for (int g0 = 0; g0 < G4; g0 += NBR_BLK) {
            const float4 *gX = sX + g0;
            uint32_t m8[QT];
#pragma unroll
            for (int j = 0; j < QT; ++j) m8[j] = 0u;
#pragma unroll
            for (int u = 0; u < NBR_BLK; ++u) {
                const float4 cX = X, cY = Y, cZ = Z, cW = W;
                // prefetch the next group (one group past the tile at the very end: harmless,
                // still inside this CTA's shared memory, never used)
                X = gX[u + 1];
                Y = gX[G4 + u + 1];
                Z = gX[2 * G4 + u + 1];
                W = gX[3 * G4 + u + 1];
#pragma unroll
                for (int j = 0; j < QT; ++j)
                    if (filter4(q[j], cX, cY, cZ, cW) < thr[j]) m8[j] |= (0x80u >> u);
            }
#pragma unroll
            for (int j = 0; j < QT; ++j) {
                if (m8[j] != 0u && cnt[j] < SCAN_CAP)
                    pend[j * (SCAN_CAP * 32) + nbr_pend_off(cnt[j])] = ent | m8[j];
                if (m8[j] != 0u) ++cnt[j];  // keeps counting past the capacity: overflow marker
            }
            ent += 1u << 8;
        }
        // this warp is done with the stage: refill it with the tile STAGES ahead
        __syncwarp();
        if (lane == 0 && t + STAGES < ntiles) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            issue_tile(t + STAGES);
        }
    }
    uint32_t *pc = p.pend_cnt + warp_linear * (QT * 32) + lane;
#pragma unroll
    for (int j = 0; j < QT; ++j) pc[j * 32] = (uint32_t)cnt[j];
}

// ---- ball query on the two-pass path -----------------------------------------------------------
// pointnet2/src/ball_query_gpu.cu:30-44: the first `nsample` refs (ascending index) with
// d2 < radius^2; the first hit fills every slot first; idx is pre-zeroed by the caller.
// The scan runs with the uniform bound radius^2; one thread per query then walks its lists in
// order and stops at nsample hits. A query whose list overflowed before nsample hits were
// found (possible only with > SCAN_CAP flagged steps in one split) is redone by a warp that scans
// the whole cloud in order.
struct BallSelectParams {
    int *idx;  // [B,S,nsample]
    int nsample;
    float radius2;
    int *fail_count;
    int *fail_list;
    int scan_tiles;
    int force_redo;  // test hook: send every query through the exact redo kernel
};

static __global__ void __launch_bounds__(128) ball_select_kernel(NbrParams p, BallSelectParams sp) {
    const int tid = threadIdx.x, lane = tid & 31, j = tid >> 5;
    const int b = blockIdx.z;
    const int qi = blockIdx.x * 128 + tid;
    const bool valid = qi < p.S;
    QueryRegs q;
    {
        float x = 0.f, y = 0.f, z = 0.f;
        if (valid) {
            const float *src = p.q + b * p.q_sb + qi * p.q_sp;
            x = src[p.q_ox];
            y = src[p.q_oy];
            z = src[2 * p.q_sc];
        }
        q.set(x, y, z);
    }
    const float *grp = p.ws_grp + (size_t)b * 4 * p.Npad;
    const int ns = sp.nsample;
    const float r2 = sp.radius2;
    int *row = sp.idx + ((size_t)b * p.S + (valid ? qi : 0)) * ns;
    int found = valid ? 0 : ns;
    bool must_redo = false;
    for (int s = 0; s < p.nsplit; ++s) {
        const size_t warp_linear = ((size_t)(b * p.nsplit + s) * sp.scan_tiles + blockIdx.x);
        int cnt = valid ? (int)p.pend_cnt[warp_linear * (NBR_QT * 32) + j * 32 + lane] : 0;
        // A split whose list overflowed has lost its LAST flagged steps. If its surviving entries do
        // not complete the query, hits of this split (lower indices than anything a later split
        // holds) may be missing: the query is redone exactly and consumes no later split.
        const bool capped = cnt > SCAN_CAP;
        if (capped) cnt = SCAN_CAP;
        const uint32_t *list =
            p.pend + warp_linear * (size_t)(NBR_QT * SCAN_CAP * 32) + j * (SCAN_CAP * 32) + lane * 4;
        int e = 0;
        uint32_t m8 = 0u, gs = 0u;
        while (true) {
            if (m8 == 0u && e < cnt && found < ns) {
                const uint32_t ent = list[nbr_pend_off(e)];
                m8 = ent & 0xffu;
                gs = ent >> 8;
                ++e;
            }
            const bool has = m8 != 0u && found < ns;
            if (!__any_sync(0xffffffffu, has)) break;
            const int bit = has ? (31 - __clz((int)m8)) : 0;  // highest bit = lowest group
            m8 &= ~(1u << bit);
            const uint32_t gid = has ? gs * NBR_BLK + (uint32_t)(7 - bit) : 0u;
            float4 X, Y, Z, Wn;
            ldg256(grp + (size_t)gid * 16, X, Y);
            ldg256(grp + (size_t)gid * 16 + 8, Z, Wn);
            float d[4];
            dist4<B200PCI_DIST_DIRECT>(q, X, Y, Z, gid * 4u, p.N, d);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (has && d[i] < r2 && found < ns) {
                    if (found == 0)
                        for (int l = 0; l < ns; ++l) row[l] = (int)(gid * 4u + i);
                    row[found] = (int)(gid * 4u + i);
                    ++found;
                }
            }
        }
        if (capped && found < ns) {
            must_redo = true;
            found = ns;  // this lane is done (stays in the loop only for the warp-wide votes)
        }
    }
    if (valid && (must_redo || sp.force_redo))
        sp.fail_list[atomicAdd(sp.fail_count, 1)] = (int)((size_t)b * p.S + qi);
}

// exact redo: one warp per failed query scans the packed rows in index order
static __global__ void __launch_bounds__(128) ball_fallback_kernel(NbrParams p, BallSelectParams sp) {
    const int lane = threadIdx.x & 31;
    const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    const int nfail = *sp.fail_count;
    const int ns = sp.nsample;
    for (int f = wid; f < nfail; f += nw) {
        const int qrow = sp.fail_list[f];
        const int b = qrow / p.S, qi = qrow - b * p.S;
        const float *src = p.q + b * p.q_sb + qi * p.q_sp;
        const float qx = src[0], qy = src[p.q_sc], qz = src[2 * p.q_sc];
        const float *ws = p.ws_ref + (size_t)b * 4 * p.Npad;
        int *row = sp.idx + (size_t)qrow * ns;
        int found = 0;
        for (int base = 0; base < p.N && found < ns; base += 32) {
            const int k = base + lane;
            bool hit = false;
            if (k < p.N) {
                const float dx = __fsub_rn(ws[k], qx), dy = __fsub_rn(ws[p.Npad + k], qy),
                            dz = __fsub_rn(ws[2 * (size_t)p.Npad + k], qz);
                hit = __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy))) < sp.radius2;
            }
            const unsigned m = __ballot_sync(0xffffffffu, hit);
            if (m == 0u) continue;
            if (found == 0) {
                const int first = base + __ffs(m) - 1;
                for (int l = lane; l < ns; l += 32) row[l] = first;
                __syncwarp();
            }
            const int pos = found + __popc(m & ((1u << lane) - 1u));
            if (hit && pos < ns) row[pos] = k;
            found += __popc(m);
        }
        __syncwarp();
    }
}

}  // namespace b200pci
