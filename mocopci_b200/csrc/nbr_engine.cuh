// Shared building blocks of the neighbourhood searches (KNN, three_nn, ball_query, Chamfer) and the
// in-kernel streaming engine (DESIGN.md "Neighbourhood searches"):
//
//   * nbr_pack_refs_kernel: converts the reference cloud once to SoA rows [B][4][Npad] (x, y, z and
//     a filter addend derived from |r|^2; streamed by the scans) plus one 64-byte record per group
//     of 4 refs (gathered by exact evaluations), padded with sentinels that can never be selected;
//   * QueryRegs / filter4 / dist4: the conservative 3-FFMA2 filter and the exact 4-ref distance in
//     the reference arithmetic of either form;
//   * sort16 / bitonic_merge16 / merge_low16 / merge_full16: sorting networks on 64-bit keys
//     (sortable(distance) << 32 | index: the lowest index wins ties) held in registers;
//   * nbr_stream + TopKSink: the single-kernel engine (scan + pending lists in global memory +
//     drains + sorting-network folds) that serves k = 33..64 and the exact mode of the test hooks.
//     The big cases run on nbr_scan_tc.cuh (scan + evaluate) and nbr_topk.cuh (top-k), ball_query
//     on nbr_two_pass.cuh, the small ones on knn_mid_kernel (knn.cu).
//
// In-kernel engine: a warp owns QT*32 queries (4 per thread, in registers) of one cloud and one
// split of the refs. It streams the 128-ref tiles of the SoA rows through its OWN small
// shared-memory ring filled by 1-D TMA bulk copies; a group of 4 refs is read with broadcast
// LDS.128 and run through the filter against the thread's 4 queries; flagged groups are appended
// to the query's pending list in global memory ([entry/4][lane][4] per query slot). A DRAIN
// re-evaluates the pending groups exactly (four entries per round trip) and folds the candidates
// into the sorted best-K with the sorting networks; the best-K lives in L2 between folds.
#pragma once
#include "common.cuh"

namespace b200pci {

typedef unsigned long long u64;

constexpr int NBR_TILE = 128;      // refs per shared-memory stage (32 groups of 4)
constexpr int NBR_QT = 4;          // queries per thread
constexpr int NBR_BLK = 8;         // groups per scan step
constexpr int NBR_CAP = 64;        // pending entries per query slot (global memory)
constexpr int NBR_SAMPLE_STRIDE = 8;  // the threshold pre-pass looks at every 8th ref

// Passed by value to the search kernels. Its size is above 128 bytes, and that matters: nvcc
// lowers the reads of a by-value kernel argument of at most 128 bytes differently, which
// reschedules every kernel that takes one (knn_scan_tc_kernel<0>, issue-bound: 1392 instead of
// 1368 SASS instructions when this struct was 128 bytes).
struct NbrParams {
    int S, N, Npad;
    int nsplit, tiles_per_split, total_tiles;
    const float *q;
    long long q_sb, q_sp, q_sc;
    int q_xzy, r_xzy;      // |q|^2 / |r|^2 summed as (x^2 + z^2) + y^2 (see nbr_sqnorm)
    long long q_ox, q_oy;  // element offsets of the query's first / second coordinate: (0, q_sc), or
                           // (q_sc, 0) for DIST_DIRECT_XYZ (the kernels then see x and y swapped)
    const float *ws_ref;  // [B][4][Npad] rows (streamed by the scan)
    const float *ws_grp;  // [B][Npad/4][4][4] the same refs, one 64-byte record per group of 4
                          // (x[4] y[4] z[4] w[4]): what a drain gathers, 2 sectors per group
    const float *ws_tc;   // tensor-core scan: [B][Npad][16] split-TF32 operand, then the exact |r|^2
                          // rows [B][Npad] (nbr_pack_tc_kernel)
    const float *tau_in;  // two-pass scans: [B][S] admission bounds (null: tau_uniform for every query)
    float tau_uniform;
    uint32_t *pend;       // [warps][QT][CAP/4][32][4] pending entries
    uint32_t *pend_cnt;   // two-pass path: [warps][QT][32] list lengths
};
static_assert(sizeof(NbrParams) > 128, "NbrParams: see the size note above");

// ---- pack kernel ---------------------------------------------------------------------------
// Packed reference rows (both distance forms): x, y, z and the FILTER addend
//   w' = |r|^2 * (1 - 2^-18)   (+inf for padding),   |r|^2 = fl(fl(x*x + y*y) + z*z).
// torch.sum(p ** 2, -1) over the 3 coordinates: CPU torch adds (x^2 + y^2) + z^2, CUDA torch's
// 3-element reduction adds (x^2 + z^2) + y^2 (measured on B200, tools/gpu_probe.py) -- `xzy`
// selects the CUDA order (DIST_EXPANDED_CUDA). Filters and bounds carry 2^-16 relative slack, far
// above one ulp, so only the EXACT evaluations care which one they get.
__device__ __forceinline__ float nbr_sqnorm(float x, float y, float z, bool xzy = false) {
    return xzy ? __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(z, z)), __fmul_rn(y, y))
               : __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
}
__host__ __device__ constexpr bool mode_expanded(int mode) { return mode == B200PCI_DIST_EXPANDED || mode == B200PCI_DIST_EXPANDED_CUDA; }
// DIST_EXPANDED_CUDA is DIST_EXPANDED with per-operand norm-order flags (NbrParams::q_xzy / r_xzy):
// CUDA torch's reduction adds (a + c) + b only when the reduced dimension is the fastest-striding
// one, i.e. for a [.., N, 3]-contiguous operand; for the permuted [B, 3, N] views the model
// usually passes it loops (a + b) + c like the CPU. The exact evaluations get the ref flag packed
// into bit 30 of their ref count argument (N <= 2^29 is checked at the API).
constexpr int NBR_N_XZY = 1 << 30;

// exact_norm: row 3 holds |r|^2 itself (group records, read by the exact evaluation) instead of
// the filter addend (rows streamed by the scan)
__device__ __forceinline__ void nbr_pack_store(float *row, int Npad, int j, bool valid, float x,
                                               float y, float z, bool exact_norm = false,
                                               bool xzy = false) {
    const float inf = __int_as_float(0x7f800000);
    row[j] = valid ? x : 0.f;
    row[Npad + j] = valid ? y : 0.f;
    row[2 * Npad + j] = valid ? z : 0.f;
    const float sr = nbr_sqnorm(x, y, z, xzy);
    row[3 * Npad + j] = valid ? (exact_norm ? sr : __fmul_rn(sr, 1.0f - 0x1p-18f)) : inf;
}

// ws: [B][4][Npad] all refs; grp: [B][Npad/4][4][4]; samp (nullable): [B][4][Spad] refs 0, 8, ...
static __global__ void nbr_pack_refs_kernel(int N, int Npad, int Spad, const float *__restrict__ r,
                                     long long r_sb, long long r_sp, long long r_sc,
                                     long long r_ox, long long r_oy,
                                     float *__restrict__ ws, float *__restrict__ grp,
                                     float *__restrict__ samp, int xzy) {
    const int b = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= Npad) return;
    float x = 0.f, y = 0.f, z = 0.f;
    if (j < N) {
        const float *p = r + b * r_sb + j * r_sp;
        x = p[r_ox];
        y = p[r_oy];
        z = p[2 * r_sc];
    }
    if (ws != nullptr) {  // (null: only the sample rows are wanted)
        nbr_pack_store(ws + (size_t)b * 4 * Npad, Npad, j, j < N, x, y, z);
        // group record (j >> 2): row stride 4, element j & 3
        nbr_pack_store(grp + (size_t)b * 4 * Npad + (size_t)(j >> 2) * 16, 4, j & 3, j < N, x, y, z, true, xzy != 0);
    }
    if (samp != nullptr && (j % NBR_SAMPLE_STRIDE) == 0 && j / NBR_SAMPLE_STRIDE < Spad)
        nbr_pack_store(samp + (size_t)b * 4 * Spad, Spad, j / NBR_SAMPLE_STRIDE, j < N, x, y, z);
}

// ---- per-query constants, the cheap filter and the exact 4-ref distance evaluation -------------
//
// FILTER (main loop, 3 FFMA2 per two pairs instead of 5-6 exact instructions):
//   A' = fma(-2z,Z, fma(-2y,Y, fma(-2x,X, w')))          ~  |r|^2 - 2 q.r  (slightly low)
//   candidate  <=>  A' < thr,   thr = fl(tau - |q|^2) + 2^-18 |q|^2 + 2^-21 |fl(tau - |q|^2)|
// Conservative for BOTH exact forms: with u = 2^-24 and P = 2(|q|^2 + |r|^2) bounding every
// partial result, |D_exact - (|q|^2 + |r|^2 - 2 q.r)| <= 5uP and the three fused roundings of A'
// add <= 3uP, i.e. <= 2^-20 (|q|^2 + |r|^2) together; the 2^-18 relative slack on |r|^2 (inside
// w') and on |q|^2 (inside thr) is 4x that. So D_exact < tau implies A' < thr: the filter may
// flag a few extra groups (re-evaluated exactly and rejected in the drain) but never misses one.
struct QueryRegs {
    float fa, fb, fc;  // -2x, -2y, -2z: the filter's and the expanded form's multipliers
    float s;           // |q|^2
    __device__ __forceinline__ void set(float x, float y, float z, bool xzy = false) {
        s = nbr_sqnorm(x, y, z, xzy);
        fa = -2.f * x;
        fb = -2.f * y;
        fc = -2.f * z;
    }
    // filter threshold for admission bound tau (tau = +-inf maps to +-inf)
    __device__ __forceinline__ float threshold(float tau) const {
        const float t0 = __fsub_rn(tau, s);
        return t0 + (0x1p-18f * s + 0x1p-21f * fabsf(t0));
    }
};

// min over the 4 refs of the filter value A'
__device__ __forceinline__ float filter4(const QueryRegs &q, const float4 &X, const float4 &Y,
                                         const float4 &Z, const float4 &W) {
    const f32x2 fa = pack2(q.fa, q.fa), fb = pack2(q.fb, q.fb), fc = pack2(q.fc, q.fc);
    f32x2 t0 = fma2(pack2(X.x, X.y), fa, pack2(W.x, W.y));
    f32x2 t1 = fma2(pack2(X.z, X.w), fa, pack2(W.z, W.w));
    t0 = fma2(pack2(Y.x, Y.y), fb, t0);
    t1 = fma2(pack2(Y.z, Y.w), fb, t1);
    t0 = fma2(pack2(Z.x, Z.y), fc, t0);
    t1 = fma2(pack2(Z.z, Z.w), fc, t1);
    float d0, d1, d2, d3;
    unpack2(t0, d0, d1);
    unpack2(t1, d2, d3);
    return fminf(fminf(d0, d1), fminf(d2, d3));
}

// Exact d[0..3] for refs i0..i0+3 = (X.x..X.w, ...) in the reference arithmetic of MODE (drains
// only). Padded refs (index >= N) get d = +inf.
template <int MODE>
__device__ __forceinline__ void dist4(const QueryRegs &q, const float4 &X, const float4 &Y,
                                      const float4 &Z, uint32_t i0, int N, float (&d)[4]) {
    const bool xzy = (N & NBR_N_XZY) != 0;  // norm order of the refs (expanded form only)
    N &= NBR_N_XZY - 1;
    const f32x2 X0 = pack2(X.x, X.y), X1 = pack2(X.z, X.w), Y0 = pack2(Y.x, Y.y),
                Y1 = pack2(Y.z, Y.w), Z0 = pack2(Z.x, Z.y), Z1 = pack2(Z.z, Z.w);
    f32x2 t0, t1;
    if (mode_expanded(MODE)) {
        // t = -2*dot = fma(-2z,Z,fma(-2y,Y,(-2x)*X)); D = (t + |q|^2) + |r|^2,
        // |r|^2 = (X*X + Y*Y) + Z*Z with every operation rounded
        // (scalar intrinsics here: ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2)
        const f32x2 qa = pack2(q.fa, q.fa), qb = pack2(q.fb, q.fb), qc = pack2(q.fc, q.fc);
        const f32x2 qs = pack2(q.s, q.s);
        const f32x2 n0 = pack2(nbr_sqnorm(X.x, Y.x, Z.x, xzy), nbr_sqnorm(X.y, Y.y, Z.y, xzy));
        const f32x2 n1 = pack2(nbr_sqnorm(X.z, Y.z, Z.z, xzy), nbr_sqnorm(X.w, Y.w, Z.w, xzy));
        t0 = mul2(X0, qa);
        t1 = mul2(X1, qa);
        t0 = fma2(Y0, qb, t0);
        t1 = fma2(Y1, qb, t1);
        t0 = fma2(Z0, qc, t0);
        t1 = fma2(Z1, qc, t1);
        t0 = add2(add2(t0, qs), n0);
        t1 = add2(add2(t1, qs), n1);
    } else {
        // dx = X + (-x) = -(x - X); D = fma(dz,dz,fma(dx,dx,dy*dy)); -x = 0.5 * (-2x) exactly
        const float a = 0.5f * q.fa, b = 0.5f * q.fb, c = 0.5f * q.fc;
        const f32x2 qa = pack2(a, a), qb = pack2(b, b), qc = pack2(c, c);
        const f32x2 x0 = add2(X0, qa), x1 = add2(X1, qa), y0 = add2(Y0, qb), y1 = add2(Y1, qb),
                    z0 = add2(Z0, qc), z1 = add2(Z1, qc);
        t0 = fma2(z0, z0, fma2(x0, x0, mul2(y0, y0)));
        t1 = fma2(z1, z1, fma2(x1, x1, mul2(y1, y1)));
    }
    unpack2(t0, d[0], d[1]);
    unpack2(t1, d[2], d[3]);
    const float inf = __int_as_float(0x7f800000);
#pragma unroll
    for (int i = 0; i < 4; ++i) d[i] = (i0 + i < (uint32_t)N) ? d[i] : inf;
}

// Same, with |r|^2 of the four refs read from the group record (Wn) instead of recomputed:
// identical bits (the pack kernel evaluates the same nbr_sqnorm), 20 instructions fewer.
template <int MODE>
__device__ __forceinline__ void dist4n(const QueryRegs &q, const float4 &X, const float4 &Y,
                                       const float4 &Z, const float4 &Wn, uint32_t i0, int N,
                                       float (&d)[4]) {
    if (!mode_expanded(MODE)) {
        dist4<MODE>(q, X, Y, Z, i0, N, d);
        return;
    }
    N &= NBR_N_XZY - 1;  // (the record's norms were packed in the order the flag asks for)
    const f32x2 qa = pack2(q.fa, q.fa), qb = pack2(q.fb, q.fb), qc = pack2(q.fc, q.fc);
    const f32x2 qs = pack2(q.s, q.s);
    f32x2 t0 = mul2(pack2(X.x, X.y), qa), t1 = mul2(pack2(X.z, X.w), qa);
    t0 = fma2(pack2(Y.x, Y.y), qb, t0);
    t1 = fma2(pack2(Y.z, Y.w), qb, t1);
    t0 = fma2(pack2(Z.x, Z.y), qc, t0);
    t1 = fma2(pack2(Z.z, Z.w), qc, t1);
    t0 = add2(add2(t0, qs), pack2(Wn.x, Wn.y));
    t1 = add2(add2(t1, qs), pack2(Wn.z, Wn.w));
    unpack2(t0, d[0], d[1]);
    unpack2(t1, d[2], d[3]);
    const float inf = __int_as_float(0x7f800000);
#pragma unroll
    for (int i = 0; i < 4; ++i) d[i] = (i0 + i < (uint32_t)N) ? d[i] : inf;
}

// ---- register-array helpers (dynamic slot index without local memory) ---------------------------
template <class T>
__device__ __forceinline__ T sel_qt(const T (&a)[NBR_QT], int j) {
    T r = a[0];
#pragma unroll
    for (int i = 1; i < NBR_QT; ++i) r = (j == i) ? a[i] : r;
    return r;
}
template <class T>
__device__ __forceinline__ void put_qt(T (&a)[NBR_QT], int j, T v) {
#pragma unroll
    for (int i = 0; i < NBR_QT; ++i) a[i] = (j == i) ? v : a[i];
}

// ---- drain: walk one query slot's pending list ------------------------------------------------
struct DrainCtx {
    const float *grp;    // group records of this cloud
    int N;               // refs in the cloud (indices >= N are padding)
    bool ring_all;       // the whole split is resident in the ring: re-read from shared memory
    const float *tiles;  // this warp's ring
    uint32_t tile0;      // first tile of the split
    __device__ __forceinline__ void load_group(uint32_t gid, float4 &X, float4 &Y, float4 &Z) const {
        constexpr int G4 = NBR_TILE / 4;
        if (ring_all) {
            const uint32_t t = gid / G4 - tile0, g = gid % G4;
            const float4 *base = reinterpret_cast<const float4 *>(tiles + (size_t)(t * 4) * NBR_TILE);
            X = base[g];
            Y = base[G4 + g];
            Z = base[2 * G4 + g];
        } else {
            const float4 *rec = reinterpret_cast<const float4 *>(grp) + (size_t)gid * 4;
            X = __ldg(rec);
            Y = __ldg(rec + 1);
            Z = __ldg(rec + 2);
        }
    }
};

// offset (in uint32) of pending entry e inside a slot's list [CAP/4][32 lanes][4], lane 0
__device__ __forceinline__ uint32_t nbr_pend_off(int e) { return (uint32_t)(e + (e >> 2) * 124); }

// Walks the slot's `cnt` pending entries (group indices, ascending) and calls
//   consume(has, d[4], first_ref_index)   for every entry, warp-synchronously,
//   after_batch()                         after every batch of NBR_DB entries per lane.
// A batch is one quad of entries (one LDG.128, fetched a batch ahead); its row loads are issued
// together, so a batch costs one L2 round trip, not one per group. All lanes walk their lists in
// lockstep (entry index = 4 * batch + i), which keeps every load's destination register free of
// cross-lane scoreboard dependencies.
constexpr int NBR_DB = 4;
template <int MODE, class Consume, class AfterBatch>
__device__ __forceinline__ void nbr_drain_items(const DrainCtx &c, const QueryRegs &q,
                                                const uint32_t *pend, int cnt, Consume &&consume,
                                                AfterBatch &&after_batch) {
    const uint4 *quads = reinterpret_cast<const uint4 *>(pend);  // this lane: quad i at [i * 32]
    const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
    const uint32_t dummy = c.tile0 * (NBR_TILE / 4);  // any valid group of this split
    const int nbatch = (warp_max_i(cnt) + NBR_DB - 1) / NBR_DB;
    uint4 wn = (cnt > 0) ? quads[0] : zero4;
    for (int bt = 0; bt < nbatch; ++bt) {
        const uint4 w = wn;
        wn = ((bt + 1) * NBR_DB < cnt) ? quads[(size_t)(bt + 1) * 32] : zero4;
        const uint32_t ent[NBR_DB] = {w.x, w.y, w.z, w.w};
        bool has[NBR_DB];
        uint32_t gid[NBR_DB];
        float4 X[NBR_DB], Y[NBR_DB], Z[NBR_DB];
#pragma unroll
        for (int i = 0; i < NBR_DB; ++i) {
            has[i] = bt * NBR_DB + i < cnt;
            gid[i] = has[i] ? ent[i] : dummy;
            c.load_group(gid[i], X[i], Y[i], Z[i]);
        }
#pragma unroll
        for (int i = 0; i < NBR_DB; ++i) {
            float d[4];
            dist4<MODE>(q, X[i], Y[i], Z[i], gid[i] * 4u, c.N, d);
            consume(has[i], d, gid[i] * 4u);
        }
        after_batch();
    }
}

// ---- sorting networks on 64-bit keys in registers ------------------------------------------------
__device__ __forceinline__ void ce64(u64 &a, u64 &b) {
    const bool p = b < a;
    const u64 lo = p ? b : a, hi = p ? a : b;
    a = lo;
    b = hi;
}
// 60-comparator, 10-layer network (verified exhaustively with the 0-1 principle)
__device__ __forceinline__ void sort16(u64 (&v)[16]) {
#define B200PCI_CE(i, j) ce64(v[i], v[j])
    B200PCI_CE(0, 13); B200PCI_CE(1, 12); B200PCI_CE(2, 15); B200PCI_CE(3, 14); B200PCI_CE(4, 8); B200PCI_CE(5, 6); B200PCI_CE(7, 11); B200PCI_CE(9, 10);
    B200PCI_CE(0, 5); B200PCI_CE(1, 7); B200PCI_CE(2, 9); B200PCI_CE(3, 4); B200PCI_CE(6, 13); B200PCI_CE(8, 14); B200PCI_CE(10, 15); B200PCI_CE(11, 12);
    B200PCI_CE(0, 1); B200PCI_CE(2, 3); B200PCI_CE(4, 5); B200PCI_CE(6, 8); B200PCI_CE(7, 9); B200PCI_CE(10, 11); B200PCI_CE(12, 13); B200PCI_CE(14, 15);
    B200PCI_CE(0, 2); B200PCI_CE(1, 3); B200PCI_CE(4, 10); B200PCI_CE(5, 11); B200PCI_CE(6, 7); B200PCI_CE(8, 9); B200PCI_CE(12, 14); B200PCI_CE(13, 15);
    B200PCI_CE(1, 2); B200PCI_CE(3, 12); B200PCI_CE(4, 6); B200PCI_CE(5, 7); B200PCI_CE(8, 10); B200PCI_CE(9, 11); B200PCI_CE(13, 14);
    B200PCI_CE(1, 4); B200PCI_CE(2, 6); B200PCI_CE(5, 8); B200PCI_CE(7, 10); B200PCI_CE(9, 13); B200PCI_CE(11, 14);
    B200PCI_CE(2, 4); B200PCI_CE(3, 6); B200PCI_CE(9, 12); B200PCI_CE(11, 13);
    B200PCI_CE(3, 5); B200PCI_CE(6, 8); B200PCI_CE(7, 9); B200PCI_CE(10, 12);
    B200PCI_CE(3, 4); B200PCI_CE(5, 6); B200PCI_CE(7, 8); B200PCI_CE(9, 10); B200PCI_CE(11, 12);
    B200PCI_CE(6, 7); B200PCI_CE(8, 9);
#undef B200PCI_CE
}
// bitonic sequence of 16 -> ascending
__device__ __forceinline__ void bitonic_merge16(u64 (&v)[16]) {
#pragma unroll
    for (int s = 8; s > 0; s >>= 1)
#pragma unroll
        for (int i = 0; i < 16; ++i)
            if ((i & s) == 0) ce64(v[i], v[i + s]);
}
// a, c sorted ascending  ->  a = the 16 smallest of a U c, sorted (c is left untouched)
__device__ __forceinline__ void merge_low16(u64 (&a)[16], const u64 (&c)[16]) {
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = (c[15 - i] < a[i]) ? c[15 - i] : a[i];
    bitonic_merge16(a);
}
// a, c sorted ascending  ->  a = the 16 smallest, c = the 16 largest of a U c, both sorted
__device__ __forceinline__ void merge_full16(u64 (&a)[16], u64 (&c)[16]) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {  // reverse c
        const u64 t = c[i];
        c[i] = c[15 - i];
        c[15 - i] = t;
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) ce64(a[i], c[i]);
    bitonic_merge16(a);
    bitonic_merge16(c);
}

__device__ __forceinline__ u64 sel16(const u64 (&v)[16], int k) {
    u64 r = v[0];
#pragma unroll
    for (int i = 1; i < 16; ++i) r = (k == i) ? v[i] : r;
    return r;
}

// Fold the buffered candidates buf[first .. first+16) (nb valid in total; this lane's column,
// stride 32) into the sorted best-K of one query slot (sj: [NBLK*16][32], this lane's column),
// block by block from the top; returns the kout-th best distance. Out of line: one copy per kernel.
template <int NBLK>
__device__ __noinline__ float topk_fold16(u64 *sj, const u64 *buf, int first, int nb, int kout) {
    u64 C[16], A[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) C[i] = (first + i < nb) ? buf[(first + i) * 32] : ~0ull;
    sort16(C);
#pragma unroll
    for (int i = 0; i < 16; ++i) A[i] = sj[(size_t)((NBLK - 1) * 16 + i) * 32];
    merge_low16(A, C);  // the 16 largest of (top block U chunk) drop out
    const int kb = (kout - 1) >> 4, ko = (kout - 1) & 15;  // block / offset of the kout-th key
    u64 kth = B200PCI_KEY_INF;
#pragma unroll 1
    for (int bk = NBLK - 2; bk >= 0; --bk) {
#pragma unroll
        for (int i = 0; i < 16; ++i) C[i] = sj[(size_t)(bk * 16 + i) * 32];
        merge_full16(C, A);  // C = low half (moves on), A = high half = new block bk+1
        if (kb == bk + 1) kth = sel16(A, ko);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            sj[(size_t)((bk + 1) * 16 + i) * 32] = A[i];
            A[i] = C[i];
        }
    }
    if (kb == 0) kth = sel16(A, ko);
#pragma unroll
    for (int i = 0; i < 16; ++i) sj[(size_t)i * 32] = A[i];
    return sortable2f((uint32_t)(kth >> 32));
}

// ---- sinks -----------------------------------------------------------------------------------
// Identity of the work a warp is doing, passed to the sinks' drain.
struct NbrWho {
    int b, S, nsplit, split;
    size_t warp_linear;  // linear warp index over the grid (workspace addressing)
};

// Top-k of 64-bit keys. K <= 4: sorted list in registers, direct insertion. K = 16/32/64: a 32-deep
// candidate buffer per lane in shared memory; after a batch of groups, if some lane holds more
// than 16 candidates, every lane folds its buffer (16 at a time) into its sorted best-K with the
// sorting networks above. The best-K lives in `state` ([K][32] per query slot, L2-resident) in
// blocks of 16 that are streamed through registers during a fold.
template <int K>
struct TopKSink {
    static constexpr bool NET = K > 4;
    static constexpr int NBLK = NET ? K / 16 : 1;
    static constexpr int BUF = 32;                       // candidate buffer depth per lane
    static constexpr int cap_first = NBR_BLK;  // exact streaming: first drain after one step
    static constexpr int cap_max = NBR_CAP;
    static_assert(!NET || K % 16 == 0, "K must be 1..4 or a multiple of 16");
    static_assert(4 * NBR_DB <= BUF / 2, "a batch must fit the free half of the buffer");
    struct Params {
        void *idx;    // final: int64/int32 [B,S,kout]   (nsplit == 1)
        float *dist;  // final, nullable
        int idx_is_int64;
        u64 *part;        // partial keys [B,S,nsplit,kout] (nsplit > 1)
        u64 *state;       // [warps][QT][K][32]
        int kout;         // number of neighbours the caller asked for (<= K)
    };
    static __host__ __device__ constexpr size_t smem_bytes_per_warp() {
        return NET ? (size_t)BUF * 32 * sizeof(u64) : 0;
    }
    Params p;
    u64 *buf;  // [BUF][32] candidate buffer, this lane's column
    u64 *st;   // state of slot 0, this lane's column

    __device__ __forceinline__ void init(const Params &params, unsigned char *smem_warp, int lane,
                                         const NbrWho &who) {
        p = params;
        buf = reinterpret_cast<u64 *>(smem_warp) + lane;
        st = p.state + who.warp_linear * (size_t)(NBR_QT * K * 32) + lane;
        for (int i = 0; i < NBR_QT * K; ++i) st[(size_t)i * 32] = B200PCI_KEY_INF;
    }
    __device__ __forceinline__ void setup(int, bool) {}
    __device__ __forceinline__ float tau0(int) const { return __int_as_float(0x7f800000); }

    // Drain one query slot; returns its new admission bound.
    template <int MODE>
    __device__ __forceinline__ float drain_slot(const DrainCtx &c, const NbrWho &who, int j,
                                                const QueryRegs &q, int qidx, const uint32_t *pend,
                                                int cnt, float tau, bool final) {
        u64 *sj = st + (size_t)j * (K * 32);
        float tcur = tau;
        const int kl = p.kout - 1;
        if constexpr (NET) {
            int nb = 0;
            auto fold_all = [&]() {
                tcur = fminf(tcur, topk_fold16<NBLK>(sj, buf, 0, nb, p.kout));
                if (__any_sync(0xffffffffu, nb > 16))
                    tcur = fminf(tcur, topk_fold16<NBLK>(sj, buf, 16, nb, p.kout));
                nb = 0;
            };
            nbr_drain_items<MODE>(
                c, q, pend, cnt,
                [&](bool has, float (&d)[4], uint32_t i0) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        if (has && d[i] < tcur) {
                            buf[nb * 32] = make_key(d[i], i0 + i);
                            ++nb;
                        }
                    }
                },
                [&]() {
                    if (__any_sync(0xffffffffu, nb > BUF / 2)) fold_all();
                });
            if (__any_sync(0xffffffffu, nb > 0)) fold_all();
        } else {
            u64 S0[K];
#pragma unroll
            for (int i = 0; i < K; ++i) S0[i] = sj[(size_t)i * 32];
            nbr_drain_items<MODE>(
                c, q, pend, cnt,
                [&](bool has, float (&d)[4], uint32_t i0) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const bool h = has && d[i] < tcur;
                        if (__any_sync(0xffffffffu, h)) {
                            u64 key = h ? make_key(d[i], i0 + i) : ~0ull;
#pragma unroll
                            for (int s = 0; s < K; ++s) ce64(S0[s], key);
                            u64 kth = S0[0];
#pragma unroll
                            for (int s = 1; s < K; ++s) kth = (kl == s) ? S0[s] : kth;
                            tcur = fminf(tcur, sortable2f((uint32_t)(kth >> 32)));
                        }
                    }
                },
                [&]() {});
#pragma unroll
            for (int i = 0; i < K; ++i) sj[(size_t)i * 32] = S0[i];
        }
        if (final && qidx >= 0) {
            const size_t qrow = (size_t)who.b * who.S + qidx;
            const int kout = p.kout;
            constexpr int OB = (K < 16) ? K : 16;  // keys loaded per round trip
            for (int i0 = 0; i0 < kout; i0 += OB) {
                u64 key[OB];
#pragma unroll
                for (int i = 0; i < OB; ++i)
                    key[i] = (i0 + i < kout) ? sj[(size_t)(i0 + i) * 32] : B200PCI_KEY_INF;
#pragma unroll
                for (int i = 0; i < OB; ++i) {
                    if (i0 + i >= kout) break;
                    const size_t o = qrow * kout + i0 + i;
                    if (who.nsplit > 1) {
                        p.part[(qrow * who.nsplit + who.split) * kout + i0 + i] = key[i];
                    } else {
                        const uint32_t id = (uint32_t)key[i];
                        if (p.idx_is_int64)
                            reinterpret_cast<long long *>(p.idx)[o] = (long long)id;
                        else
                            reinterpret_cast<int *>(p.idx)[o] = (int)id;
                        if (p.dist) p.dist[o] = sortable2f((uint32_t)(key[i] >> 32));
                    }
                }
            }
        }
        return tcur;
    }
};

// ---- the streaming kernel --------------------------------------------------------------------
template <int CW, int STAGES, class Sink>
struct NbrSmem {
    static constexpr size_t warp_ring_bytes = (size_t)STAGES * 4 * NBR_TILE * sizeof(float);
    static constexpr size_t tiles_bytes = warp_ring_bytes * CW;
    static constexpr size_t ctrl_bytes = (size_t)((CW * STAGES * sizeof(uint64_t) + 127) / 128) * 128;
    static constexpr size_t tau_off = tiles_bytes + ctrl_bytes;  // [CW][QT][32] admission bounds
    static constexpr size_t sink_off = tau_off + (size_t)CW * NBR_QT * 32 * sizeof(float);
    static constexpr size_t total = sink_off + Sink::smem_bytes_per_warp() * CW;
};

template <int MODE, int CW, int STAGES, class Sink>
__device__ __forceinline__ void nbr_stream(const NbrParams &p, const typename Sink::Params &sp) {
    using SM = NbrSmem<CW, STAGES, Sink>;
    constexpr int NT = CW * 32;
    constexpr int QT = NBR_QT;
    constexpr int G4 = NBR_TILE / 4;  // float4 per row per stage
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float *tiles = reinterpret_cast<float *>(smem + (size_t)warp * SM::warp_ring_bytes);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + SM::tiles_bytes) + warp * STAGES;

    NbrWho who;
    who.b = blockIdx.z;
    who.split = blockIdx.y;
    who.S = p.S;
    who.nsplit = p.nsplit;
    who.warp_linear =
        ((size_t)(blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * CW + warp;
    const int tile0 = who.split * p.tiles_per_split;
    const int ntiles = min(p.tiles_per_split, p.total_tiles - tile0);
    const float *ws = p.ws_ref + (size_t)who.b * 4 * p.Npad;
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

    Sink sink;
    sink.init(sp, smem + SM::sink_off + (size_t)warp * Sink::smem_bytes_per_warp(), lane, who);

    // Per-slot state kept in registers across the scan: the filter multipliers, the filter
    // threshold and the list length. Everything a drain needs beyond that is recomputed there
    // (|q|^2, the query index) or parked in shared memory (the admission bound tau).
    QueryRegs q[QT];
    float thr[QT];
    int cnt[QT];
    float *tau_s = reinterpret_cast<float *>(smem + SM::tau_off) + warp * (QT * 32) + lane;
    const int qi0 = (blockIdx.x * CW + warp) * (QT * 32) + lane;  // slot j: + 32 * j
    // this lane's base in slot 0's pending list; slot j: + j * CAP * 32, entry e: + nbr_pend_off(e)
    uint32_t *pend = p.pend + who.warp_linear * (size_t)(QT * NBR_CAP * 32) + lane * 4;
#pragma unroll
    for (int j = 0; j < QT; ++j) {
        const int qi = qi0 + 32 * j;
        float x = 0.f, y = 0.f, z = 0.f;
        if (qi < p.S) {
            const float *src = p.q + who.b * p.q_sb + qi * p.q_sp;
            x = src[p.q_ox];
            y = src[p.q_oy];
            z = src[2 * p.q_sc];
        }
        q[j].set(x, y, z, p.q_xzy != 0);
        sink.setup(j, qi < p.S);
        float t0 = sink.tau0(j);
        t0 = (qi < p.S) ? t0 : __int_as_float(0xff800000);
        tau_s[j * 32] = t0;
        thr[j] = q[j].threshold(t0);
        cnt[j] = 0;
    }

    DrainCtx dc;
    dc.grp = p.ws_grp + (size_t)who.b * 4 * p.Npad;
    dc.N = p.N | (p.r_xzy ? NBR_N_XZY : 0);
    dc.ring_all = ntiles <= STAGES;
    dc.tiles = tiles;
    dc.tile0 = (uint32_t)tile0;

    // Exact streaming starts with tau = +inf (everything is flagged): drain early at first, then
    // let the lists grow as the bound tightens.
    int cap_now = Sink::cap_first;

    auto drain_all = [&](bool final) {
#ifdef NBR_DBG_NO_DRAIN  // developer timing variant: scan + appends only (results are garbage)
        if (!final || p.S > 0)
            for (int j = 0; j < QT; ++j) cnt[j] = 0;
        if (p.S > 0) return;
#endif
#pragma unroll 1
        for (int j = 0; j < QT; ++j) {
            QueryRegs qs;
            qs.fa = q[0].fa, qs.fb = q[0].fb, qs.fc = q[0].fc;
#pragma unroll
            for (int i = 1; i < QT; ++i) {
                qs.fa = (j == i) ? q[i].fa : qs.fa;
                qs.fb = (j == i) ? q[i].fb : qs.fb;
                qs.fc = (j == i) ? q[i].fc : qs.fc;
            }
            qs.s = nbr_sqnorm(-0.5f * qs.fa, -0.5f * qs.fb, -0.5f * qs.fc, p.q_xzy != 0);  // = |q|^2 exactly
            const int qi = qi0 + 32 * j;
            const int qj = (qi < p.S) ? qi : -1;
            float tj = sink.template drain_slot<MODE>(dc, who, j, qs, qj,
                                                      pend + (size_t)j * (NBR_CAP * 32),
                                                      sel_qt(cnt, j), tau_s[j * 32], final);
            tj = (qj >= 0) ? tj : __int_as_float(0xff800000);
            tau_s[j * 32] = tj;
            put_qt(thr, j, qs.threshold(tj));
        }
#pragma unroll
        for (int j = 0; j < QT; ++j) cnt[j] = 0;
        cap_now = min(2 * cap_now, (int)Sink::cap_max);
    };

    // One STEP = 8 groups (32 refs) against the 4 queries; 4 steps per tile.
    constexpr int SPT = G4 / NBR_BLK;
    const int nsteps = ntiles * SPT;
    const float4 *sX = reinterpret_cast<const float4 *>(tiles);
    float4 X = make_float4(0.f, 0.f, 0.f, 0.f), Y = X, Z = X, W = X;
#ifdef NBR_DBG_NO_APPEND
    uint32_t dbg_acc = 0u;
#endif
#pragma unroll 1
    for (int step = 0; step < nsteps;) {
        const int g0 = (step % SPT) * NBR_BLK;
        if (g0 == 0) {
            const int t = step / SPT, s = t % STAGES;
            mbar_wait(&full[s], (t / STAGES) & 1);
            sX = reinterpret_cast<const float4 *>(tiles + (size_t)(s * 4) * NBR_TILE);
            X = sX[0], Y = sX[G4], Z = sX[2 * G4], W = sX[3 * G4];
        }
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
        // append one entry (the group index) per flagged group: the first one of every slot
        // with predicated stores, the (rare) further ones in a loop behind a single vote
#ifdef NBR_DBG_NO_APPEND  // developer timing variant (tools/variants.sh): scan only
#pragma unroll
        for (int j = 0; j < QT; ++j) dbg_acc += m8[j];  // keep the scan alive
#else
        const uint32_t gbase = ((uint32_t)tile0 * SPT + (uint32_t)step) * NBR_BLK + 7u;
        uint32_t rest = 0u;
#pragma unroll
        for (int j = 0; j < QT; ++j) {
            if (m8[j]) {
                const int bit = 31 - __clz((int)m8[j]);  // highest bit = lowest group
                m8[j] &= ~(1u << bit);
                pend[j * (NBR_CAP * 32) + nbr_pend_off(cnt[j])] = gbase - (uint32_t)bit;
                ++cnt[j];
            }
            rest |= m8[j];
        }
        if (__any_sync(0xffffffffu, rest != 0u)) {
#pragma unroll
            for (int j = 0; j < QT; ++j) {
                uint32_t mm = m8[j];
                while (mm) {
                    const int bit = 31 - __clz((int)mm);
                    mm &= ~(1u << bit);
                    pend[j * (NBR_CAP * 32) + nbr_pend_off(cnt[j])] = gbase - (uint32_t)bit;
                    ++cnt[j];
                }
            }
        }
#endif
        ++step;
        if (step % SPT == 0) {
            // this warp is done with the stage: refill it with the tile STAGES ahead
            const int t = step / SPT - 1;
            __syncwarp();
            if (lane == 0 && t + STAGES < ntiles) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                issue_tile(t + STAGES);
            }
        }
        // a step adds at most NBR_BLK entries to a list: drain when one could overflow during
        // the next step, and after the last step
        const bool last = step == nsteps;
        bool over = false;
#pragma unroll
        for (int j = 0; j < QT; ++j) over |= cnt[j] > cap_now - NBR_BLK;
        if (last || __any_sync(0xffffffffu, over)) drain_all(last);
    }
#ifdef NBR_DBG_NO_APPEND
    pend[0] = dbg_acc;
#endif
}

}  // namespace b200pci
