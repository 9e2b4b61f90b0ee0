// KNN / three_nn / ball_query / Chamfer entry points on top of the neighbourhood engine.
#include <math.h>

#include <algorithm>

#include "nbr_engine.cuh"
#include "nbr_two_pass.cuh"
#include "nbr_topk.cuh"
#include "nbr_scan_tc.cuh"
#include "knn_grad.cuh"

extern int g_fps_single_cta;  // fps.cu (test hook)
int b200pci_gather_debug_set(int key, double value);  // gather.cu (developer hooks 15, 16)
int b200pci_emd_debug_set(int key, double value);  // emd.cu (developer hook 19)

namespace b200pci {

// One warp per CTA (128 queries, 4 per thread), <= 128 registers per thread: up to 16 resident
// warps per SM, and no warp ever waits for another. A CTA needs 4 KB of ring + 8 KB of candidate
// buffer. The refs of a cloud are split over several CTAs whenever the query tiles alone would
// leave fewer than ~3 warps per SM sub-partition (B=8 x 16384 queries: 1024 tiles x 2 splits).
constexpr int KNN_MAX_SPLIT = 16;
constexpr int KNN_SAFE_MIN_N = 2048;  // k <= 4: two-pass path from here (and from 2^25 pairs),
constexpr long long KNN_SAFE_MIN_PAIRS = 1LL << 25;  // one-launch kernel below (measured cross-over: tools/time_safe_threshold.py)
#ifndef KNN_CTAS_PER_SM_V  // (developer variants: tools/variants.sh)
#define KNN_CTAS_PER_SM_V 16
#endif
#ifndef KNN_STAGES_V
#define KNN_STAGES_V 2
#endif
#ifndef KNN_CW_V
#define KNN_CW_V 1
#endif
constexpr int KNN_CTAS_PER_SM = KNN_CTAS_PER_SM_V;
constexpr int KNN_STAGES = KNN_STAGES_V;  // per-warp ring depth (128-ref tiles)
constexpr int KNN_CW = KNN_CW_V;

template <int MODE, int K>
__global__ void __launch_bounds__(KNN_CW * 32, KNN_CTAS_PER_SM)
    knn_kernel(NbrParams p, typename TopKSink<K>::Params sp) {
    nbr_stream<MODE, KNN_CW, KNN_STAGES, TopKSink<K>>(p, sp);
}

__global__ void __launch_bounds__(KNN_CW * 32, KNN_CTAS_PER_SM) knn_scan_kernel(NbrParams p) {
    nbr_scan<KNN_CW, KNN_STAGES>(p);
}

// the two-pass KNN's scan: filter on the tensor cores, exact evaluation of what it flags (nbr_scan_tc.cuh)
template <int MODE>
__global__ void __launch_bounds__(TC_THREADS, TC_UNITS == 1 ? 2 : 1)
    knn_scan_tc_kernel(NbrParams p, ScanEvalParams ep) {
    nbr_scan_tc<MODE>(p, ep);
}

template <int RMAX>
__global__ void __launch_bounds__(TAU_THREADS, 2)
    knn_tau_tc_kernel(NbrParams p, const float *tcs, int SpadT, int R, float *tau_out, float tau_scale,
                      float slack_rel) {
    nbr_tau_tc<RMAX>(p, tcs, SpadT, R, tau_out, tau_scale, slack_rel);
}

// One-launch kernel for everything too small for the two-pass path (N < 2048 or fewer than 2^25
// pairs: the model's coarser pyramid levels, three_nn on the coarse levels, Chamfer on
// small sets), where launch latency and parallelism matter, not FLOPs. A CTA owns 32 queries
// (one per lane) and splits the refs over its P warps; every warp stages its part through its own
// shared-memory slice (float4 x, y, z, |r|^2 per ref, read back as broadcast LDS.128), evaluates
// every pair in the exact reference arithmetic and keeps the candidates that beat its running
// k-th distance in a 16-deep per-lane buffer, folded into a sorted best-K in registers by the
// sorting networks of nbr_engine.cuh. The P partial results are merged through shared memory.
constexpr int MID_MAXP = 16;
constexpr int REDO_SPARSE_MAX = 2048;  // failed queries up to which the per-query redo kernel is used
#ifndef MID_SUB_V
#define MID_SUB_V 512
#endif
constexpr int MID_SUB = MID_SUB_V;  // refs staged per warp at a time
constexpr size_t MID_WARP_SMEM = (size_t)MID_SUB * 16 + 16 * 32 * sizeof(unsigned long long);
struct MidArgs {
    int S, N, P;
    const float *q;
    long long q_sb, q_sp, q_sc;
    const float *r;
    long long r_sb, r_sp, r_sc;
    int swap_xy;  // DIST_DIRECT_XYZ: first and second coordinate change places (see NbrParams::q_ox)
    int q_xzy, r_xzy;  // norm order of the expanded form (see NbrParams)
    void *idx;
    int idx_is_int64;
    float *dist;
    int kout;
    const int *redo;       // redo mode: [B*S] flags of the queries to recompute (else null)
    const int *tile_list;  // redo mode: 32-query tiles (b * tiles_per_cloud + tile) with a flagged query
    const int *tile_count;
};

// one 32-query tile of cloud b (all threads of the CTA)
template <int MODE, int K>
__device__ __forceinline__ void knn_mid_tile(const MidArgs &a, int b, int tile) {
    const int S = a.S, N = a.N, P = a.P, kout = a.kout, idx_is_int64 = a.idx_is_int64;
    const float *__restrict__ q = a.q;
    const float *__restrict__ r = a.r;
    const long long q_sb = a.q_sb, q_sp = a.q_sp, q_sc = a.q_sc, r_sb = a.r_sb, r_sp = a.r_sp,
                    r_sc = a.r_sc;
    const long long q_ox = a.swap_xy ? q_sc : 0, q_oy = a.swap_xy ? 0 : q_sc;
    const long long r_ox = a.swap_xy ? r_sc : 0, r_oy = a.swap_xy ? 0 : r_sc;
    void *idx = a.idx;
    float *dist = a.dist;
    const int *__restrict__ redo = a.redo;
    constexpr int NBLK = K / 16;
    static_assert(K == 16 || K == 32, "knn_mid_kernel: K = 16 or 32");
    static_assert((size_t)K * 32 * sizeof(u64) <= MID_WARP_SMEM, "hand-over area fits a warp slice");
    extern __shared__ __align__(16) unsigned char mid_smem[];
    const int tid = threadIdx.x, lane = tid & 31, part = tid >> 5;
    const int qi = tile * 32 + lane;
    unsigned char *slice = mid_smem + (size_t)part * MID_WARP_SMEM;
    float4 *sref = reinterpret_cast<float4 *>(slice);
    u64 *buf = reinterpret_cast<u64 *>(slice + (size_t)MID_SUB * 16) + lane;  // [16][32]

    // redo mode (exact redo of the two-pass path): only the flagged queries are live
    bool live = qi < S;
    if (redo != nullptr) live = live && redo[(size_t)b * S + qi] != 0;
    float x = 0.f, y = 0.f, z = 0.f;
    if (live) {
        const float *src = q + b * q_sb + qi * q_sp;
        x = src[q_ox];
        y = src[q_oy];
        z = src[2 * q_sc];
    }
    QueryRegs qr;
    qr.set(x, y, z, a.q_xzy != 0);
    u64 S0[16], S1[NBLK > 1 ? 16 : 1];
#pragma unroll
    for (int i = 0; i < 16; ++i) S0[i] = B200PCI_KEY_INF;
    if constexpr (NBLK > 1) {
#pragma unroll
        for (int i = 0; i < 16; ++i) S1[i] = B200PCI_KEY_INF;
    }
    auto merge_sorted16 = [&](u64 (&C)[16]) {
        if constexpr (NBLK == 1) {
            merge_low16(S0, C);
        } else {
            merge_low16(S1, C);    // S1 = 16 smallest of (top block U chunk)
            merge_full16(S0, S1);  // S0 = low half, S1 = high half
        }
    };
    const int kl = kout - 1;
    float tcur = live ? __int_as_float(0x7f800000) : __int_as_float(0xff800000);  // dead: admit nothing
    int nb = 0;
    auto fold = [&]() {
        u64 C[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) C[i] = (i < nb) ? buf[i * 32] : ~0ull;
        nb = 0;
        sort16(C);
        merge_sorted16(C);
        u64 kth;
        if constexpr (NBLK == 1)
            kth = sel16(S0, kl);
        else
            kth = (kl < 16) ? sel16(S0, kl) : sel16(S1, kl - 16);
        tcur = fminf(tcur, sortable2f((uint32_t)(kth >> 32)));
    };

    const int per = ((N + P - 1) / P + 3) & ~3;  // refs per part, a multiple of 4
    const int n0 = part * per, n1 = min(N, n0 + per);
    for (int c0 = n0; c0 < n1; c0 += MID_SUB) {
        const int len = min(MID_SUB, n1 - c0);
        __syncwarp();
        for (int i = lane; i < len; i += 32) {
            const float *pr = r + b * r_sb + (long long)(c0 + i) * r_sp;
            const float X = pr[r_ox], Y = pr[r_oy], Z = pr[2 * r_sc];
            sref[i] = make_float4(X, Y, Z, nbr_sqnorm(X, Y, Z, a.r_xzy != 0));
        }
        __syncwarp();
        for (int i0 = 0; i0 < len; i0 += 4) {
            float d[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {  // four independent distance chains first ...
                const float4 R = sref[min(i0 + u, len - 1)];
                if (mode_expanded(MODE)) {
                    float t = __fmul_rn(R.x, qr.fa);
                    t = __fmaf_rn(R.y, qr.fb, t);
                    t = __fmaf_rn(R.z, qr.fc, t);
                    d[u] = __fadd_rn(__fadd_rn(t, qr.s), R.w);
                } else if (MODE == B200PCI_DIST_SQDIFF || MODE == B200PCI_DIST_SQDIFF_CUDA) {
                    // squares and sums all rounded; the 3-element sum in CPU torch's / CUDA torch's order
                    const float dx = __fsub_rn(x, R.x), dy = __fsub_rn(y, R.y), dz = __fsub_rn(z, R.z);
                    d[u] = nbr_sqnorm(dx, dy, dz, MODE == B200PCI_DIST_SQDIFF_CUDA);
                } else {
                    const float dx = __fsub_rn(R.x, x), dy = __fsub_rn(R.y, y), dz = __fsub_rn(R.z, z);
                    d[u] = __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {  // ... then the (rare) appends, in index order
                // ascending index inside a part: an equal distance never displaces an earlier ref
                if (i0 + u < len && d[u] < tcur) {
                    buf[nb * 32] = make_key(d[u], (uint32_t)(c0 + i0 + u));
                    ++nb;
                }
            }
            if (__any_sync(0xffffffffu, nb > 12)) fold();
        }
    }
    if (__any_sync(0xffffffffu, nb > 0)) fold();

    // hand-over: parts 1..P-1 -> part 0 through the (now free) warp slices
    __syncthreads();
    u64 *xch = reinterpret_cast<u64 *>(slice) + lane;  // [K][32]
    if (part > 0) {
#pragma unroll
        for (int i = 0; i < 16; ++i) xch[i * 32] = S0[i];
        if constexpr (NBLK > 1) {
#pragma unroll
            for (int i = 0; i < 16; ++i) xch[(16 + i) * 32] = S1[i];
        }
    }
    __syncthreads();
    if (part == 0 && live) {
    for (int pp = 1; pp < P; ++pp) {
        const u64 *src = reinterpret_cast<const u64 *>(mid_smem + (size_t)pp * MID_WARP_SMEM) + lane;
#pragma unroll 1
        for (int blk = 0; blk < NBLK; ++blk) {
            u64 C[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) C[i] = src[(blk * 16 + i) * 32];
            merge_sorted16(C);
        }
    }
    const size_t qrow = (size_t)b * S + qi;
#pragma unroll
    for (int i = 0; i < K; ++i) {
        if (i < kout) {
            u64 key;
            if constexpr (NBLK > 1)
                key = (i < 16) ? S0[i < 16 ? i : 0] : S1[i >= 16 ? i - 16 : 0];
            else
                key = S0[i];
            const size_t o = qrow * kout + i;
            const uint32_t id = (uint32_t)key;
            if (idx_is_int64)
                reinterpret_cast<long long *>(idx)[o] = (long long)id;
            else
                reinterpret_cast<int *>(idx)[o] = (int)id;
            if (dist) dist[o] = sortable2f((uint32_t)(key >> 32));
        }
    }
    }
}

template <int MODE, int K>
__global__ void __launch_bounds__(32 * MID_MAXP) knn_mid_kernel(MidArgs a) {
    knn_mid_tile<MODE, K>(a, blockIdx.y, blockIdx.x);
}

// exact redo of the two-pass path: persistent CTAs walk the list of tiles with a flagged query
template <int MODE, int K>
__global__ void __launch_bounds__(32 * MID_MAXP) knn_redo_kernel(MidArgs a) {
    if (a.tile_count[1] <= REDO_SPARSE_MAX) return;  // few failures: knn_fallback_kernel does them
    const int ntile = *a.tile_count;
    const int tiles_per_cloud = (a.S + 31) / 32;
    for (int t = blockIdx.x; t < ntile; t += gridDim.x) {
        const int id = a.tile_list[t];
        knn_mid_tile<MODE, K>(a, id / tiles_per_cloud, id % tiles_per_cloud);
        __syncthreads();  // the shared-memory slices are reused by the next tile
    }
}

// Threshold pre-pass over the 1-in-8 sample rows. The sample is cut into 32 consecutive buckets;
// a thread keeps, for each of its 4 queries, the running minimum (filter-form) distance of the
// current bucket (one FMNMX3 pair per 4-ref group, no compare, no candidate lists) and inserts it
// into a sorted list of the RMAX smallest bucket minima when the bucket ends. tau_out[b,q] = the
// R-th smallest bucket minimum: an ESTIMATE of a bound admitting >= k refs of the full cloud
// (the top-k pass verifies it; under-filled queries are redone exactly), or, with R = k <= 4 and
// the filter's error bound added, a guaranteed bound (DESIGN.md "Bounds").
#ifndef TAU_CW_V  // (developer variants: tools/variants.sh)
#define TAU_CW_V 2
#endif
constexpr int TAU_CW = TAU_CW_V;
constexpr int TAU_BUCKETS = 32;
constexpr int TAU_PIECE = 256;  // refs staged per step (sample too big for shared memory)
constexpr int TAU_QT = 4;       // queries per thread
template <int RMAX>
__global__ void __launch_bounds__(TAU_CW * 32)
    knn_tau_kernel(NbrParams p, const float *__restrict__ samp, int Spad, int R, int resident,
                   float *tau_out, float tau_scale, float slack_rel) {
    constexpr int ROWS = 4;
    constexpr int QT = TAU_QT;
    constexpr int NT = TAU_CW * 32;
    __shared__ __align__(16) float tile[ROWS * TAU_PIECE];
    const int tid = threadIdx.x, b = blockIdx.z;
    const float *rows = samp + (size_t)b * ROWS * Spad;
    const float inf = __int_as_float(0x7f800000);
    QueryRegs q[QT];
    float top[QT][RMAX];  // the RMAX smallest bucket minima so far, ascending
#pragma unroll
    for (int j = 0; j < QT; ++j) {
        const int qi = (blockIdx.x * QT + j) * NT + tid;
        float x = 0.f, y = 0.f, z = 0.f;
        if (qi < p.S) {
            const float *src = p.q + b * p.q_sb + qi * p.q_sp;
            x = src[p.q_ox];
            y = src[p.q_oy];
            z = src[2 * p.q_sc];
        }
        q[j].set(x, y, z);
#pragma unroll
        for (int r = 0; r < RMAX; ++r) top[j][r] = inf;
    }
    auto insert = [&](float (&m)[QT]) {  // end of a bucket: fold its minima into the sorted lists
#pragma unroll
        for (int j = 0; j < QT; ++j) {
            float v = m[j];
#pragma unroll
            for (int r = 0; r < RMAX; ++r) {
                const float lo = fminf(top[j][r], v);
                v = fmaxf(top[j][r], v);
                top[j][r] = lo;
            }
            m[j] = inf;
        }
    };
    const int bucket = Spad / TAU_BUCKETS;  // refs per bucket (Spad is a multiple of 256)
    extern __shared__ __align__(16) float whole[];  // [ROWS][Spad] when the sample fits (resident)
    float m[QT];
#pragma unroll
    for (int j = 0; j < QT; ++j) m[j] = inf;
    if (resident) {
        // the whole sample is staged once; the bucket loop then runs without barriers
        for (int i = tid; i < ROWS * (Spad / 4); i += NT)
            reinterpret_cast<float4 *>(whole)[i] = __ldg(reinterpret_cast<const float4 *>(rows) + i);
        __syncthreads();
        const float4 *sX = reinterpret_cast<const float4 *>(whole);
        const float4 *sY = sX + Spad / 4, *sZ = sY + Spad / 4, *sW = sZ + Spad / 4;
        const int gpb = bucket / 4;
#pragma unroll 1
        for (int c = 0; c < TAU_BUCKETS; ++c) {
#pragma unroll 4
            for (int g = c * gpb; g < (c + 1) * gpb; ++g) {
                const float4 X = sX[g], Y = sY[g], Z = sZ[g], W = sW[g];
#pragma unroll
                for (int j = 0; j < QT; ++j) m[j] = fminf(m[j], filter4(q[j], X, Y, Z, W));
            }
            insert(m);
        }
    } else {
#pragma unroll 1
        for (int c = 0; c < TAU_BUCKETS; ++c) {
            for (int r0 = 0; r0 < bucket; r0 += TAU_PIECE) {
                const int len = min(TAU_PIECE, bucket - r0);  // multiple of 8
                __syncthreads();
                for (int i = tid; i < ROWS * (len / 4); i += NT) {
                    const int r = i / (len / 4), g = i - r * (len / 4);
                    reinterpret_cast<float4 *>(tile + r * TAU_PIECE)[g] = __ldg(
                        reinterpret_cast<const float4 *>(rows + (size_t)r * Spad + c * bucket + r0) + g);
                }
                __syncthreads();
                const float4 *sX = reinterpret_cast<const float4 *>(tile);
                const float4 *sY = sX + TAU_PIECE / 4, *sZ = sY + TAU_PIECE / 4, *sW = sZ + TAU_PIECE / 4;
#pragma unroll 2
                for (int g = 0; g < len / 4; ++g) {
                    const float4 X = sX[g], Y = sY[g], Z = sZ[g], W = sW[g];
#pragma unroll
                    for (int j = 0; j < QT; ++j)  // filter form: ~ D - |q|^2, fine for an estimate
                        m[j] = fminf(m[j], filter4(q[j], X, Y, Z, W));
                }
            }
            insert(m);
        }
    }
#pragma unroll
    for (int j = 0; j < QT; ++j) {
        const int qi = (blockIdx.x * QT + j) * NT + tid;
        float t = top[j][0];  // R-th smallest bucket minimum
#pragma unroll
        for (int r = 1; r < RMAX; ++r) t = (r == R - 1) ? top[j][r] : t;
        t += q[j].s;  // back to a distance
        // guaranteed-bound mode (R = k): the filter form reads slightly low; 2^-16 (|q|^2 + |t|)
        // covers its distance to the exact arithmetic, so that at least the k sample refs behind
        // t pass the strict test d < tau
        t += slack_rel * (q[j].s + fabsf(t));
        // tau_scale is a test hook (1.0 in production): < 1 forces the exact-redo path
        if (qi < p.S) tau_out[(size_t)b * p.S + qi] = (tau_scale == 1.0f) ? t : t * tau_scale;
    }
}

// Exact redo of the (rare) queries whose estimated bound admitted fewer than k refs (k <= 32): one
// CTA of 512 threads per query, two passes over the packed rows and two small sorts, no serial
// insertion (the previous generation kept a sorted list per warp and inserted candidates one by
// one through shuffles: 31-36 us per query, the critical path of a single-pair call).
//   pass 1  thread t evaluates refs t, t + 512, ... (at most 32 of a 16384-ref segment) and keeps the
//           smallest KEY (distance, index). The k-th smallest of the 512 thread minima, T, is an
//           upper bound of the k-th smallest key of the segment: k different threads hold a key <= T.
//   pass 2  the same refs again (L1/L2 hits): keys <= T go to a shared list. Keys are unique, so
//           exactly k threads contribute and the list holds at most 32 k entries (typically ~k).
//   sort    bitonic sort of the list in shared memory; the first k entries are the segment's best.
// Clouds of more than 16384 refs are walked segment by segment, the best k carried as candidates.
constexpr int FB_THREADS = 512;
constexpr int FB_PER_THREAD = 32;
constexpr int FB_SEG = FB_THREADS * FB_PER_THREAD;
constexpr int FB_LIST = 2048;  // >= 32 * 32 (one segment's worst case) + 32 (carried), a power of two

// ascending bitonic sort of n (a power of two >= 64) keys in shared memory by the whole CTA. Thread
// t owns pair t of every step; for distances j <= 32 the 32 pairs of a warp lie inside one 64-key
// block that no other warp touches until the next j >= 64 step, so those steps synchronise the warp
// only: 9 CTA barriers for 512 keys instead of 45.
__device__ __forceinline__ void cta_bitonic_sort(unsigned long long *s, int n) {
    for (int k2 = 2; k2 <= n; k2 <<= 1) {
        for (int j = k2 >> 1; j > 0; j >>= 1) {
            for (int t = threadIdx.x; t < n / 2; t += FB_THREADS) {
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                const int l = i | j;
                const unsigned long long x = s[i], y = s[l];
                if ((x > y) == ((i & k2) == 0)) {
                    s[i] = y;
                    s[l] = x;
                }
            }
            // a CTA barrier after every step that crossed 64-key blocks (j >= 64: the next step reads
            // what other warps wrote) and before the first such step of the next k2; else the warp's
            if (j >= 64 || (j == 1 && k2 >= 64))
                __syncthreads();
            else
                __syncwarp();
        }
    }
    __syncthreads();
}

template <int MODE>
__global__ void __launch_bounds__(FB_THREADS)
    knn_fallback_kernel(NbrParams p, const int *__restrict__ fail_count,
                        const int *__restrict__ fail_list, int kout, void *idx, int idx_is_int64,
                        float *dist) {
    constexpr int ROWS = 4;
    __shared__ unsigned long long mins[FB_THREADS];
    __shared__ unsigned long long list[FB_LIST];
    __shared__ int nlist;
    const int tid = threadIdx.x;
    const int nfail = *fail_count;
    if (nfail > REDO_SPARSE_MAX) return;  // mass failure: knn_redo_kernel does it by tiles
    for (int f = blockIdx.x; f < nfail; f += gridDim.x) {
        const int qrow = fail_list[f];
        const int b = qrow / p.S, qi = qrow - b * p.S;
        const float *src = p.q + b * p.q_sb + qi * p.q_sp;
        QueryRegs q;
        q.set(src[p.q_ox], src[p.q_oy], src[2 * p.q_sc], p.q_xzy != 0);
        const float *ws = p.ws_ref + (size_t)b * ROWS * p.Npad;
        auto key_of = [&](int j) {  // j < Npad
            const float X = ws[j], Y = ws[p.Npad + j], Z = ws[2 * (size_t)p.Npad + j],
                        W = ws[3 * (size_t)p.Npad + j];
            float d;
            if (mode_expanded(MODE)) {
                float t = __fmul_rn(X, q.fa);
                t = __fmaf_rn(Y, q.fb, t);
                t = __fmaf_rn(Z, q.fc, t);
                t = __fadd_rn(t, q.s);
                d = __fadd_rn(t, nbr_sqnorm(X, Y, Z, p.r_xzy != 0));
            } else {
                const float dx = __fadd_rn(X, 0.5f * q.fa), dy = __fadd_rn(Y, 0.5f * q.fb),
                            dz = __fadd_rn(Z, 0.5f * q.fc);
                d = __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
            }
            if (W == __int_as_float(0x7f800000)) d = W;  // padding
            return make_key(d, (uint32_t)j);
        };
        int nbest = 0;  // keys carried from the previous segments: list[0 .. nbest)
        for (int seg0 = 0; seg0 < p.Npad; seg0 += FB_SEG) {
            unsigned long long keys[FB_PER_THREAD], mn = ~0ull;
#pragma unroll
            for (int i = 0; i < FB_PER_THREAD; ++i) {
                const int j = seg0 + i * FB_THREADS + tid;
                keys[i] = j < p.Npad ? key_of(j) : ~0ull;
                mn = keys[i] < mn ? keys[i] : mn;
            }
            mins[tid] = mn;
            if (tid == 0) nlist = nbest;
            __syncthreads();
            cta_bitonic_sort(mins, FB_THREADS);
            const unsigned long long T = mins[kout - 1];
            if (mn <= T && mn != ~0ull) {  // (k threads get here)
#pragma unroll
                for (int i = 0; i < FB_PER_THREAD; ++i)
                    if (keys[i] <= T && keys[i] != ~0ull) list[atomicAdd(&nlist, 1)] = keys[i];
            }
            __syncthreads();
            const int n = nlist;
            int P2 = 64;
            while (P2 < n) P2 <<= 1;
            for (int t = n + tid; t < P2; t += FB_THREADS) list[t] = ~0ull;
            __syncthreads();
            cta_bitonic_sort(list, P2);
            nbest = n < kout ? n : kout;
        }
        if (tid < kout) {
            const unsigned long long k = list[tid];
            const uint32_t id = (uint32_t)k;
            const size_t o = (size_t)qrow * kout + tid;
            if (idx_is_int64)
                reinterpret_cast<long long *>(idx)[o] = (long long)id;
            else
                reinterpret_cast<int *>(idx)[o] = (int)id;
            if (dist) dist[o] = sortable2f((uint32_t)(k >> 32));
        }
        __syncthreads();
    }
}

// merge the per-split sorted key lists of one query: thread per query.
__global__ void knn_merge_kernel(long long nq, int nsplit, int kout,
                                 const unsigned long long *__restrict__ part, void *idx,
                                 int idx_is_int64, float *dist) {
    const long long qrow = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (qrow >= nq) return;
    const unsigned long long *src = part + (size_t)qrow * nsplit * kout;
    int head[KNN_MAX_SPLIT];
#pragma unroll
    for (int s = 0; s < KNN_MAX_SPLIT; ++s) head[s] = 0;
    for (int i = 0; i < kout; ++i) {
        unsigned long long best = ~0ull;
        int bs = 0;
#pragma unroll
        for (int s = 0; s < KNN_MAX_SPLIT; ++s) {
            if (s < nsplit && head[s] < kout) {
                const unsigned long long v = src[(size_t)s * kout + head[s]];
                if (v < best) {
                    best = v;
                    bs = s;
                }
            }
        }
#pragma unroll
        for (int s = 0; s < KNN_MAX_SPLIT; ++s)
            if (s == bs) ++head[s];
        const uint32_t id = (uint32_t)best;
        if (idx_is_int64)
            reinterpret_cast<long long *>(idx)[(size_t)qrow * kout + i] = (long long)id;
        else
            reinterpret_cast<int *>(idx)[(size_t)qrow * kout + i] = (int)id;
        if (dist) dist[(size_t)qrow * kout + i] = sortable2f((uint32_t)(best >> 32));
    }
}

// ---- host-side planning --------------------------------------------------------------------
struct KnnPlan {
    int Npad, total_tiles, nsplit, tiles_per_split, Kc, qpb;
    int use_est, safe, Spad, R;  // use_est: two-pass path; safe: its bound is guaranteed (k <= 4)
    int cap;                     // two-pass path: candidate keys per (query, split)
    int tau_tc, SpadT;           // threshold pre-pass on the tensor cores: sample slots (multiple of 1024)
    long long warps;  // warps of the streaming grid (one per 128 queries per split per cloud)
    size_t ws_ref_bytes, samp_bytes, tau_bytes, fail_bytes, part_bytes, pend_bytes, state_bytes;
    size_t cand_bytes;  // two-pass KNN: candidate lists + counters (shares the pend/state region)
    size_t tc_bytes;    // split-TF32 operand of the refs (tensor-core filter)
    size_t tcs_bytes;   // ... and of the pre-pass sample
    size_t total() const {
        const size_t a = pend_bytes + state_bytes;
        return ws_ref_bytes + samp_bytes + tau_bytes + fail_bytes + part_bytes +
               (a > cand_bytes ? a : cand_bytes) + tc_bytes + tcs_bytes;
    }
};

// test / measurement hooks (b200pci_debug_set / b200pci_debug_get): not used in production
static float g_tau_scale = 1.0f;
static int g_force_exact = 0;
static long long g_safe_min_pairs = KNN_SAFE_MIN_PAIRS;  // key 7 (tests lower it)
static int g_ball_force_redo = 0;
static int g_R_override = 0;  // key 11 (developer): R of the estimated bound
// k = 5..32: the two-pass path (estimated bound) pays from 8192 refs on, and from 2048 refs when the
// problem has at least 2^25 pairs (measured cross-over against the one-launch kernel with the
// tensor-core scan: tools/time_est_threshold.py). Keys 12 / 13 (developer) move the second rule.
static int g_est_min_n = 2048;
static long long g_est_min_pairs = 1LL << 25;
static bool est_path_pays(int B, int S, int N) {
    return N >= 8192 || (N >= g_est_min_n && (long long)B * S * N >= g_est_min_pairs);
}
static int g_topk_balance = 1;  // key 20 (tests): 0 = thread t of the top-k kernel takes query t
static int g_topk_split = 1;  // key 18 (tests): 0 = always the thread-per-query top-k kernel
// developer: redo counters of the calling thread's last two-pass call (debug_get 5 / 6); every
// two-pass call writes it, so it is per thread like the library's other state
static thread_local const int *g_last_fail = nullptr;
// key 3: time the dominant kernel of every b200pci_knn call (knn_scan_kernel on the two-pass path,
// knn_kernel otherwise) with CUDA events on the launching stream; b200pci_debug_get(3) -> accumulated ms, (4) -> number of timed launches.
static int g_time_kernel = 0;
static const int KT_MAX = 256;
static cudaEvent_t g_kt_ev[KT_MAX][2];
static int g_kt_n = 0, g_kt_alloc = 0;
static bool kt_begin(cudaStream_t st) {
    if (!g_time_kernel || g_kt_n >= KT_MAX) return false;
    if (g_kt_n >= g_kt_alloc) {
        if (cudaEventCreate(&g_kt_ev[g_kt_n][0]) != cudaSuccess ||
            cudaEventCreate(&g_kt_ev[g_kt_n][1]) != cudaSuccess)
            return false;
        g_kt_alloc = g_kt_n + 1;
    }
    return cudaEventRecord(g_kt_ev[g_kt_n][0], st) == cudaSuccess;
}
static void kt_end(cudaStream_t st) {
    if (cudaEventRecord(g_kt_ev[g_kt_n][1], st) == cudaSuccess) ++g_kt_n;
}

static int round_k(int k) {
    const int ks[] = {1, 3, 4, 16, 32, 64};
    for (int v : ks)
        if (k <= v) return v;
    return -1;
}

// Split the refs of one cloud over several CTAs when the query tiles alone cannot fill the GPU
// (small B*S), trading a merge pass for occupancy: pick the smallest split count that brings
// the wave efficiency units / (slots * ceil(units / slots)) above 90 %, if one exists.
// tc_split = false: the split rule of ball query's scan (knn_scan_kernel, one warp per 128 queries)
// instead of the tensor-core scan's.
static KnnPlan make_plan(int B, int S, int N, int k, int rows, bool allow_split, bool tc_split = true) {
    KnnPlan pl;
    pl.total_tiles = ceil_div(N > 0 ? N : 1, NBR_TILE);
    pl.Npad = pl.total_tiles * NBR_TILE;
    pl.Kc = round_k(k);
    pl.qpb = NBR_QT * 32 * KNN_CW;
    const long long ctas = (long long)ceil_div(S > 0 ? S : 1, pl.qpb) * B;
    const long long slots = (long long)sm_count() * KNN_CTAS_PER_SM;
    // Split the refs when the query tiles alone give fewer than 3 warps per SM sub-partition:
    // the largest split count that still fits one resident wave (keeping >= 1024 refs per split).
    pl.safe = pl.Kc <= 4;  // R-th smallest bucket minimum with R = k bounds the k-th distance
    pl.use_est = allow_split && !g_force_exact && pl.Kc <= 32 &&
                 (pl.safe ? (N >= KNN_SAFE_MIN_N && (long long)B * S * N >= g_safe_min_pairs)
                          : est_path_pays(B, S, N)) &&
                 (long long)B * S < (1LL << 31);
    int nsplit = 1;
    if (pl.use_est && tc_split) {
        // one CTA per SM, 512 queries per CTA: the split count with the cheapest schedule
        // (waves x (tiles per split + a start-up cost of ~6 tiles))
        const long long tcc = (long long)ceil_div(S, 128 * TC_UNITS) * B;
        int maxn = pl.total_tiles / 8;
        if (maxn > KNN_MAX_SPLIT) maxn = KNN_MAX_SPLIT;
        long long best = -1;
        for (int n = 1; n <= (maxn > 1 ? maxn : 1); ++n) {
            const long long waves = (tcc * n + sm_count() - 1) / sm_count();
            const long long cost = waves * (ceil_div(pl.total_tiles, n) + 6);
            if (best < 0 || cost < best) {
                best = cost;
                nsplit = n;
            }
        }
    } else if (allow_split && ctas < (long long)sm_count() * 4 * 3) {
        int maxn = pl.total_tiles / 8;
        if (maxn > KNN_MAX_SPLIT) maxn = KNN_MAX_SPLIT;
        for (int n = 2; n <= maxn; ++n)
            if (ctas * n <= slots) nsplit = n;
    }
    pl.tiles_per_split = ceil_div(pl.total_tiles, nsplit);
    pl.nsplit = ceil_div(pl.total_tiles, pl.tiles_per_split);
    pl.warps = (long long)ceil_div(S > 0 ? S : 1, pl.qpb) * KNN_CW * pl.nsplit * B;
    const int cap = SCAN_CAP > NBR_CAP ? SCAN_CAP : NBR_CAP;
    pl.pend_bytes = align_up((size_t)pl.warps * NBR_QT * cap * 32 * sizeof(uint32_t), 256) +
                    align_up((size_t)pl.warps * NBR_QT * 32 * sizeof(uint32_t), 256);
    pl.state_bytes = align_up((size_t)pl.warps * NBR_QT * pl.Kc * 32 * sizeof(unsigned long long), 256);
    // two copies of the packed refs: SoA rows for the scan, 64-byte group records for the drains
    pl.ws_ref_bytes = align_up((size_t)2 * B * rows * pl.Npad * sizeof(float), 256);
    pl.part_bytes = pl.nsplit > 1
                        ? align_up((size_t)B * S * pl.nsplit * k * sizeof(unsigned long long), 256)
                        : 0;
    // Estimated admission bound (threshold pre-pass on every 16th ref) for the big selections:
    // R-th smallest of 32 bucket minima of the 1-in-8 sample; simulated (tools/tau_sim.py) to admit
    // ~42 / 61 / 104 refs for k = 8 / 16 / 32 with P(fewer than k) ~ 1e-3 or less.
    pl.R = pl.safe ? k : (k <= 8 ? 5 : (k <= 16 ? 7 : 10));
    if (!pl.safe && g_R_override > 0) pl.R = g_R_override;
    pl.Spad = pl.use_est ? ceil_div(ceil_div(N, NBR_SAMPLE_STRIDE), 256) * 256 : 0;
    pl.samp_bytes = pl.use_est ? align_up((size_t)B * rows * pl.Spad * sizeof(float), 256) : 0;
    pl.tau_bytes = pl.use_est ? align_up((size_t)B * S * sizeof(float), 256) : 0;
    // redo bookkeeping: counters (256 B: [0] flagged tiles, [1] flagged queries), per-query flags
    // [B*S], flagged-tile list [B*ceil(S/32)], flagged-query list [B*S]
    pl.fail_bytes = pl.use_est ? 256 + align_up(((size_t)2 * B * S + (size_t)B * ceil_div(S, 32)) * sizeof(int), 256) : 0;
    pl.cand_bytes = 0;
    pl.cap = 0;
    // split-TF32 operand [B][Npad][16] followed by the exact |r|^2 row [B][Npad]
    pl.tc_bytes = pl.use_est ? align_up((size_t)B * pl.Npad * 17 * sizeof(float), 256) : 0;
    pl.tau_tc = pl.use_est && ceil_div(N, NBR_SAMPLE_STRIDE) >= 1024;
    pl.SpadT = pl.tau_tc ? ceil_div(ceil_div(N, NBR_SAMPLE_STRIDE), 1024) * 1024 : 0;
    pl.tcs_bytes = pl.tau_tc ? align_up((size_t)B * pl.SpadT * 16 * sizeof(float), 256) : 0;
    if (pl.use_est) {  // the two-pass KNN path needs neither `part` nor `state`
        pl.part_bytes = pl.state_bytes = 0;
        // (an unsplit scan puts all of a query's candidates into one list: twice the room)
        pl.cap = se_cand_cap(pl.Kc) * (pl.nsplit == 1 ? 2 : 1);
        pl.cand_bytes = align_up((size_t)pl.warps * pl.cap * 128 * sizeof(unsigned long long), 256) +
                        align_up((size_t)pl.warps * 128 * sizeof(uint32_t), 256);
    }
    return pl;
}

static int pack_refs(int B, int N, int Npad, const float *r, long long sb, long long sp,
                     long long sc, float *ws, float *grp, cudaStream_t st, int Spad = 0,
                     float *samp = nullptr, int swap_xy = 0, int xzy = 0) {
    dim3 grid(ceil_div(Npad, 256), B);
    nbr_pack_refs_kernel<<<grid, 256, 0, st>>>(N, Npad, Spad, r, sb, sp, sc, swap_xy ? sc : 0,
                                               swap_xy ? 0 : sc, ws, grp, samp, xzy);
    B200PCI_LAUNCH_CHECK("nbr_pack_refs_kernel");
    return 0;
}

template <int MODE, int K>
static int launch_knn(const NbrParams &p, int B, const typename TopKSink<K>::Params &sp,
                      cudaStream_t st) {
    using SM = NbrSmem<KNN_CW, KNN_STAGES, TopKSink<K>>;
    const size_t smem = SM::total;
    auto kern = knn_kernel<MODE, K>;
    if (smem > 48 * 1024)
        B200PCI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(ceil_div(p.S, NBR_QT * 32 * KNN_CW), p.nsplit, B);
    kern<<<grid, KNN_CW * 32, smem, st>>>(p, sp);
    B200PCI_LAUNCH_CHECK("knn_kernel");
    return 0;
}

template <int MODE>
static int dispatch_knn(int Kc, const NbrParams &p, int B, void *idx, int idx_is_int64, float *dist,
                        unsigned long long *part, unsigned long long *state, int kout,
                        cudaStream_t st) {
#define B200PCI_KNN_CASE(KK)                                            \
    case KK: {                                                          \
        typename TopKSink<KK>::Params sp;                               \
        sp.idx = idx;                                                   \
        sp.dist = dist;                                                 \
        sp.idx_is_int64 = idx_is_int64;                                 \
        sp.part = part;                                                 \
        sp.state = state;                                               \
        sp.kout = kout;                                                 \
        return launch_knn<MODE, KK>(p, B, sp, st);                      \
    }
    switch (Kc) {  // k <= 4 never gets here: one-launch kernel or two-pass path
        B200PCI_KNN_CASE(16)
        B200PCI_KNN_CASE(32)
        B200PCI_KNN_CASE(64)
    }
#undef B200PCI_KNN_CASE
    set_error("unsupported k");
    return B200PCI_EINVAL;
}

static int launch_tau(const KnnPlan &pl, const NbrParams &p, int B, const float *ws_samp,
                      float *tau, const float *ws_tcs, cudaStream_t st) {
    if (pl.tau_tc) {
        dim3 grid(ceil_div(p.S, 128 * TAU_UNITS), 1, B);
        const float slack = pl.safe ? 0x1p-16f : 0.f;
#define B200PCI_TAUTC(RM)                                                                           \
    do {                                                                                            \
        auto kern = knn_tau_tc_kernel<RM>;                                                          \
        B200PCI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,        \
                                          (int)TauTcSmem::total));                                  \
        kern<<<grid, TAU_THREADS, TauTcSmem::total, st>>>(p, ws_tcs, pl.SpadT, pl.R, tau, g_tau_scale, slack); \
    } while (0)
        if (pl.R <= 4)
            B200PCI_TAUTC(4);
        else if (pl.R <= 8)
            B200PCI_TAUTC(8);
        else
            B200PCI_TAUTC(12);
#undef B200PCI_TAUTC
        B200PCI_LAUNCH_CHECK("knn_tau_tc_kernel");
        return 0;
    }
    dim3 grid(ceil_div(p.S, TAU_QT * 32 * TAU_CW), 1, B);
    const size_t whole = (size_t)4 * pl.Spad * sizeof(float);
    const int resident = whole <= 96 * 1024;
    const size_t smem = resident ? whole : 0;
    const float slack = pl.safe ? 0x1p-16f : 0.f;
#define B200PCI_TAU(RM)                                                                           \
    do {                                                                                          \
        auto kern = knn_tau_kernel<RM>;                                                           \
        if (smem > 32 * 1024)                                                                     \
            B200PCI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,  \
                                              (int)smem));                                        \
        kern<<<grid, TAU_CW * 32, smem, st>>>(p, ws_samp, pl.Spad, pl.R, resident, tau,           \
                                              g_tau_scale, slack);                                \
    } while (0)
    if (pl.R <= 4)
        B200PCI_TAU(4);
    else if (pl.R <= 8)
        B200PCI_TAU(8);
    else
        B200PCI_TAU(12);
#undef B200PCI_TAU
    B200PCI_LAUNCH_CHECK("knn_tau_kernel");
    return 0;
}

// two-pass path: scan + exact evaluation in one kernel -> top-k over the candidate lists
template <int K>
static int launch_topk(const NbrParams &p, int B, const TopkParams &tp, cudaStream_t st) {
    dim3 grid(tp.scan_tiles, 1, B);
    if constexpr (K == 16 || K == 32) {
        // small launches (less than two CTAs per SM): one thread per (query, split group)
        const int P = tp.nsplit < 4 ? tp.nsplit : 4;
        if (g_topk_split && P >= 2 && ((long long)tp.scan_tiles * B < 2LL * sm_count() || g_topk_split == 2)) {
            const size_t smem = (size_t)(P - 1) * K * 128 * sizeof(unsigned long long);
            auto kern = knn_topk_split_kernel<K>;
            B200PCI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<grid, dim3(TOPK_THREADS, P), smem, st>>>(p.S, tp);
            B200PCI_LAUNCH_CHECK("knn_topk_split_kernel");
            return 0;
        }
    }
    knn_topk_kernel<K><<<grid, TOPK_THREADS, 0, st>>>(p.S, tp);
    B200PCI_LAUNCH_CHECK("knn_topk_kernel");
    return 0;
}

template <int MODE>
static int run_two_pass(const KnnPlan &pl, const NbrParams &p, int B, int k, void *idx,
                        int idx_is_int64, float *dist, int *fail_count, int *fail_list,
                        void *cand_region, TopkParams &tp, cudaStream_t st) {
    ScanEvalParams ep;
    ep.cand = reinterpret_cast<unsigned long long *>(cand_region);
    ep.cand_cnt = reinterpret_cast<uint32_t *>(
        reinterpret_cast<char *>(cand_region) +
        align_up((size_t)pl.warps * pl.cap * 128 * sizeof(unsigned long long), 256));
    ep.cap = pl.cap;
    auto kern = knn_scan_tc_kernel<MODE>;
    B200PCI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ScanTcSmem::total));
    dim3 tgrid(ceil_div(p.S, 128 * TC_UNITS), p.nsplit, B);
    const bool timed = kt_begin(st);  // measurement hook: the scan kernel alone
    kern<<<tgrid, TC_THREADS, ScanTcSmem::total, st>>>(p, ep);
    if (timed) kt_end(st);
    B200PCI_LAUNCH_CHECK("knn_scan_tc_kernel");
    tp.idx = idx;
    tp.dist = dist;
    tp.idx_is_int64 = idx_is_int64;
    tp.kout = k;
    tp.fail_count = fail_count;
    tp.fail_list = fail_list;
    tp.cand = ep.cand;
    tp.cand_cnt = ep.cand_cnt;
    tp.scan_tiles = ceil_div(p.S, 128);  // 128-query units of a cloud
    tp.nsplit = p.nsplit;
    tp.cap = ep.cap;
    tp.balance = g_topk_balance;
    // the queries for the exact redo kernels are known from the list lengths alone
    knn_flag_kernel<<<dim3(tp.scan_tiles, 1, B), TOPK_THREADS, 0, st>>>(p.S, tp);
    B200PCI_LAUNCH_CHECK("knn_flag_kernel");
    return 0;
}

static int run_topk(const KnnPlan &pl, const NbrParams &p, int B, const TopkParams &tp, cudaStream_t st) {
    switch (pl.Kc) {
        case 1: return launch_topk<1>(p, B, tp, st);
        case 3: return launch_topk<3>(p, B, tp, st);
        case 4: return launch_topk<4>(p, B, tp, st);
        case 16: return launch_topk<16>(p, B, tp, st);
        case 32: return launch_topk<32>(p, B, tp, st);
    }
    set_error("unsupported k");
    return B200PCI_EINVAL;
}

// Side stream of the two-pass path (per host thread and device): the exact redo of the flagged
// queries runs on it concurrently with the top-k kernel (fork after the flag kernel, join before
// the tile-wise redo). Event record / wait only, so the pattern is also legal under stream capture.
struct SideStream {
    cudaStream_t s = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
static SideStream *side_stream() {
    static thread_local SideStream side[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    SideStream &ss = side[dev];
    if (!ss.s) {
        if (cudaStreamCreateWithFlags(&ss.s, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&ss.join, cudaEventDisableTiming) != cudaSuccess) {
            ss.s = nullptr;
            return nullptr;
        }
    }
    return &ss;
}

// pack -> [tau pre-pass] -> streaming selection -> [merge] -> [exact redo of failed queries]
template <int MODE>
static int run_knn(const KnnPlan &pl, const NbrParams &p, int B, int k, const float *r,
                   long long r_sb, long long r_sp, long long r_sc, float *ws_samp, float *tau,
                   void *idx, int idx_is_int64, float *dist, unsigned long long *part,
                   unsigned long long *state, int *fail_count, int *fail_list, float *ws_tc,
                   cudaStream_t st) {
    const int swap_xy = p.q_ox != 0;
    if (pl.use_est) {
        dim3 grid(ceil_div(pl.Npad, 256), B);
        nbr_pack_tc_kernel<<<grid, 256, 0, st>>>(p.N, pl.Npad, r, r_sb, r_sp, r_sc, swap_xy ? r_sc : 0,
                                                 swap_xy ? 0 : r_sc, ws_tc,
                                                 pl.tau_tc ? ws_tc + pl.tc_bytes / sizeof(float) : nullptr, pl.SpadT,
                                                 ws_tc + (size_t)B * pl.Npad * 16, p.r_xzy);
        B200PCI_LAUNCH_CHECK("nbr_pack_tc_kernel");
    }
    int rc = pack_refs(B, p.N, pl.Npad, r, r_sb, r_sp, r_sc, const_cast<float *>(p.ws_ref),
                       const_cast<float *>(p.ws_grp), st, pl.Spad,
                       (pl.use_est && !pl.tau_tc) ? ws_samp : nullptr, swap_xy, p.r_xzy);
    if (rc) return rc;
    if (pl.use_est) {
        g_last_fail = fail_count;
        B200PCI_CUDA(cudaMemsetAsync(fail_count, 0, 256 + (size_t)B * p.S * sizeof(int), st));  // count + flags
        rc = launch_tau(pl, p, B, ws_samp, tau, ws_tc + pl.tc_bytes / sizeof(float), st);
        if (rc) return rc;
    }
    TopkParams tp;
    if (pl.use_est) {
        rc = run_two_pass<MODE>(pl, p, B, k, idx, idx_is_int64, dist, fail_count, fail_list, p.pend, tp, st);
    } else {
        const bool timed = kt_begin(st);
        rc = dispatch_knn<MODE>(pl.Kc, p, B, idx, idx_is_int64, dist, part, state, k, st);
        if (timed) kt_end(st);
    }
    if (rc) return rc;
    if (pl.nsplit > 1 && !pl.use_est) {
        const long long nq = (long long)B * p.S;
        knn_merge_kernel<<<(unsigned)((nq + 127) / 128), 128, 0, st>>>(
            nq, pl.nsplit, k, part, idx, idx_is_int64, dist);
        B200PCI_LAUNCH_CHECK("knn_merge_kernel");
    }
    if (pl.use_est) {
        // exact redo of the flagged queries (under-filled estimate / overflowed list). Normally a
        // few hundred: one CTA per query, its warps striding over the refs (knn_fallback_kernel).
        // Degenerate inputs can flag most queries (e.g. a cloud of identical points): then
        // persistent CTAs redo whole 32-query tiles instead (knn_redo_kernel). Both are launched;
        // the failure count on the device decides which one works.
        // The per-query redo runs on the side stream while the top-k kernel (which skips the flagged
        // rows) runs on the caller's.
        int *qlist = fail_list + (size_t)B * p.S + (size_t)B * ceil_div(p.S, 32);
        SideStream *ss = side_stream();
        cudaStream_t fst = st;
        if (ss) {
            B200PCI_CUDA(cudaEventRecord(ss->fork, st));
            B200PCI_CUDA(cudaStreamWaitEvent(ss->s, ss->fork, 0));
            fst = ss->s;
        }
        knn_fallback_kernel<MODE><<<4 * sm_count(), FB_THREADS, 0, fst>>>(p, fail_count + 1, qlist, k, idx,
                                                                  idx_is_int64, dist);
        B200PCI_LAUNCH_CHECK("knn_fallback_kernel");
        if (ss) B200PCI_CUDA(cudaEventRecord(ss->join, ss->s));
        rc = run_topk(pl, p, B, tp, st);
        if (rc) return rc;
        if (ss) B200PCI_CUDA(cudaStreamWaitEvent(st, ss->join, 0));
        int P = MID_MAXP;
        while (P > 1 && p.N / P < 64) P /= 2;
        const size_t smem = (size_t)P * MID_WARP_SMEM;
        const MidArgs ma = {p.S, p.N, P, p.q, p.q_sb, p.q_sp, p.q_sc, r, r_sb, r_sp, r_sc, swap_xy, p.q_xzy, p.r_xzy, idx,
                            idx_is_int64, dist, k, fail_list, fail_list + (size_t)B * p.S, fail_count};
        if (pl.Kc <= 16) {
            auto kern = knn_redo_kernel<MODE, 16>;
            B200PCI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<sm_count(), 32 * P, smem, st>>>(ma);
        } else {
            auto kern = knn_redo_kernel<MODE, 32>;
            B200PCI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<sm_count(), 32 * P, smem, st>>>(ma);
        }
        B200PCI_LAUNCH_CHECK("knn_mid_kernel (redo)");
    }
    return B200PCI_OK;
}

// Generic search used by knn, three_nn and Chamfer.
static int knn_impl(int B, int S, int N, int k, int mode, const float *q, long long q_sb,
                    long long q_sp, long long q_sc, const float *r, long long r_sb, long long r_sp,
                    long long r_sc, void *idx, int idx_is_int64, float *dist, void *workspace,
                    size_t workspace_bytes, cudaStream_t st) {
    B200PCI_CHECK_ARG(B >= 0 && S >= 0 && N >= 0, "knn: negative size");
    B200PCI_CHECK_ARG(k >= 1 && k <= 64, "knn: k=%d outside [1,64]", k);
    B200PCI_CHECK_ARG(mode >= B200PCI_DIST_EXPANDED && mode <= B200PCI_DIST_EXPANDED_CUDA,
                      "knn: bad dist_mode %d", mode);
    // DIRECT_XYZ is DIRECT with the first two coordinates exchanged on the way in
    const int swap_xy = mode == B200PCI_DIST_DIRECT_XYZ;
    if (swap_xy) mode = B200PCI_DIST_DIRECT;
    // SQDIFF (no fused multiply-add; pointT_layer2's 2048-point clouds) exists in the one-launch kernel only
    const bool sqdiff = mode == B200PCI_DIST_SQDIFF || mode == B200PCI_DIST_SQDIFF_CUDA;
    B200PCI_CHECK_ARG(!sqdiff || k <= 32, "knn: DIST_SQDIFF supports k <= 32 (got %d)", k);
    const bool expanded = mode == B200PCI_DIST_EXPANDED || mode == B200PCI_DIST_EXPANDED_CUDA;
    // CUDA torch sums |p|^2 as (x^2 + z^2) + y^2 only where the coordinate is the fastest-striding
    // dimension of the operand; permuted [B,3,N] views get the sequential (x^2 + y^2) + z^2
    int q_xzy = (mode == B200PCI_DIST_EXPANDED_CUDA && q_sc == 1) ? 1 : 0;
    int r_xzy = (mode == B200PCI_DIST_EXPANDED_CUDA && r_sc == 1) ? 1 : 0;
    if (mode == B200PCI_DIST_EXPANDED_CUDA) mode = B200PCI_DIST_EXPANDED;
    if (mode == B200PCI_DIST_SQDIFF_CUDA && !(q_sc == 1 && r_sc == 1)) mode = B200PCI_DIST_SQDIFF;
    if (expanded)
        B200PCI_CHECK_ARG(k <= N, "selected index k out of range (k=%d > N=%d)", k, N);
    if (B == 0 || S == 0) return B200PCI_OK;
    B200PCI_CHECK_ARG(q && r && idx, "knn: null pointer");
    B200PCI_CHECK_ARG((long long)N <= (1LL << 29), "knn: N too large");
    B200PCI_CHECK_ARG(B <= 65535, "knn: batch too large");
    const bool small_k_small_job =
        k <= 4 && (N < KNN_SAFE_MIN_N || (long long)B * S * N < g_safe_min_pairs || g_force_exact);
    if (sqdiff || small_k_small_job ||
        (k > 4 && k <= 32 && (!est_path_pays(B, S, N) || g_force_exact == 2))) {
        // the one-launch kernel (no workspace); k <= 4 runs in the K = 16 instantiation, where the
        // admission test against the k-th best keeps folds rare
        const long long qwarps = (long long)B * ceil_div(S, 32);
        int P = 1;
        while (P < 8 && qwarps * P < 8LL * sm_count() && N / (2 * P) >= 64) P *= 2;
        const size_t smem = (size_t)P * MID_WARP_SMEM;
        dim3 grid(ceil_div(S, 32), B);
        const MidArgs ma = {S, N, P, q, q_sb, q_sp, q_sc, r, r_sb, r_sp, r_sc, swap_xy, q_xzy, r_xzy, idx,
                            idx_is_int64, dist, k, nullptr, nullptr, nullptr};
#define B200PCI_MID(MM, KK)                                                                       \
    do {                                                                                          \
        auto kern = knn_mid_kernel<MM, KK>;                                                       \
        if (smem > 48 * 1024)                                                                     \
            B200PCI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,  \
                                              (int)smem));                                        \
        kern<<<grid, 32 * P, smem, st>>>(ma);                                                     \
    } while (0)
        if (mode == B200PCI_DIST_EXPANDED) {
            if (k <= 16) B200PCI_MID(B200PCI_DIST_EXPANDED, 16);
            else B200PCI_MID(B200PCI_DIST_EXPANDED, 32);
        } else if (mode == B200PCI_DIST_SQDIFF) {
            if (k <= 16) B200PCI_MID(B200PCI_DIST_SQDIFF, 16);
            else B200PCI_MID(B200PCI_DIST_SQDIFF, 32);
        } else if (mode == B200PCI_DIST_SQDIFF_CUDA) {
            if (k <= 16) B200PCI_MID(B200PCI_DIST_SQDIFF_CUDA, 16);
            else B200PCI_MID(B200PCI_DIST_SQDIFF_CUDA, 32);
        } else {
            if (k <= 16) B200PCI_MID(B200PCI_DIST_DIRECT, 16);
            else B200PCI_MID(B200PCI_DIST_DIRECT, 32);
        }
#undef B200PCI_MID
        B200PCI_LAUNCH_CHECK("knn_mid_kernel");
        return B200PCI_OK;
    }
    const int rows = 4;
    const KnnPlan pl = make_plan(B, S, N, k, rows, true);
    if (!workspace || workspace_bytes < pl.total() ||
        (reinterpret_cast<uintptr_t>(workspace) & 255)) {
        set_error("knn: workspace of %zu bytes (256-B aligned) required, got %zu", pl.total(),
                  workspace_bytes);
        return B200PCI_EWORKSPACE;
    }
    char *wsb = reinterpret_cast<char *>(workspace);
    float *ws_ref = reinterpret_cast<float *>(wsb);
    float *ws_samp = reinterpret_cast<float *>(wsb + pl.ws_ref_bytes);
    float *tau = reinterpret_cast<float *>(wsb + pl.ws_ref_bytes + pl.samp_bytes);
    int *fail_count = reinterpret_cast<int *>(wsb + pl.ws_ref_bytes + pl.samp_bytes + pl.tau_bytes);
    int *fail_list = fail_count + 64;
    char *wsp = wsb + pl.ws_ref_bytes + pl.samp_bytes + pl.tau_bytes + pl.fail_bytes;
    unsigned long long *part = reinterpret_cast<unsigned long long *>(wsp);
    uint32_t *pend = reinterpret_cast<uint32_t *>(wsp + pl.part_bytes);
    unsigned long long *state =
        reinterpret_cast<unsigned long long *>(wsp + pl.part_bytes + pl.pend_bytes);
    if (!pl.use_est) fail_count = fail_list = nullptr;
    const size_t shared_region = pl.pend_bytes + pl.state_bytes > pl.cand_bytes ? pl.pend_bytes + pl.state_bytes : pl.cand_bytes;
    float *ws_tc = reinterpret_cast<float *>(wsp + pl.part_bytes + shared_region);

    NbrParams p;
    p.S = S;
    p.N = N;
    p.Npad = pl.Npad;
    p.nsplit = pl.nsplit;
    p.tiles_per_split = pl.tiles_per_split;
    p.total_tiles = pl.total_tiles;
    p.q = q;
    p.q_sb = q_sb;
    p.q_sp = q_sp;
    p.q_sc = q_sc;
    p.q_ox = swap_xy ? q_sc : 0;
    p.q_oy = swap_xy ? 0 : q_sc;
    p.q_xzy = q_xzy;
    p.r_xzy = r_xzy;
    p.ws_ref = ws_ref;
    p.ws_grp = ws_ref + (size_t)B * 4 * pl.Npad;
    p.ws_tc = ws_tc;
    p.tau_in = pl.use_est ? tau : nullptr;
    p.pend = pend;
    p.pend_cnt = pend + (size_t)pl.warps * NBR_QT * (SCAN_CAP > NBR_CAP ? SCAN_CAP : NBR_CAP) * 32;

    int rc = (mode == B200PCI_DIST_EXPANDED)
                 ? run_knn<B200PCI_DIST_EXPANDED>(pl, p, B, k, r, r_sb, r_sp, r_sc, ws_samp, tau, idx,
                                                  idx_is_int64, dist, part, state, fail_count,
                                                  fail_list, ws_tc, st)
                 : run_knn<B200PCI_DIST_DIRECT>(pl, p, B, k, r, r_sb, r_sp, r_sc, ws_samp, tau, idx,
                                                idx_is_int64, dist, part, state, fail_count,
                                                fail_list, ws_tc, st);
    return rc;
}

static size_t knn_ws_bytes(int B, int S, int N, int k, int rows) {
    if (B <= 0 || S <= 0 || N < 0 || k < 1 || k > 64) return 256;
    const KnnPlan pl = make_plan(B, S, N, k, rows, true);
    return pl.total();
}

// ---- Chamfer reduction ---------------------------------------------------------------------
// partial[b] = sum_i dist_x[b,i] / N + sum_j dist_y[b,j] / M (FP64), then loss = mean_b.
__global__ void chamfer_reduce_kernel(int B, int N, int M, const float *__restrict__ dx,
                                      const float *__restrict__ dy, double *partial) {
    __shared__ double sh[32];
    const int b = blockIdx.x;
    double sx = 0.0, sy = 0.0;
    for (int i = threadIdx.x; i < N; i += blockDim.x) sx += (double)dx[(size_t)b * N + i];
    for (int i = threadIdx.x; i < M; i += blockDim.x) sy += (double)dy[(size_t)b * M + i];
    double v = (N > 0 ? sx / N : 0.0) + (M > 0 ? sy / M : 0.0);
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x < 32) {
        v = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : 0.0;
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0) partial[b] = v;
    }
}
__global__ void chamfer_final_kernel(int B, const double *__restrict__ partial, float *loss) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double s = 0.0;
        for (int b = 0; b < B; ++b) s += partial[b];
        loss[0] = (float)(s / (B > 0 ? B : 1));
    }
}

// grad wrt x: 2*(x_i - y_nn(i)) * g/(B*N), plus scatter of the y->x direction; same for y.
__global__ void chamfer_backward_kernel(int B, int N, int M, const float *__restrict__ x,
                                        const float *__restrict__ y, const int *__restrict__ idx_x,
                                        const int *__restrict__ idx_y,
                                        const float *__restrict__ grad_loss, float *grad_x,
                                        float *grad_y, int phase) {
    const int b = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const float g = grad_loss[0];
    if (phase == 0) {  // x -> y direction
        if (i >= N) return;
        const float w = 2.f * g / ((float)B * (float)N);
        const int j = idx_x[(size_t)b * N + i];
        const float *xi = x + ((size_t)b * N + i) * 3, *yj = y + ((size_t)b * M + j) * 3;
        for (int c = 0; c < 3; ++c) {
            const float d = w * (xi[c] - yj[c]);
            atomicAdd(grad_x + ((size_t)b * N + i) * 3 + c, d);
            atomicAdd(grad_y + ((size_t)b * M + j) * 3 + c, -d);
        }
    } else {  // y -> x direction
        if (i >= M) return;
        const float w = 2.f * g / ((float)B * (float)M);
        const int j = idx_y[(size_t)b * M + i];
        const float *yi = y + ((size_t)b * M + i) * 3, *xj = x + ((size_t)b * N + j) * 3;
        for (int c = 0; c < 3; ++c) {
            const float d = w * (yi[c] - xj[c]);
            atomicAdd(grad_y + ((size_t)b * M + i) * 3 + c, d);
            atomicAdd(grad_x + ((size_t)b * N + j) * 3 + c, -d);
        }
    }
}

// Backward of b200pci_knn's distances: thread per query (knn_grad.cuh); grad_r (pre-zeroed) gets
// -d(i,k) of every live slot through atomics, in no particular order.
template <typename I>
__global__ void __launch_bounds__(256)
    knn_backward_kernel(KnnGradArgs a, const I *__restrict__ idx, float *__restrict__ grad_r) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (i >= a.S) return;
    float *gr = grad_r + (size_t)b * a.N * 3;
    knn_grad_query(a, b, i, idx, [&](long long j, float dx, float dy, float dz) {
        atomicAdd(gr + j * 3, -dx);
        atomicAdd(gr + j * 3 + 1, -dy);
        atomicAdd(gr + j * 3 + 2, -dz);
    });
}

}  // namespace b200pci

using namespace b200pci;

// ============================================================================================
// C ABI
// ============================================================================================
extern "C" size_t b200pci_knn_workspace_bytes(int B, int S, int N, int k) {
    return knn_ws_bytes(B, S, N, k, 4);
}

extern "C" int b200pci_knn(int B, int S, int N, int k, int dist_mode, const float *q, int64_t q_sb,
                           int64_t q_sp, int64_t q_sc, const float *r, int64_t r_sb, int64_t r_sp,
                           int64_t r_sc, void *idx, int idx_is_int64, float *dist, void *workspace,
                           size_t workspace_bytes, void *stream) {
    return knn_impl(B, S, N, k, dist_mode, q, q_sb, q_sp, q_sc, r, r_sb, r_sp, r_sc, idx,
                    idx_is_int64, dist, workspace, workspace_bytes, (cudaStream_t)stream);
}

// Per host thread and device: copy stream, events and a device buffer that is kept (and only ever
// grown) across calls, so that a call costs no allocation. thread_local => re-entrant across host
// threads without locks; b200pci_host_release() frees the calling thread's contexts.
constexpr int HOST_MAX_CHUNKS = 16;
struct HostCtx {
    cudaStream_t cs = nullptr, hs = nullptr;  // device-to-host / host-to-device copy streams
    cudaEvent_t ev[HOST_MAX_CHUNKS] = {};     // chunk computed
    cudaEvent_t evh[HOST_MAX_CHUNKS] = {};    // chunk copied in
    cudaEvent_t ev_free = nullptr;
    char *buf = nullptr;
    size_t cap = 0;
};
static thread_local HostCtx g_host[64];
static int g_host_chunks = 0;  // key 14 (developer): D2H pipeline depth, 0 = default

// chunk sizes of one b200pci_knn_host call (see there); returns the number of chunks
static int host_schedule(int B, int *sizes) {
    if (g_host_chunks > 0 || B < 24) {  // (developer hook) / small batches: equal chunks of >= 4 clouds
        int n = g_host_chunks > 0 ? g_host_chunks : (B + 3) / 4;
        n = std::max(1, std::min(std::min(n, 8), B));
        const int bc = ceil_div(B, n);
        n = ceil_div(B, bc);
        for (int c = 0; c < n; ++c) sizes[c] = (c + 1 < n) ? bc : B - bc * (n - 1);
        return n;
    }
    const double r = 0.65;
    const int first = std::max(2, B / 20), rem = B - first;
    int n = 2;
    double a = 0.0;
    for (int t = 2; t <= HOST_MAX_CHUNKS - 1; ++t) {  // the longest taper whose last chunk has >= 3 clouds
        const double at = rem * (1.0 - r) / (1.0 - pow(r, t));
        if (at * pow(r, t - 1) < 3.0 && t > 2) break;
        n = t;
        a = at;
    }
    sizes[0] = first;
    int used = first;
    for (int i = 0; i < n; ++i) {
        int sz = std::max(1, (int)(a * pow(r, i) + 0.5));
        if (i + 1 == n || used + sz > B) sz = B - used;
        sizes[1 + i] = sz;
        used += sz;
    }
    int cnt = 1 + n;
    while (cnt > 1 && sizes[cnt - 1] <= 0) --cnt;  // (rounding can exhaust the batch early)
    return cnt;
}

extern "C" int b200pci_host_release(void) {
    int cur = 0;
    if (cudaGetDevice(&cur) != cudaSuccess) return B200PCI_ECUDA;
    for (int d = 0; d < 64; ++d) {
        HostCtx &c = g_host[d];
        if (!c.cs && !c.buf) continue;
        cudaSetDevice(d);
        if (c.cs) cudaStreamSynchronize(c.cs);
        if (c.hs) cudaStreamSynchronize(c.hs);
        if (c.buf) cudaFree(c.buf);
        for (auto &e : c.ev)
            if (e) cudaEventDestroy(e);
        for (auto &e : c.evh)
            if (e) cudaEventDestroy(e);
        if (c.ev_free) cudaEventDestroy(c.ev_free);
        if (c.cs) cudaStreamDestroy(c.cs);
        if (c.hs) cudaStreamDestroy(c.hs);
        c = HostCtx();
    }
    cudaSetDevice(cur);
    return B200PCI_OK;
}

extern "C" int b200pci_knn_host(int B, int S, int N, int k, int dist_mode, const float *q_host,
                                const float *r_host, void *idx_host, int idx_is_int64, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    B200PCI_CHECK_ARG(B >= 0 && S >= 0 && N >= 0 && k >= 1 && k <= 64, "knn_host: bad sizes");
    if (B == 0 || S == 0) return B200PCI_OK;
    B200PCI_CHECK_ARG(q_host && r_host && idx_host, "knn_host: null pointer");
    // The clouds are processed in chunks so that the copy-in of the next chunk and the copy-out of
    // the previous one (the largest transfer: 8 bytes x k per query) overlap the kernels of the
    // current chunk; the copies run on their own streams (one per direction: separate copy
    // engines), ordered by events; the kernels of all chunks run on the caller's stream. What
    // cannot overlap is the copy-in of the first chunk and the copy-out of the last, and every
    // chunk costs ~60 us of small serial kernels and partial waves, so a large batch starts with
    // a small chunk and then tapers off from a large one: sizes fall geometrically (x 0.65; the
    // copy-out of a chunk takes 0.7 x its kernels, so it ends before the next, smaller, chunk is
    // computed) down to about 3 clouds. (Alternating the chunks between two kernel streams was
    // measured slower: the grids fill the GPU in submission order anyway, and the small tail
    // kernels of one chunk queue behind the next chunk's scan, which delays its copy-out.)
    int sizes[HOST_MAX_CHUNKS];
    const int nchunk = host_schedule(B, sizes);
    const size_t isz = idx_is_int64 ? sizeof(int64_t) : sizeof(int);
    const size_t qb = (size_t)B * S * 3 * sizeof(float), rb = (size_t)B * N * 3 * sizeof(float);
    const size_t ib = (size_t)B * S * k * isz;
    // make_plan is not monotonic in the batch: a smaller chunk can need MORE scratch
    size_t wb = 0;
    for (int c = 0; c < nchunk; ++c) {
        bool seen = false;
        for (int d = 0; d < c; ++d) seen |= sizes[d] == sizes[c];
        if (seen) continue;
        const size_t w = align_up(knn_ws_bytes(sizes[c], S, N, k, 4), 256);
        if (w > wb) wb = w;
    }
    const size_t o_q = 0, o_r = align_up(qb, 256), o_i = o_r + align_up(rb, 256),
                 o_w = o_i + align_up(ib, 256);
    int devid = 0;
    B200PCI_CUDA(cudaGetDevice(&devid));
    B200PCI_CHECK_ARG(devid >= 0 && devid < 64, "knn_host: device ordinal %d not supported", devid);
    HostCtx &hc = g_host[devid];
    if (!hc.cs) {
        B200PCI_CUDA(cudaStreamCreateWithFlags(&hc.cs, cudaStreamNonBlocking));
        B200PCI_CUDA(cudaStreamCreateWithFlags(&hc.hs, cudaStreamNonBlocking));
        for (auto &e : hc.ev) B200PCI_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto &e : hc.evh) B200PCI_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        B200PCI_CUDA(cudaEventCreateWithFlags(&hc.ev_free, cudaEventDisableTiming));
    }
    if (hc.cap < o_w + wb) {
        if (hc.buf) {
            B200PCI_CUDA(cudaStreamSynchronize(hc.cs));
            B200PCI_CUDA(cudaStreamSynchronize(hc.hs));
            B200PCI_CUDA(cudaFree(hc.buf));
            hc.buf = nullptr;
            hc.cap = 0;
        }
        B200PCI_CUDA(cudaMalloc((void **)&hc.buf, o_w + wb));
        hc.cap = o_w + wb;
    }
    char *dev = hc.buf;
    cudaStream_t cs = hc.cs, hs = hc.hs;
    int rc = B200PCI_OK;
    cudaError_t e;
    // the copy-in stream starts after everything already queued on the caller's stream
    if ((e = cudaEventRecord(hc.ev_free, st)) != cudaSuccess ||
        (e = cudaStreamWaitEvent(hs, hc.ev_free, 0)) != cudaSuccess)
        rc = cuda_fail(e, "H2D pipeline");
    for (int c = 0, b0 = 0; c < nchunk && !rc; b0 += sizes[c], ++c) {  // all copy-ins are queued up front
        const int nb = sizes[c];
        const size_t qo = (size_t)b0 * S * 3 * sizeof(float), ro = (size_t)b0 * N * 3 * sizeof(float);
        if ((e = cudaMemcpyAsync(dev + o_q + qo, reinterpret_cast<const char *>(q_host) + qo,
                                 (size_t)nb * S * 3 * sizeof(float), cudaMemcpyHostToDevice, hs)) != cudaSuccess ||
            (e = cudaMemcpyAsync(dev + o_r + ro, reinterpret_cast<const char *>(r_host) + ro,
                                 (size_t)nb * N * 3 * sizeof(float), cudaMemcpyHostToDevice, hs)) != cudaSuccess ||
            (e = cudaEventRecord(hc.evh[c], hs)) != cudaSuccess)
            rc = cuda_fail(e, "cudaMemcpyAsync H2D");
    }
    for (int c = 0, b0 = 0; c < nchunk && !rc; b0 += sizes[c], ++c) {
        const int nb = sizes[c];
        const size_t qo = (size_t)b0 * S * 3 * sizeof(float), ro = (size_t)b0 * N * 3 * sizeof(float);
        const size_t io = (size_t)b0 * S * k * isz;
        if ((e = cudaStreamWaitEvent(st, hc.evh[c], 0)) != cudaSuccess) {
            rc = cuda_fail(e, "H2D pipeline");
            break;
        }
        rc = knn_impl(nb, S, N, k, dist_mode, (const float *)(dev + o_q + qo), (long long)S * 3, 3, 1,
                      (const float *)(dev + o_r + ro), (long long)N * 3, 3, 1, dev + o_i + io,
                      idx_is_int64, nullptr, dev + o_w, wb, st);
        if (rc) break;
        if ((e = cudaEventRecord(hc.ev[c], st)) != cudaSuccess ||
            (e = cudaStreamWaitEvent(cs, hc.ev[c], 0)) != cudaSuccess ||
            (e = cudaMemcpyAsync(reinterpret_cast<char *>(idx_host) + io, dev + o_i + io,
                                 (size_t)nb * S * k * isz, cudaMemcpyDeviceToHost, cs)) != cudaSuccess)
            rc = cuda_fail(e, "D2H pipeline");
    }
    // all three streams are idle on return: the buffer can be reused by the next call right away
    if ((e = cudaStreamSynchronize(hs)) != cudaSuccess && !rc) rc = cuda_fail(e, "cudaStreamSynchronize");
    if ((e = cudaStreamSynchronize(cs)) != cudaSuccess && !rc) rc = cuda_fail(e, "cudaStreamSynchronize");
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess && !rc) rc = cuda_fail(e, "cudaStreamSynchronize");
    return rc;
}

extern "C" size_t b200pci_three_nn_workspace_bytes(int b, int n, int m) {
    return knn_ws_bytes(b, n, m, 3, 4);
}

extern "C" int b200pci_three_nn(int b, int n, int m, const float *unknown, const float *known,
                                float *dist2, int *idx, void *workspace, size_t workspace_bytes,
                                void *stream) {
    B200PCI_CHECK_ARG(dist2 != nullptr || b == 0 || n == 0, "three_nn: null dist2");
    return knn_impl(b, n, m, 3, B200PCI_DIST_DIRECT, unknown, (long long)n * 3, 3, 1, known,
                    (long long)m * 3, 3, 1, idx, 0, dist2, workspace, workspace_bytes,
                    (cudaStream_t)stream);
}

// T3: the caller-side inverse-distance weights of pointnet2/pointnet2_modules.py:139-144 on the
// three_nn result: dist = sqrt(d2) (pointnet2_utils.py:97), r = 1/(dist + eps),
// w = r / ((r0 + r2) + r1) -- the same IEEE operations, in the order CUDA torch evaluates them
// (its reduction over a last dimension of 3 adds elements 0 and 2 first; three_nn only exists on
// CUDA in the reference, so that is the composition to match).
__global__ void three_nn_finish_kernel(long long rows, float eps, float *__restrict__ d2_to_dist,
                                       float *__restrict__ weight) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows) return;
    float *d = d2_to_dist + i * 3;
    const float s0 = __fsqrt_rn(d[0]), s1 = __fsqrt_rn(d[1]), s2 = __fsqrt_rn(d[2]);
    const float r0 = __fdiv_rn(1.0f, __fadd_rn(s0, eps)), r1 = __fdiv_rn(1.0f, __fadd_rn(s1, eps)),
                r2 = __fdiv_rn(1.0f, __fadd_rn(s2, eps));
    const float norm = __fadd_rn(__fadd_rn(r0, r2), r1);  // CUDA torch's 3-element sum (tools/gpu_probe.py)
    d[0] = s0;
    d[1] = s1;
    d[2] = s2;
    float *w = weight + i * 3;
    w[0] = __fdiv_rn(r0, norm);
    w[1] = __fdiv_rn(r1, norm);
    w[2] = __fdiv_rn(r2, norm);
}

extern "C" int b200pci_three_nn_weights(int b, int n, int m, const float *unknown, const float *known,
                                        float eps, float *dist, float *weight, int *idx,
                                        void *workspace, size_t workspace_bytes, void *stream) {
    B200PCI_CHECK_ARG(b == 0 || n == 0 || (dist && weight), "three_nn_weights: null output");
    int rc = knn_impl(b, n, m, 3, B200PCI_DIST_DIRECT, unknown, (long long)n * 3, 3, 1, known,
                      (long long)m * 3, 3, 1, idx, 0, dist, workspace, workspace_bytes,
                      (cudaStream_t)stream);
    if (rc || b == 0 || n == 0) return rc;
    const long long rows = (long long)b * n;
    three_nn_finish_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rows, eps, dist, weight);
    B200PCI_LAUNCH_CHECK("three_nn_finish_kernel");
    return B200PCI_OK;
}

static size_t ball_fail_bytes(int b, int m) {
    return 256 + align_up((size_t)(b > 0 ? b : 1) * (m > 0 ? m : 1) * sizeof(int), 256);
}

extern "C" size_t b200pci_ball_query_workspace_bytes(int b, int n, int m, int nsample) {
    (void)nsample;
    if (b <= 0 || n < 0 || m < 0) return 256;
    const KnnPlan pl = make_plan(b, m, n, 1, 4, true, false);
    return pl.ws_ref_bytes + pl.pend_bytes + ball_fail_bytes(b, m);
}

// Two-pass path (nbr_two_pass.cuh): scan with the uniform bound r^2 -> one thread per query takes
// the first nsample hits of its lists -> exact redo of overflowed queries.
extern "C" int b200pci_ball_query(int b, int n, int m, float radius, int nsample,
                                  const float *new_xyz, const float *xyz, int *idx, void *workspace,
                                  size_t workspace_bytes, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    B200PCI_CHECK_ARG(b >= 0 && n >= 0 && m >= 0 && nsample >= 0, "ball_query: negative size");
    if (b == 0 || m == 0 || nsample == 0) return B200PCI_OK;
    B200PCI_CHECK_ARG(new_xyz && xyz && idx, "ball_query: null pointer");
    B200PCI_CHECK_ARG(b <= 65535, "ball_query: batch too large");
    const KnnPlan pl = make_plan(b, m, n, 1, 4, true, false);
    const size_t need = pl.ws_ref_bytes + pl.pend_bytes + ball_fail_bytes(b, m);
    if (!workspace || workspace_bytes < need || (reinterpret_cast<uintptr_t>(workspace) & 255)) {
        set_error("ball_query: workspace of %zu bytes (256-B aligned) required, got %zu", need,
                  workspace_bytes);
        return B200PCI_EWORKSPACE;
    }
    char *wsb = reinterpret_cast<char *>(workspace);
    float *ws_ref = reinterpret_cast<float *>(wsb);
    int rc = pack_refs(b, n, pl.Npad, xyz, (long long)n * 3, 3, 1, ws_ref,
                       ws_ref + (size_t)b * 4 * pl.Npad, st);
    if (rc) return rc;
    NbrParams p;
    p.S = m;
    p.N = n;
    p.Npad = pl.Npad;
    p.nsplit = pl.nsplit;
    p.tiles_per_split = pl.tiles_per_split;
    p.total_tiles = pl.total_tiles;
    p.q = new_xyz;
    p.q_sb = (long long)m * 3;
    p.q_sp = 3;
    p.q_sc = 1;
    p.q_ox = 0;
    p.q_oy = 1;
    p.q_xzy = p.r_xzy = 0;
    p.ws_ref = ws_ref;
    p.ws_grp = ws_ref + (size_t)b * 4 * pl.Npad;
    p.ws_tc = nullptr;
    p.tau_in = nullptr;
    p.tau_uniform = radius * radius;  // FP32, ball_query_gpu.cu:24
    p.pend = reinterpret_cast<uint32_t *>(wsb + pl.ws_ref_bytes);
    p.pend_cnt = p.pend + (size_t)pl.warps * NBR_QT * (SCAN_CAP > NBR_CAP ? SCAN_CAP : NBR_CAP) * 32;
    int *fail_count = reinterpret_cast<int *>(wsb + pl.ws_ref_bytes + pl.pend_bytes);
    B200PCI_CUDA(cudaMemsetAsync(fail_count, 0, sizeof(int), st));
    const size_t smem = (size_t)KNN_CW * KNN_STAGES * 4 * NBR_TILE * sizeof(float) + 128;
    dim3 grid(ceil_div(m, NBR_QT * 32 * KNN_CW), pl.nsplit, b);
    knn_scan_kernel<<<grid, KNN_CW * 32, smem, st>>>(p);
    B200PCI_LAUNCH_CHECK("knn_scan_kernel");
    BallSelectParams sp;
    sp.idx = idx;
    sp.nsample = nsample;
    sp.radius2 = p.tau_uniform;
    sp.fail_count = fail_count;
    sp.fail_list = fail_count + 64;
    sp.scan_tiles = (int)grid.x;
    sp.force_redo = g_ball_force_redo;
    ball_select_kernel<<<dim3(grid.x, 1, b), 128, 0, st>>>(p, sp);
    B200PCI_LAUNCH_CHECK("ball_select_kernel");
    ball_fallback_kernel<<<sm_count(), 128, 0, st>>>(p, sp);
    B200PCI_LAUNCH_CHECK("ball_fallback_kernel");
    return B200PCI_OK;
}

extern "C" size_t b200pci_chamfer_workspace_bytes(int B, int N, int M) {
    const size_t a = knn_ws_bytes(B, N, M, 1, 4), b = knn_ws_bytes(B, M, N, 1, 4);
    return (a > b ? a : b) + align_up((size_t)(B > 0 ? B : 1) * sizeof(double), 256);
}

extern "C" int b200pci_chamfer_forward(int B, int N, int M, const float *x, int64_t x_sb,
                                       int64_t x_sp, int64_t x_sc, const float *y, int64_t y_sb,
                                       int64_t y_sp, int64_t y_sc, float *dist_x, int *idx_x,
                                       float *dist_y, int *idx_y, float *loss, void *workspace,
                                       size_t workspace_bytes, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    B200PCI_CHECK_ARG(B >= 0 && N >= 0 && M >= 0, "chamfer: negative size");
    B200PCI_CHECK_ARG(dist_x && idx_x && dist_y && idx_y && loss, "chamfer: null output");
    if (B == 0) return B200PCI_OK;
    const size_t need = b200pci_chamfer_workspace_bytes(B, N, M);
    if (!workspace || workspace_bytes < need) {
        set_error("chamfer: workspace of %zu bytes required, got %zu", need, workspace_bytes);
        return B200PCI_EWORKSPACE;
    }
    const size_t pbytes = align_up((size_t)B * sizeof(double), 256);
    double *partial = reinterpret_cast<double *>(workspace);
    char *ws = reinterpret_cast<char *>(workspace) + pbytes;
    // pytorch3d's arithmetic, like knn_points: the per-point minima and NN indices are those of
    // knn_points(x, y, K=1) and knn_points(y, x, K=1) bit for bit
    int rc = knn_impl(B, N, M, 1, B200PCI_DIST_DIRECT_XYZ, x, x_sb, x_sp, x_sc, y, y_sb, y_sp, y_sc,
                      idx_x, 0, dist_x, ws, workspace_bytes - pbytes, st);
    if (rc) return rc;
    rc = knn_impl(B, M, N, 1, B200PCI_DIST_DIRECT_XYZ, y, y_sb, y_sp, y_sc, x, x_sb, x_sp, x_sc, idx_y,
                  0, dist_y, ws, workspace_bytes - pbytes, st);
    if (rc) return rc;
    chamfer_reduce_kernel<<<B, 1024, 0, st>>>(B, N, M, dist_x, dist_y, partial);
    B200PCI_LAUNCH_CHECK("chamfer_reduce_kernel");
    chamfer_final_kernel<<<1, 32, 0, st>>>(B, partial, loss);
    B200PCI_LAUNCH_CHECK("chamfer_final_kernel");
    return B200PCI_OK;
}

extern "C" int b200pci_chamfer_backward(int B, int N, int M, const float *x, const float *y,
                                        const int *idx_x, const int *idx_y, const float *grad_loss,
                                        float *grad_x, float *grad_y, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    B200PCI_CHECK_ARG(B >= 0 && N >= 0 && M >= 0, "chamfer_backward: negative size");
    if (B == 0 || (N == 0 && M == 0)) return B200PCI_OK;
    B200PCI_CHECK_ARG(x && y && idx_x && idx_y && grad_loss && grad_x && grad_y,
                      "chamfer_backward: null pointer");
    B200PCI_CUDA(cudaMemsetAsync(grad_x, 0, (size_t)B * N * 3 * sizeof(float), st));
    B200PCI_CUDA(cudaMemsetAsync(grad_y, 0, (size_t)B * M * 3 * sizeof(float), st));
    if (N > 0 && M > 0) {
        chamfer_backward_kernel<<<dim3(ceil_div(N, 256), B), 256, 0, st>>>(
            B, N, M, x, y, idx_x, idx_y, grad_loss, grad_x, grad_y, 0);
        chamfer_backward_kernel<<<dim3(ceil_div(M, 256), B), 256, 0, st>>>(
            B, N, M, x, y, idx_x, idx_y, grad_loss, grad_x, grad_y, 1);
        B200PCI_LAUNCH_CHECK("chamfer_backward_kernel");
    }
    return B200PCI_OK;
}

extern "C" int b200pci_knn_backward(int B, int S, int N, int K, const float *q, int64_t q_sb, int64_t q_sp,
                                    int64_t q_sc, const float *r, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                                    const void *idx, int idx_is_int64, const float *grad_dist, float *grad_q,
                                    float *grad_r, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    bool nothing;
    if (int rc = knn_grad_check(B, S, N, K, q, r, idx, grad_dist, grad_q, grad_r, "knn_backward", &nothing))
        return rc;
    if (nothing) return B200PCI_OK;
    B200PCI_CUDA(cudaMemsetAsync(grad_r, 0, (size_t)B * N * 3 * sizeof(float), st));
    if (S == 0) return B200PCI_OK;
    if (K == 0 || N == 0) {  // no live slot
        B200PCI_CUDA(cudaMemsetAsync(grad_q, 0, (size_t)B * S * 3 * sizeof(float), st));
        return B200PCI_OK;
    }
    const KnnGradArgs a{S, N, K, q, q_sb, q_sp, q_sc, r, r_sb, r_sp, r_sc, grad_dist, grad_q};
    const dim3 grid(ceil_div(S, 256), B);
    if (idx_is_int64)
        knn_backward_kernel<long long><<<grid, 256, 0, st>>>(a, reinterpret_cast<const long long *>(idx), grad_r);
    else
        knn_backward_kernel<int><<<grid, 256, 0, st>>>(a, reinterpret_cast<const int *>(idx), grad_r);
    B200PCI_LAUNCH_CHECK("knn_backward_kernel");
    return B200PCI_OK;
}

// Test hooks (every key is listed in include/b200pci.h): key 1 = scale applied to the estimated
// admission bound (1.0 = production), key 2 = 1 disables the estimate (exact streaming only), key 6 =
// 1 sends every ball query through the exact redo kernel, key 7 = pair count from which k <= 4 takes
// the two-pass path (0 = default), key 3 = 1 starts (and resets) CUDA-event timing of the selection
// kernel. A key not listed there returns B200PCI_EINVAL. Process-global, not thread-safe.
extern "C" int b200pci_debug_set(int key, double value) {
    if (key == 1)
        g_tau_scale = (float)value;
    else if (key == 2)
        g_force_exact = (int)value;  // 1: in-kernel engine, 2: one-launch kernels for any N
    else if (key == 3) {
        g_time_kernel = value != 0.0;
        g_kt_n = 0;
    } else if (key == 5)
        ::g_fps_single_cta = value != 0.0;
    else if (key == 6)
        g_ball_force_redo = value != 0.0;
    else if (key == 7)
        g_safe_min_pairs = value > 0.0 ? (long long)value : KNN_SAFE_MIN_PAIRS;
    else if (key == 12)
        g_est_min_n = value > 0.0 ? (int)value : 2048;
    else if (key == 13)
        g_est_min_pairs = value > 0.0 ? (long long)value : (1LL << 25);
    else if (key == 11)
        g_R_override = (int)value;
    else if (key == 18)
        g_topk_split = (int)value;
    else if (key == 20)
        g_topk_balance = (int)value;
    else if (key == 14)
        g_host_chunks = (int)value;
    else if (key == 15 || key == 16)
        return b200pci_gather_debug_set(key, value);
    else if (key == 19)
        return b200pci_emd_debug_set(key, value);
    else
        return B200PCI_EINVAL;
    return B200PCI_OK;
}

extern "C" double b200pci_debug_get(int key) {
    if (key == 3) {  // accumulated selection-kernel time (ms) of the launches timed so far
        double ms = 0.0;
        for (int i = 0; i < g_kt_n; ++i) {
            float t = 0.f;
            if (cudaEventSynchronize(g_kt_ev[i][1]) != cudaSuccess ||
                cudaEventElapsedTime(&t, g_kt_ev[i][0], g_kt_ev[i][1]) != cudaSuccess)
                return -1.0;
            ms += t;
        }
        return ms;
    }
    if (key == 4) return (double)g_kt_n;
    if ((key == 5 || key == 6) && g_last_fail != nullptr) {  // developer: flagged tiles / queries of the last call
        int v[2] = {0, 0};
        if (cudaDeviceSynchronize() != cudaSuccess ||
            cudaMemcpy(v, g_last_fail, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess)
            return -1.0;
        return (double)v[key - 5];
    }
    return -1.0;
}
