// KNN two-pass path, second pass: top-k over the candidate lists.
//
// The tensor-core scan (knn_scan_tc_kernel, nbr_scan_tc.cuh) evaluates the pairs its filter flags
// exactly and appends every candidate below the query's bound to the query's list in global memory
// (ScanEvalParams: one list per query and ref split, layout [slot][query]). Then:
//
//   knn_flag_kernel        flags the queries with fewer than k candidates below an ESTIMATED bound,
//                          or with an overflowed list, for the exact redo kernels (knn.cu).
//   knn_topk_kernel        one thread per query reads its candidate keys 16 at a time (coalesced)
//                          and folds them into a sorted best-K in registers with the sorting
//                          networks of nbr_engine.cuh. Keys are sortable(distance) << 32 | index, so
//                          the result does not depend on the order in which the candidates were
//                          appended, and the lowest index wins ties.
//   knn_topk_split_kernel  the same for launches that leave most of the GPU idle: one thread per
//                          (query, group of ref splits).
#pragma once
#include "nbr_engine.cuh"

namespace b200pci {

// candidate keys per (query, split): about 3x the expected count below the bound (k <= 4: ~8k with
// the guaranteed bound; k <= 16: ~30; k <= 32: ~52 with two splits)
__host__ __device__ constexpr int se_cand_cap(int K) { return K <= 4 ? 64 : (K <= 16 ? 96 : 160); }

struct ScanEvalParams {
    u64 *cand;           // [units][cap][128]  candidate keys (a unit: 128 queries x one ref split)
    uint32_t *cand_cnt;  // [units][128]       candidates appended (> cap: overflow)
    int cap;
};

// ---- pass 2: top-k over the candidate lists (one thread per query) ------------------------------
struct TopkParams {
    void *idx;    // int64/int32 [B,S,kout]
    float *dist;  // nullable
    int idx_is_int64;
    int kout;
    int *fail_count;  // [0] flagged tiles, [1] flagged queries (pre-zeroed)
    int *fail_list;   // [B*S] redo flags (pre-zeroed), then the flagged-tile list, then the query list
    const u64 *cand;
    const uint32_t *cand_cnt;
    int scan_tiles;  // query tiles of the scan grid
    int nsplit;
    int cap;  // candidate list capacity per (query, split)
    int balance;  // top-k kernel: hand the queries of a CTA out in order of their list length
};

constexpr int TOPK_THREADS = 128;  // = the 128 queries of one scan unit
template <int K>
__global__ void __launch_bounds__(TOPK_THREADS) knn_topk_kernel(int S, TopkParams tp) {
    constexpr bool NET = K > 4;
    constexpr int NBLK = NET ? K / 16 : 1;
    constexpr int KR = NET ? 16 : K;
    static_assert(NBLK <= 2, "top-k kernel: K <= 32");
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.z, tile = blockIdx.x;
    // Which of the CTA's 128 queries this thread takes. A warp walks ceil(max n / 16) chunks, so 32
    // queries with list lengths drawn at random (mean ~61, maximum of 32 ~110 for k = 16) waste almost
    // half of the lanes' work: the queries are handed out in order of their total list length
    // (bitonic sort of 128 (length, query) words in shared memory), so a warp's 32 lists are alike.
    int tid = threadIdx.x;
    if (tp.balance) {
        __shared__ uint32_t order[TOPK_THREADS];
        uint32_t total = 0u;
        for (int s = 0; s < tp.nsplit; ++s) {
            const size_t warp_linear = (size_t)(b * tp.nsplit + s) * tp.scan_tiles + tile;
            total += min(tp.cand_cnt[warp_linear * 128 + tid], (uint32_t)tp.cap);
        }
        order[tid] = (total << 8) | (uint32_t)tid;
        __syncthreads();
        for (int k2 = 2; k2 <= TOPK_THREADS; k2 <<= 1) {
            for (int j = k2 >> 1; j > 0; j >>= 1) {
                if (threadIdx.x < TOPK_THREADS / 2) {
                    const int t = threadIdx.x;
                    const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                    const int l = i | j;
                    const uint32_t x = order[i], y = order[l];
                    if ((x > y) == ((i & k2) == 0)) {
                        order[i] = y;
                        order[l] = x;
                    }
                }
                __syncthreads();
            }
        }
        tid = (int)(order[threadIdx.x] & 0xffu);
    }
    const int qi = tile * TOPK_THREADS + tid;
    const bool valid = qi < S;
    u64 S0[KR], S1[NBLK > 1 ? 16 : 1];
#pragma unroll
    for (int i = 0; i < KR; ++i) S0[i] = B200PCI_KEY_INF;
    if constexpr (NBLK > 1) {
#pragma unroll
        for (int i = 0; i < 16; ++i) S1[i] = B200PCI_KEY_INF;
    }
    for (int s = 0; s < tp.nsplit; ++s) {
        const size_t warp_linear = (size_t)(b * tp.nsplit + s) * tp.scan_tiles + tile;
        const uint32_t ntot = tp.cand_cnt[warp_linear * 128 + tid];
        const int n = (int)min(ntot, (uint32_t)tp.cap);
        const u64 *col = tp.cand + warp_linear * (size_t)tp.cap * 128 + tid;
        if constexpr (NET) {
            const int nchunk = (warp_max_i(n) + 15) / 16;
            for (int c = 0; c < nchunk; ++c) {
                u64 C[16];
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    C[i] = (c * 16 + i < n) ? col[(size_t)(c * 16 + i) * 128] : ~0ull;
                sort16(C);
                if constexpr (NBLK == 1) {
                    merge_low16(S0, C);
                } else {
                    merge_low16(S1, C);    // S1 = 16 smallest of (top block U chunk)
                    merge_full16(S0, S1);  // S0 = low half, S1 = high half
                }
            }
        } else {
            const int nmax = warp_max_i(n);
            for (int c = 0; c < nmax; ++c) {
                u64 key = (c < n) ? col[(size_t)c * 128] : ~0ull;
#pragma unroll
                for (int r = 0; r < K; ++r) ce64(S0[r], key);
            }
        }
    }
    const size_t qrow = (size_t)b * S + (valid ? qi : 0);
    const int kout = tp.kout;
    // rows flagged by knn_flag_kernel belong to the exact redo kernels (which may be running
    // concurrently on another stream): not written here
    const bool mine = valid && tp.fail_list[qrow] == 0;
#pragma unroll
    for (int i = 0; i < K; ++i) {
        if (i < kout && mine) {
            u64 key;
            if constexpr (NBLK > 1)
                key = (i < 16) ? S0[i < 16 ? i : 0] : S1[i >= 16 ? i - 16 : 0];
            else
                key = S0[i];
            const size_t o = qrow * kout + i;
            const uint32_t id = (uint32_t)key;
            if (tp.idx_is_int64)
                reinterpret_cast<long long *>(tp.idx)[o] = (long long)id;
            else
                reinterpret_cast<int *>(tp.idx)[o] = (int)id;
            if (tp.dist) tp.dist[o] = sortable2f((uint32_t)(key >> 32));
        }
    }
}

// The same for launches that leave most of the GPU idle (one frame pair: 128 CTAs of 4 warps, each
// thread walking the lists of all ref splits one after the other -- 53 us against 7 us per cloud in
// a 64-pair launch): one thread per (query, split group). blockDim = (128, P); thread (q, p) folds
// the lists of splits p, p + P, ...; groups p > 0 leave their sorted block(s) in shared memory and
// group 0 folds them in, 16 keys at a time (each block is sorted, which is all the fold needs).
// The selected set and its order do not depend on how the keys were grouped: same result.
// dynamic shared memory: (P - 1) * K * 128 keys.
template <int K>
__global__ void __launch_bounds__(TOPK_THREADS * 4) knn_topk_split_kernel(int S, TopkParams tp) {
    static_assert(K == 16 || K == 32, "split top-k: K = 16 or 32");
    constexpr int NBLK = K / 16;
    extern __shared__ __align__(16) u64 tk_lists[];  // [P-1][K][128]
    const int tid = threadIdx.x, part = threadIdx.y, P = blockDim.y;
    const int b = blockIdx.z, tile = blockIdx.x;
    const int qi = tile * TOPK_THREADS + tid;
    const bool valid = qi < S;
    u64 S0[16], S1[NBLK > 1 ? 16 : 1];
#pragma unroll
    for (int i = 0; i < 16; ++i) S0[i] = B200PCI_KEY_INF;
    if constexpr (NBLK > 1) {
#pragma unroll
        for (int i = 0; i < 16; ++i) S1[i] = B200PCI_KEY_INF;
    }
    auto fold = [&](u64(&C)[16]) {  // C sorted ascending
        if constexpr (NBLK == 1) {
            merge_low16(S0, C);
        } else {
            merge_low16(S1, C);    // S1 = 16 smallest of (top block U chunk)
            merge_full16(S0, S1);  // S0 = low half, S1 = high half
        }
    };
    for (int s = part; s < tp.nsplit; s += P) {
        const size_t warp_linear = (size_t)(b * tp.nsplit + s) * tp.scan_tiles + tile;
        const uint32_t ntot = tp.cand_cnt[warp_linear * 128 + tid];
        const int n = (int)min(ntot, (uint32_t)tp.cap);
        const u64 *col = tp.cand + warp_linear * (size_t)tp.cap * 128 + tid;
        const int nchunk = (warp_max_i(n) + 15) / 16;
        for (int c = 0; c < nchunk; ++c) {
            u64 C[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) C[i] = (c * 16 + i < n) ? col[(size_t)(c * 16 + i) * 128] : ~0ull;
            sort16(C);
            fold(C);
        }
    }
    if (part > 0) {
        u64 *mine = tk_lists + (size_t)(part - 1) * K * 128 + tid;
#pragma unroll
        for (int i = 0; i < 16; ++i) mine[(size_t)i * 128] = S0[i];
        if constexpr (NBLK > 1) {
#pragma unroll
            for (int i = 0; i < 16; ++i) mine[(size_t)(16 + i) * 128] = S1[i];
        }
    }
    __syncthreads();
    if (part > 0) return;
    for (int o = 0; o + 1 < P; ++o) {
        const u64 *theirs = tk_lists + (size_t)o * K * 128 + tid;
#pragma unroll
        for (int blk = 0; blk < NBLK; ++blk) {
            u64 C[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) C[i] = theirs[(size_t)(blk * 16 + i) * 128];
            fold(C);
        }
    }
    const size_t qrow = (size_t)b * S + (valid ? qi : 0);
    const int kout = tp.kout;
    const bool mine_row = valid && tp.fail_list[qrow] == 0;  // flagged rows belong to the exact redo
#pragma unroll
    for (int i = 0; i < K; ++i) {
        if (i < kout && mine_row) {
            u64 key;
            if constexpr (NBLK > 1)
                key = (i < 16) ? S0[i < 16 ? i : 0] : S1[i >= 16 ? i - 16 : 0];
            else
                key = S0[i];
            const size_t o = qrow * kout + i;
            const uint32_t id = (uint32_t)key;
            if (tp.idx_is_int64)
                reinterpret_cast<long long *>(tp.idx)[o] = (long long)id;
            else
                reinterpret_cast<int *>(tp.idx)[o] = (int)id;
            if (tp.dist) tp.dist[o] = sortable2f((uint32_t)(key >> 32));
        }
    }
}

// Queries to redo exactly, known as soon as the scan has published the list lengths: fewer than k
// candidates below an estimated bound, or an overflowed list. Writes a flag per query, the query
// list and (once per warp = one 32-query tile) the tile list.
static __global__ void __launch_bounds__(TOPK_THREADS) knn_flag_kernel(int S, TopkParams tp) {
    const int tid = threadIdx.x, lane = tid & 31;
    const int b = blockIdx.z, tile = blockIdx.x;
    const int qi = tile * TOPK_THREADS + tid;
    const bool valid = qi < S;
    uint32_t total = 0u;
    bool overflow = false;
    for (int s = 0; s < tp.nsplit; ++s) {
        const size_t warp_linear = (size_t)(b * tp.nsplit + s) * tp.scan_tiles + tile;
        const uint32_t ntot = tp.cand_cnt[warp_linear * 128 + tid];
        overflow |= ntot > (uint32_t)tp.cap;
        total += min(ntot, (uint32_t)tp.cap);
    }
    const size_t qrow = (size_t)b * S + (valid ? qi : 0);
    const bool redo = valid && (total < (uint32_t)tp.kout || overflow);
    const int tiles_per_cloud = (S + 31) / 32;
    int *tile_list = tp.fail_list + (size_t)gridDim.z * S;
    int *query_list = tile_list + (size_t)gridDim.z * tiles_per_cloud;
    if (redo) {
        tp.fail_list[qrow] = 1;
        query_list[atomicAdd(tp.fail_count + 1, 1)] = (int)qrow;
    }
    if (__any_sync(0xffffffffu, redo) && lane == 0)
        tile_list[atomicAdd(tp.fail_count, 1)] = b * tiles_per_cloud + qi / 32;
}

}  // namespace b200pci
