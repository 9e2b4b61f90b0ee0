// KNN two-pass path, third generation: the FILTER runs on the tensor cores.
//
// The filter value  D = w' - 2 q.r - thr  is a depth-4 contraction over (x, y, z, 1) -- the
// reference itself forms it with a batched matmul (models/pointconv_util.py:81-85). Here it is a
// tcgen05 TF32 MMA with FP32 accumulation in tensor memory: every FP32 operand is split into
// exact TF32 pieces (a piece = the value with the low 13 mantissa bits cleared, the next piece =
// the exact remainder), laid out over K = 16:
//
//   A row (query m): [qh.x qh.y qh.z 1 | qh.x qh.y qh.z 1 | ql.x ql.y ql.z 1 | t1 t2 t3 0]
//   B row (ref n):   [rh.x rh.y rh.z wh | rl.x rl.y rl.z wl | rh.x rh.y rh.z wll | 1 1 1 0]
//
// (q~ = -2q = qh + ql, r = rh + rl, w' = wh + wl + wll, -thr = t1 + t2 + t3). The result matches
// the real-number value to ~2^-20 (|q|^2 + |r|^2) (measured: tools/mb/mb_tc_tile.cu, 2^-20.4;
// bound: the dropped ql.rl term plus one FP32 ulp of the largest addend per addition). The filter
// stays CONSERVATIVE through a 2^-16 relative slack on |r|^2 (inside w') and on |q|^2 (inside
// thr), 14x that bound: no pair below the admission bound is ever missed, candidate <=> D < 0. The
// flagged groups are re-evaluated in the exact reference arithmetic (FP32 pipe, dist4 of
// nbr_engine.cuh) and the candidates go to the lists that the top-k kernels of nbr_topk.cuh read.
//
// Operand layout: K-major, no swizzle. A tile of 128 rows is [k/4][row][4 floats]: 8 rows x 16 B
// form one 128-byte core matrix, SBO = 128 B between 8-row groups, LBO = 2048 B between the four
// K chunks. nbr_pack_tc_kernel writes the ref tiles in exactly this layout, so a tile is one
// contiguous 8 KB block in HBM / L2 and one 1-D TMA bulk copy (no tensor map).
//
// knn_scan_tc_kernel: a CTA (18 warps, one per SM: it allocates all 512 TMEM columns) owns 256
// queries = two 128-row units, each with TWO 128-column accumulators, and one split of the refs.
//   warp 16      TMA producer: operand tiles into a 4-stage ring, the tiles' exact x, y, z rows
//                (for the drain) into a 64-stage ring
//   warp 17      MMA issuer: per tile and unit two tcgen05.mma (M = N = 128, K = 8), a
//                tcgen05.commit onto the accumulator's mbarrier, and one onto the operand stage's
//   warps 0..15  epilogue: warp w owns unit w / 8, column half (w / 4) % 2, TMEM lanes
//                32 (w % 4) .. +31 (one query per thread). Per tile: two tcgen05.ld.32x32b.x32,
//                release the accumulator, min over each group of 4 refs (FMNMX3 + FMNMX), its
//                sign bit shifted into the step mask (one SHF.L.W), ballot-compact the
//                (query, tile) items into the warp's circular work queue; drain rounds of 32 items
//                (tc_drain) when enough are queued, when an item's tile has to leave the ring, and
//                while waiting for an accumulator.
// knn_tau_tc_kernel: the threshold pre-pass on the same pipeline over the packed 1-in-8 sample.
#pragma once
#include "nbr_topk.cuh"

namespace b200pci {

#ifndef TC_UNITS_V  // (developer variants: tools/variants.sh)
#define TC_UNITS_V 2
#endif
#ifndef TC_STAGES_V
#define TC_STAGES_V 64
#endif
#ifndef TC_BSTAGES_V
#define TC_BSTAGES_V 4
#endif
constexpr int TC_UNITS = TC_UNITS_V;                  // 128-query units per CTA, each with two 128-column accumulators
// Two rings: the 8 KB operand tiles leave as soon as their MMAs are done (TC_BSTAGES), the 2 KB of
// exact x, y, z, |r|^2 rows stay until every warp has drained the items that point into them (TC_STAGES)
constexpr int TC_BSTAGES = TC_BSTAGES_V;
constexpr int TC_STAGES = TC_STAGES_V;                  // SoA ring depth (tiles); a warp may hold back TC_HOLD of them
constexpr int TC_HOLD_PAIRS = TC_STAGES / 2 - 4;  // tile pairs a warp lets its oldest queued item age
constexpr int TC_HOLD = TC_STAGES - 3;         // tiles a warp lets its oldest queued item age before draining
constexpr int TC_QCAP = 256;                   // circular work queue per epilogue warp (items)
constexpr int TC_EPI_WARPS = TC_UNITS * 8;      // per unit: 4 TMEM lane quarters x 2 column halves
constexpr int TC_THREADS = (TC_EPI_WARPS + 2) * 32;
constexpr uint32_t TC_B_BYTES = NBR_TILE * 16 * sizeof(float);    // split-TF32 operand of one tile
constexpr uint32_t TC_SOA_BYTES = 4 * NBR_TILE * sizeof(float);   // exact x, y, z (+ |r|^2, expanded forms) rows of one tile
constexpr uint32_t TC_KCHUNK_BYTES = NBR_TILE * 16;               // LBO: one K chunk of 4 (16 B) x 128 rows
constexpr uint32_t TC_TMEM_COLS = 2 * TC_UNITS * NBR_TILE;        // 512
// instruction descriptor: FP32 accumulate, TF32 x TF32, both K-major, N = 128, M = 128
constexpr int TC_HALF = NBR_TILE / 2;  // columns per epilogue warp
constexpr uint32_t TC_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((NBR_TILE >> 3) << 17) | ((128u >> 4) << 24);

static_assert((TC_STAGES & (TC_STAGES - 1)) == 0 && TC_STAGES <= 64, "SoA ring depth: power of two, 6-bit tile tags");
static_assert((TC_BSTAGES & (TC_BSTAGES - 1)) == 0, "operand ring depth: power of two");

#ifndef TC_SHADOW_V  // drain rounds while waiting for an accumulator
#define TC_SHADOW_V 0
#endif
#ifndef TC_ROUNDS_V  // drain rounds per tile (the last tile of a split drains everything)
#define TC_ROUNDS_V (1 << 30)
#endif
#ifndef TC_DRAIN_AT_V
#define TC_DRAIN_AT_V 32u
#endif

struct ScanTcSmem {
    static constexpr size_t bring = (size_t)TC_BSTAGES * TC_B_BYTES;
    static constexpr size_t sring = (size_t)TC_STAGES * TC_SOA_BYTES;
    static constexpr size_t ring = bring + sring;
    static constexpr size_t aop = (size_t)TC_UNITS * TC_B_BYTES;
    static constexpr size_t qtab = (size_t)TC_UNITS * 5 * 128 * sizeof(float);
    static constexpr size_t queue = (size_t)TC_EPI_WARPS * 2 * TC_QCAP * sizeof(uint32_t);
    static constexpr size_t cnt = (size_t)TC_UNITS * 128 * sizeof(uint32_t);
    static constexpr size_t ctrl = 2048;  // mbarriers (1152 B), TMEM slot
    static constexpr size_t used = ring + aop + qtab + queue + cnt + ctrl;
    // two units: more than half of the SM's shared memory, one CTA per SM (it allocates all of TMEM)
    static constexpr size_t total = (TC_UNITS == 1 || used > 120 * 1024) ? used : 120 * 1024;
};

__device__ __forceinline__ float tf32_hi(float v) { return __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); }

// packed B operand of the ref tiles: [B][tiles][4 chunks][128 refs][4]
__device__ __forceinline__ void tc_pack_store(float *tc_tile, int n, bool valid, float x, float y, float z,
                                              float wscale) {
    float4 c0, c1, c2, c3;
    if (valid) {
        const float w = __fmul_rn(nbr_sqnorm(x, y, z), wscale);
        const float xh = tf32_hi(x), yh = tf32_hi(y), zh = tf32_hi(z), wh = tf32_hi(w);
        const float xl = tf32_hi(__fsub_rn(x, xh)), yl = tf32_hi(__fsub_rn(y, yh)), zl = tf32_hi(__fsub_rn(z, zh));
        const float w1 = __fsub_rn(w, wh), wl = tf32_hi(w1), wll = tf32_hi(__fsub_rn(w1, wl));
        c0 = make_float4(xh, yh, zh, wh);
        c1 = make_float4(xl, yl, zl, wl);
        c2 = make_float4(xh, yh, zh, wll);
        c3 = make_float4(1.f, 1.f, 1.f, 0.f);
    } else {  // padding: +inf, never flagged
        c0 = make_float4(0.f, 0.f, 0.f, __int_as_float(0x7f800000));
        c1 = c2 = c3 = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float4 *dst = reinterpret_cast<float4 *>(tc_tile) + n;
    dst[0] = c0;
    dst[NBR_TILE] = c1;
    dst[2 * NBR_TILE] = c2;
    dst[3 * NBR_TILE] = c3;
}

// tcs (nullable): the same operand for the threshold pre-pass's sample (refs 0, 8, 16, ...; SpadT
// slots, padded; exact |r|^2, the pre-pass adds its own slack)
// nrm (nullable): [B][Npad] the exact |r|^2 of every ref in the reference's summation order (xzy: see
// nbr_sqnorm) -- the fourth row of the drain's SoA stages, so that the exact evaluation of the
// expanded forms adds it instead of recomputing three squares and two sums per ref
static __global__ void nbr_pack_tc_kernel(int N, int Npad, const float *__restrict__ r, long long r_sb, long long r_sp,
                                   long long r_sc, long long r_ox, long long r_oy, float *__restrict__ tc,
                                   float *__restrict__ tcs, int SpadT, float *__restrict__ nrm = nullptr,
                                   int xzy = 0) {
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
    if (tc != nullptr)  // (null: only the sample operand is wanted)
        tc_pack_store(tc + ((size_t)b * Npad + (size_t)(j / NBR_TILE) * NBR_TILE) * 16, j % NBR_TILE, j < N, x, y, z,
                      1.0f - 0x1p-16f);
    if (nrm != nullptr) nrm[(size_t)b * Npad + j] = nbr_sqnorm(x, y, z, xzy != 0);
    if (tcs != nullptr && j < SpadT) {  // sample slot j <- ref 8 j
        const long long src = (long long)j * NBR_SAMPLE_STRIDE;
        x = y = z = 0.f;
        if (src < N) {
            const float *p = r + b * r_sb + src * r_sp;
            x = p[r_ox];
            y = p[r_oy];
            z = p[2 * r_sc];
        }
        tc_pack_store(tcs + ((size_t)b * SpadT + (size_t)(j / NBR_TILE) * NBR_TILE) * 16, j % NBR_TILE, src < N, x, y, z, 1.0f);
    }
}

// ---- tcgen05 wrappers ------------------------------------------------------------------------
__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t saddr) {  // K-major, no swizzle
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)(TC_KCHUNK_BYTES >> 4) << 16) |
           ((uint64_t)(128u >> 4) << 32) | ((uint64_t)1 << 46);
}
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(TC_IDESC), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// 32 consecutive columns of this thread's TMEM lane (asynchronous: tc_ld_wait before use)
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,"
        "%26,%27,%28,%29,%30,%31}, [%32];"
        : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]),
          "=f"(v[8]), "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]),
          "=f"(v[15]), "=f"(v[16]), "=f"(v[17]), "=f"(v[18]), "=f"(v[19]), "=f"(v[20]), "=f"(v[21]),
          "=f"(v[22]), "=f"(v[23]), "=f"(v[24]), "=f"(v[25]), "=f"(v[26]), "=f"(v[27]), "=f"(v[28]),
          "=f"(v[29]), "=f"(v[30]), "=f"(v[31])
        : "r"(taddr)
        : "memory");
}
// wait for the outstanding tcgen05.ld; the registers are threaded through so that no use moves above
__device__ __forceinline__ void tc_ld_wait(float (&v)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]),
                   "+f"(v[7]), "+f"(v[8]), "+f"(v[9]), "+f"(v[10]), "+f"(v[11]), "+f"(v[12]), "+f"(v[13]),
                   "+f"(v[14]), "+f"(v[15]), "+f"(v[16]), "+f"(v[17]), "+f"(v[18]), "+f"(v[19]),
                   "+f"(v[20]), "+f"(v[21]), "+f"(v[22]), "+f"(v[23]), "+f"(v[24]), "+f"(v[25]),
                   "+f"(v[26]), "+f"(v[27]), "+f"(v[28]), "+f"(v[29]), "+f"(v[30]), "+f"(v[31])
                 :
                 : "memory");
}

// compiler-only barrier for a second register block covered by the same tcgen05.wait::ld
__device__ __forceinline__ void tc_ld_pin(float (&v)[32]) {
    asm volatile(""
                 : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]),
                   "+f"(v[7]), "+f"(v[8]), "+f"(v[9]), "+f"(v[10]), "+f"(v[11]), "+f"(v[12]), "+f"(v[13]),
                   "+f"(v[14]), "+f"(v[15]), "+f"(v[16]), "+f"(v[17]), "+f"(v[18]), "+f"(v[19]),
                   "+f"(v[20]), "+f"(v[21]), "+f"(v[22]), "+f"(v[23]), "+f"(v[24]), "+f"(v[25]),
                   "+f"(v[26]), "+f"(v[27]), "+f"(v[28]), "+f"(v[29]), "+f"(v[30]), "+f"(v[31])
                 :
                 : "memory");
}

// Flagged-group mask of one 32-ref step (bit 7 - u <=> group u has a negative filter value D' =
// A' - thr): min over the group (FMNMX3 + FMNMX), then its sign bit goes into the mask. The
// variant kept for comparison (TC_MASK_SHF_V = 0) tests the sign on the FMA pipe: sat(min * -inf) is
// exactly 1.0 for min < 0 and 0.0 otherwise (+-0 and NaN give NaN -> 0), one FFMA per group.
__device__ __forceinline__ float tc_sign_ind(float m) {
    float r;
    asm("mul.sat.f32 %0, %1, %2;" : "=f"(r) : "f"(m), "f"(__int_as_float(0xff800000)));
    return r;
}
#ifndef TC_WAIT_SYNCWARP_V  // (developer variant) 1: __syncwarp() between the accumulator wait and tcgen05.ld
#define TC_WAIT_SYNCWARP_V 0
#endif
#ifndef TC_MASK_SHF_V  // (developer variant) 1: the sign bit of the group minimum is shifted into the mask
#define TC_MASK_SHF_V 1  //                     (one funnel shift per group), 0: FMA-pipe indicator + FFMA
#endif
__device__ __forceinline__ uint32_t tc_step_mask(const float (&v)[32]) {
#if TC_MASK_SHF_V
    // mask = (mask << 1) | sign(min of the group): bit 7 - u <=> group u, one SHF per group. The sign
    // bit also flags a minimum of -0.0 (the exact evaluation then rejects it): still conservative.
    uint32_t mask = 0u;
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const float g = fminf(fminf(fminf(v[4 * u], v[4 * u + 1]), v[4 * u + 2]), v[4 * u + 3]);
        mask = __funnelshift_l(__float_as_uint(g), mask, 1);
    }
    return mask;
#else
    float acc[2] = {0.f, 0.f};
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const float g = fminf(fminf(fminf(v[4 * u], v[4 * u + 1]), v[4 * u + 2]), v[4 * u + 3]);
        acc[u & 1] = fmaf(tc_sign_ind(g), (float)(0x80u >> u), acc[u & 1]);
    }
    return __float2uint_rz(acc[0] + acc[1]);
#endif
}

// Work queue of an epilogue warp: one item per (query, PAIR of tiles 2p, 2p+1) with a flagged group,
//   mask: bit 31 - g <=> group (g & 15) of the warp's column half in tile 2p + (g >> 4) is flagged
//   meta: lane of the query | (p & 63) << 5
// kept in a circular buffer ACROSS tiles, so that a drain round always has 32 items: lane e takes
// item e, evaluates its first flagged group exactly against the tile's SoA rows (still in the
// ring) and appends the candidates below the query's bound to the query's list; items with more
// flagged groups go back to the head of the queue for the next round.
// Runs rounds while at least 32 items are queued, or the oldest item is from a tile before
// `min_tile` (the tile has to leave the ring). Returns the tile of the oldest item left.
template <int MODE>
__device__ __noinline__ int tc_drain(uint32_t *qm, uint32_t *qi, uint32_t &qhead, uint32_t qtail, int min_tile, int max_rounds,
                                     const float *qt, int quarter, int half, const unsigned char *ring, int t_now,
                                     int tile0, int N, uint32_t *ccnt, u64 *cand_unit, uint32_t cap) {
    constexpr int G4 = NBR_TILE / 4;
    const int lane = threadIdx.x & 31;
    const uint32_t lt_mask = (1u << lane) - 1u;
    int oldest = t_now + 1;
    for (int round = 0;; ++round) {
        const uint32_t size = qtail - qhead;
        if (size == 0u) {
            oldest = t_now + 1;
            break;
        }
        oldest = t_now - ((t_now - (int)(qi[qhead & (TC_QCAP - 1)] >> 5)) & 63);
        if ((size < 32u && oldest >= min_tile) || round >= max_rounds) break;
        const uint32_t n = size < 32u ? size : 32u;
        const bool e = (uint32_t)lane < n;
        const uint32_t pos = (qhead + lane) & (TC_QCAP - 1);
        uint32_t m = e ? qm[pos] : 0u;
        const uint32_t meta = e ? qi[pos] : 0u;
        const int owner = quarter * 32 + (int)(meta & 31u);
        const int pair = t_now - ((t_now - (int)(meta >> 5)) & 63);
        QueryRegs q;
        q.fa = qt[owner];
        q.fb = qt[128 + owner];
        q.fc = qt[256 + owner];
        q.s = qt[384 + owner];
        const float tau = qt[512 + owner];
        const uint32_t gb = e ? (uint32_t)__clz((int)m) : 0u;
        m &= ~(0x80000000u >> gb);
        const int tile = 2 * pair + (int)(gb >> 4);
        const uint32_t g = (uint32_t)half * 16u + (gb & 15u);  // group inside the tile
        const float4 *sX = reinterpret_cast<const float4 *>(ring + (size_t)(tile & (TC_STAGES - 1)) * TC_SOA_BYTES);
        const float4 X = sX[g], Y = sX[G4 + g], Z = sX[2 * G4 + g];
        const float4 Wn = mode_expanded(MODE) ? sX[3 * G4 + g] : make_float4(0.f, 0.f, 0.f, 0.f);
        float d[4];
        const uint32_t i0 = ((uint32_t)(tile0 + tile) * G4 + g) * 4u;
        dist4n<MODE>(q, X, Y, Z, Wn, i0, N, d);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (e && d[i] < tau) {
                const uint32_t slot = atomicAdd(&ccnt[owner], 1u);
                if (slot < cap) cand_unit[(size_t)slot * 128 + owner] = make_key(d[i], i0 + i);
            }
        }
        const bool left = m != 0u;
        const unsigned bal = __ballot_sync(0xffffffffu, left);
        const uint32_t newhead = qhead + n - (uint32_t)__popc(bal);
        __syncwarp();
        if (left) {
            const uint32_t w = (newhead + __popc(bal & lt_mask)) & (TC_QCAP - 1);
            qm[w] = m;
            qi[w] = meta;
        }
        __syncwarp();
        qhead = newhead;
    }
    return oldest;
}

template <int MODE>
__device__ __forceinline__ void nbr_scan_tc(const NbrParams &p, const ScanEvalParams &ep) {
    using SM = ScanTcSmem;
    constexpr int G4 = NBR_TILE / 4;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned char *ring = smem;
    float *aop = reinterpret_cast<float *>(smem + SM::ring);
    float *qtab_all = reinterpret_cast<float *>(smem + SM::ring + SM::aop);
    uint32_t *queue_all = reinterpret_cast<uint32_t *>(smem + SM::ring + SM::aop + SM::qtab);
    uint32_t *ccnt_all = reinterpret_cast<uint32_t *>(smem + SM::ring + SM::aop + SM::qtab + SM::queue);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + SM::ring + SM::aop + SM::qtab + SM::queue + SM::cnt);
    uint64_t *full = bars, *empty = bars + TC_STAGES;  // SoA ring
    uint64_t *bfull = bars + 2 * TC_STAGES, *bempty = bfull + TC_BSTAGES;  // operand ring
    uint64_t *acc_full = bempty + TC_BSTAGES, *acc_empty = acc_full + 2 * TC_UNITS;  // [unit][buffer]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_empty + 2 * TC_UNITS);
    unsigned char *sring = ring + ScanTcSmem::bring;

    const int b = blockIdx.z, split = blockIdx.y;
    const int tile0 = split * p.tiles_per_split;
    const int ntiles = min(p.tiles_per_split, p.total_tiles - tile0);
    const int scan_units = (p.S + 127) / 128;  // 128-query units of a cloud (= top-k kernel's grid)

    if (tid == 0) {
        for (int s = 0; s < TC_STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], TC_EPI_WARPS);
        }
        for (int s = 0; s < TC_BSTAGES; ++s) {
            mbar_init(&bfull[s], 1);
            mbar_init(&bempty[s], 1);
        }
        for (int j = 0; j < 2 * TC_UNITS; ++j) {
            mbar_init(&acc_full[j], 1);
            mbar_init(&acc_empty[j], 8);
        }
        mbar_fence_init();
    }
    if (warp == TC_EPI_WARPS + 1) {  // the MMA warp owns the tensor-memory allocation
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(TC_TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }

    // epilogue threads: query constants, A operand row, per-query tables
    const int unit = warp >> 3, half = (warp >> 2) & 1, quarter = warp & 3;
    const int owner = quarter * 32 + lane;  // row inside the unit = TMEM lane
    float thr = __int_as_float(0xff800000);  // -inf: never flagged
    if (warp < TC_EPI_WARPS) {
        const int qi = (blockIdx.x * TC_UNITS + unit) * 128 + owner;
        float x = 0.f, y = 0.f, z = 0.f, t0 = __int_as_float(0xff800000);
        if (qi < p.S) {
            const float *src = p.q + b * p.q_sb + qi * p.q_sp;
            x = src[p.q_ox];
            y = src[p.q_oy];
            z = src[2 * p.q_sc];
            t0 = p.tau_in ? p.tau_in[(size_t)b * p.S + qi] : p.tau_uniform;
        }
        QueryRegs q;
        q.set(x, y, z, p.q_xzy != 0);
        const float d0 = __fsub_rn(t0, q.s);
        thr = d0 + (0x1p-16f * q.s + 0x1p-21f * fabsf(d0));
        if (half == 0) {  // (both column halves hold the same queries)
        float *qt = qtab_all + unit * (5 * 128);
        qt[owner] = q.fa;
        qt[128 + owner] = q.fb;
        qt[256 + owner] = q.fc;
        qt[384 + owner] = q.s;
        qt[512 + owner] = t0;
        ccnt_all[unit * 128 + owner] = 0u;
        const float ah = tf32_hi(q.fa), bh = tf32_hi(q.fb), ch = tf32_hi(q.fc);
        const float al = tf32_hi(__fsub_rn(q.fa, ah)), bl = tf32_hi(__fsub_rn(q.fb, bh)),
                    cl = tf32_hi(__fsub_rn(q.fc, ch));
        float4 *arow = reinterpret_cast<float4 *>(aop + (size_t)unit * (TC_B_BYTES / 4)) + owner;
        // -thr in three exact TF32 pieces (invalid query / tau = -inf: +inf, never flagged)
        float n1 = __int_as_float(0x7f800000), n2 = 0.f, n3 = 0.f;
        if (fabsf(thr) < __int_as_float(0x7f800000)) {
            n1 = tf32_hi(-thr);
            const float r1 = __fsub_rn(-thr, n1);
            n2 = tf32_hi(r1);
            n3 = tf32_hi(__fsub_rn(r1, n2));
        } else if (thr > 0.f) {
            n1 = -n1;  // tau = +inf: every real ref is a candidate
        }
        arow[0] = make_float4(ah, bh, ch, 1.f);
        arow[NBR_TILE] = make_float4(ah, bh, ch, 1.f);
        arow[2 * NBR_TILE] = make_float4(al, bl, cl, 1.f);
        arow[3 * NBR_TILE] = make_float4(n1, n2, n3, 0.f);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // operand writes -> tensor core reads
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == TC_EPI_WARPS) {
        // ---- TMA producer ----
        if (lane == 0) {
            const float *tc_cloud = p.ws_tc + (size_t)b * p.Npad * 16;
            const float *ws = p.ws_ref + (size_t)b * 4 * p.Npad;
            // exact |r|^2 row (behind the operands of all clouds): only the expanded forms read it
            const float *nrm = p.ws_tc + (size_t)gridDim.z * p.Npad * 16 + (size_t)b * p.Npad;
            constexpr uint32_t soa_tx = (mode_expanded(MODE) ? 4u : 3u) * NBR_TILE * sizeof(float);
            for (int t = 0; t < ntiles; ++t) {
                const int s = t & (TC_STAGES - 1), sb = t & (TC_BSTAGES - 1);
                const int pp = t >> 1, ps = pp & (TC_STAGES / 2 - 1);  // the SoA barriers count tile PAIRS
                if (t >= TC_BSTAGES) mbar_wait_suspend(&bempty[sb], ((t / TC_BSTAGES) - 1) & 1);
                mbar_arrive_expect_tx(&bfull[sb], TC_B_BYTES);
                const int ta = tile0 + t;  // absolute tile
                tma_load_1d(ring + (size_t)sb * TC_B_BYTES, tc_cloud + (size_t)ta * NBR_TILE * 16, TC_B_BYTES, &bfull[sb]);
                unsigned char *st = sring + (size_t)s * TC_SOA_BYTES;
                if ((t & 1) == 0) {
                    if (t >= TC_STAGES) mbar_wait_suspend(&empty[ps], ((pp / (TC_STAGES / 2)) - 1) & 1);
                    mbar_arrive_expect_tx(&full[ps], (t + 1 < ntiles ? 2u : 1u) * soa_tx);
                }
#pragma unroll
                for (int r = 0; r < 3; ++r)
                    tma_load_1d(st + r * NBR_TILE * sizeof(float),
                                ws + (size_t)r * p.Npad + (size_t)ta * NBR_TILE,
                                NBR_TILE * sizeof(float), &full[ps]);
                if (mode_expanded(MODE))
                    tma_load_1d(st + 3 * NBR_TILE * sizeof(float), nrm + (size_t)ta * NBR_TILE,
                                NBR_TILE * sizeof(float), &full[ps]);
            }
        }
    } else if (warp == TC_EPI_WARPS + 1) {
        // ---- MMA issuer ----
        if (lane == 0) {
            for (int t = 0; t < ntiles; ++t) {
                const int sb = t & (TC_BSTAGES - 1);
                mbar_wait_suspend(&bfull[sb], (t / TC_BSTAGES) & 1);
                tc_fence_after();
                const uint32_t bsm = smem_u32(ring + (size_t)sb * TC_B_BYTES);
                const int buf = t & 1;
#pragma unroll
                for (int j = 0; j < TC_UNITS; ++j) {
                    if (t >= 2) {
                        mbar_wait_suspend(&acc_empty[2 * j + buf], ((t >> 1) - 1) & 1);
                        tc_fence_after();
                    }
                    const uint32_t asm_ = smem_u32(aop) + j * TC_B_BYTES;
                    const uint32_t d = tmem_base + (2 * j + buf) * NBR_TILE;
                    tc_mma(d, tc_smem_desc(asm_), tc_smem_desc(bsm), 0u);
                    tc_mma(d, tc_smem_desc(asm_ + 2 * TC_KCHUNK_BYTES), tc_smem_desc(bsm + 2 * TC_KCHUNK_BYTES), 1u);
                    tc_commit(&acc_full[2 * j + buf]);
                }
                tc_commit(&bempty[sb]);  // the operand stage is free once these MMAs have read it
            }
        }
    } else {
        // ---- epilogue: filter compare, queue, exact drain ----
        const int unit_index = blockIdx.x * TC_UNITS + unit;
        const bool unit_valid = unit_index < scan_units;
        const size_t unit_linear = (size_t)(blockIdx.z * gridDim.y + blockIdx.y) * scan_units + (unit_valid ? unit_index : 0);
        u64 *cand_unit = ep.cand + unit_linear * (size_t)ep.cap * 128;
        const float *qt = qtab_all + unit * (5 * 128);
        uint32_t *ccnt = ccnt_all + unit * 128;
        uint32_t *qm = queue_all + warp * (2 * TC_QCAP), *qi = qm + TC_QCAP;
        const uint32_t lt_mask = (1u << lane) - 1u;
        const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) + 2 * unit * NBR_TILE + half * TC_HALF;
        uint32_t qhead = 0u, qtail = 0u;
        int t_oldest = 0;   // tile of the oldest queued item (queue not empty)
        int released = 0;   // ring stages of tile pairs < released have been handed back
        // (t_oldest, t_now of tc_drain count tile PAIRS here)
        const int npairs = (ntiles + 1) / 2;
#pragma unroll 1
        for (int pr = 0; pr < npairs; ++pr) {
            uint32_t m32 = 0u;
#pragma unroll
            for (int buf = 0; buf < 2; ++buf) {  // tiles 2 pr (accumulator 0) and 2 pr + 1 (accumulator 1)
                const int t = 2 * pr + buf;
                if (t < ntiles) {
                    float va[32], vb[32];
                    // wait for the accumulator; while it is not there, do pending exact work (one round at a time)
#if TC_SHADOW_V
                    bool ready = false;
                    while (!ready) {
                        ready = __all_sync(0xffffffffu, mbar_try_wait(&acc_full[2 * unit + buf], pr & 1));
                        if (!ready && qtail - qhead >= 32u)
                            t_oldest = tc_drain<MODE>(qm, qi, qhead, qtail, -0x40000000, 1, qt, quarter, half, sring, pr, tile0,
                                                      p.N | (p.r_xzy ? NBR_N_XZY : 0), ccnt, cand_unit, (uint32_t)ep.cap);
                    }
#else
                    mbar_wait(&acc_full[2 * unit + buf], pr & 1);
#if TC_WAIT_SYNCWARP_V
                    __syncwarp();  // (the wait loop reconverges on its own; the explicit barrier costs 6 issue slots per tile)
#endif
#endif
                    tc_fence_after();
                    tc_ld32(trow + buf * NBR_TILE, va);
                    tc_ld32(trow + buf * NBR_TILE + 32, vb);
                    tc_ld_wait(va);
                    tc_ld_pin(vb);
                    // this warp's 64 columns are in registers: release the accumulator
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc_empty[2 * unit + buf]);
                    m32 |= ((tc_step_mask(va) << 8) | tc_step_mask(vb)) << (16 - 16 * buf);
                }
            }
            // the pair's SoA rows (TMA writes, one barrier per pair), for the drain
            mbar_wait(&full[(uint32_t)pr & (TC_STAGES / 2 - 1)], ((uint32_t)pr / (TC_STAGES / 2)) & 1);
            // queue the (query, tile pair) items
            const bool f = m32 != 0u;
            const unsigned bal = __ballot_sync(0xffffffffu, f);
            if (qhead == qtail) t_oldest = pr;
            if (f) {
                const uint32_t w = (qtail + __popc(bal & lt_mask)) & (TC_QCAP - 1);
                qm[w] = m32;
                qi[w] = (uint32_t)lane | ((uint32_t)(pr & 63) << 5);
            }
            qtail += __popc(bal);
            __syncwarp();
            // exact evaluation in full rounds of 32 items; older items when their tiles have to
            // leave the ring; everything when the split ends
            const uint32_t size = qtail - qhead;
            const bool last = pr == npairs - 1;
            if (size >= TC_DRAIN_AT_V || (size > 0u && (pr - t_oldest >= TC_HOLD_PAIRS || last)))
                t_oldest = tc_drain<MODE>(qm, qi, qhead, qtail, last ? pr + 1 : pr - TC_HOLD_PAIRS + 1, last ? (1 << 30) : TC_ROUNDS_V, qt,
                                          quarter, half, sring, pr, tile0, p.N | (p.r_xzy ? NBR_N_XZY : 0), ccnt, cand_unit, (uint32_t)ep.cap);
            const int p_free = (qhead != qtail) ? t_oldest : pr + 1;  // pairs < p_free leave the ring
            __syncwarp();
            if (lane == 0) {
#pragma unroll 1
                for (uint32_t r = (uint32_t)released; r < (uint32_t)p_free; ++r) mbar_arrive(&empty[r & (TC_STAGES / 2 - 1)]);
            }
            released = p_free;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp < TC_EPI_WARPS && half == 0) {  // both column halves have appended: publish the list lengths
        const int unit_index = blockIdx.x * TC_UNITS + unit;
        if (unit_index < scan_units)
            ep.cand_cnt[((size_t)(blockIdx.z * gridDim.y + blockIdx.y) * scan_units + unit_index) * 128 + owner] =
                ccnt_all[unit * 128 + owner];
    }
    if (warp == TC_EPI_WARPS + 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TC_TMEM_COLS) : "memory");
    }
}

// ---- threshold pre-pass on the tensor cores -----------------------------------------------------
// The same MMA pipeline over the SAMPLE operand (refs 0, 8, 16, ... packed like the ref tiles,
// SpadT slots = a multiple of 1024): the epilogue keeps, per query, the running minimum of the
// filter value over a bucket (G consecutive 32-column chunks of the warp's column half; 16 buckets
// per half, 32 per query -- at 16384 refs exactly the 64-ref buckets of knn_tau_kernel) and the
// RMAX smallest bucket minima in a sorted list; the two column halves merge their lists through
// shared memory. tau[b,q] = R-th smallest bucket minimum + |q|^2 (+ slack in guaranteed-bound mode).
// The pre-pass has only Spad / 128 (16 at 16384 refs) tiles per CTA, so CTA start-up and tear-down
// matter: its CTAs own ONE 128-query unit (256 TMEM columns, 10 warps, 79 KB of shared memory), two
// of them share an SM and overlap each other's prologue.
constexpr int TAU_TC_STAGES = 8;
constexpr int TAU_UNITS = 1;
constexpr int TAU_EPI_WARPS = TAU_UNITS * 8;
constexpr int TAU_THREADS = (TAU_EPI_WARPS + 2) * 32;
constexpr uint32_t TAU_TMEM_COLS = 2 * TAU_UNITS * NBR_TILE;
struct TauTcSmem {
    static constexpr size_t ring = (size_t)TAU_TC_STAGES * TC_B_BYTES;
    static constexpr size_t aop = (size_t)TAU_UNITS * TC_B_BYTES;
    static constexpr size_t merge = (size_t)12 * TAU_UNITS * 128 * sizeof(float);
    static constexpr size_t ctrl = 512;
    static constexpr size_t total = ring + aop + merge + ctrl;
};

__device__ __forceinline__ float tc_min32(const float (&v)[32]) {
    float m[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        m[c] = fminf(fminf(v[8 * c], v[8 * c + 1]), v[8 * c + 2]);
        m[c] = fminf(fminf(m[c], v[8 * c + 3]), v[8 * c + 4]);
        m[c] = fminf(fminf(m[c], v[8 * c + 5]), v[8 * c + 6]);
        m[c] = fminf(m[c], v[8 * c + 7]);
    }
    return fminf(fminf(fminf(m[0], m[1]), m[2]), m[3]);
}

// one 32-column chunk's minimum: extend the current bucket; when the bucket ends (G chunks), fold
// its minimum into the sorted list of the RMAX smallest bucket minima
template <int RMAX>
__device__ __forceinline__ void tau_chunk(float v, float &m, int &cib, int G, float (&top)[RMAX]) {
    m = fminf(m, v);
    if (++cib == G) {
        float x = m;
#pragma unroll
        for (int r = 0; r < RMAX; ++r) {
            const float lo = fminf(top[r], x);
            x = fmaxf(top[r], x);
            top[r] = lo;
        }
        m = __int_as_float(0x7f800000);
        cib = 0;
    }
}

template <int RMAX>
__device__ __forceinline__ void nbr_tau_tc(const NbrParams &p, const float *tcs, int SpadT, int R, float *tau_out,
                                           float tau_scale, float slack_rel) {
    using SM = TauTcSmem;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned char *ring = smem;
    float *aop = reinterpret_cast<float *>(smem + SM::ring);
    float *merge = reinterpret_cast<float *>(smem + SM::ring + SM::aop);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + SM::ring + SM::aop + SM::merge);
    uint64_t *full = bars, *empty = bars + TAU_TC_STAGES, *acc_full = bars + 2 * TAU_TC_STAGES,
             *acc_empty = bars + 2 * TAU_TC_STAGES + 2 * TAU_UNITS;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * TAU_TC_STAGES + 4 * TAU_UNITS);
    const int b = blockIdx.z;
    const int ntiles = SpadT / NBR_TILE;
    const int G = SpadT / 1024;  // 32-column chunks per bucket
    const float inf = __int_as_float(0x7f800000);

    if (tid == 0) {
        for (int s = 0; s < TAU_TC_STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], TAU_EPI_WARPS);
        }
        for (int j = 0; j < 2 * TAU_UNITS; ++j) {
            mbar_init(&acc_full[j], 1);
            mbar_init(&acc_empty[j], 8);
        }
        mbar_fence_init();
    }
    if (warp == TAU_EPI_WARPS + 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(TAU_TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    const int unit = warp >> 3, half = (warp >> 2) & 1, quarter = warp & 3;
    const int owner = quarter * 32 + lane;
    const int qi = (blockIdx.x * TAU_UNITS + unit) * 128 + owner;
    float qs = 0.f;
    if (warp < TAU_EPI_WARPS) {
        float x = 0.f, y = 0.f, z = 0.f;
        if (qi < p.S) {
            const float *src = p.q + b * p.q_sb + qi * p.q_sp;
            x = src[p.q_ox];
            y = src[p.q_oy];
            z = src[2 * p.q_sc];
        }
        QueryRegs q;
        q.set(x, y, z);
        qs = q.s;
        if (half == 0) {
            const float ah = tf32_hi(q.fa), bh = tf32_hi(q.fb), ch = tf32_hi(q.fc);
            const float al = tf32_hi(__fsub_rn(q.fa, ah)), bl = tf32_hi(__fsub_rn(q.fb, bh)),
                        cl = tf32_hi(__fsub_rn(q.fc, ch));
            float4 *arow = reinterpret_cast<float4 *>(aop + (size_t)unit * (TC_B_BYTES / 4)) + owner;
            arow[0] = make_float4(ah, bh, ch, 1.f);
            arow[NBR_TILE] = make_float4(ah, bh, ch, 1.f);
            arow[2 * NBR_TILE] = make_float4(al, bl, cl, 1.f);
            arow[3 * NBR_TILE] = make_float4(0.f, 0.f, 0.f, 0.f);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    float top[RMAX];  // the RMAX smallest bucket minima of this thread's column half, ascending
#pragma unroll
    for (int r = 0; r < RMAX; ++r) top[r] = inf;

    if (warp == TAU_EPI_WARPS) {
        if (lane == 0) {  // TMA producer
            const float *cloud = tcs + (size_t)b * SpadT * 16;
            for (int t = 0; t < ntiles; ++t) {
                const int s = t % TAU_TC_STAGES;
                if (t >= TAU_TC_STAGES) mbar_wait_suspend(&empty[s], ((t / TAU_TC_STAGES) - 1) & 1);
                mbar_arrive_expect_tx(&full[s], TC_B_BYTES);
                tma_load_1d(ring + (size_t)s * TC_B_BYTES, cloud + (size_t)t * NBR_TILE * 16, TC_B_BYTES, &full[s]);
            }
        }
    } else if (warp == TAU_EPI_WARPS + 1) {
        if (lane == 0) {  // MMA issuer
            for (int t = 0; t < ntiles; ++t) {
                const int s = t % TAU_TC_STAGES;
                mbar_wait_suspend(&full[s], (t / TAU_TC_STAGES) & 1);
                tc_fence_after();
                const uint32_t bsm = smem_u32(ring + (size_t)s * TC_B_BYTES);
                const int buf = t & 1;
#pragma unroll
                for (int j = 0; j < TAU_UNITS; ++j) {
                    if (t >= 2) {
                        mbar_wait_suspend(&acc_empty[2 * j + buf], ((t >> 1) - 1) & 1);
                        tc_fence_after();
                    }
                    const uint32_t asm_ = smem_u32(aop) + j * TC_B_BYTES;
                    const uint32_t d = tmem_base + (2 * j + buf) * NBR_TILE;
                    tc_mma(d, tc_smem_desc(asm_), tc_smem_desc(bsm), 0u);
                    tc_mma(d, tc_smem_desc(asm_ + 2 * TC_KCHUNK_BYTES), tc_smem_desc(bsm + 2 * TC_KCHUNK_BYTES), 1u);
                    tc_commit(&acc_full[2 * j + buf]);
                }
            }
        }
    } else {
        const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) + 2 * unit * NBR_TILE + half * TC_HALF;
        float m = inf;
        int cib = 0;  // chunks in the current bucket
#pragma unroll 1
        for (int t = 0; t < ntiles; ++t) {
            const int buf = t & 1;
            float va[32], vb[32];
            mbar_wait(&acc_full[2 * unit + buf], (t >> 1) & 1);
            tc_fence_after();
            tc_ld32(trow + buf * NBR_TILE, va);
            tc_ld32(trow + buf * NBR_TILE + 32, vb);
            tc_ld_wait(va);
            tc_ld_pin(vb);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&acc_empty[2 * unit + buf]);
                mbar_arrive(&empty[t % TAU_TC_STAGES]);  // (the MMA that filled this accumulator has read the stage)
            }
            tau_chunk<RMAX>(tc_min32(va), m, cib, G, top);
            tau_chunk<RMAX>(tc_min32(vb), m, cib, G, top);
        }
        if (half == 1) {
#pragma unroll
            for (int r = 0; r < RMAX; ++r) merge[(r * TAU_UNITS + unit) * 128 + owner] = top[r];
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp < TAU_EPI_WARPS && half == 0) {
#pragma unroll
        for (int i = 0; i < RMAX; ++i) {
            float x = merge[(i * TAU_UNITS + unit) * 128 + owner];
#pragma unroll
            for (int r = 0; r < RMAX; ++r) {
                const float lo = fminf(top[r], x);
                x = fmaxf(top[r], x);
                top[r] = lo;
            }
        }
        float t = top[0];
#pragma unroll
        for (int r = 1; r < RMAX; ++r) t = (r == R - 1) ? top[r] : t;
        t += qs;                                // back to a distance
        t += slack_rel * (qs + fabsf(t));       // guaranteed-bound mode (see knn_tau_kernel)
        if (qi < p.S) tau_out[(size_t)b * p.S + qi] = (tau_scale == 1.0f) ? t : t * tau_scale;
    }
    if (warp == TAU_EPI_WARPS + 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TAU_TMEM_COLS) : "memory");
    }
}

}  // namespace b200pci
