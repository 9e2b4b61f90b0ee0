// Furthest point sampling -- replaces pointnet2/src/sampling_gpu.cu:93-253.
//
// One CTA per cloud. Every thread keeps its points (x, y, z) and their running min-distance
// `temp` in registers for the whole call (the reference re-reads both from global memory in each
// of the npoint-1 iterations, sampling_gpu.cu:123-131); the cloud is mirrored once in shared
// memory so the coordinates of the last pick are a broadcast LDS. The block-wide argmax is two
// REDUX rounds on a 64-bit key per level and ONE __syncthreads per iteration (the reference
// runs a 10-step shared-memory tree with a barrier per step, :143-203).
//
// Tie order == the reference's: inside a reference thread the lowest k wins (:136-137, strict >);
// across threads the tree keeps the left operand on equality (:86-91), i.e. among equal distances
// the candidate whose reference thread id (k mod block, block = opt_n_threads(N),
// cuda_utils.h:10-14) has the smallest BIT-REVERSED value wins. The key encodes exactly that:
//   key = dist_bits << 32 | ~prio,   prio = bitrev(k mod block) << hb | (k / block).
#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace b200pci {

constexpr int FPS_MAX_THREADS = 1024;
}  // namespace b200pci
extern int g_fps_single_cta;
namespace b200pci {

struct FpsGeom {
    int log2bs;  // log2 of the reference block size
    int hb;      // bits for k / block
};

__device__ __forceinline__ uint32_t fps_prio(uint32_t k, const FpsGeom g) {
    const uint32_t t = k & ((1u << g.log2bs) - 1u);
    const uint32_t rb = g.log2bs ? (__brev(t) >> (32 - g.log2bs)) : 0u;
    return (rb << g.hb) | (k >> g.log2bs);
}
__device__ __forceinline__ uint32_t fps_unprio(uint32_t prio, const FpsGeom g) {
    const uint32_t hi = prio & ((1u << g.hb) - 1u);
    const uint32_t rb = prio >> g.hb;
    const uint32_t t = g.log2bs ? (__brev(rb) >> (32 - g.log2bs)) : 0u;
    return (hi << g.log2bs) | t;
}

// (max dist, then max low) over the warp; returns the packed key in every lane.
__device__ __forceinline__ unsigned long long warp_argmax_key(uint32_t db, uint32_t low) {
    const uint32_t m1 = __reduce_max_sync(0xffffffffu, db);
    const uint32_t m2 = __reduce_max_sync(0xffffffffu, (db == m1) ? low : 0u);
    return ((unsigned long long)m1 << 32) | m2;
}

// PT > 0: points in registers (n <= PT * blockDim.x). PT == 0: points stay in global memory.
template <int PT, bool XYZ_SMEM>
__global__ void __launch_bounds__(FPS_MAX_THREADS, 1)
    fps_kernel(int n, int m, const float *__restrict__ xyz_all, float *__restrict__ temp_all,
               int *__restrict__ idx_all, FpsGeom g) {
    extern __shared__ float sxyz[];  // [3n] when XYZ_SMEM
    __shared__ unsigned long long part[2][32];
    const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, warp = tid >> 5;
    const int nwarps = nth >> 5;
    const float *xyz = xyz_all + (size_t)blockIdx.x * n * 3;
    float *temp = temp_all + (size_t)blockIdx.x * n;
    int *idx = idx_all + (size_t)blockIdx.x * m;

    constexpr int PTR = PT > 0 ? PT : 1;
    float px[PTR], py[PTR], pz[PTR], pt[PTR];
    if (PT > 0) {
#pragma unroll
        for (int i = 0; i < PTR; ++i) {
            const int k = tid + i * nth;
            if (k < n) {
                px[i] = xyz[k * 3 + 0];
                py[i] = xyz[k * 3 + 1];
                pz[i] = xyz[k * 3 + 2];
                pt[i] = temp[k];
            } else {
                px[i] = py[i] = pz[i] = 0.f;
                pt[i] = -1.f;  // min(d,-1) = -1 can never beat a real point (d2 >= 0)
            }
        }
    }
    if (XYZ_SMEM)
        for (int t = tid; t < 3 * n; t += nth) sxyz[t] = xyz[t];
    if (tid == 0) idx[0] = 0;
    __syncthreads();

    int old = 0;
    for (int j = 1; j < m; ++j) {
        float x1, y1, z1;
        if (XYZ_SMEM) {
            x1 = sxyz[old * 3 + 0];
            y1 = sxyz[old * 3 + 1];
            z1 = sxyz[old * 3 + 2];
        } else {
            x1 = __ldg(xyz + old * 3 + 0);
            y1 = __ldg(xyz + old * 3 + 1);
            z1 = __ldg(xyz + old * 3 + 2);
        }
        float best = -1.f;
        int bk = 0;
        if (PT > 0) {
            int bi = 0;
#pragma unroll
            for (int i = 0; i < PTR; ++i) {
                const float dx = __fsub_rn(px[i], x1), dy = __fsub_rn(py[i], y1),
                            dz = __fsub_rn(pz[i], z1);
                const float d = __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
                const float d2 = fminf(d, pt[i]);
                pt[i] = d2;
                const bool gt = d2 > best;
                bi = gt ? i : bi;
                best = gt ? d2 : best;
            }
            bk = tid + bi * nth;
        } else {
            for (int k = tid; k < n; k += nth) {
                const float dx = __fsub_rn(xyz[k * 3 + 0], x1), dy = __fsub_rn(xyz[k * 3 + 1], y1),
                            dz = __fsub_rn(xyz[k * 3 + 2], z1);
                const float d = __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
                const float d2 = fminf(d, temp[k]);
                temp[k] = d2;
                const bool gt = d2 > best;
                bk = gt ? k : bk;
                best = gt ? d2 : best;
            }
        }
        // Threads of OUR block own several reference threads' worth of points only when the
        // reference block is 1024 too (then k mod 1024 == tid for all of them), so "lowest local
        // slot wins" above is the reference's in-thread rule; for smaller clouds PT == 1.
        const bool has = best >= 0.f;
        const uint32_t db = has ? __float_as_uint(best) : 0u;
        const uint32_t low = has ? ~fps_prio((uint32_t)bk, g) : 0u;
        const unsigned long long wk = warp_argmax_key(db, low);
        if (lane == 0) part[j & 1][warp] = wk;
        __syncthreads();
        const unsigned long long v = (lane < nwarps) ? part[j & 1][lane] : 0ull;
        const unsigned long long fk = warp_argmax_key((uint32_t)(v >> 32), (uint32_t)v);
        old = (int)fps_unprio(~(uint32_t)fk, g);
        if (tid == 0) idx[j] = old;
    }
    if (PT > 0 && m > 1) {
#pragma unroll
        for (int i = 0; i < PTR; ++i) {
            const int k = tid + i * nth;
            if (k < n) temp[k] = pt[i];
        }
    }
}

// ---- thread-block-cluster variant -------------------------------------------------------------
// One cloud per cluster of FPS_CS CTAs (one CTA per SM): a single CTA per cloud leaves all but B of
// the 148 SMs idle and needs 16 points per thread at N=16384. Here CTA r owns the contiguous point
// range [r*chunk, (r+1)*chunk) in registers and every CTA mirrors the whole cloud in shared
// memory. Per iteration each CTA reduces its own best key (REDUX + one __syncthreads) and sends
// the 8-byte key to EVERY CTA of the cluster with `st.async` (a DSMEM store that also completes
// bytes on the receiver's mbarrier); a CTA waits on its own mbarrier only, then all CTAs pick the
// same winner from the 8 keys and read its coordinates from their mirror. No cluster-wide
// barrier in the loop. The key is the same 64-bit (distance, reference tie priority) as above.
#ifndef FPS_CS_V  // (developer variants: tools/variants.sh)
#define FPS_CS_V 8
#endif
#ifndef FPS_CT_V
#define FPS_CT_V 512
#endif
constexpr int FPS_CS = FPS_CS_V;
constexpr int FPS_CT = FPS_CT_V;  // threads per CTA

__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_async_u64(uint32_t remote_addr, unsigned long long v,
                                             uint32_t remote_bar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];" ::"r"(
                     remote_addr),
                 "l"(v), "r"(remote_bar)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}

template <int PT, bool MIRROR, int CS, int CT>
__global__ void __launch_bounds__(CT, 1)
    fps_cluster_kernel(int n, int m, int chunk, const float *__restrict__ xyz_all,
                       float *__restrict__ temp_all, int *__restrict__ idx_all, FpsGeom g) {
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned rank = cluster.block_rank();
    const int cloud = blockIdx.x / CS;
    extern __shared__ float sxyz[];  // the whole cloud, [3n] (MIRROR)
    __shared__ unsigned long long part[CT / 32];
    __shared__ __align__(8) unsigned long long rec[2][CS];
    __shared__ __align__(8) uint64_t bar[2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *xyz = xyz_all + (size_t)cloud * n * 3;
    float *temp = temp_all + (size_t)cloud * n;
    int *idx = idx_all + (size_t)cloud * m;
    const int k0 = rank * chunk, k1 = min(n, k0 + chunk);

    float px[PT], py[PT], pz[PT], pt[PT];
    uint32_t plow[PT];  // ~priority of the point (0 = no point)
#pragma unroll
    for (int i = 0; i < PT; ++i) {
        const int k = k0 + tid + i * CT;
        if (k < k1) {
            px[i] = xyz[k * 3 + 0];
            py[i] = xyz[k * 3 + 1];
            pz[i] = xyz[k * 3 + 2];
            pt[i] = temp[k];
            plow[i] = ~fps_prio((uint32_t)k, g);
        } else {
            px[i] = py[i] = pz[i] = 0.f;
            pt[i] = -1.f;
            plow[i] = 0u;
        }
    }
    if (MIRROR)
        for (int t = tid; t < 3 * n; t += CT) sxyz[t] = xyz[t];
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        mbar_fence_init();
        if (rank == 0) idx[0] = 0;
    }
    float x1 = xyz[0], y1 = xyz[1], z1 = xyz[2];
    __syncthreads();
    cluster.sync();  // every CTA's barriers are initialised before the first remote store

    for (int j = 1; j < m; ++j) {
        const int s = j & 1;
        if (tid == 0) mbar_arrive_expect_tx(&bar[s], CS * sizeof(unsigned long long));
        uint32_t bd = 0u, bl = 0u;  // best (distance bits, ~priority) of this thread
#pragma unroll
        for (int i = 0; i < PT; ++i) {
            const float dx = __fsub_rn(px[i], x1), dy = __fsub_rn(py[i], y1), dz = __fsub_rn(pz[i], z1);
            const float d = __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
            const float d2 = fminf(d, pt[i]);
            pt[i] = d2;
            const uint32_t db = (d2 >= 0.f) ? __float_as_uint(d2) : 0u;  // -1 marks "no point"
            const bool better = (db > bd) || (db == bd && plow[i] > bl);
            bd = better ? db : bd;
            bl = better ? plow[i] : bl;
        }
        const unsigned long long wk = warp_argmax_key(bd, bl);
        if (lane == 0) part[warp] = wk;
        __syncthreads();
        if (warp == 0) {
            const unsigned long long v = (lane < CT / 32) ? part[lane] : 0ull;
            const unsigned long long ck = warp_argmax_key((uint32_t)(v >> 32), (uint32_t)v);
            if (lane < CS)  // lane l sends this CTA's key to CTA l (including itself)
                st_async_u64(mapa_u32(smem_u32(&rec[s][rank]), lane), ck,
                             mapa_u32(smem_u32(&bar[s]), lane));
        }
        while (!mbar_try_wait_cluster(&bar[s], ((j - 1) >> 1) & 1)) {
        }
        // all CTAs see the same 8 keys -> the same winner
        unsigned long long best = 0ull;
#pragma unroll
        for (int r = 0; r < CS; ++r) {
            const unsigned long long c = rec[s][r];
            best = c > best ? c : best;
        }
        const int old = (int)fps_unprio(~(uint32_t)best, g);
        if (MIRROR) {
            x1 = sxyz[old * 3 + 0];
            y1 = sxyz[old * 3 + 1];
            z1 = sxyz[old * 3 + 2];
        } else {
            x1 = __ldg(xyz + old * 3 + 0);
            y1 = __ldg(xyz + old * 3 + 1);
            z1 = __ldg(xyz + old * 3 + 2);
        }
        if (rank == 0 && tid == 0) idx[j] = old;
    }
    if (m > 1) {
#pragma unroll
        for (int i = 0; i < PT; ++i) {
            const int k = k0 + tid + i * CT;
            if (k < k1) temp[k] = pt[i];
        }
    }
    cluster.sync();  // no CTA exits while a peer may still write into it
}

// ---- pytorch3d form (b200pci_fps_p3d) ------------------------------------------------------------
// The cluster scheme above with pytorch3d's sample_farthest_points rules: per cloud n = lengths[b]
// points and m = min(K[b], n) picks (both read here, on the device), the first pick start[b], the
// running minimum starts at +inf (no temp buffer), d = fma(dz,dz,fma(dy,dy,dx*dx)), and the tie key
// is the point index itself (~k: the lowest index wins). Picks m..M-1 are written as -1 with zero
// rows. Points are read through element strides; the mirror holds them as [n][3].
constexpr int FPS3_CS = 8, FPS3_CT = 512;

struct Fps3Args {
    int N, M, chunk;
    const float *xyz;
    long long sb, sp, sc;
    const long long *lengths, *K, *start;  // [B] each, nullable
    long long *idx;                        // [B, M]
    float *sel;                            // [B, M, 3], nullable
};

template <int PT, bool MIRROR>
__global__ void __launch_bounds__(FPS3_CT, 1) fps_p3d_cluster_kernel(Fps3Args a) {
    constexpr int CS = FPS3_CS, CT = FPS3_CT;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned rank = cluster.block_rank();
    const int cloud = blockIdx.x / CS;
    extern __shared__ float sxyz[];  // the cloud's n points, [n][3] (MIRROR)
    __shared__ unsigned long long part[CT / 32];
    __shared__ __align__(8) unsigned long long rec[2][CS];
    __shared__ __align__(8) uint64_t bar[2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *xyz = a.xyz + cloud * a.sb;
    const long long nl = a.lengths ? a.lengths[cloud] : a.N;
    const int n = (int)(nl < 0 ? 0 : (nl > a.N ? a.N : nl));
    const long long kl = a.K ? a.K[cloud] : a.M;
    const int m = (int)min((long long)n, kl < 0 ? 0 : (kl > a.M ? a.M : kl));
    long long *idx = a.idx + (size_t)cloud * a.M;
    float *sel = a.sel ? a.sel + (size_t)cloud * a.M * 3 : nullptr;
    const int k0 = rank * a.chunk, k1 = min(n, k0 + a.chunk);

    if (rank == 0)
        for (int j = m + tid; j < a.M; j += CT) {
            idx[j] = -1;
            if (sel) sel[3 * j] = sel[3 * j + 1] = sel[3 * j + 2] = 0.f;
        }
    float px[PT], py[PT], pz[PT], pt[PT];
    uint32_t plow[PT];  // ~index of the point (0 = no point)
#pragma unroll
    for (int i = 0; i < PT; ++i) {
        const int k = k0 + tid + i * CT;
        if (k < k1) {
            const float *p = xyz + k * a.sp;
            px[i] = p[0];
            py[i] = p[a.sc];
            pz[i] = p[2 * a.sc];
            pt[i] = __int_as_float(0x7f800000);
            plow[i] = ~(uint32_t)k;
        } else {
            px[i] = py[i] = pz[i] = 0.f;
            pt[i] = -1.f;
            plow[i] = 0u;
        }
    }
    if (MIRROR)
        for (int k = tid; k < n; k += CT) {
            const float *p = xyz + k * a.sp;
            sxyz[3 * k] = p[0];
            sxyz[3 * k + 1] = p[a.sc];
            sxyz[3 * k + 2] = p[2 * a.sc];
        }
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        mbar_fence_init();
    }
    int old = 0;
    float x1 = 0.f, y1 = 0.f, z1 = 0.f;
    if (m > 0) {
        const long long s = a.start ? a.start[cloud] : 0;
        old = (int)(s < 0 ? 0 : (s >= n ? n - 1 : s));
        const float *p = xyz + old * a.sp;
        x1 = p[0];
        y1 = p[a.sc];
        z1 = p[2 * a.sc];
        if (rank == 0 && tid == 0) {
            idx[0] = old;
            if (sel) sel[0] = x1, sel[1] = y1, sel[2] = z1;
        }
    }
    __syncthreads();
    cluster.sync();  // every CTA's barriers are initialised before the first remote store

    for (int j = 1; j < m; ++j) {
        const int s = j & 1;
        if (tid == 0) mbar_arrive_expect_tx(&bar[s], CS * sizeof(unsigned long long));
        uint32_t bd = 0u, bl = 0u;  // best (distance bits, ~index) of this thread
#pragma unroll
        for (int i = 0; i < PT; ++i) {
            const float dx = __fsub_rn(px[i], x1), dy = __fsub_rn(py[i], y1), dz = __fsub_rn(pz[i], z1);
            const float d = __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
            const float d2 = fminf(d, pt[i]);
            pt[i] = d2;
            const uint32_t db = (d2 >= 0.f) ? __float_as_uint(d2) : 0u;  // -1 marks "no point"
            const bool better = (db > bd) || (db == bd && plow[i] > bl);
            bd = better ? db : bd;
            bl = better ? plow[i] : bl;
        }
        const unsigned long long wk = warp_argmax_key(bd, bl);
        if (lane == 0) part[warp] = wk;
        __syncthreads();
        if (warp == 0) {
            const unsigned long long v = (lane < CT / 32) ? part[lane] : 0ull;
            const unsigned long long ck = warp_argmax_key((uint32_t)(v >> 32), (uint32_t)v);
            if (lane < CS)
                st_async_u64(mapa_u32(smem_u32(&rec[s][rank]), lane), ck,
                             mapa_u32(smem_u32(&bar[s]), lane));
        }
        while (!mbar_try_wait_cluster(&bar[s], ((j - 1) >> 1) & 1)) {
        }
        unsigned long long best = 0ull;
#pragma unroll
        for (int r = 0; r < CS; ++r) {
            const unsigned long long c = rec[s][r];
            best = c > best ? c : best;
        }
        old = (int)~(uint32_t)best;
        if (MIRROR) {
            x1 = sxyz[old * 3 + 0];
            y1 = sxyz[old * 3 + 1];
            z1 = sxyz[old * 3 + 2];
        } else {
            const float *p = xyz + old * a.sp;
            x1 = __ldg(p);
            y1 = __ldg(p + a.sc);
            z1 = __ldg(p + 2 * a.sc);
        }
        if (rank == 0 && tid == 0) {
            idx[j] = old;
            if (sel) sel[3 * j] = x1, sel[3 * j + 1] = y1, sel[3 * j + 2] = z1;
        }
    }
    cluster.sync();  // no CTA exits while a peer may still write into it
}

template <int PT>
static int launch_fps_p3d(int b, const Fps3Args &a, cudaStream_t st) {
    const size_t smem = (size_t)a.N * 3 * sizeof(float);
    const bool mirror = smem <= 200 * 1024;
    auto kern = mirror ? fps_p3d_cluster_kernel<PT, true> : fps_p3d_cluster_kernel<PT, false>;
    const size_t dyn = mirror ? smem : 0;
    if (dyn > 40 * 1024)
        B200PCI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(b * FPS3_CS);
    cfg.blockDim = dim3(FPS3_CT);
    cfg.dynamicSmemBytes = dyn;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = FPS3_CS;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    B200PCI_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
    return B200PCI_OK;
}

template <int PT, bool MIRROR, int CS, int CT>
static int launch_fps_cluster_impl(int b, int n, int m, int chunk, const float *xyz, float *temp,
                                   int *idx, FpsGeom g, cudaStream_t st) {
    const size_t smem = MIRROR ? (size_t)n * 3 * sizeof(float) : 0;
    auto kern = fps_cluster_kernel<PT, MIRROR, CS, CT>;
    if (smem > 40 * 1024)
        B200PCI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (CS > 8)
        B200PCI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(b * CS);
    cfg.blockDim = dim3(CT);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    B200PCI_CUDA(cudaLaunchKernelEx(&cfg, kern, n, m, chunk, xyz, temp, idx, g));
    return B200PCI_OK;
}

template <int PT, int CS, int CT>
static int launch_fps_cluster(int b, int n, int m, int chunk, const float *xyz, float *temp, int *idx,
                              FpsGeom g, cudaStream_t st) {
    if ((size_t)n * 3 * sizeof(float) <= 200 * 1024)
        return launch_fps_cluster_impl<PT, true, CS, CT>(b, n, m, chunk, xyz, temp, idx, g, st);
    return launch_fps_cluster_impl<PT, false, CS, CT>(b, n, m, chunk, xyz, temp, idx, g, st);
}

// cluster of CS CTAs x CT threads per cloud, PT = points per thread
template <int CS, int CT>
static int dispatch_fps_cluster(int b, int n, int m, const float *xyz, float *temp, int *idx, FpsGeom g,
                                cudaStream_t st) {
    const int chunk = (n + CS - 1) / CS;
    const int need = (chunk + CT - 1) / CT;
    if (need <= 2) return launch_fps_cluster<2, CS, CT>(b, n, m, chunk, xyz, temp, idx, g, st);
    if (need <= 4) return launch_fps_cluster<4, CS, CT>(b, n, m, chunk, xyz, temp, idx, g, st);
    if (need <= 8) return launch_fps_cluster<8, CS, CT>(b, n, m, chunk, xyz, temp, idx, g, st);
    if (need <= 16) return launch_fps_cluster<16, CS, CT>(b, n, m, chunk, xyz, temp, idx, g, st);
    return launch_fps_cluster<32, CS, CT>(b, n, m, chunk, xyz, temp, idx, g, st);
}

static int ref_opt_n_threads(int work_size) {  // cuda_utils.h:10-14, same double arithmetic
    const int pow_2 = (int)(std::log((double)work_size) / std::log(2.0));
    int t = 1 << pow_2;
    if (t > 1024) t = 1024;
    if (t < 1) t = 1;
    return t;
}

template <int PT>
static int launch_fps(int b, int n, int m, const float *xyz, float *temp, int *idx, FpsGeom g,
                      int threads, cudaStream_t st) {
    const size_t xyz_bytes = (size_t)n * 3 * sizeof(float);
    if (xyz_bytes <= 200 * 1024) {
        auto kern = fps_kernel<PT, true>;
        if (xyz_bytes > 40 * 1024)
            B200PCI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                              (int)xyz_bytes));
        kern<<<b, threads, xyz_bytes, st>>>(n, m, xyz, temp, idx, g);
    } else {
        fps_kernel<PT, false><<<b, threads, 0, st>>>(n, m, xyz, temp, idx, g);
    }
    B200PCI_LAUNCH_CHECK("fps_kernel");
    return B200PCI_OK;
}

}  // namespace b200pci

using namespace b200pci;

// test hook (b200pci_debug_set key 5): force the single-CTA kernel
int g_fps_single_cta = 0;

extern "C" int b200pci_furthest_point_sampling(int b, int n, int m, const float *xyz, float *temp,
                                               int *idx, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    B200PCI_CHECK_ARG(b >= 0 && n >= 0 && m >= 0, "fps: negative size");
    if (b == 0 || m <= 0) return B200PCI_OK;  // sampling_gpu.cu:100
    B200PCI_CHECK_ARG(n >= 1, "fps: empty cloud");
    B200PCI_CHECK_ARG(xyz && temp && idx, "fps: null pointer");
    const int bs = ref_opt_n_threads(n);
    FpsGeom g;
    g.log2bs = 0;
    while ((1 << g.log2bs) < bs) ++g.log2bs;
    const int cnt = (n + bs - 1) / bs;
    g.hb = 0;
    while ((1 << g.hb) < cnt) ++g.hb;
    if (n >= 4096 && n <= FPS_CS * FPS_CT * 32 && !g_fps_single_cta) {
        // Few clouds: clusters of 16 CTAs x 256 threads (non-portable size) shorten the per-CTA part
        // of an iteration (B=1, 16384 -> 2048: 1.44 -> 1.30 ms); from 5 clouds on they no longer fit
        // the GPU in one wave (B=8: 5.2 vs 2.8 ms). If the launch is refused (cluster size not
        // available on this device / partition), fall back to the portable size.
        if (b <= 4 && FPS_CS == 8 && n <= 16 * 256 * 32) {
            const int rc16 = dispatch_fps_cluster<16, 256>(b, n, m, xyz, temp, idx, g, st);
            if (rc16 == B200PCI_OK) return rc16;
            (void)cudaGetLastError();
        }
        return dispatch_fps_cluster<FPS_CS, FPS_CT>(b, n, m, xyz, temp, idx, g, st);
    }
    int threads = (n + 31) / 32 * 32;
    if (threads > FPS_MAX_THREADS) threads = FPS_MAX_THREADS;
    const int need = (n + threads - 1) / threads;
    if (need <= 1) return launch_fps<1>(b, n, m, xyz, temp, idx, g, threads, st);
    if (need <= 2) return launch_fps<2>(b, n, m, xyz, temp, idx, g, threads, st);
    if (need <= 4) return launch_fps<4>(b, n, m, xyz, temp, idx, g, threads, st);
    if (need <= 8) return launch_fps<8>(b, n, m, xyz, temp, idx, g, threads, st);
    if (need <= 16) return launch_fps<16>(b, n, m, xyz, temp, idx, g, threads, st);
    if (need <= 32) return launch_fps<32>(b, n, m, xyz, temp, idx, g, threads, st);
    return launch_fps<0>(b, n, m, xyz, temp, idx, g, threads, st);
}

extern "C" int b200pci_fps_p3d(int B, int P, int M, const float *points, int64_t p_sb, int64_t p_sp,
                               int64_t p_sc, const int64_t *lengths, const int64_t *K,
                               const int64_t *start, int64_t *idx, float *selected, void *stream) {
    B200PCI_CHECK_ARG(B >= 0 && P >= 0 && M >= 0, "fps_p3d: negative size");
    if (B == 0 || M == 0) return B200PCI_OK;
    B200PCI_CHECK_ARG(idx && (points || P == 0), "fps_p3d: null pointer");
    B200PCI_CHECK_ARG(P <= FPS3_CS * FPS3_CT * 32, "fps_p3d: more than %d points per cloud",
                      FPS3_CS * FPS3_CT * 32);
    B200PCI_CHECK_ARG(B <= (1 << 27), "fps_p3d: batch too large");
    Fps3Args a;
    a.N = P;
    a.M = M;
    a.chunk = (P + FPS3_CS - 1) / FPS3_CS;
    a.xyz = points;
    a.sb = p_sb;
    a.sp = p_sp;
    a.sc = p_sc;
    a.lengths = reinterpret_cast<const long long *>(lengths);
    a.K = reinterpret_cast<const long long *>(K);
    a.start = reinterpret_cast<const long long *>(start);
    a.idx = reinterpret_cast<long long *>(idx);
    a.sel = selected;
    cudaStream_t st = (cudaStream_t)stream;
    const int need = (a.chunk + FPS3_CT - 1) / FPS3_CT;
    if (need <= 2) return launch_fps_p3d<2>(B, a, st);
    if (need <= 4) return launch_fps_p3d<4>(B, a, st);
    if (need <= 8) return launch_fps_p3d<8>(B, a, st);
    if (need <= 16) return launch_fps_p3d<16>(B, a, st);
    return launch_fps_p3d<32>(B, a, st);
}
