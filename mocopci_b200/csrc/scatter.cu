// Deterministic (fixed-order) versions of the scatter-add gradients: gather / group, three_interpolate,
// the [B,N,C] row gathers and Chamfer. The atomic kernels (gather.cu, knn.cu) add the contributions
// to one destination in whatever order the threads arrive, so the last bits of a gradient change
// from run to run. Here each destination sums its contributions sequentially in FP32, in ascending
// source position, every product rounded before it is added (include/b200pci.h, "_det").
//
// Both steps run on the caller's stream with the caller's scratch (no allocation, no host sync):
//  1. inverse index of idx per cloud, a CSR: offsets[b, 0..N] and the source positions of each
//     destination sorted ascending. Histogram (integer atomics), exclusive scan per cloud, fill
//     through atomic cursors, then each bucket is sorted: the (idx, t) pairs are distinct, so the
//     sorted list does not depend on the order of the fill.
//  2. one fixed-order reduction over that CSR per output.
#include <limits.h>

#include <algorithm>

#include "common.cuh"

namespace b200pci {

constexpr int SC_THREADS = 256;
constexpr int SC_SCAN_THREADS = 1024;
constexpr int SC_SORT_THREADS = 512;
constexpr int SC_SMALL = 32;     // buckets up to this length: insertion sort by one thread
constexpr int SC_SMEM = 4096;    // up to this length: bitonic sort of the bucket in shared memory
                                 // beyond: the bucket is rebuilt in order by a scan over idx
constexpr int SC_CCHUNK = 8;     // channels per thread of the [B,C,N] reductions

// Carved from the caller's workspace (b200pci_scatter_workspace_bytes).
struct Csr {
    int *cursor;     // [B,N]: counts, then fill cursors
    int *offsets;    // [B,N+1]: bucket i of cloud b is list[b*T + offsets[b,i] .. offsets[b,i+1])
    int *list;       // [B,T]: source positions t, ascending within a bucket
    long long *work; // [B*N]: buckets longer than SC_SMALL (b*N + i), in no particular order
    int *nwork;      // [1]
};

static size_t csr_bytes(long long B, long long N, long long T) {
    return align_up((size_t)(B * N) * sizeof(int), 256) + align_up((size_t)(B * (N + 1)) * sizeof(int), 256) +
           align_up((size_t)(B * T) * sizeof(int), 256) + align_up((size_t)(B * N) * sizeof(long long), 256) + 256;
}

static Csr csr_carve(void *ws, long long B, long long N, long long T) {
    char *p = reinterpret_cast<char *>(ws);
    Csr c;
    c.cursor = reinterpret_cast<int *>(p);
    p += align_up((size_t)(B * N) * sizeof(int), 256);
    c.offsets = reinterpret_cast<int *>(p);
    p += align_up((size_t)(B * (N + 1)) * sizeof(int), 256);
    c.list = reinterpret_cast<int *>(p);
    p += align_up((size_t)(B * T) * sizeof(int), 256);
    c.work = reinterpret_cast<long long *>(p);
    p += align_up((size_t)(B * N) * sizeof(long long), 256);
    c.nwork = reinterpret_cast<int *>(p);
    return c;
}

template <typename I>
__device__ __forceinline__ long long load_idx(const I *idx, size_t k) {
    return (long long)__ldg(idx + k);
}

template <typename I>
__global__ void __launch_bounds__(SC_THREADS)
    scatter_hist_kernel(int N, long long T, const I *__restrict__ idx, int *__restrict__ cnt) {
    const long long t = (long long)blockIdx.x * SC_THREADS + threadIdx.x;
    const int b = blockIdx.y;
    if (t >= T) return;
    const long long v = load_idx(idx, (size_t)b * T + t);
    if (v >= 0 && v < N) atomicAdd(cnt + (size_t)b * N + v, 1);
}

// One CTA per cloud: offsets = exclusive scan of the counts; the counts become the fill cursors;
// buckets longer than SC_SMALL go to the work list of the long-bucket sort.
__global__ void __launch_bounds__(SC_SCAN_THREADS)
    scatter_scan_kernel(int N, int *__restrict__ cnt, int *__restrict__ offsets, long long *__restrict__ work,
                        int *__restrict__ nwork) {
    __shared__ int warp_sum[SC_SCAN_THREADS / 32];
    __shared__ int carry_sh;
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int *c = cnt + (size_t)b * N;
    int *o = offsets + (size_t)b * (N + 1);
    if (threadIdx.x == 0) carry_sh = 0;
    __syncthreads();
    constexpr int ITEMS = 4;
    for (long long base = 0; base < N; base += (long long)SC_SCAN_THREADS * ITEMS) {
        const long long i0 = base + (long long)threadIdx.x * ITEMS;
        int v[ITEMS], s = 0;
#pragma unroll
        for (int u = 0; u < ITEMS; ++u) {
            v[u] = (i0 + u < N) ? c[i0 + u] : 0;
            s += v[u];
        }
        int incl = s;  // inclusive scan of the per-thread sums within the warp
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += y;
        }
        if (lane == 31) warp_sum[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int w = warp_sum[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, w, d);
                if (lane >= d) w += y;
            }
            warp_sum[lane] = w;  // inclusive over warps
        }
        __syncthreads();
        const int carry = carry_sh;
        int run = carry + (warp > 0 ? warp_sum[warp - 1] : 0) + incl - s;
#pragma unroll
        for (int u = 0; u < ITEMS; ++u) {
            if (i0 + u < N) {
                o[i0 + u] = run;
                c[i0 + u] = run;  // fill cursor
                if (v[u] > SC_SMALL) work[atomicAdd(nwork, 1)] = (long long)b * N + i0 + u;
            }
            run += v[u];
        }
        __syncthreads();
        if (threadIdx.x == SC_SCAN_THREADS - 1) carry_sh = run;
        __syncthreads();
    }
    if (threadIdx.x == 0) o[N] = carry_sh;
}

template <typename I>
__global__ void __launch_bounds__(SC_THREADS)
    scatter_fill_kernel(int N, long long T, const I *__restrict__ idx, int *__restrict__ cursor,
                        int *__restrict__ list) {
    const long long t = (long long)blockIdx.x * SC_THREADS + threadIdx.x;
    const int b = blockIdx.y;
    if (t >= T) return;
    const long long v = load_idx(idx, (size_t)b * T + t);
    if (v >= 0 && v < N) list[(size_t)b * T + atomicAdd(cursor + (size_t)b * N + v, 1)] = (int)t;
}

// Buckets of up to SC_SMALL entries: insertion sort by one thread.
__global__ void __launch_bounds__(SC_THREADS)
    scatter_sort_small_kernel(int N, long long T, const int *__restrict__ offsets, int *__restrict__ list) {
    const int i = blockIdx.x * SC_THREADS + threadIdx.x;
    const int b = blockIdx.y;
    if (i >= N) return;
    const int beg = offsets[(size_t)b * (N + 1) + i], end = offsets[(size_t)b * (N + 1) + i + 1];
    if (end - beg > SC_SMALL || end - beg < 2) return;
    int *l = list + (size_t)b * T;
    for (int p = beg + 1; p < end; ++p) {
        const int x = l[p];
        int q = p - 1;
        while (q >= beg && l[q] > x) {
            l[q + 1] = l[q];
            --q;
        }
        l[q + 1] = x;
    }
}

// Longer buckets, one CTA each (grid-stride over the work list): up to SC_SMEM entries a bitonic
// sort in shared memory; beyond that the bucket is rebuilt in order by an ordered compaction of
// idx (O(T) per such bucket, and there are at most T / SC_SMEM of them).
template <typename I>
__global__ void __launch_bounds__(SC_SORT_THREADS)
    scatter_sort_long_kernel(int N, long long T, const I *__restrict__ idx, const int *__restrict__ offsets,
                             int *__restrict__ list, const long long *__restrict__ work,
                             const int *__restrict__ nwork) {
    __shared__ int s[SC_SMEM];
    __shared__ int warp_cnt[SC_SORT_THREADS / 32];
    const int nw = *nwork;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int w = blockIdx.x; w < nw; w += gridDim.x) {
        const long long key = work[w];
        const int b = (int)(key / N), i = (int)(key - (long long)b * N);
        const int beg = offsets[(size_t)b * (N + 1) + i], L = offsets[(size_t)b * (N + 1) + i + 1] - beg;
        int *l = list + (size_t)b * T + beg;
        if (L <= SC_SMEM) {
            int P = 1;
            while (P < L) P <<= 1;
            for (int x = threadIdx.x; x < P; x += SC_SORT_THREADS) s[x] = x < L ? l[x] : INT_MAX;
            __syncthreads();
            for (int k = 2; k <= P; k <<= 1)
                for (int j = k >> 1; j > 0; j >>= 1) {
                    for (int x = threadIdx.x; x < P; x += SC_SORT_THREADS) {
                        const int y = x ^ j;
                        if (y > x) {
                            const int a = s[x], c = s[y];
                            if ((a > c) == ((x & k) == 0)) {
                                s[x] = c;
                                s[y] = a;
                            }
                        }
                    }
                    __syncthreads();
                }
            for (int x = threadIdx.x; x < L; x += SC_SORT_THREADS) l[x] = s[x];
        } else {
            constexpr int ITEMS = 4;
            const I *ib = idx + (size_t)b * T;
            int written = 0;  // same value in every thread
            for (long long base = 0; base < T; base += (long long)SC_SORT_THREADS * ITEMS) {
                const long long t0 = base + (long long)threadIdx.x * ITEMS;
                unsigned hit = 0;
#pragma unroll
                for (int u = 0; u < ITEMS; ++u)
                    if (t0 + u < T && load_idx(ib, t0 + u) == i) hit |= 1u << u;
                const int mine = __popc(hit);
                int incl = mine;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int y = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += y;
                }
                if (lane == 31) warp_cnt[warp] = incl;
                __syncthreads();
                int before = 0, total = 0;
                for (int q = 0; q < SC_SORT_THREADS / 32; ++q) {
                    const int v = warp_cnt[q];
                    before += q < warp ? v : 0;
                    total += v;
                }
                int pos = written + before + incl - mine;
#pragma unroll
                for (int u = 0; u < ITEMS; ++u)
                    if (hit & (1u << u)) l[pos++] = (int)(t0 + u);
                written += total;
                __syncthreads();
            }
        }
        __syncthreads();
    }
}

template <typename I>
static int csr_build(int B, int N, long long T, const I *idx, const Csr &c, cudaStream_t st) {
    B200PCI_CUDA(cudaMemsetAsync(c.cursor, 0, (size_t)B * N * sizeof(int), st));
    B200PCI_CUDA(cudaMemsetAsync(c.nwork, 0, sizeof(int), st));
    const dim3 tgrid((unsigned)((T + SC_THREADS - 1) / SC_THREADS), B);
    scatter_hist_kernel<I><<<tgrid, SC_THREADS, 0, st>>>(N, T, idx, c.cursor);
    B200PCI_LAUNCH_CHECK("scatter_hist_kernel");
    scatter_scan_kernel<<<B, SC_SCAN_THREADS, 0, st>>>(N, c.cursor, c.offsets, c.work, c.nwork);
    B200PCI_LAUNCH_CHECK("scatter_scan_kernel");
    scatter_fill_kernel<I><<<tgrid, SC_THREADS, 0, st>>>(N, T, idx, c.cursor, c.list);
    B200PCI_LAUNCH_CHECK("scatter_fill_kernel");
    scatter_sort_small_kernel<<<dim3(ceil_div(N, SC_THREADS), B), SC_THREADS, 0, st>>>(N, T, c.offsets, c.list);
    B200PCI_LAUNCH_CHECK("scatter_sort_small_kernel");
    // at most T / (SC_SMALL + 1) long buckets per cloud; the CTAs stride over however many there are
    const long long most = (long long)B * std::min<long long>(N, T / (SC_SMALL + 1));
    const int grid = (int)std::max<long long>(1, std::min<long long>(most, 4LL * sm_count()));
    scatter_sort_long_kernel<I><<<grid, SC_SORT_THREADS, 0, st>>>(N, T, idx, c.offsets, c.list, c.work, c.nwork);
    B200PCI_LAUNCH_CHECK("scatter_sort_long_kernel");
    return B200PCI_OK;
}

// ---- fixed-order reductions -------------------------------------------------------------------
// [B,C,N] outputs (gather / group): one thread per destination point, SC_CCHUNK channels each (grid.y),
// so one CSR serves every channel. grad_points[b,c,i] += grad_out[b,c,t] for t ascending.
__global__ void __launch_bounds__(SC_THREADS)
    group_grad_det_kernel(int C, int N, long long T, const float *__restrict__ grad_out, const int *__restrict__ offsets,
                          const int *__restrict__ list, float *__restrict__ grad_points) {
    const int i = blockIdx.x * SC_THREADS + threadIdx.x;
    const int b = blockIdx.z;
    const int c0 = blockIdx.y * SC_CCHUNK;
    const int cc = min(SC_CCHUNK, C - c0);
    if (i >= N) return;
    const int beg = offsets[(size_t)b * (N + 1) + i], end = offsets[(size_t)b * (N + 1) + i + 1];
    const int *l = list + (size_t)b * T;
    const float *g = grad_out + ((size_t)b * C + c0) * T;
    float *dst = grad_points + ((size_t)b * C + c0) * N + i;
    float acc[SC_CCHUNK];
#pragma unroll
    for (int u = 0; u < SC_CCHUNK; ++u) acc[u] = u < cc ? dst[(size_t)u * N] : 0.f;
    for (int p = beg; p < end; ++p) {
        const long long t = __ldg(l + p);
#pragma unroll
        for (int u = 0; u < SC_CCHUNK; ++u)
            if (u < cc) acc[u] = __fadd_rn(acc[u], __ldg(g + (size_t)u * T + t));
    }
#pragma unroll
    for (int u = 0; u < SC_CCHUNK; ++u)
        if (u < cc) dst[(size_t)u * N] = acc[u];
}

// three_interpolate: source position s = 3 i + j of idx [B,n,3]; contribution fl(grad_out[b,c,i] *
// weight[b,i,j]) added for s ascending.
__global__ void __launch_bounds__(SC_THREADS)
    three_interpolate_grad_det_kernel(int C, int n, int m, const float *__restrict__ grad_out,
                                      const float *__restrict__ weight, const int *__restrict__ offsets,
                                      const int *__restrict__ list, float *__restrict__ grad_points) {
    const int i = blockIdx.x * SC_THREADS + threadIdx.x;
    const int b = blockIdx.z;
    const int c0 = blockIdx.y * SC_CCHUNK;
    const int cc = min(SC_CCHUNK, C - c0);
    if (i >= m) return;
    const long long T = 3LL * n;
    const int beg = offsets[(size_t)b * (m + 1) + i], end = offsets[(size_t)b * (m + 1) + i + 1];
    const int *l = list + (size_t)b * T;
    const float *g = grad_out + ((size_t)b * C + c0) * n;
    const float *w = weight + (size_t)b * T;
    float *dst = grad_points + ((size_t)b * C + c0) * m + i;
    float acc[SC_CCHUNK];
#pragma unroll
    for (int u = 0; u < SC_CCHUNK; ++u) acc[u] = u < cc ? dst[(size_t)u * m] : 0.f;
    for (int p = beg; p < end; ++p) {
        const int s = __ldg(l + p);
        const int src = s / 3;
        const float ws = __ldg(w + s);
#pragma unroll
        for (int u = 0; u < SC_CCHUNK; ++u)
            if (u < cc) acc[u] = __fadd_rn(acc[u], __fmul_rn(__ldg(g + (size_t)u * n + src), ws));
    }
#pragma unroll
    for (int u = 0; u < SC_CCHUNK; ++u)
        if (u < cc) dst[(size_t)u * m] = acc[u];
}

// [B,N,C] rows: `width` lanes (a power of two <= 32) per destination row, lanes across channels so
// that the loads of a grad_out row are coalesced; every lane walks the row's bucket in order.
constexpr int RD_UNROLL = 4;
__global__ void __launch_bounds__(SC_THREADS)
    rows_grad_det_kernel(int N, long long T, int C, int wshift, const float *__restrict__ grad_out,
                         const int *__restrict__ offsets, const int *__restrict__ list,
                         float *__restrict__ grad_points) {
    const int b = blockIdx.y;
    const long long gt = (long long)blockIdx.x * SC_THREADS + threadIdx.x;
    const int width = 1 << wshift;
    const long long i = gt >> wshift;
    const int lane = (int)(gt & (width - 1));
    if (i >= N) return;
    const int beg = offsets[(size_t)b * (N + 1) + i], end = offsets[(size_t)b * (N + 1) + i + 1];
    const int *l = list + (size_t)b * T;
    const float *g = grad_out + (size_t)b * T * C;
    float *dst = grad_points + ((size_t)b * N + i) * C;
    for (int c0 = lane; c0 < C; c0 += width * RD_UNROLL) {
        float acc[RD_UNROLL];
#pragma unroll
        for (int u = 0; u < RD_UNROLL; ++u) {
            const int c = c0 + u * width;
            acc[u] = c < C ? dst[c] : 0.f;
        }
        for (int p = beg; p < end; ++p) {
            const float *row = g + (size_t)__ldg(l + p) * C;
#pragma unroll
            for (int u = 0; u < RD_UNROLL; ++u) {
                const int c = c0 + u * width;
                if (c < C) acc[u] = __fadd_rn(acc[u], __ldg(row + c));
            }
        }
#pragma unroll
        for (int u = 0; u < RD_UNROLL; ++u) {
            const int c = c0 + u * width;
            if (c < C) dst[c] = acc[u];
        }
    }
}

// Chamfer: one thread per point of the direction's own cloud P (grad_p overwritten). Its own term
// d_p(i) = fl(w_p * fl(p_i - q_{idx_p[i]})), w_p = fl(fl(2 g) / fl(B * P)), then minus the terms
// d_q(j) = fl(w_q * fl(q_j - p_i)) of the points j of Q whose nearest point is i, j ascending.
__global__ void __launch_bounds__(SC_THREADS)
    chamfer_grad_det_kernel(int B, int P, int Q, const float *__restrict__ p, const float *__restrict__ q,
                            const int *__restrict__ idx_p, const float *__restrict__ grad_loss,
                            const int *__restrict__ offsets, const int *__restrict__ list,
                            float *__restrict__ grad_p) {
    const int i = blockIdx.x * SC_THREADS + threadIdx.x;
    const int b = blockIdx.y;
    if (i >= P) return;
    const float g2 = __fmul_rn(2.f, __ldg(grad_loss));
    const float wp = __fdiv_rn(g2, __fmul_rn((float)B, (float)P));
    const float wq = __fdiv_rn(g2, __fmul_rn((float)B, (float)Q));
    const float *pi = p + ((size_t)b * P + i) * 3;
    const float px = __ldg(pi), py = __ldg(pi + 1), pz = __ldg(pi + 2);
    float ax = 0.f, ay = 0.f, az = 0.f;
    const int j = __ldg(idx_p + (size_t)b * P + i);
    if (j >= 0 && j < Q) {
        const float *qj = q + ((size_t)b * Q + j) * 3;
        ax = __fadd_rn(ax, __fmul_rn(wp, __fsub_rn(px, __ldg(qj))));
        ay = __fadd_rn(ay, __fmul_rn(wp, __fsub_rn(py, __ldg(qj + 1))));
        az = __fadd_rn(az, __fmul_rn(wp, __fsub_rn(pz, __ldg(qj + 2))));
    }
    const int beg = offsets[(size_t)b * (P + 1) + i], end = offsets[(size_t)b * (P + 1) + i + 1];
    const int *l = list + (size_t)b * Q;
    for (int e = beg; e < end; ++e) {
        const float *qk = q + ((size_t)b * Q + __ldg(l + e)) * 3;
        ax = __fsub_rn(ax, __fmul_rn(wq, __fsub_rn(__ldg(qk), px)));
        ay = __fsub_rn(ay, __fmul_rn(wq, __fsub_rn(__ldg(qk + 1), py)));
        az = __fsub_rn(az, __fmul_rn(wq, __fsub_rn(__ldg(qk + 2), pz)));
    }
    float *dst = grad_p + ((size_t)b * P + i) * 3;
    dst[0] = ax;
    dst[1] = ay;
    dst[2] = az;
}

static int check_ws(void *workspace, size_t have, size_t need, const char *what) {
    if (!workspace || have < need) {
        set_error("%s: workspace of %zu bytes required, got %zu", what, need, have);
        return B200PCI_EWORKSPACE;
    }
    return B200PCI_OK;
}

static int group_grad_det_impl(int b, int c, int n, long long T, const float *grad_out, const int *idx,
                               float *grad_points, void *workspace, size_t workspace_bytes, cudaStream_t st,
                               const char *what) {
    B200PCI_CHECK_ARG(b >= 0 && c >= 0 && n >= 0 && T >= 0, "%s: negative size", what);
    if (b == 0 || c == 0 || T == 0) return B200PCI_OK;
    B200PCI_CHECK_ARG(grad_out && idx && grad_points, "%s: null pointer", what);
    B200PCI_CHECK_ARG(b <= 65535 && ceil_div(c, SC_CCHUNK) <= 65535, "%s: batch or channels exceed the grid", what);
    B200PCI_CHECK_ARG(T < (1LL << 31), "%s: 2^31 or more source positions per cloud", what);
    if (n == 0) return B200PCI_OK;
    if (int rc = check_ws(workspace, workspace_bytes, csr_bytes(b, n, T), what)) return rc;
    const Csr csr = csr_carve(workspace, b, n, T);
    if (int rc = csr_build<int>(b, n, T, idx, csr, st)) return rc;
    group_grad_det_kernel<<<dim3(ceil_div(n, SC_THREADS), ceil_div(c, SC_CCHUNK), b), SC_THREADS, 0, st>>>(
        c, n, T, grad_out, csr.offsets, csr.list, grad_points);
    B200PCI_LAUNCH_CHECK("group_grad_det_kernel");
    return B200PCI_OK;
}

}  // namespace b200pci

using namespace b200pci;

extern "C" size_t b200pci_scatter_workspace_bytes(int B, int N, long long T) {
    if (B < 0 || N < 0 || T < 0) return 0;
    return csr_bytes(B, N, T);
}

extern "C" int b200pci_gather_points_grad_det(int b, int c, int n, int npoints, const float *grad_out,
                                              const int *idx, float *grad_points, void *workspace,
                                              size_t workspace_bytes, void *stream) {
    return group_grad_det_impl(b, c, n, npoints, grad_out, idx, grad_points, workspace, workspace_bytes,
                               (cudaStream_t)stream, "gather_points_grad_det");
}

extern "C" int b200pci_group_points_grad_det(int b, int c, int n, int npoints, int nsample, const float *grad_out,
                                             const int *idx, float *grad_points, void *workspace,
                                             size_t workspace_bytes, void *stream) {
    B200PCI_CHECK_ARG(npoints >= 0 && nsample >= 0, "group_points_grad_det: negative size");
    return group_grad_det_impl(b, c, n, (long long)npoints * nsample, grad_out, idx, grad_points, workspace,
                               workspace_bytes, (cudaStream_t)stream, "group_points_grad_det");
}

extern "C" int b200pci_three_interpolate_grad_det(int b, int c, int n, int m, const float *grad_out, const int *idx,
                                                  const float *weight, float *grad_points, void *workspace,
                                                  size_t workspace_bytes, void *stream) {
    const char *what = "three_interpolate_grad_det";
    cudaStream_t st = (cudaStream_t)stream;
    B200PCI_CHECK_ARG(b >= 0 && c >= 0 && n >= 0 && m >= 0, "%s: negative size", what);
    if (b == 0 || c == 0 || n == 0) return B200PCI_OK;
    B200PCI_CHECK_ARG(grad_out && idx && weight && grad_points, "%s: null pointer", what);
    B200PCI_CHECK_ARG(b <= 65535 && ceil_div(c, SC_CCHUNK) <= 65535, "%s: batch or channels exceed the grid", what);
    const long long T = 3LL * n;
    B200PCI_CHECK_ARG(T < (1LL << 31), "%s: 2^31 or more source positions per cloud", what);
    if (m == 0) return B200PCI_OK;
    if (int rc = check_ws(workspace, workspace_bytes, csr_bytes(b, m, T), what)) return rc;
    const Csr csr = csr_carve(workspace, b, m, T);
    if (int rc = csr_build<int>(b, m, T, idx, csr, st)) return rc;
    three_interpolate_grad_det_kernel<<<dim3(ceil_div(m, SC_THREADS), ceil_div(c, SC_CCHUNK), b), SC_THREADS, 0,
                                        st>>>(c, n, m, grad_out, weight, csr.offsets, csr.list, grad_points);
    B200PCI_LAUNCH_CHECK("three_interpolate_grad_det_kernel");
    return B200PCI_OK;
}

extern "C" int b200pci_index_points_rows_grad_det(int B, int N, long long T, int C, const float *grad_out,
                                                  const void *idx, int idx_is_int64, float *grad_points,
                                                  void *workspace, size_t workspace_bytes, void *stream) {
    const char *what = "index_points_rows_grad_det";
    cudaStream_t st = (cudaStream_t)stream;
    B200PCI_CHECK_ARG(B >= 0 && N >= 0 && T >= 0 && C >= 0, "%s: negative size", what);
    if (B == 0 || T == 0 || C == 0) return B200PCI_OK;
    B200PCI_CHECK_ARG(grad_out && idx && grad_points, "%s: null pointer", what);
    B200PCI_CHECK_ARG(B <= 65535, "%s: batch too large", what);
    B200PCI_CHECK_ARG(T < (1LL << 31), "%s: 2^31 or more source positions per cloud", what);
    if (N == 0) return B200PCI_OK;
    if (int rc = check_ws(workspace, workspace_bytes, csr_bytes(B, N, T), what)) return rc;
    const Csr csr = csr_carve(workspace, B, N, T);
    int rc = idx_is_int64 ? csr_build<long long>(B, N, T, reinterpret_cast<const long long *>(idx), csr, st)
                          : csr_build<int>(B, N, T, reinterpret_cast<const int *>(idx), csr, st);
    if (rc) return rc;
    int wshift = 5;  // lanes per row: 32, or the least power of two >= C
    while (wshift > 0 && (1 << (wshift - 1)) >= C) --wshift;
    const long long threads = (long long)N << wshift;
    B200PCI_CHECK_ARG((threads + SC_THREADS - 1) / SC_THREADS < (1LL << 31), "%s: too many rows", what);
    rows_grad_det_kernel<<<dim3((unsigned)((threads + SC_THREADS - 1) / SC_THREADS), B), SC_THREADS, 0, st>>>(
        N, T, C, wshift, grad_out, csr.offsets, csr.list, grad_points);
    B200PCI_LAUNCH_CHECK("rows_grad_det_kernel");
    return B200PCI_OK;
}

extern "C" size_t b200pci_chamfer_backward_det_workspace_bytes(int B, int N, int M) {
    if (B < 0 || N < 0 || M < 0) return 0;
    return csr_bytes(B, N, M) + csr_bytes(B, M, N);
}

extern "C" int b200pci_chamfer_backward_det(int B, int N, int M, const float *x, const float *y, const int *idx_x,
                                            const int *idx_y, const float *grad_loss, float *grad_x, float *grad_y,
                                            void *workspace, size_t workspace_bytes, void *stream) {
    const char *what = "chamfer_backward_det";
    cudaStream_t st = (cudaStream_t)stream;
    B200PCI_CHECK_ARG(B >= 0 && N >= 0 && M >= 0, "%s: negative size", what);
    if (B == 0 || (N == 0 && M == 0)) return B200PCI_OK;
    B200PCI_CHECK_ARG(x && y && idx_x && idx_y && grad_loss && grad_x && grad_y, "%s: null pointer", what);
    B200PCI_CHECK_ARG(B <= 65535, "%s: batch too large", what);
    if (int rc = check_ws(workspace, workspace_bytes, b200pci_chamfer_backward_det_workspace_bytes(B, N, M), what))
        return rc;
    if (N == 0 || M == 0) {  // no neighbours: the gradient is zero (as b200pci_chamfer_backward)
        B200PCI_CUDA(cudaMemsetAsync(grad_x, 0, (size_t)B * N * 3 * sizeof(float), st));
        B200PCI_CUDA(cudaMemsetAsync(grad_y, 0, (size_t)B * M * 3 * sizeof(float), st));
        return B200PCI_OK;
    }
    // by_x: the y points grouped by their nearest x (idx_y over N buckets); by_y the mirror image
    const Csr by_x = csr_carve(workspace, B, N, M);
    const Csr by_y = csr_carve(reinterpret_cast<char *>(workspace) + csr_bytes(B, N, M), B, M, N);
    if (int rc = csr_build<int>(B, N, M, idx_y, by_x, st)) return rc;
    if (int rc = csr_build<int>(B, M, N, idx_x, by_y, st)) return rc;
    chamfer_grad_det_kernel<<<dim3(ceil_div(N, SC_THREADS), B), SC_THREADS, 0, st>>>(
        B, N, M, x, y, idx_x, grad_loss, by_x.offsets, by_x.list, grad_x);
    B200PCI_LAUNCH_CHECK("chamfer_grad_det_kernel");
    chamfer_grad_det_kernel<<<dim3(ceil_div(M, SC_THREADS), B), SC_THREADS, 0, st>>>(
        B, M, N, y, x, idx_y, grad_loss, by_y.offsets, by_y.list, grad_y);
    B200PCI_LAUNCH_CHECK("chamfer_grad_det_kernel");
    return B200PCI_OK;
}
