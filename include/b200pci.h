/* b200pci -- B200-native (sm_100a) point-set neighbourhood kernels for MoCoPCI: C ABI.
 *
 * This is the drop-in boundary (SURVEY.md section 8b). Every entry point takes raw DEVICE pointers,
 * plain sizes and a CUDA stream (passed as void* == cudaStream_t), launches asynchronously on that
 * stream and returns 0 or a negative B200PCI_E* code; it never exits the process (the reference's
 * launchers fprintf+exit(-1), e.g. pointnet2/src/sampling_gpu.cu:39-43). No torch types appear.
 * All entry points are re-entrant across host threads. State the library keeps, all of it
 * thread-local (nothing is shared between host threads in production use):
 *   - the error string of b200pci_last_error();
 *   - per device, a side stream + two events used by the KNN path to run the exact redo of a few
 *     queries next to the top-k kernel (event fork/join, legal under stream capture);
 *   - per device, the copy stream, events and device buffer of b200pci_knn_host (kept warm across
 *     calls; b200pci_host_release() frees them).
 * The b200pci_debug_* hooks at the end of this file are process-global and NOT thread-safe; they
 * exist for tests and measurements and are never needed in production.
 *
 * Each function cites the reference interface it replaces (paths relative to the reference
 * repository root). INTEGRATION.md shows the ctypes / pybind stubs a maintainer would add.
 */
#ifndef B200PCI_H
#define B200PCI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200PCI_VERSION 100

#define B200PCI_OK 0
#define B200PCI_EINVAL (-1)     /* bad argument (shape, null pointer, k out of range ...) */
#define B200PCI_ECUDA (-2)      /* a CUDA runtime call / launch failed; see b200pci_last_error() */
#define B200PCI_EWORKSPACE (-3) /* workspace missing or too small */

/* Distance arithmetic (bit-exact contracts, DESIGN.md "Arithmetic"):
 *  EXPANDED: torch square_distance, models/pointconv_util.py:67-88 --
 *            D = fl(fl(-2*fma(z,Z,fma(y,Y,x*X)) + ((x*x+y*y)+z*z)) + ((X*X+Y*Y)+Z*Z))
 *  DIRECT:   the pointnet2 kernels' form, pointnet2/src/interpolate_gpu.cu:37 as compiled --
 *            D = fma(dz,dz,fma(dx,dx,dy*dy)),  d* = query - ref                                  */
#define B200PCI_DIST_EXPANDED 0
#define B200PCI_DIST_DIRECT 1
/*  DIRECT_XYZ: pytorch3d 0.7.5's CUDA knn (`dist += diff*diff` over d = 0,1,2 as nvcc contracts it;
 *            pytorch3d/csrc/knn/knn.cu, not vendored by the reference) --
 *            D = fma(dz,dz,fma(dy,dy,dx*dx))
 *  SQDIFF:   torch.sum((src[:,:,None] - dst[:,None]) ** 2, -1), models/pointT_layer2.py:20 --
 *            D = fl(fl(dx*dx + dy*dy) + dz*dz), every product and sum rounded (k <= 32)        */
#define B200PCI_DIST_DIRECT_XYZ 2
#define B200PCI_DIST_SQDIFF 3
/*  The two torch-defined forms exist in torch's CPU and CUDA evaluation order: torch.sum over a
 *  last dimension of 3 adds (a+b)+c on the CPU and (a+c)+b on CUDA (measured, tools/gpu_probe.py;
 *  the K = 3 matmul gives the same bits on both). EXPANDED / SQDIFF above are the CPU orders (what
 *  BASELINE's CPU torch path and the committed golden vectors hold); the _CUDA variants reproduce the
 *  reference as it runs on a GPU -- |p|^2 = fl(fl(x*x + z*z) + y*y), D = fl(fl(dx*dx + dz*dz) + dy*dy)
 *  for an operand whose coordinate is its fastest-striding dimension ([.., N, 3] contiguous); CUDA
 *  torch reduces a permuted [B, 3, N] view sequentially, (a+b)+c, and so do these modes, operand by
 *  operand, from the strides they are given -- and are what mocopci_b200.install() binds, so a model moved from the reference's CUDA path to
 *  these kernels sees bit-identical neighbour distances.                                          */
#define B200PCI_DIST_SQDIFF_CUDA 4
#define B200PCI_DIST_EXPANDED_CUDA 5

int b200pci_version(void);
/* Message for the last non-zero return on the calling thread ("" if none). */
const char *b200pci_last_error(void);

/* ------------------------------------------------------------------------------------------ */
/* K2 (+K1): fused distance + top-k. Replaces models/pointconv_util.py:129-140 knn_point        */
/* (square_distance :67-88 + torch.topk), its copy models/m_models/mocopci.py:1158-1169, and    */
/* with DIST_DIRECT_XYZ pytorch3d.ops.knn_points as called at models/pointconv_util.py:910,      */
/* with DIST_SQDIFF the neighbour search of models/pointT_layer2.py:62-63.                       */
/*                                                                                              */
/* query (b,i,c) is at q[b*q_sb + i*q_sp + c*q_sc] (element strides, so both [B,S,3] and the    */
/* permuted [B,3,S] views the model passes work without a copy); same for ref.                   */
/* Output per query: the k nearest refs sorted ascending by (distance, index) -- the lowest     */
/* index wins ties. idx is int64 [B,S,k] if idx_is_int64 else int32; dist (nullable) float      */
/* [B,S,k] holds the distances in the chosen arithmetic. Requires 1 <= k <= 64 and, for         */
/* EXPANDED(_CUDA), k <= N (torch.topk raises otherwise -> EINVAL). With DIRECT and k > N the missing   */
/* slots are (inf, 0) like three_nn's m<3 case.                                                 */
/* workspace: device scratch of at least b200pci_knn_workspace_bytes(B,S,N,k), 256-B aligned.   */
/* ------------------------------------------------------------------------------------------ */
size_t b200pci_knn_workspace_bytes(int B, int S, int N, int k);
int b200pci_knn(int B, int S, int N, int k, int dist_mode,
                const float *q, int64_t q_sb, int64_t q_sp, int64_t q_sc,
                const float *r, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                void *idx, int idx_is_int64, float *dist,
                void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------ */
/* f2: feature-space cosine k-NN. Replaces models/pointconv_util.py:142-153 knn_point_cosine     */
/* (cosine_distance :111-127 = normalise both clouds with x / sqrt(sum x^2 + 1e-8), 1 - bmm; then */
/* torch.topk). q [B,S,C], r [B,N,C] float32 given by element strides (the model passes permuted   */
/* [B,C,N] views), C a multiple of 16 (<= 1024), k <= 32, k <= N <= 4096. idx int64/int32         */
/* [B,S,k] sorted ascending by (distance, index); dist (nullable) [B,S,k] = 1 - cosine.           */
/* The contraction runs on the tensor cores (tcgen05 TF32, operands split hi/lo: FP32-level        */
/* accuracy); cuBLAS' summation order in the reference is unspecified, so parity is to ~1e-6, not  */
/* bitwise. workspace_bytes() returns 0 for unsupported shapes (the caller keeps the reference     */
/* path for those).                                                                               */
/* ------------------------------------------------------------------------------------------ */
size_t b200pci_knn_cosine_workspace_bytes(int B, int S, int N, int C, int k);
int b200pci_knn_cosine(int B, int S, int N, int C, int k,
                       const float *q, int64_t q_sb, int64_t q_sn, int64_t q_sc,
                       const float *r, int64_t r_sb, int64_t r_sn, int64_t r_sc,
                       void *idx, int idx_is_int64, float *dist,
                       void *workspace, size_t workspace_bytes, void *stream);

/* Same op with HOST buffers (pinned or pageable): q [B,S,3], r [B,N,3] contiguous float32,
 * idx [B,S,k] on the host, int64 (what knn_point returns) if idx_is_int64 else int32 (half the
 * device-to-host bytes). Copies in, runs b200pci_knn in chunks of clouds so that the copy-out of
 * one chunk overlaps the kernels of the next, and synchronises `stream` before returning. The
 * device buffer, copy stream and events are created on first use per (host thread, device) and
 * reused by later calls; b200pci_host_release() frees the calling thread's.
 * This is what bench.py's `e2e` figure times. */
int b200pci_knn_host(int B, int S, int N, int k, int dist_mode, const float *q_host,
                     const float *r_host, void *idx_host, int idx_is_int64, void *stream);
int b200pci_host_release(void);

/* ------------------------------------------------------------------------------------------ */
/* pointnet2_cuda replacements. Argument order == the reference launchers                       */
/* (pointnet2/src/*_gpu.h), which is also the order of the pybind wrappers                      */
/* (pointnet2/src/pointnet2_api.cpp:10-24) after the tensors are unwrapped.                     */
/* The three neighbourhood searches need scratch: *_workspace_bytes().                          */
/* ------------------------------------------------------------------------------------------ */

/* F1: furthest_point_sampling_wrapper -> sampling_gpu.cu:93-253. xyz [B,N,3], temp [B,N]
 * in/out (caller pre-fills 1e10), idx int32 [B,M]. Tie order identical to the reference's
 * shared-memory tree (DESIGN.md "FPS"). */
int b200pci_furthest_point_sampling(int b, int n, int m, const float *xyz, float *temp, int *idx,
                                    void *stream);

/* F2: gather_points_wrapper / gather_points_grad_wrapper -> sampling_gpu.cu:8-83.
 * points [B,C,N], idx int32 [B,M] -> out [B,C,M]; grad_points [B,C,N] must be pre-zeroed. */
int b200pci_gather_points(int b, int c, int n, int npoints, const float *points, const int *idx,
                          float *out, void *stream);
int b200pci_gather_points_grad(int b, int c, int n, int npoints, const float *grad_out,
                               const int *idx, float *grad_points, void *stream);

/* Q1: ball_query_wrapper -> ball_query_gpu.cu:9-64. new_xyz [B,M,3], xyz [B,N,3],
 * idx int32 [B,M,nsample] pre-zeroed by the caller (pointnet2_utils.py:218). */
size_t b200pci_ball_query_workspace_bytes(int b, int n, int m, int nsample);
int b200pci_ball_query(int b, int n, int m, float radius, int nsample, const float *new_xyz,
                       const float *xyz, int *idx, void *workspace, size_t workspace_bytes,
                       void *stream);

/* G1: group_points_wrapper / group_points_grad_wrapper -> group_points_gpu.cu:8-86.
 * points [B,C,N], idx int32 [B,npoints,nsample] -> out [B,C,npoints,nsample]. */
int b200pci_group_points(int b, int c, int n, int npoints, int nsample, const float *points,
                         const int *idx, float *out, void *stream);
int b200pci_group_points_grad(int b, int c, int n, int npoints, int nsample,
                              const float *grad_out, const int *idx, float *grad_points,
                              void *stream);

/* Q2: the grouping half of QueryAndGroup.forward (pointnet2/pointnet2_utils.py:250-264: transpose of
 * the cloud, grouping_operation, `-= new_xyz`, grouping_operation on the features, torch.cat) in
 * two launches writing straight into the concatenated tensor: xyz [B,N,3] (row-major, no transposed
 * copy), new_xyz [B,npoints,3], features [B,C,N] (NULL with c = 0), idx int32 [B,npoints,nsample]
 * (b200pci_ball_query's output) -> out [B, 3 + C, npoints, nsample] (use_xyz != 0) or
 * [B, C, npoints, nsample]; channels 0..2 hold xyz[idx] - new_xyz, one IEEE subtraction each, the
 * rest are copies: bit-identical to the reference composition. */
int b200pci_query_group(int b, int n, int npoints, int nsample, int c, const float *xyz,
                        const float *new_xyz, const float *features, const int *idx, float *out,
                        int use_xyz, void *stream);

/* T1: three_nn_wrapper -> interpolate_gpu.cu:9-74. unknown [B,n,3], known [B,m,3] ->
 * dist2 [B,n,3] (squared), idx int32 [B,n,3]. */
size_t b200pci_three_nn_workspace_bytes(int b, int n, int m);
int b200pci_three_nn(int b, int n, int m, const float *unknown, const float *known, float *dist2,
                     int *idx, void *workspace, size_t workspace_bytes, void *stream);

/* T3 (optional fused path): three_nn followed by the inverse-distance weights its only in-repo
 * caller computes with five torch ops (pointnet2/pointnet2_modules.py:139-144 on top of
 * pointnet2_utils.py:97): dist = sqrt(dist2), r = 1/(dist + eps), weight = r / sum_j r_j.
 * dist [B,n,3] (NOT squared), weight [B,n,3], idx int32 [B,n,3]; same workspace as three_nn.
 * Bitwise equal to the torch composition on CUDA (IEEE sqrt / divide, sum as (r0+r2)+r1). */
int b200pci_three_nn_weights(int b, int n, int m, const float *unknown, const float *known,
                             float eps, float *dist, float *weight, int *idx, void *workspace,
                             size_t workspace_bytes, void *stream);

/* T2: three_interpolate_wrapper / _grad_wrapper -> interpolate_gpu.cu:77-161.
 * points [B,C,m], idx int32 [B,n,3], weight [B,n,3] -> out [B,C,n];
 * out = fma(w2,p2,fma(w0,p0,w1*p1)) exactly as the reference compiles. */
int b200pci_three_interpolate(int b, int c, int m, int n, const float *points, const int *idx,
                              const float *weight, float *out, void *stream);
int b200pci_three_interpolate_grad(int b, int c, int n, int m, const float *grad_out,
                                   const int *idx, const float *weight, float *grad_points,
                                   void *stream);

/* ------------------------------------------------------------------------------------------ */
/* K3 / K4: index_points_group / index_points_gather, models/pointconv_util.py:168-192 (copies   */
/* models/m_models/mocopci.py:1190-1215): out[b,t,:] = points[b, idx[b,t], :] in the [B,N,C]      */
/* layout the model keeps its features in. The reference transposes to [B,C,N] (a copy), casts   */
/* the int64 KNN indices to int32, gathers into [B,C,S,K] and returns a permuted view; here one   */
/* kernel reads the strided `points` view (element strides p_sb, p_sn, p_sc), takes int64 or     */
/* int32 idx [B,T] (T = S*K, or S for the gather) and writes contiguous [B,T,C].                  */
/* _grad: grad_points [B,N,C] contiguous, pre-zeroed by the caller, accumulated with atomics.     */
/* ------------------------------------------------------------------------------------------ */
int b200pci_index_points_rows(int B, int N, long long T, int C, const float *points,
                              int64_t p_sb, int64_t p_sn, int64_t p_sc, const void *idx,
                              int idx_is_int64, float *out, void *stream);
int b200pci_index_points_rows_grad(int B, int N, long long T, int C, const float *grad_out,
                                   const void *idx, int idx_is_int64, float *grad_points,
                                   void *stream);

/* f1: group / group_query, models/pointconv_util.py:194-241 (copies models/m_models/mocopci.py:
 * 1218-1266), after the neighbour search: out[b,s,k,:] = [xyz[b,idx[b,s,k],:] - centre[b,s,:] |
 * points[b,idx[b,s,k],:]] ([B,S,K,3+D] contiguous) and norm[b,s,k,:] = the first three ([B,S,K,3],
 * nullable). xyz [B,N,3], centre [B,S,3], points [B,N,D] (nullable when D = 0) are strided views
 * (element strides batch / point / channel); idx int64 or int32 [B,S,K]. One kernel instead of the
 * reference's two gathers (each with a transpose copy and an index cast), the broadcast
 * subtraction and torch.cat. out may be null when only norm is wanted. */
int b200pci_group_concat(int B, int N, int S, int K, int D, const float *xyz, int64_t x_sb, int64_t x_sn,
                         int64_t x_sc, const float *centre, int64_t c_sb, int64_t c_sn, int64_t c_sc,
                         const float *points, int64_t p_sb, int64_t p_sn, int64_t p_sc, const void *idx,
                         int idx_is_int64, float *out, float *norm, void *stream);

/* ------------------------------------------------------------------------------------------ */
/* C1: Chamfer. Replaces pytorch3d.loss.chamfer_distance as used by models/utils.py:36-45        */
/* (defaults: squared L2, point_reduction="mean", batch_reduction="mean").                       */
/* x [B,N,3], y [B,M,3] (strided like b200pci_knn). Outputs: per-point squared NN distance and   */
/* NN index in each direction (dist_x [B,N], idx_x int32 [B,N], dist_y [B,M], idx_y [B,M]) and   */
/* loss[0] = mean_b(mean_i dist_x + mean_j dist_y) accumulated in FP64 then rounded.             */
/* Both searches are K = 1 in DIST_DIRECT_XYZ, pytorch3d's fma(dz,dz,fma(dy,dy,dx*dx)) with      */
/* d = point - candidate; among equal distances the lowest index wins. So dist_x / idx_x equal   */
/* b200pci_knn(K=1, DIST_DIRECT_XYZ) with queries x and refs y bit for bit (knn_points), and     */
/* dist_y / idx_y the same with x and y exchanged.                                              */
/* ------------------------------------------------------------------------------------------ */
size_t b200pci_chamfer_workspace_bytes(int B, int N, int M);
int b200pci_chamfer_forward(int B, int N, int M,
                            const float *x, int64_t x_sb, int64_t x_sp, int64_t x_sc,
                            const float *y, int64_t y_sb, int64_t y_sp, int64_t y_sc,
                            float *dist_x, int *idx_x, float *dist_y, int *idx_y, float *loss,
                            void *workspace, size_t workspace_bytes, void *stream);
/* d loss / d x, d loss / d y given grad_loss[0]; grad_x [B,N,3], grad_y [B,M,3] contiguous,
 * overwritten. x, y contiguous [B,N,3] / [B,M,3]. */
int b200pci_chamfer_backward(int B, int N, int M, const float *x, const float *y,
                             const int *idx_x, const int *idx_y, const float *grad_loss,
                             float *grad_x, float *grad_y, void *stream);

/* ------------------------------------------------------------------------------------------ */
/* D1: deterministic gradients (_det). The scatter-add backwards above add their contributions   */
/* with float atomics, so the last bits of a gradient vary from run to run. Each _det twin takes */
/* the same arguments plus device scratch and gives the same sums in ONE fixed order: every      */
/* destination element is accumulated sequentially in FP32, starting from the value the output  */
/* holds (callers pre-zero it; Chamfer overwrites), contributions in ascending source position,  */
/* each product rounded before it is added (no FMA). Every such sum is one of the orders the     */
/* atomic kernels can produce. Bit for bit reproducible across runs, streams and GPUs of one     */
/* architecture. Entries of idx outside [0, N) contribute nothing.                               */
/* Scratch: an inverse index (CSR) of idx per cloud, built on the stream from integer counts;    */
/* no allocation, no host synchronisation (stream-ordered, graph capturable).                    */
/* Returns EWORKSPACE for missing or short scratch, EINVAL for 2^31 or more source positions     */
/* per cloud and for the arguments the atomic twin rejects.                                      */
/* ------------------------------------------------------------------------------------------ */
/* Scratch of a CSR over N destinations of T source positions per cloud (B clouds): the gather,
 * group and rows twins need (B, N, T), three_interpolate (B, m, 3n). 256-B aligned. */
size_t b200pci_scatter_workspace_bytes(int B, int N, long long T);
/* grad_points[b,c,i] = ((g0 + grad_out[b,c,t1]) + grad_out[b,c,t2]) + ...,  t1 < t2 < ... the
 * positions with idx[b,t] == i (t over npoints, or npoints*nsample for group); g0 the value
 * grad_points holds: a sequential loop over t. */
int b200pci_gather_points_grad_det(int b, int c, int n, int npoints, const float *grad_out,
                                   const int *idx, float *grad_points, void *workspace,
                                   size_t workspace_bytes, void *stream);
int b200pci_group_points_grad_det(int b, int c, int n, int npoints, int nsample,
                                  const float *grad_out, const int *idx, float *grad_points,
                                  void *workspace, size_t workspace_bytes, void *stream);
/* grad_points[b,c,k] = g0 + fl(grad_out[b,c,i] * weight[b,i,j]) + ... over the (i, j) with
 * idx[b,i,j] == k, ascending (i, j), j the slot 0..2 (the repeated slots of three_nn's m < 3 case
 * in slot order). Scratch b200pci_scatter_workspace_bytes(b, m, 3 n). */
int b200pci_three_interpolate_grad_det(int b, int c, int n, int m, const float *grad_out,
                                       const int *idx, const float *weight, float *grad_points,
                                       void *workspace, size_t workspace_bytes, void *stream);
/* grad_points[b,i,c] = ((g0 + grad_out[b,t1,c]) + grad_out[b,t2,c]) + ..., t ascending;
 * grad_points [B,N,C] contiguous, pre-zeroed; idx int64 or int32 [B,T]. */
int b200pci_index_points_rows_grad_det(int B, int N, long long T, int C, const float *grad_out,
                                       const void *idx, int idx_is_int64, float *grad_points,
                                       void *workspace, size_t workspace_bytes, void *stream);
/* Chamfer, overwriting grad_x / grad_y. Per-point terms as b200pci_chamfer_backward computes
 * them: w_x = fl(fl(2 g) / fl(B N)), d_x(i) = fl(w_x * fl(x_i - y_{idx_x[i]})), the same for y
 * with M. grad_x[b,i] = ((0 + d_x(i)) - d_y(j1)) - d_y(j2) - ..., j1 < j2 < ... the points of y
 * whose nearest x is i; grad_y the mirror image. */
size_t b200pci_chamfer_backward_det_workspace_bytes(int B, int N, int M);
int b200pci_chamfer_backward_det(int B, int N, int M, const float *x, const float *y,
                                 const int *idx_x, const int *idx_y, const float *grad_loss,
                                 float *grad_x, float *grad_y, void *workspace,
                                 size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------ */
/* K5: backward of b200pci_knn's distances (any dist_mode; pytorch3d knn_points' backward, the   */
/* dists of models/pointconv_util.py:910 under autograd). q [B,S,3], r [B,N,3] strided like      */
/* b200pci_knn; idx int64/int32 [B,S,K] contiguous (b200pci_knn's output); grad_dist [B,S,K]     */
/* contiguous. grad_q [B,S,3], grad_r [B,N,3] contiguous, OVERWRITTEN.                            */
/* Arithmetic, for slot (i, k) with j = idx[b,i,k] and each coordinate c:                         */
/*   d(i,k)_c = fl( fl(2 * grad_dist[b,i,k]) * fl(q[b,i,c] - r[b,j,c]) ), no FMA -- the form of   */
/*   pytorch3d's KNN backward kernel, 2 * grad_dist * (p1 - p2) (PARITY UNPINNED, as the forward); */
/*   grad_q[b,i,c] = ((0 + d(i,0)_c) + d(i,1)_c) + ..., k ascending;                              */
/*   grad_r[b,j,c] = ((0 - d(t1)_c) - d(t2)_c) - ..., over the flat slots t = i*K + k with        */
/*   idx == j, t ascending (the _det order; the atomic variant adds the same terms in any order).  */
/* A slot contributes nothing when k >= N (the (inf, 0) padding of the DIRECT modes for K > N) or */
/* when j is outside [0, N). grad_q has the same bits from both entry points (one thread walks a  */
/* query's slots in order, no atomics); only grad_r differs.                                      */
/* Both: EINVAL for negative sizes, null pointers, B > 65535 or S*K >= 2^31; B = 0 or S = N = 0   */
/* is a no-op. _det: scratch of b200pci_scatter_workspace_bytes(B, N, S*K) (EWORKSPACE when      */
/* missing or short), the D1 guarantees above (no allocation, no host synchronisation).           */
/* ------------------------------------------------------------------------------------------ */
int b200pci_knn_backward(int B, int S, int N, int K,
                         const float *q, int64_t q_sb, int64_t q_sp, int64_t q_sc,
                         const float *r, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                         const void *idx, int idx_is_int64, const float *grad_dist,
                         float *grad_q, float *grad_r, void *stream);
int b200pci_knn_backward_det(int B, int S, int N, int K,
                             const float *q, int64_t q_sb, int64_t q_sp, int64_t q_sc,
                             const float *r, int64_t r_sb, int64_t r_sp, int64_t r_sc,
                             const void *idx, int idx_is_int64, const float *grad_dist,
                             float *grad_q, float *grad_r, void *workspace,
                             size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------ */
/* P1 / P2: pytorch3d.ops.ball_query and pytorch3d.ops.sample_farthest_points (0.7.5, PARITY     */
/* UNPINNED as for knn_points: the contract below is this library's own). Ragged batches: the    */
/* per-cloud lengths are int64 [B] DEVICE arrays, read by the kernels and clamped to [0, P]      */
/* (NULL: every cloud has P points). Neither call allocates, needs scratch or synchronises with  */
/* the host; both are graph capturable and launch one kernel on `stream`.                        */
/* ------------------------------------------------------------------------------------------ */
/* P1: p1 [B,P1,3], p2 [B,P2,3] float32 through element strides (like b200pci_knn). For query    */
/* i < lengths1[b], the slots of idx[b,i,:] hold, in ascending j, the first K refs j < lengths2[b] */
/* with d2 < r2 (strict), d2 = fma(dz,dz,fma(dy,dy,dx*dx)), d = p1[b,i] - p2[b,j] (DIST_DIRECT_XYZ) */
/* and r2 = radius * radius rounded in FP32; dists holds those d2. Slots past the hits, and every   */
/* slot of a query i >= lengths1[b], are idx = -1, dists = 0. idx int64 [B,P1,K], dists float32    */
/* [B,P1,K], nn (nullable) float32 [B,P1,K,3] = p2[b, idx] row by row (zeros where idx = -1).     */
/* Every output element is written. EINVAL: negative sizes, K < 1, radius < 0 or NaN, null        */
/* pointers, B > 65535. B = 0 or P1 = 0 is a no-op. The distance backward is b200pci_knn_backward */
/* (_det) with this idx as is: -1 slots contribute nothing, and a query has at most P2 hits, so    */
/* none sits in a slot k >= P2.                                                                   */
/* ------------------------------------------------------------------------------------------ */
int b200pci_ball_query_p3d(int B, int P1, int P2, int K, float radius,
                           const float *p1, int64_t p1_sb, int64_t p1_sp, int64_t p1_sc,
                           const float *p2, int64_t p2_sb, int64_t p2_sp, int64_t p2_sc,
                           const int64_t *lengths1, const int64_t *lengths2,
                           int64_t *idx, float *dists, float *nn, void *stream);
/* P2: points [B,P,3] float32 through element strides. Per cloud n = lengths[b] points and         */
/* m = min(K[b], n) picks (K: int64 [B] device array, values clamped to [0, M]; NULL: M for every */
/* cloud). idx[b,0] = start[b] (int64 [B] device array clamped to [0, n-1]; NULL: 0); pick t > 0   */
/* is the argmax over j < n of the running minimum, over the earlier picks, of                   */
/* d2 = fma(dz,dz,fma(dy,dy,dx*dx)) (the minimum starts at +inf); among equal values the LOWEST   */
/* index wins (b200pci_furthest_point_sampling keeps the reference's bit-reversed thread order    */
/* instead). Picks m..M-1 are -1. idx int64 [B,M]; selected (nullable) float32 [B,M,3] = the      */
/* picked points' rows, zeros for -1. EINVAL: negative sizes, null pointers, P > 131072,          */
/* B > 2^27. B = 0 or M = 0 is a no-op.                                                            */
int b200pci_fps_p3d(int B, int P, int M, const float *points, int64_t p_sb, int64_t p_sp,
                    int64_t p_sc, const int64_t *lengths, const int64_t *K, const int64_t *start,
                    int64_t *idx, float *selected, void *stream);

/* ------------------------------------------------------------------------------------------ */
/* E1-E3: emd_cuda replacements (models/EMD/cuda/emd.cpp:23-27, emd_kernel.cu).                  */
/* xyz1 [B,n,3], xyz2 [B,m,3] contiguous. match [B,m,n]; temp: scratch of                        */
/* b200pci_emd_workspace_bytes(B,n,m). Launches on `stream` (the reference uses the legacy       */
/* default stream, emd_kernel.cu:192). All four return EINVAL for negative sizes, null pointers   */
/* or B > 65535 (one grid row per pair).                                                         */
/* ------------------------------------------------------------------------------------------ */
size_t b200pci_emd_workspace_bytes(int B, int n, int m);
int b200pci_emd_approxmatch(int B, int n, int m, const float *xyz1, const float *xyz2,
                            float *match, void *workspace, size_t workspace_bytes, void *stream);
int b200pci_emd_matchcost(int B, int n, int m, const float *xyz1, const float *xyz2,
                          const float *match, float *cost, void *workspace,
                          size_t workspace_bytes, void *stream);
int b200pci_emd_matchcost_grad(int B, int n, int m, const float *grad_cost, const float *xyz1,
                               const float *xyz2, const float *match, float *grad1, float *grad2,
                               void *stream);
/* Forward-only cost[b] = matchcost(approxmatch(xyz1, xyz2)) for the eval metric EMD()
 * (models/utils.py:223-235 -> emd_kernel.cu:175-197,261-283) WITHOUT materialising match
 * (1.07 GB per pair at 16384 x 16384): the per-level increments of match are weighted with the
 * squared distance and summed on the fly (FP64 across tiles and levels). Same workspace size. */
int b200pci_emd_cost(int B, int n, int m, const float *xyz1, const float *xyz2, float *cost,
                     void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------ */
/* Roofline probes (bench.py): measured FP32 FMA peak and device copy bandwidth.                 */
/* b200pci_probe_fp32 runs `iters` dependent-free FFMA (packed=0) or FFMA2 (packed=1) per lane   */
/* on a full grid and returns the flop count through *flops; time it with CUDA events.           */
/* ------------------------------------------------------------------------------------------ */
int b200pci_probe_fp32(int packed, int iters, float *sink, double *flops, void *stream);

/* Test / measurement hooks, never needed in production (process-global, not thread-safe).
 * b200pci_debug_set(key, value):
 *    1  scale applied to the estimated KNN admission bound (1.0; < 1 forces the exact-redo path)
 *    2  1 = in-kernel streaming engine for every KNN, 2 = one-launch kernel for every KNN (0)
 *    3  1 = start (and reset) CUDA-event timing of the dominant KNN kernel on its launching stream
 *    5  1 = force the single-CTA FPS kernel (0)
 *    6  1 = send every ball query through the exact redo kernel (0)
 *    7  pair count from which k <= 4 takes the two-pass path (0 = default 2^25)
 *   11  R of the estimated bound (0 = default by k)
 *   12 / 13  ref count / pair count from which k = 5..32 takes the two-pass path (0 = defaults)
 *   14  number of (equal) chunks of b200pci_knn_host's copy pipeline (0 = default: tapered schedule)
 *   18  0 = thread-per-query top-k kernel even for small launches (1 = one thread per (query, split group)
 *       for launches of fewer than two CTAs per SM, 2 = whenever the refs are split)
 *   20  0 = thread t of the top-k kernel takes query t (1 = queries handed out by list length)
 *   19  lanes per row of the forward-only EMD sweeps: 4, 8, 16 (default), 32
 *   15 / 16  three_interpolate: point slices of the quad kernel (0 = automatic) / 1 = rows kernel
 *   any other key: B200PCI_EINVAL, nothing changed
 * b200pci_debug_get(key): 3 = accumulated ms of the timed launches, 4 = their number;
 *    5 / 6 = flagged tiles / flagged queries of the calling thread's last two-pass KNN call
 *    (synchronises the device; -1 if this thread has made none). */
int b200pci_debug_set(int key, double value);
double b200pci_debug_get(int key);

#ifdef __cplusplus
}
#endif
#endif /* B200PCI_H */
