/* TEST INFRASTRUCTURE ONLY -- CPU restatements of the two gradients the C oracle (oracle/oracle.c)
 * does not cover, written as plain sequential loops in the summation order of the deterministic
 * entry points (include/b200pci.h, "_det"). Built by tests/grad_oracle.py with -ffp-contract=off,
 * like the oracle: every product and every sum is rounded on its own. The product never loads it.
 */
#include <stddef.h>
#include <stdint.h>

/* models/pointconv_util.py:168-192 backward: grad_points [B,N,C] (pre-zeroed) += grad_out [B,T,C]
 * rows at idx [B,T] (int64), t ascending; indices outside [0, N) are skipped. */
void orc_index_rows_grad(int B, int N, long long T, int C, const float *grad_out, const int64_t *idx,
                         float *grad_points) {
    for (int b = 0; b < B; ++b)
        for (long long t = 0; t < T; ++t) {
            const int64_t i = idx[(size_t)b * T + t];
            if (i < 0 || i >= N) continue;
            float *gp = grad_points + ((size_t)b * N + i) * C;
            const float *g = grad_out + ((size_t)b * T + t) * C;
            for (int c = 0; c < C; ++c) gp[c] += g[c];
        }
}

/* d loss / d x, d loss / d y of the Chamfer loss (models/utils.py:36-45) given the nearest-neighbour
 * indices ix [B,N], iy [B,M] and d loss = grad_loss; gx [B,N,3], gy [B,M,3] overwritten.
 * w_x = fl(fl(2 g) / fl(B N)), d_x(i) = fl(w_x fl(x_i - y_{ix[i]})), the same for y with M;
 * gx[i] = ((0 + d_x(i)) - d_y(j1)) - d_y(j2) - ..., j ascending over the y points whose nearest x
 * is i; gy the mirror image. */
void orc_chamfer_backward(int B, int N, int M, const float *x, const float *y, const int32_t *ix,
                          const int32_t *iy, float grad_loss, float *gx, float *gy) {
    const float g2 = 2.f * grad_loss;
    const float wx = g2 / ((float)B * (float)N), wy = g2 / ((float)B * (float)M);
    for (size_t k = 0; k < (size_t)B * N * 3; ++k) gx[k] = 0.f;
    for (size_t k = 0; k < (size_t)B * M * 3; ++k) gy[k] = 0.f;
    for (int b = 0; b < B; ++b) {
        const float *xb = x + (size_t)b * N * 3, *yb = y + (size_t)b * M * 3;
        float *gxb = gx + (size_t)b * N * 3, *gyb = gy + (size_t)b * M * 3;
        /* each point's own term first, then the terms of the points whose nearest neighbour it is,
           in ascending order of those points */
        for (int i = 0; i < N; ++i)
            for (int c = 0; c < 3; ++c) gxb[i * 3 + c] += wx * (xb[i * 3 + c] - yb[ix[(size_t)b * N + i] * 3 + c]);
        for (int j = 0; j < M; ++j)
            for (int c = 0; c < 3; ++c) gyb[j * 3 + c] += wy * (yb[j * 3 + c] - xb[iy[(size_t)b * M + j] * 3 + c]);
        for (int j = 0; j < M; ++j) {
            const int i = iy[(size_t)b * M + j];
            for (int c = 0; c < 3; ++c) gxb[i * 3 + c] -= wy * (yb[j * 3 + c] - xb[i * 3 + c]);
        }
        for (int i = 0; i < N; ++i) {
            const int j = ix[(size_t)b * N + i];
            for (int c = 0; c < 3; ++c) gyb[j * 3 + c] -= wx * (xb[i * 3 + c] - yb[j * 3 + c]);
        }
    }
}
