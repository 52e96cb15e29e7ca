// cw_grad.cu -- backward of cobweb_rank_scores w.r.t. the query
// (src/cobweb/CobwebWrapper.py:267-294 is differentiable in x; its one consumer is
// FixedDocsRankingLoss, src/training/cobweb_query_train.py:104-126).
//
//   leaf[q,l] = sum_j w(len_l, j) * s[q, path(l, j)],   s[q,n] = -0.5 (sumlog_n + sum_d (x_qd r_nd + mb_nd)^2)
//   dL/dx[q,d] = - sum_n gs[q,n] * (x_qd r_nd + mb_nd) r_nd,   gs[q,n] = sum_{l : n in path(l)} w * dL/dleaf[q,l]
//
// Kernel 1 (path transpose): lane = query, positions in tree order; a node's descendants are a
// contiguous run of positions, so each level keeps a running sum that is flushed when the node
// at that level changes (atomicAdd only because a run may straddle two chunks).
// Kernel 2: gs^T [Q, Nn] times the node operands, 64 queries x 64 attributes per CTA, FP32 FMA.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/cobweb_b200.h"

void cw_set_error(const char *fmt, ...);
int cw_check_cuda(cudaError_t e, const char *what);

namespace cw {

// grid (position chunks, query groups of 32 per warp, 1/2/4 warps per CTA)
__global__ void __launch_bounds__(128)
paths_transpose_kernel(const float *__restrict__ G, long long nq, int n_pos, int max_len,
                       const int *__restrict__ path_pm, const int4 *__restrict__ pos_rec,
                       const double *__restrict__ level_w, float *gs, unsigned ldq, int chunk_len) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    double *lw = reinterpret_cast<double *>(sm_raw);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    float *run = reinterpret_cast<float *>(lw + max_len) + (size_t)warp * max_len * 32;       // [max_len][32]
    int *node = reinterpret_cast<int *>(reinterpret_cast<float *>(lw + max_len) + (size_t)wpb * max_len * 32) +
                (size_t)warp * max_len;                                                    // [max_len]
    for (int i = threadIdx.x; i < max_len; i += blockDim.x) lw[i] = level_w[i];
    __syncthreads();
    const long long g = (long long)blockIdx.y * wpb + warp;
    if (g * 32 >= nq) return;
    const long long q = g * 32 + lane;
    const bool qvalid = q < nq;
    const int p0 = blockIdx.x * chunk_len, p1 = min(n_pos, p0 + chunk_len);
    int open_len = 0;  // levels currently holding an open run
    for (int p = p0; p <= p1; p++) {
        int len = 0, m = 0;
        int4 rc = make_int4(0, 0, 0, 0);
        if (p < p1) {
            rc = pos_rec[p];
            len = rc.x;
            m = (p == p0) ? 0 : rc.y;
            // the stored prefix is 0 when the lengths differ although the leading nodes may still be
            // shared; recompute against the open run so that shared ancestors are not flushed early
            if (p != p0 && m == 0) {
                while (m < len && m < open_len && path_pm[(size_t)p * max_len + m] == node[m]) m++;
            }
        }
        // flush levels m .. open_len-1 of the previous path
        for (int j = m; j < open_len; j++) {
            if (qvalid) atomicAdd(&gs[(size_t)(unsigned)node[j] * ldq + q], run[j * 32 + lane]);
        }
        __syncwarp();
        if (p == p1) break;
        const float gq = qvalid ? G[q * n_pos + rc.w] : 0.0f;
        const double dlen = (double)len;
        for (int j = 0; j < len; j++) {
            const float w = (float)(lw[j] / dlen);
            if (j < m) {
                run[j * 32 + lane] = fmaf(w, gq, run[j * 32 + lane]);
            } else {
                if (lane == 0) node[j] = path_pm[(size_t)p * max_len + j];
                run[j * 32 + lane] = w * gq;
            }
        }
        open_len = len;
        __syncwarp();
    }
}

// out[q,d] = -(x[q,d] * sum_n gs[n,q] r[n,d]^2 + sum_n gs[n,q] mb[n,d] r[n,d]); operands in the index's
// tiled layout [node tile][k tile][CW_TILE_K][CW_TILE_N]
constexpr int GQ = 64, GD = 64, GN = 16;
__global__ void __launch_bounds__(256)
rank_grad_kernel(const float *__restrict__ gs, unsigned ldq, long long nq, int nn, int D, int n_ktiles,
                 const float *__restrict__ R, const float *__restrict__ MB, const float *__restrict__ X,
                 float *__restrict__ out) {
    __shared__ float As[GN][GQ + 1], B1[GN][GD + 1], B2[GN][GD + 1];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const long long q0 = (long long)blockIdx.x * GQ;
    const int d0 = blockIdx.y * GD;
    float a1[4][4] = {}, a2[4][4] = {};
    for (int n0 = 0; n0 < nn; n0 += GN) {
        for (int i = tid; i < GN * GQ; i += 256) {
            const int r = i / GQ, c = i % GQ;
            const int n = n0 + r;
            const long long q = q0 + c;
            As[r][c] = (n < nn && q < nq) ? gs[(size_t)n * ldq + q] : 0.0f;
        }
        for (int i = tid; i < GN * GD; i += 256) {
            const int c = i / GN, r = i % GN;  // consecutive threads -> consecutive nodes (contiguous in the tile)
            const int n = n0 + r, d = d0 + c;
            float rv = 0.0f, mv = 0.0f;
            if (n < nn && d < D) {
                const size_t off = ((size_t)(n / CW_TILE_N) * n_ktiles + d / CW_TILE_K) * (CW_TILE_K * CW_TILE_N) +
                                   (size_t)(d % CW_TILE_K) * CW_TILE_N + (n % CW_TILE_N);
                rv = R[off];
                mv = MB[off];
            }
            B1[r][c] = rv * rv;
            B2[r][c] = mv * rv;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < GN; r++) {
            float av[4], b1[4], b2[4];
#pragma unroll
            for (int i = 0; i < 4; i++) { av[i] = As[r][ty * 4 + i]; b1[i] = B1[r][tx * 4 + i]; b2[i] = B2[r][tx * 4 + i]; }
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    a1[i][j] = fmaf(av[i], b1[j], a1[i][j]);
                    a2[i][j] = fmaf(av[i], b2[j], a2[i][j]);
                }
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const long long q = q0 + ty * 4 + i;
        if (q >= nq) continue;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int d = d0 + tx * 4 + j;
            if (d < D) out[q * D + d] = -(X[q * D + d] * a1[i][j] + a2[i][j]);
        }
    }
}

}  // namespace cw

extern "C" int cw_rank_scores_bwd(const cw_index *ix, const float *Q, int64_t nq, const float *grad_leaf,
                                  float *gs_scratch, int64_t ldq, float *grad_q, void *stream) {
    if (!ix || !Q || !grad_leaf || !gs_scratch || !grad_q || nq < 0 || ix->n_pos < 1 || ldq < nq || ldq > 0x7fffffffLL) {
        cw_set_error("cw_rank_scores_bwd: bad argument");
        return CW_E_ARG;
    }
    if (nq == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    // warps per CTA of the path transpose: each warp keeps a [max_len][32] run stack and a [max_len] node list in shared
    // memory, so deep trees get 2 or 1 warps per CTA (the forward path kernel accepts max_len up to 1024)
    int dev = 0, optin = 0;
    int rc = cw_check_cuda(cudaGetDevice(&dev), "cw_rank_scores_bwd: device");
    if (rc) return rc;
    rc = cw_check_cuda(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev), "cw_rank_scores_bwd: smem limit");
    if (rc) return rc;
    auto smem_of = [&](int w) {
        return (size_t)ix->max_len * sizeof(double) + (size_t)w * ix->max_len * (32 * sizeof(float) + sizeof(int));
    };
    int wpb = 4;
    while (wpb > 1 && smem_of(wpb) > (size_t)optin) wpb /= 2;
    if (smem_of(wpb) > (size_t)optin) {
        cw_set_error("cw_rank_scores_bwd: max_len=%d needs %zu bytes of shared memory with one warp per CTA, more than the %d one CTA has",
                     ix->max_len, smem_of(1), optin);
        return CW_E_ARG;
    }
    rc = cw_check_cuda(cudaMemsetAsync(gs_scratch, 0, (size_t)ix->nn * ldq * sizeof(float), st), "cw_rank_scores_bwd: memset");
    if (rc) return rc;
    const long long groups = (nq + 31) / 32, gblocks = (groups + wpb - 1) / wpb;
    long long want = (148 * 32 + groups - 1) / groups;
    if (want > (ix->n_pos + 255) / 256) want = (ix->n_pos + 255) / 256;
    if (want < 1) want = 1;
    const int chunk_len = (int)((ix->n_pos + want - 1) / want);
    const int n_chunks = (ix->n_pos + chunk_len - 1) / chunk_len;
    const size_t smem = smem_of(wpb);
    if (smem > 48 * 1024) {
        rc = cw_check_cuda(cudaFuncSetAttribute(cw::paths_transpose_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                           "cw_rank_scores_bwd: smem attribute");
        if (rc) return rc;
    }
    cw::paths_transpose_kernel<<<dim3(n_chunks, (unsigned)gblocks), wpb * 32, smem, st>>>(
        grad_leaf, nq, ix->n_pos, ix->max_len, ix->path_idx, reinterpret_cast<const int4 *>(ix->pos_rec), ix->level_w,
        gs_scratch, (unsigned)ldq, chunk_len);
    dim3 g2((unsigned)((nq + cw::GQ - 1) / cw::GQ), (unsigned)((ix->D + cw::GD - 1) / cw::GD));
    cw::rank_grad_kernel<<<g2, 256, 0, st>>>(gs_scratch, (unsigned)ldq, nq, ix->nn, ix->D, ix->n_ktiles, ix->R, ix->MB, Q, grad_q);
    return cw_check_cuda(cudaGetLastError(), "cw_rank_scores_bwd");
}
