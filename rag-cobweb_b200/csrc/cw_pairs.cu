// Exact leaf scores of chosen (query, sentence) pairs and their gradient w.r.t. the queries (cw_pair_scores,
// cw_pair_scores_bwd): the FP32 form's result for a candidate list, without scoring the rest of the index.
//
// Per query, the rows on the candidates' paths are listed once and scored once:
//   pair_list_kernel   one CTA per query: sorts the candidates by position (positions are in leaf BFS-row order: by
//                      depth, then lexicographically by path), drops each candidate's common prefix with its
//                      predecessor in that order, lists the remaining levels' index rows and writes the map
//                      (candidate, level) -> list entry;
//   fn_exact_kernel    (cw_half.cu) exact node scores of the listed rows, one warp per (query, row block);
//   pair_sum_kernel    one thread per (query, candidate): the path sum, root first, in the caller's candidate order.
// The backward runs pair_list_kernel with the incoming gradient, which turns the map into one coefficient per list entry
// (gs_e = sum over the candidates through it of G[q, c] w(len_c, level)), and pair_grad_kernel, one CTA per query:
// grad_q[q, d] = -sum_e gs_e (x_d r_ed + mb_ed) r_ed.  Every sum has a fixed order and one owner: no atomics, the same bits
// on every run.
//
// A row listed twice (the sort puts a deeper cousin after a shallower one, so their shared ancestors are listed again)
// costs a second read, never a different result: both entries get the same bits.

#include <climits>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/cobweb_b200.h"

void cw_set_error(const char *fmt, ...);
int cw_check_cuda(cudaError_t e, const char *what);
int cw_exact_rows_attr();
void cw_exact_rows_launch(const cw_index &ix, const float2 *RM, const float *Q, long long nq, const int *list,
                          const int *meta, int meta_stride, int n_word, int stride, float *out, int row_blocks,
                          cudaStream_t st);

namespace cwp {

constexpr int PL_THREADS = 256, PL_WARPS = PL_THREADS / 32, PL_PER = CW_PAIR_MAX_M / PL_THREADS;
constexpr int GR_THREADS = 256, GR_PER = CW_MAX_D / GR_THREADS;  // attributes per thread of pair_grad_kernel
static_assert(CW_PAIR_MAX_M % PL_THREADS == 0, "slots per thread of the scan");

struct PairArgs {
    const int *path_idx;   // [n_pos, max_len]
    const int4 *pos_rec;   // [n_pos] {len, common prefix, leaf row, sentence id}
    const double *level_w; // [max_len]
    int n_pos, max_len;
    const int *pos_of_sid; // [n_sid]
    int n_sid;
    const int *cand;       // [nq, m]
    long long nq;
    int m;
    int E;                 // list entries per query: m * max_len
    const float *grad_out; // [nq, m] (backward)
    int *n_rows;           // [nq]
    int *list;             // [nq, E] index rows
    float *val;            // [nq, E] exact node scores (forward) or coefficients (backward)
    int *map;              // [nq, m, max_len] (candidate, level) -> entry (forward)
};

// position of candidate c of query q, or -1 for padding and for any id outside [0, n_sid)
__device__ __forceinline__ int pos_of(const PairArgs &a, long long q, int c) {
    const int sid = a.cand[q * a.m + c];
    if (sid < 0 || sid >= a.n_sid) return -1;
    const int p = a.pos_of_sid[sid];
    return p >= 0 && p < a.n_pos ? p : -1;
}

template <bool GRAD>
__global__ void __launch_bounds__(PL_THREADS) pair_list_kernel(const PairArgs a) {
    __shared__ int key[CW_PAIR_MAX_M];  // by candidate: position, INT_MAX for padding
    __shared__ int s_c[CW_PAIR_MAX_M], s_pos[CW_PAIR_MAX_M], s_len[CW_PAIR_MAX_M], s_cp[CW_PAIR_MAX_M],
        s_start[CW_PAIR_MAX_M];  // by sorted slot
    __shared__ int warp_tot[PL_WARPS];
    const long long q = blockIdx.x;
    const int m = a.m, ML = a.max_len, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int c = tid; c < m; c += PL_THREADS) {
        const int p = pos_of(a, q, c);
        key[c] = p < 0 ? INT_MAX : p;
    }
    __syncthreads();
    // slot of a candidate = its rank in (position, candidate index) order; padding ranks last
    int nvalid = 0;
    for (int base = 0; base < m; base += PL_THREADS) {
        const int c = base + tid;
        if (c < m) {
            const int k = key[c];
            int r = 0;
            for (int j = 0; j < m; j++) {
                const int kj = key[j];
                r += kj < k || (kj == k && j < c);
            }
            s_c[r] = c;
        }
        nvalid += __syncthreads_count(c < m && key[c] != INT_MAX);
    }
    // common prefix with the previous slot: levels [0, cp) are the same index rows, and equal rows at one level mean
    // equal rows at every level above it, so a binary search finds cp
    for (int t = tid; t < nvalid; t += PL_THREADS) {
        const int p = key[s_c[t]], len = a.pos_rec[p].x;
        int cp = 0;
        if (t > 0) {
            const int pp = key[s_c[t - 1]];
            const int *pa = a.path_idx + (size_t)p * ML, *pb = a.path_idx + (size_t)pp * ML;
            int lo = 0, hi = min(len, a.pos_rec[pp].x);
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (pa[mid - 1] == pb[mid - 1]) lo = mid; else hi = mid - 1;
            }
            cp = lo;
        }
        s_pos[t] = p;
        s_len[t] = len;
        s_cp[t] = cp;
    }
    __syncthreads();
    // list offsets: exclusive scan of the new levels (len - cp) over the slots, PL_PER consecutive slots per thread
    int loc = 0;
    for (int i = 0; i < PL_PER; i++) {
        const int t = tid * PL_PER + i;
        if (t < nvalid) loc += s_len[t] - s_cp[t];
    }
    int inc = loc;
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    int run = inc - loc, total = 0;
    for (int w = 0; w < PL_WARPS; w++) {
        run += w < warp ? warp_tot[w] : 0;
        total += warp_tot[w];
    }
    for (int i = 0; i < PL_PER; i++) {
        const int t = tid * PL_PER + i;
        if (t < nvalid) { s_start[t] = run; run += s_len[t] - s_cp[t]; }
    }
    if (tid == 0) a.n_rows[q] = total;
    __syncthreads();
    int *list = a.list + q * a.E;
    for (int t = warp; t < nvalid; t += PL_WARPS) {
        const int p = s_pos[t], cp = s_cp[t], len = s_len[t], st = s_start[t];
        for (int j = cp + lane; j < len; j += 32) list[st + j - cp] = a.path_idx[(size_t)p * ML + j];
    }
    // one thread per level walks the slots in order: a slot whose new levels include j opens entry start + j - cp, the
    // slots after it share that entry until the next one opens.  Forward: write the map; backward: sum G w per entry.
    for (int j = tid; j < ML; j += PL_THREADS) {
        int cur = -1;
        float g = 0.0f;
        for (int t = 0; t < nvalid; t++) {
            const int len = s_len[t];
            if (j >= len) continue;
            const int cp = s_cp[t];
            if (j >= cp) {
                if (GRAD && cur >= 0) a.val[q * a.E + cur] = g;
                cur = s_start[t] + j - cp;
                g = 0.0f;
            }
            if (GRAD)
                g = __fmaf_rn(a.grad_out[q * m + s_c[t]], (float)(a.level_w[j] / (double)len), g);
            else
                a.map[(q * m + s_c[t]) * ML + j] = cur;
        }
        if (GRAD && cur >= 0) a.val[q * a.E + cur] = g;
    }
}

// leaf score of (q, c): acc = fma((float)(level_w[j] / len), s_j, acc) root first from 0, as cw_dense_paths_topk
__global__ void __launch_bounds__(256) pair_sum_kernel(const PairArgs a, float *out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.nq * a.m) return;
    const long long q = i / a.m;
    const int p = pos_of(a, q, (int)(i - q * a.m));
    if (p < 0) { out[i] = -__int_as_float(0x7f800000); return; }
    const int len = a.pos_rec[p].x;
    const int *mp = a.map + i * a.max_len;
    const float *s = a.val + q * a.E;
    float acc = 0.0f;
    for (int j = 0; j < len; j++) acc = __fmaf_rn((float)(a.level_w[j] / (double)len), s[mp[j]], acc);
    out[i] = acc;
}

// grad_q[q, d] = -sum_e gs_e (x_d r_ed + mb_ed) r_ed over the query's list in list order; thread = attributes
// tid, tid + 256, ...
__global__ void __launch_bounds__(GR_THREADS) pair_grad_kernel(const PairArgs a, const float2 *__restrict__ RM,
                                                                const float *__restrict__ Q, int D, float *grad_q) {
    const long long q = blockIdx.x;
    const int n = a.n_rows[q], tid = threadIdx.x;
    const int *list = a.list + q * a.E;
    const float *gs = a.val + q * a.E;
    float x[GR_PER], acc[GR_PER];
#pragma unroll
    for (int k = 0; k < GR_PER; k++) {
        const int d = tid + k * GR_THREADS;
        x[k] = d < D ? Q[q * D + d] : 0.0f;
        acc[k] = 0.0f;
    }
#pragma unroll 2
    for (int e = 0; e < n; e++) {
        const float2 *row = RM + (size_t)list[e] * D;
        const float g = gs[e];
#pragma unroll
        for (int k = 0; k < GR_PER; k++) {
            const int d = tid + k * GR_THREADS;
            if (d < D) {
                const float2 v = row[d];
                const float t = __fmaf_rn(x[k], v.x, v.y);
                acc[k] = __fmaf_rn(__fmul_rn(g, t), v.x, acc[k]);
            }
        }
    }
#pragma unroll
    for (int k = 0; k < GR_PER; k++) {
        const int d = tid + k * GR_THREADS;
        if (d < D) grad_q[q * D + d] = -acc[k];
    }
}

static int pair_check(const char *what, const cw_index *ix, const float *rows, const int32_t *pos_of_sid, int32_t n_sid,
                      const float *Q, int64_t nq, const int32_t *cand, int32_t m, const void *out, const int32_t *scratch) {
    if (m < 0 || m > CW_PAIR_MAX_M) {
        cw_set_error("%s: m=%d candidates per query, outside 0..%d (CW_PAIR_MAX_M: split wider lists into column blocks)",
                     what, m, CW_PAIR_MAX_M);
        return CW_E_ARG;
    }
    if (nq < 0 || nq > INT_MAX) {
        cw_set_error("%s: nq=%lld queries, outside 0..%d per call", what, (long long)nq, INT_MAX);
        return CW_E_ARG;
    }
    if (!ix || ix->n_pos < 1 || !ix->path_idx || !ix->pos_rec || !ix->level_w || !ix->sumlog || ix->D < 1 ||
        ix->D > CW_MAX_D || n_sid < 0) {
        cw_set_error("%s: bad index (no positions, D=%d outside 1..%d, or n_sid=%d < 0)", what, ix ? ix->D : -1, CW_MAX_D,
                     n_sid);
        return CW_E_ARG;
    }
    if (ix->max_len < 1 || ix->max_len > CW_PAIR_MAX_LEN) {
        cw_set_error("%s: max_len=%d outside 1..%d", what, ix->max_len, CW_PAIR_MAX_LEN);
        return CW_E_ARG;
    }
    if (nq > 0 && m > 0 && (!rows || !pos_of_sid || !Q || !cand || !out || !scratch)) {
        cw_set_error("%s: null pointer", what);
        return CW_E_ARG;
    }
    if (reinterpret_cast<uintptr_t>(rows) % 16) {  // fn_exact_kernel fetches the rows with bulk copies
        cw_set_error("%s: rows must be 16-byte aligned", what);
        return CW_E_ARG;
    }
    return 0;
}

static PairArgs pair_args(const cw_index *ix, const int32_t *pos_of_sid, int32_t n_sid, int64_t nq, const int32_t *cand,
                          int32_t m, int32_t *scratch) {
    PairArgs a;
    a.path_idx = ix->path_idx;
    a.pos_rec = reinterpret_cast<const int4 *>(ix->pos_rec);
    a.level_w = ix->level_w;
    a.n_pos = ix->n_pos;
    a.max_len = ix->max_len;
    a.pos_of_sid = pos_of_sid;
    a.n_sid = n_sid;
    a.cand = cand;
    a.nq = nq;
    a.m = m;
    a.E = m * ix->max_len;
    a.grad_out = nullptr;
    a.n_rows = scratch;
    a.list = scratch + nq;
    a.val = reinterpret_cast<float *>(a.list + nq * a.E);
    a.map = reinterpret_cast<int *>(a.val + nq * a.E);
    return a;
}

}  // namespace cwp

using namespace cwp;

extern "C" int64_t cw_pair_scratch_words(int64_t nq, int32_t m, int32_t max_len) {
    if (nq < 0 || m < 0 || m > CW_PAIR_MAX_M || max_len < 1 || max_len > CW_PAIR_MAX_LEN) {
        cw_set_error("cw_pair_scratch_words: nq=%lld, m=%d (0..%d) or max_len=%d (1..%d) out of range", (long long)nq, m,
                     CW_PAIR_MAX_M, max_len, CW_PAIR_MAX_LEN);
        return CW_E_ARG;
    }
    return nq * (1 + 3LL * m * max_len);
}

extern "C" int cw_pair_scores(const cw_index *ix, const float *rows, const int32_t *pos_of_sid, int32_t n_sid,
                              const float *Q, int64_t nq, const int32_t *cand, int32_t m, float *out, int32_t *scratch,
                              void *stream) {
    int rc = pair_check("cw_pair_scores", ix, rows, pos_of_sid, n_sid, Q, nq, cand, m, out, scratch);
    if (rc || nq == 0 || m == 0) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = cw_exact_rows_attr())) return rc;
    const PairArgs a = pair_args(ix, pos_of_sid, n_sid, nq, cand, m, scratch);
    // (query, row block) work items: a few per resident warp of the GPU, however few queries there are
    long long blocks = (148LL * 48 + nq - 1) / nq;
    blocks = blocks < (a.E + 15) / 16 ? blocks : (a.E + 15) / 16;
    blocks = blocks < 65535 ? (blocks > 0 ? blocks : 1) : 65535;
    pair_list_kernel<false><<<(unsigned)nq, PL_THREADS, 0, st>>>(a);
    cw_exact_rows_launch(*ix, reinterpret_cast<const float2 *>(rows), Q, nq, a.list, a.n_rows, 1, 0, a.E, a.val,
                         (int)blocks, st);
    pair_sum_kernel<<<(unsigned)((nq * m + 255) / 256), 256, 0, st>>>(a, out);
    return cw_check_cuda(cudaGetLastError(), "cw_pair_scores");
}

extern "C" int cw_pair_scores_bwd(const cw_index *ix, const float *rows, const int32_t *pos_of_sid, int32_t n_sid,
                                  const float *Q, int64_t nq, const int32_t *cand, int32_t m, const float *grad_out,
                                  float *grad_q, int32_t *scratch, void *stream) {
    int rc = pair_check("cw_pair_scores_bwd", ix, rows, pos_of_sid, n_sid, Q, nq, cand, m, grad_q, scratch);
    if (rc || nq == 0) return rc;
    if (m > 0 && !grad_out) {
        cw_set_error("cw_pair_scores_bwd: null pointer");
        return CW_E_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (m == 0) return cw_check_cuda(cudaMemsetAsync(grad_q, 0, (size_t)nq * ix->D * sizeof(float), st), "cw_pair_scores_bwd");
    PairArgs a = pair_args(ix, pos_of_sid, n_sid, nq, cand, m, scratch);
    a.grad_out = grad_out;
    pair_list_kernel<true><<<(unsigned)nq, PL_THREADS, 0, st>>>(a);
    pair_grad_kernel<<<(unsigned)nq, GR_THREADS, 0, st>>>(a, reinterpret_cast<const float2 *>(rows), Q, ix->D, grad_q);
    return cw_check_cuda(cudaGetLastError(), "cw_pair_scores_bwd");
}
