// cw_dense.cu -- batched dense predict (CobwebWrapper.cobweb_predict_indexed /
// cobweb_rank_scores, src/cobweb/CobwebWrapper.py:210-294): every query of a batch against
// every node, path product, top-k.
//
// Kernel 1  dense_score_kernel: node_scores[q,b] = -0.5*(sumlog[b] + sum_d (x_qd*r_bd + mb_bd)^2)
//           with r = 1/sqrt(var), mb = -mean*r, i.e. the reference's (x-mean)^2/var evaluated as
//           TWO FFMAs per (query, node, attribute) on the FP32 pipe.  (x-mean) has to be formed
//           per (q, n, d) triple, so this is not a tensor-core contraction; the GEMM form
//           sum x^2/var - 2 sum x*mean/var + sum mean^2/var cancels catastrophically exactly
//           where ranking matters (query close to a leaf) -- DESIGN.md "Dense predict".
//           128x128 output tile per CTA, 8x8 per thread, operands pre-tiled k-major in HBM so
//           each pipeline stage is three contiguous 8 KB blocks fetched with cp.async.bulk
//           (TMA bulk copy, mbarrier completion), 4 stages.
// Kernel 2  paths_topk_kernel: leaf score = sequential FMA of path_w * node score, root first
//           (bit-identical to torch.sparse.mm on the reference's side), fused with a per-chunk
//           top-k; kernel 3 merges the chunk candidates.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/cobweb_b200.h"
#include "cw_nvtx.h"

void cw_set_error(const char *fmt, ...);
int cw_check_cuda(cudaError_t e, const char *what);

namespace cw {

constexpr int TQ = 128, TN = CW_TILE_N, TK = CW_TILE_K, STAGES = 4, SCORE_THREADS = 256;

// ------------------------------------------------------------------ PTX helpers (mbarrier + bulk copy)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// 1-D TMA bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

struct __align__(128) ScoreStage {
    float x[TK][TQ];
    float r[TK][TN];
    float mb[TK][TN];
};

// packed fp32x2 arithmetic (Blackwell FFMA2): one instruction = two FMAs, operands are aligned
// 64-bit register pairs, so three-operand FMAs no longer collide in the two register banks.
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}

// Refill protocol: every warp bumps a per-stage counter when it is done with the stage; the
// warp that arrives last re-arms the stage's mbarrier and issues the three bulk copies for the
// k-tile STAGES ahead.  No thread ever blocks waiting for the others (v1 had thread 0 wait on
// an "empty" mbarrier, which put 35 % of warp time into mbarrier waits -- profiles/r01_*).
//
// grid: (query tiles, node tiles) -- query tile fastest so that concurrently resident CTAs
// share one node tile through L2 and the node matrices stream from HBM exactly once.
// Warp w owns a 32-query x 64-node sub-tile (4 x 2 warps); lane (tx = lane%8, ty = lane/8)
// owns queries {ty*4.., 16+ty*4..} x nodes {tx*4.., 32+tx*4..}: every LDS.128 touches one
// 128-byte line per half-warp (2 wavefronts instead of 4).
__global__ void __launch_bounds__(SCORE_THREADS, 2)
dense_score_kernel(const float *__restrict__ XT, const float *__restrict__ R, const float *__restrict__ MB,
                   const float *__restrict__ sumlog, float *__restrict__ out, long long ldq, int n_ktiles) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    ScoreStage *st = reinterpret_cast<ScoreStage *>(smem_raw);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw + STAGES * sizeof(ScoreStage));
    int *done = reinterpret_cast<int *>(full + STAGES);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int qt = blockIdx.x, nt = blockIdx.y;
    const float *xsrc = XT + (size_t)qt * n_ktiles * (TK * TQ);
    const float *rsrc = R + (size_t)nt * n_ktiles * (TK * TN);
    const float *msrc = MB + (size_t)nt * n_ktiles * (TK * TN);
    constexpr uint32_t XB = TK * TQ * 4, NB = TK * TN * 4;
    constexpr int NWARPS = SCORE_THREADS / 32;

    if (tid == 0) {
        for (int s = 0; s < STAGES; s++) {
            mbar_init(&full[s], 1);
            done[s] = 0;
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        for (int s = 0; s < STAGES && s < n_ktiles; s++) {
            mbar_arrive_expect_tx(&full[s], XB + 2 * NB);
            bulk_g2s(st[s].x, xsrc + (size_t)s * (TK * TQ), XB, &full[s]);
            bulk_g2s(st[s].r, rsrc + (size_t)s * (TK * TN), NB, &full[s]);
            bulk_g2s(st[s].mb, msrc + (size_t)s * (TK * TN), NB, &full[s]);
        }
    }

    const int tx = lane & 7, ty = lane >> 3;
    const int qb = (warp >> 1) * 32 + ty * 4;  // first query of this thread inside the tile (second group: +16)
    const int nb = (warp & 1) * 64 + tx * 4;   // first node (second group: +32)
    uint64_t acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
        for (int p = 0; p < 4; p++) acc[i][p] = 0ull;

    for (int kt = 0; kt < n_ktiles; kt++) {
        const int s = kt % STAGES;
        const uint32_t ph = (kt / STAGES) & 1;
        mbar_wait(&full[s], ph);
        const ScoreStage &S = st[s];
#pragma unroll 4
        for (int kk = 0; kk < TK; kk++) {
            const float4 xa = *reinterpret_cast<const float4 *>(&S.x[kk][qb]);
            const float4 xb = *reinterpret_cast<const float4 *>(&S.x[kk][qb + 16]);
            const ulonglong2 ra = *reinterpret_cast<const ulonglong2 *>(&S.r[kk][nb]);
            const ulonglong2 rb = *reinterpret_cast<const ulonglong2 *>(&S.r[kk][nb + 32]);
            const ulonglong2 ma = *reinterpret_cast<const ulonglong2 *>(&S.mb[kk][nb]);
            const ulonglong2 mb = *reinterpret_cast<const ulonglong2 *>(&S.mb[kk][nb + 32]);
            const float xv[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
            const uint64_t r2[4] = {ra.x, ra.y, rb.x, rb.y};
            const uint64_t m2[4] = {ma.x, ma.y, mb.x, mb.y};
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const uint64_t xx = pack2(xv[i], xv[i]);
                uint64_t u[4];
#pragma unroll
                for (int p = 0; p < 4; p++) u[p] = ffma2(xx, r2[p], m2[p]);  // four independent FFMA2 ...
#pragma unroll
                for (int p = 0; p < 4; p++) acc[i][p] = ffma2(u[p], u[p], acc[i][p]);  // ... before their consumers
            }
        }
        // release the stage; the last warp to get here refills it
        __syncwarp();
        if (lane == 0) {
            __threadfence_block();
            const int prev = atomicAdd(&done[s], 1);
            if (prev == NWARPS - 1) {
                atomicExch(&done[s], 0);
                const int k2 = kt + STAGES;
                if (k2 < n_ktiles) {
                    __threadfence_block();
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    mbar_arrive_expect_tx(&full[s], XB + 2 * NB);
                    bulk_g2s(st[s].x, xsrc + (size_t)k2 * (TK * TQ), XB, &full[s]);
                    bulk_g2s(st[s].r, rsrc + (size_t)k2 * (TK * TN), NB, &full[s]);
                    bulk_g2s(st[s].mb, msrc + (size_t)k2 * (TK * TN), NB, &full[s]);
                }
            }
        }
    }

    // epilogue: -0.5 * (sumlog + quad)   (CobwebWrapper.py:232-236), written NODE-major:
    // out[node * ldq + query], so the path kernel reads 32 queries of one node as one 128-byte line
    const int b0 = nt * TN + nb;
    const float4 sla = *reinterpret_cast<const float4 *>(sumlog + b0);
    const float4 slb = *reinterpret_cast<const float4 *>(sumlog + b0 + 32);
    const float sl[8] = {sla.x, sla.y, sla.z, sla.w, slb.x, slb.y, slb.z, slb.w};
    float o[8][8];  // [query][node]
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
        for (int p = 0; p < 4; p++) {
            float lo, hi;
            unpack2(acc[i][p], lo, hi);
            o[i][2 * p] = -0.5f * (sl[2 * p] + lo);
            o[i][2 * p + 1] = -0.5f * (sl[2 * p + 1] + hi);
        }
    float *col = out + (long long)qt * TQ + qb;
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const long long b = b0 + (j < 4 ? j : 32 + (j - 4));
        float *row = col + b * ldq;
        *reinterpret_cast<float4 *>(row) = make_float4(o[0][j], o[1][j], o[2][j], o[3][j]);
        *reinterpret_cast<float4 *>(row + 16) = make_float4(o[4][j], o[5][j], o[6][j], o[7][j]);
    }
}

// Q [nq, D] row-major -> XT [q tile][k tile][TK][TQ], zero padded (same tiling as the index)
__global__ void __launch_bounds__(256)
tile_queries_kernel(const float *__restrict__ Q, long long nq, int D, int n_ktiles, float *XT) {
    __shared__ float t[TK][TQ + 1];
    const int qt = blockIdx.x, kt = blockIdx.y, tid = threadIdx.x;
    const int ql = tid >> 1, half = tid & 1;
    const long long q = (long long)qt * TQ + ql;
#pragma unroll
    for (int e = 0; e < 8; e++) {
        const int kk = half * 8 + e, d = kt * TK + kk;
        t[kk][ql] = (q < nq && d < D) ? Q[q * D + d] : 0.0f;
    }
    __syncthreads();
    const size_t tile = ((size_t)qt * n_ktiles + kt) * (TK * TQ);
    for (int i = tid; i < TK * TQ; i += 256) XT[tile + i] = t[i / TQ][i % TQ];
}

// ------------------------------------------------------------------ path product + top-k
constexpr int PT_MAXLEN = 1024, PT_SLOTS = CW_MAX_K / 32;

// order: score desc, then sentence id asc; sid < 0 = empty
__device__ __forceinline__ bool cand_better(float as, int ai, float bs, int bi) {
    if (bi < 0) return ai >= 0;
    if (ai < 0) return false;
    if (as != bs) return as > bs;
    return ai < bi;
}

// order-preserving float <-> int key (for atomicMax on scores)
__device__ __forceinline__ int float_key(float f) {
    const int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float key_float(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }

// Rare path of the kernel below (the path length changes a handful of times per chunk); kept out
// of line so that its binary64 division does not inflate the hot loop's register allocation.
__device__ __noinline__ void fill_weight_row(float *wl, const double *lw, int len, int lane) {
    for (int j = lane; j < len; j += 32) wl[j] = (float)(lw[j] / (double)len);
}

// 4-byte asynchronous copy global -> shared (LDGSTS): the prefetch ring of the path kernel
__device__ __forceinline__ void cp_async4(float *dst, const float *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

constexpr int PF_DIST = 6, PF_RING = 8, PF_LEVELS = 3, PF_RECS = 64;
struct __align__(16) PathRec {
    int len, m, leaf, sid;  // path length, levels shared with the previous position, leaf row, sentence id
    int par, gpar, pad0, pad1;  // rows of levels len-2 / len-3 when they are not shared
};

// grid (position chunks, groups of `wpb` query groups): warp = 32 queries (lane = query) x one
// chunk of sentence positions.  Positions are in tree order, so consecutive paths share a
// prefix (siblings differ only in the leaf); the index stores per position
// {len, common prefix m with the previous position, leaf row, sentence id} in one 16-byte
// record.  The FMA chain's partial sums are kept per level in a lane-private shared-memory
// stack and a position recomputes only levels m..len-1 -- the same operations in the same order
// as a full root-to-leaf chain (bit-equal to torch.sparse.mm on the reference's side).  Each
// level is one coalesced 128-byte read of the node-major score matrix.  Every lane keeps its
// query's sorted top-k in shared memory ([rank][lane]) behind a register threshold.
//
// The score reads are the kernel's only long-latency operations and each depends on the record of
// its position, so they are software-pipelined: records are loaded 32 positions at a time (lane =
// position, one block ahead) into a shared-memory ring, and the scores of the last three levels of
// position p + PF_DIST are in flight (cp.async into a per-lane ring) while position p is consumed.
// Deeper non-shared levels (an ancestor above the grandparent changed: ~1 position in 60) are read
// on demand.
// TAGGED: a position is offered to its query's list only if its sentence is eligible (pos_tags & qtags[q]); the path
// sums of every position are still formed, since the next positions build on them.  The tag rides in the record's pad0.
template <bool LEAF, bool K32, bool TAGGED>
__global__ void __launch_bounds__(256, 3)
paths_topk_kernel(const float *__restrict__ ST, unsigned ldq, long long nq, int n_pos, int max_len,
                  const int *__restrict__ path_pm, const int4 *__restrict__ pos_rec,
                  const double *__restrict__ level_w, int k, float *leaf_scores, float *cand_s, int *cand_i,
                  int n_chunks, int chunk_len, int *shared_thr, const int *__restrict__ nq_dev,
                  const unsigned *__restrict__ qtags, const unsigned *__restrict__ pos_tags) {
    extern __shared__ __align__(16) unsigned char pt_smem[];
    if (nq_dev) nq = min(nq, (long long)*nq_dev);  // count decided on the device (flagged queries of the fused mode)
    // level weights in binary64; the path weight of level j on a path of length len is
    // (float)(level_w[j] / len), the fp32 value the reference stores in its sparse path matrix
    double *lw = reinterpret_cast<double *>(pt_smem);  // [max_len]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    PathRec *recs = reinterpret_cast<PathRec *>(lw + ((max_len + 1) & ~1)) + (size_t)warp * PF_RECS;            // [PF_RECS]
    float *wt = reinterpret_cast<float *>(reinterpret_cast<PathRec *>(lw + ((max_len + 1) & ~1)) + (size_t)wpb * PF_RECS);
    float *ring = wt + (size_t)warp * (PF_RING * PF_LEVELS * 32);                                               // [PF_RING][PF_LEVELS][32]
    wt += (size_t)wpb * (PF_RING * PF_LEVELS * 32);
    float *Ls = wt + (size_t)warp * k * 32;                                                // [32 lanes][k]
    int *Li = reinterpret_cast<int *>(wt + (size_t)wpb * k * 32) + (size_t)warp * k * 32;  // [32 lanes][k]
    float *St = wt + (size_t)2 * wpb * k * 32 + (size_t)warp * max_len * 32;               // [max_len][32]
    float *wl = wt + (size_t)2 * wpb * k * 32 + (size_t)wpb * max_len * 32 + (size_t)warp * max_len;  // [max_len]
    for (int i = threadIdx.x; i < max_len; i += blockDim.x) lw[i] = level_w[i];
    const float NEG_INF = -__int_as_float(0x7f800000);
    for (int i = lane; i < 32 * k; i += 32) { Ls[i] = NEG_INF; Li[i] = -1; }
    __syncthreads();
    const long long g = (long long)blockIdx.y * wpb + warp;
    if (g * 32 >= nq) return;
    const long long q = g * 32 + lane;
    const bool qvalid = q < nq;
    const float *col = ST + (qvalid ? q : g * 32);
    const int chunk = blockIdx.x;
    const int p0 = chunk * chunk_len, p1 = min(n_pos, p0 + chunk_len);
    const int n = p1 - p0;
    // k-th best of this lane's query so far; while the list is not full: (-inf, INT_MAX), which every finite
    // candidate beats (sentence ids compare as unsigned, so the empty id -1 also loses every tie)
    float thr_s = NEG_INF;
    int thr_i = 0x7fffffff;
    const bool collect = k > 0 && qvalid;
    const unsigned qtag = TAGGED && qvalid ? qtags[q] : 0u;
    // Threshold shared by the chunks of a query: the k-th best of ANY chunk's full list is a lower bound of the k-th
    // best over all positions, so a score strictly below it cannot be in the final top-k.  Each lane publishes its own
    // k-th best (atomicMax on an order-preserving integer key) and re-reads the shared bound once per 32 positions;
    // without it every chunk pays the k ln(n/k) warm-up insertions of a cold list.  The merged result is the exact
    // top-k whatever the timing.
    float gthr = NEG_INF, published = NEG_INF;
    int *gslot = shared_thr + (qvalid ? q : 0);
    int wl_len = -1;  // path length the per-warp weight row wl[] was computed for

    // record of position p0 + r (lane-parallel): the first position of a chunk recomputes its whole path
    auto load_rec = [&](int r) {
        PathRec R;
        R.len = 0; R.m = 0; R.leaf = 0; R.sid = -1; R.par = 0; R.gpar = 0; R.pad0 = 0; R.pad1 = 0;
        if (r < n) {
            const int4 rc = pos_rec[p0 + r];
            R.len = rc.x; R.m = r == 0 ? 0 : rc.y; R.leaf = rc.z; R.sid = rc.w;
            const int *path = path_pm + (size_t)(p0 + r) * max_len;
            if (R.m <= R.len - 2) R.par = path[R.len - 2];
            if (R.m <= R.len - 3) R.gpar = path[R.len - 3];
            if (TAGGED) R.pad0 = (int)pos_tags[p0 + r];
        }
        return R;
    };
    auto prefetch = [&](int r) {  // scores of the last (up to three) non-shared levels of position p0 + r
        if (r < n) {
            const PathRec R = recs[r & (PF_RECS - 1)];
            float *slot = ring + (r & (PF_RING - 1)) * (PF_LEVELS * 32) + lane;
            const int nl = R.len - R.m;
            if (nl >= 1) cp_async4(slot, col + (size_t)(unsigned)R.leaf * ldq);
            if (nl >= 2) {
                cp_async4(slot + 32, col + (size_t)(unsigned)R.par * ldq);
                if (nl >= 3) cp_async4(slot + 64, col + (size_t)(unsigned)R.gpar * ldq);
            }
        }
        cp_async_commit();
    };
    recs[lane] = load_rec(lane);
    recs[32 + lane] = load_rec(32 + lane);
    __syncwarp();
    for (int r = 0; r < PF_DIST; r++) prefetch(r);
    PathRec nb;  // records of the block after the next one, in flight
    // The common position differs from its predecessor in the leaf only: its score is one FMA on top of the
    // partial sum through the parent level, kept in a register together with the leaf-level weight.
    float base = 0.0f, wleaf = 0.0f, last_acc = 0.0f;

    // record ring = two blocks of 32 positions.  At the start of block B: the records of block B+1, fetched one
    // block ago, take the slots of the finished block B-1, and the fetch of block B+2 is issued.
    for (int rb = 0; rb < n; rb += 32) {
      if (rb > 0) {
          recs[((rb + 32) & (PF_RECS - 1)) + lane] = nb;
          __syncwarp();
      }
      nb = load_rec(rb + 64 + lane);
      if (collect) {
          if (thr_i != 0x7fffffff && thr_s > published) {  // list full and its k-th best moved: publish
              published = thr_s;
              atomicMax(gslot, float_key(thr_s));
          }
          gthr = fmaxf(gthr, key_float(__ldcg(gslot)));
      }
      const int re = min(n, rb + 32);
      for (int r = rb; r < re; r++) {
        prefetch(r + PF_DIST);
        cp_async_wait<PF_DIST>();
        const PathRec R = recs[r & (PF_RECS - 1)];
        const float *slot = ring + (r & (PF_RING - 1)) * (PF_LEVELS * 32) + lane;
        const int len = R.len, m = R.m;
        float acc;
        if (m == len - 1 && len == wl_len) {
            acc = __fmaf_rn(wleaf, slot[0], base);
        } else if (m == len && len == wl_len) {  // another sentence of the previous position's leaf
            acc = last_acc;
        } else {
            // levels m .. len-2 changed (or the path length did, then m = 0): rebuild the partial sums
            const int p = p0 + r;
            if (len != wl_len) {  // rare: positions are sorted by depth, so len changes a handful of times per chunk
                __syncwarp();
                fill_weight_row(wl, lw, len, lane);
                wl_len = len;
                __syncwarp();
            }
            float a = m > 0 ? St[(m - 1) * 32 + lane] : 0.0f;
            for (int j = m; j < len - 3; j++) {  // rare: an ancestor above the grandparent changed as well
                const int b = path_pm[(size_t)p * max_len + j];
                a = __fmaf_rn(wl[j], col[(size_t)(unsigned)b * ldq], a);
                St[j * 32 + lane] = a;
            }
            if (m <= len - 3) {
                a = __fmaf_rn(wl[len - 3], slot[64], a);
                St[(len - 3) * 32 + lane] = a;
            }
            if (m <= len - 2) {
                a = __fmaf_rn(wl[len - 2], slot[32], a);
                St[(len - 2) * 32 + lane] = a;
            }
            base = a;
            wleaf = wl[len - 1];
            acc = __fmaf_rn(wleaf, slot[0], base);
        }
        last_acc = acc;
        const int sid = R.sid;
        if (LEAF && qvalid) leaf_scores[q * n_pos + sid] = acc;
        // top-k: lanes whose candidate beats their query's k-th best are served one at a time by
        // the whole warp (lane r handles rank r of that query's list): no divergent shifting loops
        unsigned need = __ballot_sync(0xffffffffu, collect && acc >= gthr &&
                                                       (acc > thr_s || (acc == thr_s && (unsigned)sid < (unsigned)thr_i)) &&
                                                       (!TAGGED || ((unsigned)R.pad0 & qtag) != 0u));
        if (K32) {
            // one rank per lane: read, ballot the insertion point, shift by one, done
            while (need) {
                const int L = __ffs(need) - 1;
                need &= need - 1;
                const float cv = __shfl_sync(0xffffffffu, acc, L);
                const int base = L * k;
                float es = NEG_INF;
                int ei = -1;
                if (lane < k) { es = Ls[base + lane]; ei = Li[base + lane]; }
                // empty ranks hold -inf, so they never beat a finite candidate
                const int pos = __popc(__ballot_sync(0xffffffffu, es > cv || (es == cv && ei < sid)));
                const float ps = __shfl_sync(0xffffffffu, es, (k - 2) & 31);
                const int pi = __shfl_sync(0xffffffffu, ei, (k - 2) & 31);
                if (lane >= pos && lane + 1 < k) { Ls[base + lane + 1] = es; Li[base + lane + 1] = ei; }
                if (lane == pos) { Ls[base + lane] = cv; Li[base + lane] = sid; }
                if (lane == L) {  // new k-th best: old rank k-2, unless the candidate itself landed on rank k-1
                    const bool cand_last = (k < 2) || (pos == k - 1);
                    thr_s = cand_last ? cv : ps;
                    thr_i = cand_last ? sid : pi;
                    if (thr_i < 0) thr_i = 0x7fffffff;  // list not full yet
                }
                __syncwarp();
            }
        }
        while (!K32 && need) {
            const int L = __ffs(need) - 1;
            need &= need - 1;
            const float cv = __shfl_sync(0xffffffffu, acc, L);
            float *ls = Ls + L * k;
            int *li = Li + L * k;
            // ranks in passes of 32, all reads before any write
            float es[PT_SLOTS];
            int ei[PT_SLOTS];
            int pos = 0;
#pragma unroll
            for (int t = 0; t < PT_SLOTS; t++) {
                if (t * 32 < k) {  // uniform: only the passes this k needs
                    const int r = t * 32 + lane;
                    es[t] = NEG_INF; ei[t] = -1;
                    if (r < k) { es[t] = ls[r]; ei[t] = li[r]; }
                    pos += __popc(__ballot_sync(0xffffffffu, r < k && cand_better(es[t], ei[t], cv, sid)));
                }
            }
            __syncwarp();
            float new_thr_s = cv;
            int new_thr_i = sid;
#pragma unroll
            for (int t = 0; t < PT_SLOTS; t++) {
                if (t * 32 >= k) continue;
                const int r = t * 32 + lane;
                if (r >= pos && r + 1 < k) { ls[r + 1] = es[t]; li[r + 1] = ei[t]; }
                if (r == pos) { ls[r] = cv; li[r] = sid; }
                // the new k-th best: the old rank k-2 unless the candidate itself landed on rank k-1
                if (k >= 2 && ((k - 2) >> 5) == t) {
                    const float ps = __shfl_sync(0xffffffffu, es[t], (k - 2) & 31);
                    const int pi = __shfl_sync(0xffffffffu, ei[t], (k - 2) & 31);
                    if (pos < k - 1) { new_thr_s = ps; new_thr_i = pi; }
                }
            }
            if (lane == L) { thr_s = new_thr_s; thr_i = new_thr_i < 0 ? 0x7fffffff : new_thr_i; }
            __syncwarp();
        }
      }
    }
    if (k > 0 && qvalid) {
        float *os = cand_s + (q * n_chunks + chunk) * k;
        int *oi = cand_i + (q * n_chunks + chunk) * k;
        for (int r = 0; r < k; r++) { os[r] = Ls[lane * k + r]; oi[r] = Li[lane * k + r]; }
    }
}

// Running top-k of one warp, kept sorted across the lanes: rank r lives in lane r%32, slot r/32
// (register arrays ls/li, fully unrolled).  Used to merge the per-chunk candidate lists.
__device__ __forceinline__ void topk_init(float (&ls)[PT_SLOTS], int (&li)[PT_SLOTS]) {
#pragma unroll
    for (int s = 0; s < PT_SLOTS; s++) { ls[s] = -__int_as_float(0x7f800000); li[s] = -1; }
}
// Offer one candidate per lane (id < 0: none).  One ballot against the current k-th best; the
// few candidates that beat it are inserted one by one.
__device__ __forceinline__ void topk_offer(float (&ls)[PT_SLOTS], int (&li)[PT_SLOTS], int k, float v, int id) {
    const int last_lane = (k - 1) & 31, last_slot = (k - 1) >> 5;
    const int lane = threadIdx.x & 31;
    float tsel = ls[0];
    int isel = li[0];
#pragma unroll
    for (int s = 1; s < PT_SLOTS; s++)
        if (last_slot == s) { tsel = ls[s]; isel = li[s]; }
    const float ts = __shfl_sync(0xffffffffu, tsel, last_lane);
    const int ti = __shfl_sync(0xffffffffu, isel, last_lane);
    unsigned m = __ballot_sync(0xffffffffu, cand_better(v, id, ts, ti));
    while (m) {
        const int src = __ffs(m) - 1;
        m &= m - 1;
        const float cv = __shfl_sync(0xffffffffu, v, src);
        const int cid = __shfl_sync(0xffffffffu, id, src);
        int pos = 0;  // rank of the candidate = number of list entries that beat it
#pragma unroll
        for (int s = 0; s < PT_SLOTS; s++) pos += __popc(__ballot_sync(0xffffffffu, cand_better(ls[s], li[s], cv, cid)));
        if (pos >= k) continue;  // an earlier insertion of this step raised the bar
        float ups[PT_SLOTS], carry_s[PT_SLOTS];
        int upi[PT_SLOTS], carry_i[PT_SLOTS];
#pragma unroll
        for (int s = 0; s < PT_SLOTS; s++) {  // all reads of the old list first
            ups[s] = __shfl_up_sync(0xffffffffu, ls[s], 1);
            upi[s] = __shfl_up_sync(0xffffffffu, li[s], 1);
            carry_s[s] = __shfl_sync(0xffffffffu, ls[s], 31);
            carry_i[s] = __shfl_sync(0xffffffffu, li[s], 31);
        }
#pragma unroll
        for (int s = 0; s < PT_SLOTS; s++) {  // shift ranks >= pos down by one, insert at pos
            float ns = ups[s];
            int ni = upi[s];
            if (s > 0 && lane == 0) { ns = carry_s[s - 1]; ni = carry_i[s - 1]; }
            const int r = s * 32 + lane;
            if (r > pos) { ls[s] = ns; li[s] = ni; }
            if (r == pos) { ls[s] = cv; li[s] = cid; }
        }
    }
}
__device__ __forceinline__ void topk_store(const float (&ls)[PT_SLOTS], const int (&li)[PT_SLOTS], int k, float *out_s,
                                           int *out_i) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int s = 0; s < PT_SLOTS; s++) {
        const int r = s * 32 + lane;
        if (r < k) { out_s[r] = ls[s]; out_i[r] = li[s]; }
    }
}

// grid (ceil(nq/8)): warp w merges the n_chunks*k candidates of one query into the final k
__global__ void __launch_bounds__(256)
merge_topk_kernel(const float *__restrict__ cand_s, const int *__restrict__ cand_i, long long nq, int n_chunks, int k,
                  int *out_sid, float *out_score, const int *__restrict__ nq_dev = nullptr) {
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (nq_dev) nq = min(nq, (long long)*nq_dev);
    const long long q = (long long)blockIdx.x * 8 + w;
    if (q >= nq) return;
    const int n = n_chunks * k;
    float ls[PT_SLOTS];
    int li[PT_SLOTS];
    topk_init(ls, li);
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        float v = 0.0f;
        int id = -1;
        if (i < n) { v = cand_s[q * n + i]; id = cand_i[q * n + i]; }
        topk_offer(ls, li, k, v, id);
    }
    topk_store(ls, li, k, out_score + q * k, out_sid + q * k);
    __syncwarp();
    // empty ranks (fewer than k sentences) report -inf
    for (int r = lane; r < k; r += 32)
        if (out_sid[q * k + r] < 0) out_score[q * k + r] = -__int_as_float(0x7f800000);
}

}  // namespace cw

using namespace cw;

static int score_smem_bytes() { return STAGES * (int)sizeof(ScoreStage) + STAGES * (int)(sizeof(uint64_t) + sizeof(int)); }

extern "C" int64_t cw_xt_floats(int64_t nq, int32_t D) {
    return ((nq + TQ - 1) / TQ) * (int64_t)((D + TK - 1) / TK) * TK * TQ;
}

extern "C" int64_t cw_score_ldq(int64_t nq) { return (nq + TQ - 1) / TQ * TQ; }

extern "C" int cw_dense_node_scores(const cw_index *ix, const float *Q, int64_t nq, float *xt_scratch,
                                    float *node_scores, int64_t ldq, void *stream) {
    CwRange range("cw_dense_node_scores");
    if (!ix || !Q || !node_scores || !xt_scratch || nq < 0 || ldq < cw_score_ldq(nq) || (ldq & 3)) {
        cw_set_error("cw_dense_node_scores: bad argument (ldq must be >= cw_score_ldq(nq) and a multiple of 4)");
        return CW_E_ARG;
    }
    if (nq == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int n_qtiles = (int)((nq + TQ - 1) / TQ);
    int rc = 0;
    // per call: the attribute is per device, and a process may drive several
    rc = cw_check_cuda(cudaFuncSetAttribute(dense_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            score_smem_bytes()),
                       "cw_dense: smem attribute");
    if (rc) return rc;
    tile_queries_kernel<<<dim3(n_qtiles, ix->n_ktiles), 256, 0, st>>>(Q, nq, ix->D, ix->n_ktiles, xt_scratch);
    dense_score_kernel<<<dim3(n_qtiles, ix->n_ntiles), SCORE_THREADS, score_smem_bytes(), st>>>(
        xt_scratch, ix->R, ix->MB, ix->sumlog, node_scores, ldq, ix->n_ktiles);
    return cw_check_cuda(cudaGetLastError(), "cw_dense_node_scores");
}

// Upper bound of position chunks per query (sizes the caller's candidate scratch); the launch
// picks fewer, larger chunks when the batch alone fills the GPU.
// one extra chunk worth of scratch holds the per-query thresholds shared between the chunks
extern "C" int64_t cw_topk_chunks(int64_t n_pos) { return (n_pos + 1023) / 1024 + 1; }

// nq_dev (optional): the number of live queries is read on the device (<= nq, which sizes the launch)
// tf (optional): offer eligible positions only (no leaf scores then)
static int paths_topk_launch(const cw_index *ix, const float *node_scores, int64_t ldq, int64_t nq, int k, float *leaf_scores,
                             int32_t *out_sid, float *out_score, int32_t *scratch, const int *nq_dev, cudaStream_t st,
                             const cw_tag_filter *tf = nullptr) {
    if (!ix || !node_scores || nq < 0 || k < 0 || k > CW_MAX_K || ix->n_pos < 1 || !ix->path_idx || !ix->pos_rec ||
        !ix->level_w || ix->max_len < 1 || ix->max_len > PT_MAXLEN || ldq < nq || ldq > 0x7fffffffLL ||
        (k > 0 && (!out_sid || !out_score || !scratch))) {
        cw_set_error("cw_dense_paths_topk: bad argument (k=%d max %d, max_len=%d max %d)", k, CW_MAX_K,
                     ix ? ix->max_len : -1, PT_MAXLEN);
        return CW_E_ARG;
    }
    if (nq == 0) return 0;
    // warps per CTA: per warp the per-lane top-k lists take k*256 bytes of shared memory, the partial-sum
    // stack max_len*128 bytes, the record and prefetch rings 5 KB; pick the CTA size that keeps most warps per SM
    const size_t per_warp = (size_t)k * 256 + (size_t)ix->max_len * 132 + PF_RECS * sizeof(PathRec) +
                            (size_t)PF_RING * PF_LEVELS * 32 * sizeof(float);
    const size_t fixed = (size_t)((ix->max_len + 1) & ~1) * sizeof(double);
    int wpb = 1, best_warps = 0;
    for (int c = 8; c >= 1; c--) {
        const size_t blk = fixed + c * per_warp;
        if (blk > 200 * 1024) continue;
        const int warps = (int)((227 * 1024) / (blk + 1024)) * c;
        if (warps > best_warps) { best_warps = warps; wpb = c; }
    }
    if (best_warps == 0) {
        cw_set_error("cw_dense_paths_topk: k=%d with max_len=%d needs more shared memory than one CTA has", k, ix->max_len);
        return CW_E_ARG;
    }
    const long long groups = (nq + 31) / 32;
    const long long gblocks = (groups + wpb - 1) / wpb;
    if (gblocks > 65535) {
        cw_set_error("cw_dense_paths_topk: too many queries per call (%lld)", (long long)nq);
        return CW_E_ARG;
    }
    // one full wave of CTAs: (CTAs per SM at this shared-memory size) x SMs, split over the query-group blocks;
    // each chunk pays k ln(n/k) top-k insertions per query, so no more chunks than that
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long long want = (long long)sms * (best_warps / wpb) / gblocks;
    const long long max_chunks = cw_topk_chunks(ix->n_pos) - 1;
    if (want > max_chunks) want = max_chunks;
    if (want < 1) want = 1;
    const int chunk_len = (int)((ix->n_pos + want - 1) / want);
    const int n_chunks = (ix->n_pos + chunk_len - 1) / chunk_len;
    float *cand_s = reinterpret_cast<float *>(scratch);
    int *cand_i = scratch + (size_t)nq * n_chunks * (k > 0 ? k : 1);
    int *shared_thr = scratch + (size_t)2 * nq * n_chunks * (k > 0 ? k : 1);  // [nq] inside the extra chunk of scratch
    if (k > 0) {
        // 0x80808080 is the key of a large negative score: below every real one
        int rc = cw_check_cuda(cudaMemsetAsync(shared_thr, 0x80, (size_t)nq * sizeof(int), st), "cw_dense_paths_topk: memset");
        if (rc) return rc;
    }
    const size_t smem = fixed + (size_t)wpb * per_warp;
    auto kern = tf ? (k <= 32 ? paths_topk_kernel<false, true, true> : paths_topk_kernel<false, false, true>)
              : leaf_scores ? (k <= 32 ? paths_topk_kernel<true, true, false> : paths_topk_kernel<true, false, false>)
                            : (k <= 32 ? paths_topk_kernel<false, true, false> : paths_topk_kernel<false, false, false>);
    if (smem > 48 * 1024) {
        int rc = cw_check_cuda(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                               "cw_dense_paths_topk: smem attribute");
        if (rc) return rc;
    }
    kern<<<dim3(n_chunks, (unsigned)gblocks), wpb * 32, smem, st>>>(
        node_scores, (unsigned)ldq, nq, ix->n_pos, ix->max_len, ix->path_idx, reinterpret_cast<const int4 *>(ix->pos_rec),
        ix->level_w, k, leaf_scores, cand_s, cand_i, n_chunks, chunk_len, shared_thr, nq_dev, tf ? tf->query_tags : nullptr,
        tf ? tf->pos_tags : nullptr);
    if (k > 0)
        merge_topk_kernel<<<(unsigned)((nq + 7) / 8), 256, 0, st>>>(cand_s, cand_i, nq, n_chunks, k, out_sid, out_score, nq_dev);
    return cw_check_cuda(cudaGetLastError(), "cw_dense_paths_topk");
}

extern "C" int cw_dense_paths_topk(const cw_index *ix, const float *node_scores, int64_t ldq, int64_t nq, int k,
                                   float *leaf_scores, int32_t *out_sid, float *out_score, int32_t *scratch,
                                   void *stream) {
    CwRange range("cw_dense_paths_topk");
    if (ldq < cw_score_ldq(nq)) {
        cw_set_error("cw_dense_paths_topk: ldq must be >= cw_score_ldq(nq)");
        return CW_E_ARG;
    }
    return paths_topk_launch(ix, node_scores, ldq, nq, k, leaf_scores, out_sid, out_score, scratch, nullptr, (cudaStream_t)stream);
}

extern "C" int cw_dense_paths_topk_tagged(const cw_index *ix, const cw_tag_filter *tf, const float *node_scores, int64_t ldq,
                                          int64_t nq, int k, int32_t *out_sid, float *out_score, int32_t *scratch, void *stream) {
    CwRange range("cw_dense_paths_topk_tagged");
    if (!tf || !tf->query_tags || !tf->pos_tags || k < 1 || ldq < cw_score_ldq(nq)) {
        cw_set_error("cw_dense_paths_topk_tagged: bad argument (query_tags and pos_tags needed, k >= 1, ldq >= cw_score_ldq(nq))");
        return CW_E_ARG;
    }
    return paths_topk_launch(ix, node_scores, ldq, nq, k, nullptr, out_sid, out_score, scratch, nullptr, (cudaStream_t)stream, tf);
}

// One call = batched cobweb_predict_fast(return_ids=True) on HOST buffers with the FP32 form
extern "C" int cw_predict_dense_host(const cw_index *ix, const cw_dense_work *w, const float *Q_host, int64_t nq, int k,
                                     int32_t *out_sid_host, float *out_score_host, void *stream) {
    CwRange range("cw_predict_dense_host");
    if (!ix || !Q_host || !w || !w->Q_dev || !w->xt_scratch || !w->node_scores || !w->out_sid_dev || !w->out_score_dev ||
        !w->scratch || !out_sid_host || !out_score_host || k < 1 || nq < 0) {
        cw_set_error("cw_predict_dense_host: bad argument");
        return CW_E_ARG;
    }
    if (nq == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = cw_check_cuda(cudaMemcpyAsync(w->Q_dev, Q_host, (size_t)nq * ix->D * sizeof(float), cudaMemcpyHostToDevice, st),
                           "cw_predict_dense_host: H2D");
    if (rc) return rc;
    const int64_t ldq = cw_score_ldq(nq);
    if ((rc = cw_dense_node_scores(ix, w->Q_dev, nq, reinterpret_cast<float *>(w->xt_scratch), w->node_scores, ldq, stream))) return rc;
    if ((rc = cw_dense_paths_topk(ix, w->node_scores, ldq, nq, k, nullptr, w->out_sid_dev, w->out_score_dev, w->scratch, stream)))
        return rc;
    if ((rc = cw_check_cuda(cudaMemcpyAsync(out_sid_host, w->out_sid_dev, (size_t)nq * k * sizeof(int32_t), cudaMemcpyDeviceToHost, st),
                            "cw_predict_dense_host: D2H ids")))
        return rc;
    if ((rc = cw_check_cuda(cudaMemcpyAsync(out_score_host, w->out_score_dev, (size_t)nq * k * sizeof(float),
                                            cudaMemcpyDeviceToHost, st), "cw_predict_dense_host: D2H scores")))
        return rc;
    return cw_check_cuda(cudaStreamSynchronize(st), "cw_predict_dense_host: sync");
}

// ------------------------------------------------------------------ exact small-batch path
// nq <= CW_SMALL_Q queries against every node with the arithmetic of dense_score_kernel (per (query, node): d ascending,
// u = fma(x, r, mb); acc = fma(u, u, acc)), but laid out for a HANDFUL of queries: thread = node, the R / MB tiles are
// streamed once with coalesced loads (16 attributes = 32 loads in flight per thread), the queries sit in shared
// memory.  One query is HBM-bound (8 bytes per node and attribute); 32 queries are FMA-bound.  Serves single-query
// cobweb_predict_fast and the flagged queries of the fused mode.
namespace cw {
constexpr int SM_DC = 256;  // attributes of the queries staged in shared memory at a time

template <int QB>
__global__ void __launch_bounds__(CW_TILE_N)
small_scores_kernel(const float *__restrict__ XQ, const float *__restrict__ R, const float *__restrict__ MB,
                    const float *__restrict__ sumlog, float *__restrict__ out, int n_ktiles, int D, int nq,
                    const int *__restrict__ nq_dev) {
    __shared__ __align__(16) float xs[SM_DC * QB];
    if (nq_dev) nq = min(nq, *nq_dev);
    if (nq <= 0) return;
    const int nt = blockIdx.x, nl = threadIdx.x;
    float acc[QB];
#pragma unroll
    for (int q = 0; q < QB; q++) acc[q] = 0.0f;
    const float *rsrc = R + (size_t)nt * n_ktiles * (TK * TN) + nl;
    const float *msrc = MB + (size_t)nt * n_ktiles * (TK * TN) + nl;
    for (int kt0 = 0; kt0 < n_ktiles; kt0 += SM_DC / TK) {
        const int d0 = kt0 * TK;
        __syncthreads();
        for (int i = threadIdx.x; i < SM_DC * QB; i += CW_TILE_N) {
            const int q = i / SM_DC, dd = i % SM_DC;  // consecutive threads read consecutive attributes of one query
            xs[dd * QB + q] = (q < nq && d0 + dd < D) ? XQ[(size_t)q * D + d0 + dd] : 0.0f;
        }
        __syncthreads();
        const int kt1 = min(n_ktiles, kt0 + SM_DC / TK);
        for (int kt = kt0; kt < kt1; kt++) {
            float r[TK], m[TK];
#pragma unroll
            for (int kk = 0; kk < TK; kk++) {
                r[kk] = rsrc[((size_t)kt * TK + kk) * TN];
                m[kk] = msrc[((size_t)kt * TK + kk) * TN];
            }
#pragma unroll
            for (int kk = 0; kk < TK; kk++) {
                const float *xr = xs + ((kt - kt0) * TK + kk) * QB;
#pragma unroll
                for (int q = 0; q < QB; q++) {
                    const float u = __fmaf_rn(xr[q], r[kk], m[kk]);
                    acc[q] = __fmaf_rn(u, u, acc[q]);
                }
            }
        }
    }
    const int b = nt * TN + nl;
    const float sl = sumlog[b];
#pragma unroll
    for (int q = 0; q < QB; q++) out[(size_t)b * CW_SMALL_Q + q] = -0.5f * (sl + acc[q]);
}

__global__ void small_gather_kernel(const float *__restrict__ Q, int D, const int *__restrict__ which, const int *__restrict__ n_dev,
                                    int off, int nq_max, float *sm_Q, int *sm_n) {
    int n = nq_max;
    if (n_dev) n = max(0, min(nq_max, *n_dev - off));
    if (blockIdx.x == 0 && threadIdx.x == 0) *sm_n = n;
    const long long total = (long long)n * D;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int q = (int)(i / D), d = (int)(i % D);
        sm_Q[i] = Q[(size_t)which[off + q] * D + d];
    }
}
__global__ void small_scatter_kernel(const int *__restrict__ which, int off, const int *__restrict__ sm_n, int k,
                                     const int *__restrict__ sm_sid, const float *__restrict__ sm_val, int *out_sid, float *out_val) {
    const int n = *sm_n;
    for (int i = threadIdx.x; i < n * k; i += blockDim.x) {
        const int q = i / k, j = i % k;
        const size_t dst = (size_t)which[off + q] * k + j;
        out_sid[dst] = sm_sid[i];
        out_val[dst] = sm_val[i];
    }
}

// Path product + per-chunk top-k for a handful of queries: lane = sentence position (32 positions per step, the
// levels of a path are independent loads of the [rows, CW_SMALL_Q] score matrix, which sits in L2), the chain
// acc = fma((float)(level_w[j]/len), s_j, acc) runs root first like paths_topk_kernel's; a warp keeps the running
// top-k of its chunk in registers (topk_offer).  grid (ceil(n_chunks / 4), queries), 4 warps = 4 chunks per CTA.
// TAGGED: only positions whose sentence is eligible (pos_tags & the query's mask) are scored and offered; query i of
// the launch is query which[which_off + i] of qtags when a which list is given.
template <bool TAGGED>
__global__ void __launch_bounds__(128)
paths_small_kernel(const float *__restrict__ ST, int nq, const int *__restrict__ nq_dev, int n_pos, int max_len,
                   const int *__restrict__ path_pm, const int4 *__restrict__ pos_rec, const double *__restrict__ level_w, int k,
                   float *cand_s, int *cand_i, int n_chunks, int chunk_len, const unsigned *__restrict__ qtags,
                   const unsigned *__restrict__ pos_tags, const int *__restrict__ which, int which_off) {
    extern __shared__ __align__(16) unsigned char ps_smem[];
    double *lw = reinterpret_cast<double *>(ps_smem);
    if (nq_dev) nq = min(nq, *nq_dev);
    const int q = blockIdx.y;
    if (q >= nq) return;
    for (int i = threadIdx.x; i < max_len; i += blockDim.x) lw[i] = level_w[i];
    __syncthreads();
    const int lane = threadIdx.x & 31, chunk = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (chunk >= n_chunks) return;
    const int p0 = chunk * chunk_len, p1 = min(n_pos, p0 + chunk_len);
    const unsigned qtag = TAGGED ? qtags[which ? which[which_off + q] : q] : 0u;
    float ls[PT_SLOTS];
    int li[PT_SLOTS];
    topk_init(ls, li);
    for (int pb = p0; pb < p1; pb += 32) {
        const int p = pb + lane;
        float acc = 0.0f;
        int sid = -1;
        if (p < p1 && (!TAGGED || (pos_tags[p] & qtag) != 0u)) {
            const int4 rc = pos_rec[p];
            const int len = rc.x;
            sid = rc.w;
            const int *path = path_pm + (size_t)p * max_len;
            const double dl = (double)len;
            for (int j = 0; j < len; j++)
                acc = __fmaf_rn((float)(lw[j] / dl), ST[(size_t)path[j] * CW_SMALL_Q + q], acc);
        }
        topk_offer(ls, li, k, acc, sid);
    }
    topk_store(ls, li, k, cand_s + ((size_t)q * n_chunks + chunk) * k, cand_i + ((size_t)q * n_chunks + chunk) * k);
}
}  // namespace cw

extern "C" int64_t cw_small_scratch_words(int64_t n_pos, int k) {
    return (int64_t)CW_SMALL_Q * cw_topk_chunks(n_pos < 1 ? 1 : n_pos) * (k > 0 ? k : 1) * 2;
}

// tf (optional): the tagged form (cw_small_predict_tagged)
int cw_small_predict_impl(const cw_index *ix, const float *Q, int64_t nq, const int32_t *which, const int32_t *n_dev,
                          int32_t which_off, int scatter, int k, float *sm_Q, float *sm_scores, int32_t *sm_scratch, int32_t *sm_sid,
                          float *sm_val, int32_t *sm_n, int32_t *out_sid, float *out_val, cudaStream_t st,
                          const cw_tag_filter *tf) {
    CwRange range("cw_small_predict");
    if (!ix || !Q || nq < 0 || nq > CW_SMALL_Q || k < 1 || k > CW_MAX_K || !sm_scores || !sm_scratch || !out_sid || !out_val ||
        (which && (!sm_Q || !sm_sid || !sm_val || !sm_n)) || (n_dev && !which) || (tf && (!tf->query_tags || !tf->pos_tags))) {
        cw_set_error("cw_small_predict: bad argument (nq=%lld, at most %d; k=%d)", (long long)nq, CW_SMALL_Q, k);
        return CW_E_ARG;
    }
    if (nq == 0) return 0;
    const float *xq = Q;
    const int *cnt = nullptr;
    if (which) {
        small_gather_kernel<<<32, 256, 0, st>>>(Q, ix->D, which, n_dev, which_off, (int)nq, sm_Q, sm_n);
        xq = sm_Q;
        cnt = sm_n;
    }
    const int qb = n_dev ? CW_SMALL_Q : (nq <= 1 ? 1 : nq <= 2 ? 2 : nq <= 4 ? 4 : nq <= 8 ? 8 : nq <= 16 ? 16 : 32);
    auto launch = [&](auto kern) {
        kern<<<ix->n_ntiles, CW_TILE_N, 0, st>>>(xq, ix->R, ix->MB, ix->sumlog, sm_scores, ix->n_ktiles, ix->D, (int)nq, cnt);
    };
    switch (qb) {
        case 1: launch(small_scores_kernel<1>); break;
        case 2: launch(small_scores_kernel<2>); break;
        case 4: launch(small_scores_kernel<4>); break;
        case 8: launch(small_scores_kernel<8>); break;
        case 16: launch(small_scores_kernel<16>); break;
        default: launch(small_scores_kernel<32>); break;
    }
    // path product + top-k: as many position chunks per query as the scratch holds (more for fewer queries)
    if (ix->n_pos < 1 || !ix->path_idx || !ix->pos_rec || !ix->level_w || ix->max_len < 1) {
        cw_set_error("cw_small_predict: the index has no sentence paths");
        return CW_E_ARG;
    }
    const long long slots = (long long)CW_SMALL_Q * (cw_topk_chunks(ix->n_pos) - 1);
    long long per_q = slots / nq;
    if (per_q > 1024) per_q = 1024;
    int chunk_len = (int)((ix->n_pos + per_q - 1) / per_q);
    if (chunk_len < 256) chunk_len = 256;
    chunk_len = (chunk_len + 31) & ~31;
    const int n_chunks = (ix->n_pos + chunk_len - 1) / chunk_len;
    float *cand_s = reinterpret_cast<float *>(sm_scratch);
    int *cand_i = sm_scratch + (size_t)nq * n_chunks * k;
    (tf ? paths_small_kernel<true> : paths_small_kernel<false>)<<<dim3((n_chunks + 3) / 4, (unsigned)nq), 128,
                                                                  (size_t)ix->max_len * sizeof(double), st>>>(
        sm_scores, (int)nq, cnt, ix->n_pos, ix->max_len, ix->path_idx, reinterpret_cast<const int4 *>(ix->pos_rec), ix->level_w, k,
        cand_s, cand_i, n_chunks, chunk_len, tf ? tf->query_tags : nullptr, tf ? tf->pos_tags : nullptr, which, which_off);
    merge_topk_kernel<<<(unsigned)((nq + 7) / 8), 256, 0, st>>>(cand_s, cand_i, nq, n_chunks, k, which ? sm_sid : out_sid,
                                                               which ? sm_val : out_val, cnt);
    int rc = cw_check_cuda(cudaGetLastError(), "cw_small_predict: paths");
    if (rc) return rc;
    if (which && scatter) small_scatter_kernel<<<1, 256, 0, st>>>(which, which_off, sm_n, k, sm_sid, sm_val, out_sid, out_val);
    return cw_check_cuda(cudaGetLastError(), "cw_small_predict");
}

extern "C" int cw_small_predict(const cw_index *ix, const float *Q, int64_t nq, const int32_t *which, const int32_t *n_dev,
                                int32_t which_off, int scatter, int k, float *sm_Q, float *sm_scores, int32_t *sm_scratch, int32_t *sm_sid,
                                float *sm_val, int32_t *sm_n, int32_t *out_sid, float *out_val, void *stream) {
    return cw_small_predict_impl(ix, Q, nq, which, n_dev, which_off, scatter, k, sm_Q, sm_scores, sm_scratch, sm_sid, sm_val, sm_n, out_sid,
                                 out_val, (cudaStream_t)stream, nullptr);
}

extern "C" int cw_small_predict_tagged(const cw_index *ix, const cw_tag_filter *tf, const float *Q, int64_t nq, const int32_t *which,
                                       const int32_t *n_dev, int32_t which_off, int scatter, int k, float *sm_Q, float *sm_scores,
                                       int32_t *sm_scratch, int32_t *sm_sid, float *sm_val, int32_t *sm_n, int32_t *out_sid,
                                       float *out_val, void *stream) {
    if (!tf) {
        cw_set_error("cw_small_predict_tagged: no tag filter");
        return CW_E_ARG;
    }
    return cw_small_predict_impl(ix, Q, nq, which, n_dev, which_off, scatter, k, sm_Q, sm_scores, sm_scratch, sm_sid, sm_val, sm_n, out_sid,
                                 out_val, (cudaStream_t)stream, tf);
}

extern "C" int cw_small_predict_host(const cw_index *ix, const float *Q_host, int64_t nq, int k, float *sm_Q, float *sm_scores,
                                     int32_t *sm_scratch, int32_t *sm_sid, float *sm_val, int32_t *sm_n, int32_t *out_sid_host,
                                     float *out_val_host, void *stream) {
    CwRange range("cw_small_predict_host");
    if (!ix || !Q_host || !sm_Q || !sm_sid || !sm_val || !out_sid_host || !out_val_host || nq < 0 || nq > CW_SMALL_Q) {
        cw_set_error("cw_small_predict_host: bad argument");
        return CW_E_ARG;
    }
    if (nq == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = cw_check_cuda(cudaMemcpyAsync(sm_Q, Q_host, (size_t)nq * ix->D * sizeof(float), cudaMemcpyHostToDevice, st),
                           "cw_small_predict_host: H2D");
    if (rc) return rc;
    if ((rc = cw_small_predict_impl(ix, sm_Q, nq, nullptr, nullptr, 0, 0, k, sm_Q, sm_scores, sm_scratch, sm_sid, sm_val, sm_n, sm_sid,
                                    sm_val, st, nullptr)))
        return rc;
    if ((rc = cw_check_cuda(cudaMemcpyAsync(out_sid_host, sm_sid, (size_t)nq * k * sizeof(int32_t), cudaMemcpyDeviceToHost, st),
                            "cw_small_predict_host: D2H ids")))
        return rc;
    if ((rc = cw_check_cuda(cudaMemcpyAsync(out_val_host, sm_val, (size_t)nq * k * sizeof(float), cudaMemcpyDeviceToHost, st),
                            "cw_small_predict_host: D2H scores")))
        return rc;
    return cw_check_cuda(cudaStreamSynchronize(st), "cw_small_predict_host: sync");
}
