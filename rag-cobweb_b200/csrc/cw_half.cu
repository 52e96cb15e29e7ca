// cw_half.cu -- the dense leaf ranking of cobweb_predict_indexed / cobweb_predict_fast
// (src/cobweb/CobwebWrapper.py:210-265) on tcgen05 with fp16 operands ("fused" mode, DESIGN.md section 5).
//
//   s[q,n]    = -0.5*(sumlog[n] + sum_d (x_qd - mu_nd)^2 / var_nd) = h[n] - 0.5 * sum_f A[q,f] * B[n,f]
//   leaf score sum_j (w_j/len) s_j = (C[parent] + w_leaf s_leaf) / len,  C[n] = sum_{j in path(n)} w_j s_j
//   C is linear in the row operands: C[n] = h'_n - 0.5 sum_f A[q,f] B'_n[f] with B'_n = sum_j w_j B_j, h'_n = sum_j w_j h_j,
//   so the internal rows carry the path-summed operands and their scores are the ancestor sums.
//
// Two operand precisions, one kernel:
//   NPROD = 3  every operand v (scaled by a per-row power of two into the fp16 range) is split v = hi + lo into two
//              fp16 numbers (22 significant bits) and a product is hi*hi + hi*lo + lo*hi -- three tcgen05.mma
//              kind::f16 (K = 16 each) per K step.  Used for the INTERNAL rows, whose scores feed every leaf below
//              them through C.  Half the MMA slots and half the operand bytes of the split-TF32 form it replaces.
//   NPROD = 1  one fp16 product.  Used for the LEAF rows (80 % of an index) as a FILTER: with round-to-nearest
//              operands |fl(a) fl(b) - a b| <= (2^-10 + 2^-22) |a b| per term (products of two fp16 numbers are
//              exact in the fp32 accumulator), so by Cauchy-Schwarz the whole contraction is off by at most
//              c1 ||a_q||_2 ||b_n||_2: a bound that costs one FMA per (query, leaf) in the epilogue.  A leaf
//              whose upper bound stays below the query's threshold is dropped; what survives (~100 of 100k leaves)
//              is re-scored exactly by the finish stage.  Leaves almost always have ONE variance for all
//              attributes (a leaf holds one vector or exact duplicates: M2 = 0, var = prior), then
//              sum_d x^2/var = |x|^2/var is a rank-one term of the epilogue and the contraction runs over D features
//              (layout F1) instead of 2D (layout F2).
//
// Kernel shape (as the split-TF32 kernel it replaces): persistent, one CTA per SM, CTA tile 256 queries x 256 rows
// = two 128 x 256 fp32 accumulators = all 512 TMEM columns; warp 0 = producer (cp.async.bulk of a 64 KB stage: the
// operands live in HBM as the exact shared-memory image, K-major rows of 64 bytes = 32 fp16, 64-byte swizzle, so a
// stage is two contiguous copies), warp 1 = MMA issuer (8 resp. 12 tcgen05.mma M128 N256 K16 per stage), warps 2-9 =
// epilogue (tcgen05.ld 32x32b.x32, lane = query, column = row).  The one-product form needs 64 B/clk of operands
// per SM at full tensor rate, above the 43 B/clk the L2 delivers: that kernel is L2->SM bound, not tensor bound.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#include <type_traits>

#include "../../include/cobweb_b200.h"
#include "cw_nvtx.h"

void cw_set_error(const char *fmt, ...);
int cw_check_cuda(cudaError_t e, const char *what);

namespace cwh {

constexpr int TQ = CW_H_TILE;   // queries per CTA tile (two UMMA M = 128 halves)
constexpr int TM = 128;         // UMMA M
constexpr int TN = CW_H_TILE;   // index rows per tile (UMMA N)
constexpr int ROWB = 64;        // bytes per operand row of a slab (32 fp16)
constexpr int IMG = CW_H_IMG_BYTES;
constexpr int SIDE = CW_H_STAGE_BYTES;  // A resp. B part of a stage: two images
constexpr int BW = 16;          // accumulator columns (index rows) an epilogue thread handles at a time
constexpr int REC_FLOATS = 8;
static_assert(IMG == TN * ROWB && SIDE == 2 * IMG, "stage geometry");
static_assert(BW * 2 == 32, "epilogue geometry");

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol error traps (the launch fails with an error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 28)) __trap();
    }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, one 128 x 256 x 16 fp16 MMA, fp32 accumulate
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): K-major operand, rows of 64 bytes, 64-byte swizzle
// (Swizzle<2,4,3>); 8-row groups 512 bytes apart.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);  // start address, 16-byte units
    d |= (uint64_t)1 << 16;                    // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(8 * ROWB >> 4) << 32;      // stride byte offset between 8-row groups
    d |= (uint64_t)1 << 46;                    // descriptor version (Blackwell)
    d |= (uint64_t)4 << 61;                    // SWIZZLE_64B
    return d;
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): D = F32 (bits 4-5 = 1), A = B = F16 (format 0), both K-major
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

#define CWH_TMEM_LD32(taddr, v)                                                                                    \
    asm volatile(                                                                                                  \
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                                  \
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "                                  \
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"                  \
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),          \
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),    \
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),  \
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])   \
        : "r"(taddr)                                                                                               \
        : "memory")

#define CWH_TMEM_LD16(taddr, v)                                                                                    \
    asm volatile(                                                                                                  \
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "                                                                  \
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"                           \
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),          \
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])     \
        : "r"(taddr)                                                                                               \
        : "memory")

// byte offset of 16-byte chunk c (0..3) of row r inside a 64-byte-swizzled operand image: address bits [7,9)
// (row / 2 within the 8-row group) are XORed into the chunk bits [4,6)
__device__ __forceinline__ int swz_off(int r, int c) { return r * ROWB + ((c ^ ((r >> 1) & 3)) << 4); }

// order-preserving float <-> int key (atomicMax on scores)
__device__ __forceinline__ int float_key(float f) {
    const int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float key_float(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }

__host__ __device__ inline int slabs_of(int D, int layout) { return layout == CW_H_F1 ? (D + 31) / 32 : (D + 15) / 16; }
__host__ __device__ inline int stages_of(int D, int layout, int nprod) {
    const int sl = slabs_of(D, layout);
    return nprod == 3 ? sl : (sl + 1) / 2;
}

// tile t -> (row tile, query tile): panels of pq query tiles, row tile outer / query tile inner within a panel
__device__ __forceinline__ void tile_coords(long long t, int n_qtiles, int n_ntiles, int pq, int &nt, int &qt) {
    const long long per_full = (long long)pq * n_ntiles;
    const int n_panels = (n_qtiles + pq - 1) / pq;
    int p = (int)(t / per_full);
    if (p > n_panels - 1) p = n_panels - 1;
    const long long rem = t - (long long)p * per_full;
    const int w = min(pq, n_qtiles - p * pq);
    nt = (int)(rem / w);
    qt = p * pq + (int)(rem % w);
}

// What the epilogue does with a finished 128 x 256 accumulator (lane = query, column = row of the operand set):
//   EPI_NODE    s = h - 0.5 acc, written row-major: out[row * ldq + q]     (internal rows: the ancestor sums C)
//   EPI_TAU     leaf score a1 of the sampled leaf tiles; per query the maximum over the rows r with r % 32 == j goes
//               to slot j (32 different leaves per query reach their slot values)
//   EPI_FILTER  a1 and its upper bound a1 + e1[row] * ||a_q||; (a1, row) appended to the query's candidate buffer when
//               the bound reaches tau[q]
// TAGGED (TAU and FILTER): a row counts only if it is eligible, leaf_tags[row] & qtags[q] != 0 (the leaf holds at least one
// sentence the query may see).  The row's tag is staged in shared memory in place of its parent row (record word 5),
// which only the staging itself reads.
enum { EPI_NODE = 0, EPI_TAU = 1, EPI_FILTER = 2 };
struct HEpi {
    float *out;           // NODE: [rows, ldq]
    long long ldq;
    const float *rc;      // per-row constants of the operand set
    const float4 *qv;     // [queries] {2^-s_leaf, |x|^2, ||a_leaf||, 2^-s_int}
    const float *C;       // TAU / FILTER: cumulative sums of the internal rows [n_int, ldq]
    int n_rows;           // real rows of the set (the rest is tile padding)
    long long nq;
    int *slots;           // TAU: [nq, 32] order-preserving keys
    const float *tau;     // FILTER: [nq]
    int cap;              // FILTER: candidate slots per query
    int *cnt;             // FILTER: [nq] candidates appended (may exceed cap: overflow)
    float *cand_val;      // FILTER: [nq, cap]
    int *cand_row;        // FILTER: [nq, cap]
};

// Two tile shapes.  FULL: 256 queries x 256 rows per CTA, one CTA per SM, all 512 TMEM columns: the least operand traffic
// per MMA (the three-product kernel of the internal rows is tensor-bound and wants exactly that).  HALF: 128 queries x
// 256 rows, TWO CTAs per SM with 256 TMEM columns each: the one-product kernels alternate between an MMA phase that waits
// on operands and an epilogue that cannot overlap it inside one CTA (the tile owns its accumulator until it is drained) --
// with two CTAs per SM one computes while the other drains, for 1.5x the operand traffic.
template <bool HALF>
struct KCfg {
    static constexpr int TQK = HALF ? 128 : 256;         // queries per CTA tile
    static constexpr int NQH = TQK / TM;                 // accumulators (128-query halves)
    static constexpr int A_IMG = HALF ? IMG / 2 : IMG;   // bytes of one query-operand image the CTA holds
    static constexpr int A_SIDE = 2 * A_IMG;
    static constexpr int STAGE = A_SIDE + SIDE;
    static constexpr int NST = HALF ? 2 : 3;
    static constexpr int EPIW = HALF ? 8 : 16;           // epilogue warps
    static constexpr int THR = 64 + 32 * EPIW;
    static constexpr int EPI_THR = 32 * EPIW;
    static constexpr int RBUFS = HALF ? 1 : 2;           // leaf-record buffers
    static constexpr int TMEM_COLS = HALF ? 256 : 512;
    static constexpr int REC = RBUFS * (TN * REC_FLOATS * 4 + TN * 8 + 64);
    static constexpr int SMEM = NST * STAGE + 1024 /* alignment slack */ + 256 /* barriers */ + REC;
    static constexpr int CTAS = HALF ? 2 : 1;
};
static_assert(KCfg<true>::SMEM * 2 + 2048 <= 227 * 1024 + 1024, "two half-tile CTAs per SM");

template <int NPROD, int MODE, bool HALF, bool TAGGED>
__global__ void __launch_bounds__(KCfg<HALF>::THR, KCfg<HALF>::CTAS)
h_score_kernel(const unsigned char *__restrict__ A, const unsigned char *__restrict__ B, const HEpi epi, int n_qtiles,
               int nt_begin, int n_ntiles, int n_stages, int pq, const unsigned *__restrict__ qtags,
               const unsigned *__restrict__ leaf_tags) {
    using K = KCfg<HALF>;
    extern __shared__ unsigned char smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;  // swizzle atoms need their natural alignment
    const uint32_t bars = base + K::NST * K::STAGE;
    // barrier words: full[NST], empty[NST], acc_full, acc_empty, then the TMEM base address
    const uint32_t full0 = bars, empty0 = bars + 8 * K::NST, accf = bars + 16 * K::NST, acce = accf + 8;
    const uint32_t tmem_slot = acce + 8;
    uint32_t *tmem_slot_ptr = reinterpret_cast<uint32_t *>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
    float4 *recs_s = reinterpret_cast<float4 *>(smem_raw + (bars + 256 - smem_u32(smem_raw)));  // [RBUFS][TN][2]
    long long *coff_s = reinterpret_cast<long long *>(recs_s + K::RBUFS * TN * 2);                // [RBUFS][TN]
    unsigned *heads_s = reinterpret_cast<unsigned *>(coff_s + K::RBUFS * TN);                     // [RBUFS][8 run heads, 8 heads to load]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < K::NST; s++) {
            mbar_init(full0 + 8 * s, 1);
            mbar_init(empty0 + 8 * s, 1);
        }
        mbar_init(accf, 1);
        mbar_init(acce, K::EPIW);  // one arrival per epilogue warp
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {  // TMEM: one 128 x 256 fp32 accumulator per 128 queries of the tile; this warp also frees them
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(K::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    const long long n_tiles = (long long)n_qtiles * n_ntiles;

    if (warp == 0) {
        // ===== producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
                int nt, qt;
                tile_coords(t, n_qtiles, n_ntiles, pq, nt, qt);
                // the query operands are stored per 256-query tile; a half tile takes rows 128 (qt & 1) .. of both images
                const unsigned char *asrc = A + (size_t)(HALF ? qt >> 1 : qt) * n_stages * SIDE + (HALF ? (qt & 1) * (IMG / 2) : 0);
                const unsigned char *bsrc = B + (size_t)(nt_begin + nt) * n_stages * SIDE;
                for (int s = 0; s < n_stages; s++) {
                    mbar_wait(empty0 + 8 * stage, phase ^ 1);
                    const uint32_t sb = base + stage * K::STAGE;
                    mbar_arrive_expect_tx(full0 + 8 * stage, K::STAGE);
                    if (HALF) {
                        bulk_g2s(sb, asrc + (size_t)s * SIDE, IMG / 2, full0 + 8 * stage);
                        bulk_g2s(sb + IMG / 2, asrc + (size_t)s * SIDE + IMG, IMG / 2, full0 + 8 * stage);
                    } else {
                        bulk_g2s(sb, asrc + (size_t)s * SIDE, SIDE, full0 + 8 * stage);
                    }
                    bulk_g2s(sb + K::A_SIDE, bsrc + (size_t)s * SIDE, SIDE, full0 + 8 * stage);
                    if (++stage == K::NST) { stage = 0; phase ^= 1; }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===== MMA issuer
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc(TM, TN);
            int stage = 0;
            uint32_t phase = 0, aphase = 0;
            for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
                mbar_wait(acce, aphase ^ 1);  // epilogue has drained the accumulators of the previous tile
                tc_fence_after();
                for (int s = 0; s < n_stages; s++) {
                    mbar_wait(full0 + 8 * stage, phase);
                    tc_fence_after();
                    const uint32_t sb = base + stage * K::STAGE;
                    if (NPROD == 3) {
                        // images: A hi, A lo | B hi, B lo of one slab
                        const uint64_t b_hi = make_smem_desc(sb + K::A_SIDE), b_lo = make_smem_desc(sb + K::A_SIDE + IMG);
#pragma unroll
                        for (int qh = 0; qh < K::NQH; qh++) {  // the 128-query halves of the tile, one accumulator each
                            const uint32_t d = tmem_base + (uint32_t)(qh * TN);
                            const uint64_t a_hi = make_smem_desc(sb + qh * (TM * ROWB));
                            const uint64_t a_lo = make_smem_desc(sb + K::A_IMG + qh * (TM * ROWB));
#pragma unroll
                            for (int k = 0; k < ROWB / 32; k++) {  // 16 fp16 = 32 bytes per MMA; +2 in 16-byte address units
                                const uint64_t ko = (uint64_t)(2 * k);
                                tc_mma_f16(d, a_hi + ko, b_hi + ko, idesc, (s | k) != 0);
                                tc_mma_f16(d, a_hi + ko, b_lo + ko, idesc, 1);
                                tc_mma_f16(d, a_lo + ko, b_hi + ko, idesc, 1);
                            }
                        }
                    } else {
                        // images: A slab 2s, A slab 2s+1 | B slab 2s, B slab 2s+1
#pragma unroll
                        for (int g = 0; g < 2; g++) {
                            const uint64_t b_g = make_smem_desc(sb + K::A_SIDE + g * IMG);
#pragma unroll
                            for (int qh = 0; qh < K::NQH; qh++) {
                                const uint32_t d = tmem_base + (uint32_t)(qh * TN);
                                const uint64_t a_g = make_smem_desc(sb + g * K::A_IMG + qh * (TM * ROWB));
#pragma unroll
                                for (int k = 0; k < ROWB / 32; k++) {
                                    const uint64_t ko = (uint64_t)(2 * k);
                                    tc_mma_f16(d, a_g + ko, b_g + ko, idesc, (s | g | k) != 0);
                                }
                            }
                        }
                    }
                    tc_commit(empty0 + 8 * stage);  // stage free once these MMAs have read it
                    if (s == n_stages - 1) tc_commit(accf);
                    if (++stage == K::NST) { stage = 0; phase ^= 1; }
                }
                aphase ^= 1;
            }
        }
        __syncwarp();
    } else {
        // ===== epilogue: sixteen warps (eight for a half tile); warp w reads TMEM lanes 32*(w%4) .. +31 (lane = query of
        // the 128-query half), the warps of a lane quarter take 16-column blocks in turn.  The work per (query, row) is a dozen
        // dependent instructions on two shared-memory reads: latency-bound, so the more warps the better; 16 columns at
        // a time keep a thread under the 112 registers that 576 threads per SM allow.
        const int quarter = warp & 3, sub = (warp - 2) >> 2;  // sub 0 .. EPIW/4 - 1
        constexpr int WPQ = K::EPIW / 4;                       // warps per lane quarter
        uint32_t aphase = 0;
        int rbuf = 0;
        const long long ldq = epi.ldq;
        for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
            int nt, qt;
            tile_coords(t, n_qtiles, n_ntiles, pq, nt, qt);
            const long long n0 = (long long)(nt_begin + nt) * TN;
            const long long qbase = (long long)qt * K::TQK + quarter * 32 + lane;
            if (MODE == EPI_NODE) {
                const float2 *rc2 = reinterpret_cast<const float2 *>(epi.rc);
                mbar_wait(accf, aphase);
                tc_fence_after();
#pragma unroll 1
                for (int qh = 0; qh < K::NQH; qh++) {
                    const long long q0 = (long long)qt * K::TQK + qh * TM;
                    if (q0 >= ldq) break;  // a half-tile of pure padding past the score matrix
                    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(qh * TN);
                    const long long q = qbase + qh * TM;
                    const float sa = epi.qv[q].w;
#pragma unroll 1
                    for (int cb = sub; cb < TN / BW; cb += WPQ) {
                        uint32_t v[BW];
                        CWH_TMEM_LD16(taddr + (uint32_t)(cb * BW), v);
                        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                        for (int j = 0; j < BW; j++) {
                            const long long n = n0 + cb * BW + j;
                            const float2 r = __ldg(rc2 + n);
                            epi.out[n * ldq + q] = fmaf(__uint_as_float(v[j]) * sa, r.y, r.x);
                        }
                    }
                }
            } else {
                // the tile's leaf records go to shared memory while the MMAs of the tile are still running; two
                // buffers, so that one named barrier per tile also protects the buffer of the tile before
                if (K::RBUFS == 1 && t != (long long)blockIdx.x)
                    asm volatile("bar.sync 1, %0;" ::"n"(K::EPI_THR) : "memory");  // one buffer: everyone is done with the previous tile's records
                const float4 *recs = recs_s + rbuf * (TN * 2);
                const long long *coff = coff_s + rbuf * TN;
                const unsigned *heads = heads_s + rbuf * 16;
                {
                    // rows are in tree order, siblings adjacent: a row whose parent is the previous row's re-uses that
                    // row's ancestor sum.  heads[c] bit j = row 32 c + j starts a new run of equal parents; heads[8 + c] =
                    // those of them that have a parent row to load; coff = byte offset of that row of C.
                    const int e = threadIdx.x - 64;  // the first 256 epilogue threads: one row each
                    if (e < TN) {
                        const float4 *src = reinterpret_cast<const float4 *>(epi.rc) + (n0 + e) * 2;
                        const float4 r1 = __ldg(src + 1);
                        recs_s[rbuf * (TN * 2) + e * 2] = __ldg(src);
                        if (TAGGED) {
                            float4 r1t = r1;
                            r1t.y = __uint_as_float(n0 + e < epi.n_rows ? leaf_tags[n0 + e] : 0u);
                            recs_s[rbuf * (TN * 2) + e * 2 + 1] = r1t;
                        } else {
                            recs_s[rbuf * (TN * 2) + e * 2 + 1] = r1;
                        }
                        const int par = __float_as_int(r1.y), prev = __shfl_up_sync(0xffffffffu, par, 1);
                        coff_s[rbuf * TN + e] = (long long)(par < 0 ? 0 : par) * ldq * 4;
                        const bool head = (lane & (BW - 1)) == 0 || par != prev;
                        const unsigned hm = __ballot_sync(0xffffffffu, head), lm = __ballot_sync(0xffffffffu, head && par >= 0);
                        if (lane == 0) { heads_s[rbuf * 16 + (e >> 5)] = hm; heads_s[rbuf * 16 + 8 + (e >> 5)] = lm; }
                    }
                    asm volatile("bar.sync 1, %0;" ::"n"(K::EPI_THR) : "memory");
                    if (K::RBUFS == 2) rbuf ^= 1;
                }
                // This warp's eight batches of 16 rows: b -> (query half b / 4, column block sub + 4 (b % 4)).  The
                // ancestor sums C[parent][q] of a batch do not depend on the accumulator, so they are fetched one batch
                // ahead -- the first batch while the MMAs of the tile are still running -- and only for the run heads
                // (predicated loads, all in flight together); the other rows carry their predecessor's value along.
                // batch b of this warp -> (query half, 16-column block)
                auto half_of = [&](int b) { return HALF ? 0 : b >> 2; };
                auto block_of = [&](int b) { return HALF ? sub + WPQ * b : sub + WPQ * (b & 3); };
                auto heads_of = [&](int b) { const int cb = block_of(b); return (heads[cb >> 1] >> ((cb & 1) * BW)) & 0xffffu; };
                auto fetch_cp = [&](int b, float (&cp)[BW]) {
                    const int qh = half_of(b), cb = block_of(b);
                    const bool qok = (long long)qt * K::TQK + qh * TM < ldq;
                    const char *Cq = reinterpret_cast<const char *>(epi.C + qbase + qh * TM);
                    const unsigned lm = qok ? (heads[8 + (cb >> 1)] >> ((cb & 1) * BW)) & 0xffffu : 0u;
#pragma unroll
                    for (int j = 0; j < BW; j++) {
                        const char *ptr = Cq + coff[cb * BW + j];  // broadcast read
                        const unsigned go = lm & (1u << j);
                        float val = 0.0f;
                        asm volatile(
                            "{\n"
                            ".reg .pred p;\n"
                            "setp.ne.u32 p, %2, 0;\n"
                            "@p ld.global.nc.f32 %0, [%1];\n"
                            "}\n"
                            : "+f"(val)
                            : "l"(ptr), "r"(go));
                        cp[j] = val;
                    }
                };
                float4 qv0 = make_float4(0.f, 0.f, 0.f, 0.f), qv1 = qv0;
                float tau0 = 0.0f, tau1 = 0.0f;
                const bool live0 = qbase < epi.nq, live1 = qbase + TM < epi.nq;
                if (live0) qv0 = epi.qv[qbase];
                if (live1) qv1 = epi.qv[qbase + TM];
                if (MODE == EPI_FILTER) {
                    if (live0) tau0 = epi.tau[qbase];
                    if (live1) tau1 = epi.tau[qbase + TM];
                }
                unsigned qtag0 = 0u, qtag1 = 0u;
                if (TAGGED) {
                    if (live0) qtag0 = qtags[qbase];
                    if (live1) qtag1 = qtags[qbase + TM];
                }
                float smax[BW];  // TAU: this warp only ever sees the rows r with (r / 16) % 4 == sub: slots (sub & 1) * 16 + j
#pragma unroll
                for (int j = 0; j < BW; j++) smax[j] = -__int_as_float(0x7f800000);
                float cpn[BW];
                fetch_cp(0, cpn);
                mbar_wait(accf, aphase);
                tc_fence_after();
#pragma unroll 1
                for (int b = 0; b < 8; b++) {
                    const int qh = half_of(b), cb = block_of(b);
                    if ((long long)qt * K::TQK + qh * TM >= ldq) break;  // a half-tile of pure padding past the score matrix
                    const long long q = qbase + qh * TM;
                    uint32_t v[BW];
                    CWH_TMEM_LD16(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(qh * TN + cb * BW), v);
                    float cur[BW];
#pragma unroll
                    for (int j = 0; j < BW; j++) cur[j] = cpn[j];
                    const unsigned hm = heads_of(b);
                    if (b + 1 < 8) fetch_cp(b + 1, cpn);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    const float4 qv = qh ? qv1 : qv0;
                    const float tau = qh ? tau1 : tau0;
                    const bool live = qh ? live1 : live0;
                    const unsigned qtag = qh ? qtag1 : qtag0;
                    float sc[BW];
                    unsigned hit = 0;
                    float c = 0.0f;
#pragma unroll
                    for (int j = 0; j < BW; j++) {
                        const float4 r0 = recs[(cb * BW + j) * 2];      // {alpha, beta, gamma, delta}, broadcast read
                        float e1 = 0.0f;
                        bool elig = true;
                        if (TAGGED && MODE == EPI_TAU) {
                            elig = (__float_as_uint(recs[(cb * BW + j) * 2 + 1].y) & qtag) != 0u;
                        } else if (TAGGED) {
                            const float2 r1 = *reinterpret_cast<const float2 *>(recs + (cb * BW + j) * 2 + 1);  // {e1, tag}
                            e1 = r1.x;
                            elig = (__float_as_uint(r1.y) & qtag) != 0u;
                        } else {
                            e1 = recs[(cb * BW + j) * 2 + 1].x;
                        }
                        c = (hm & (1u << j)) ? cur[j] : c;             // ancestor sum of this row's run
                        const float t0 = fmaf(r0.z, qv.y, r0.y);       // beta + gamma |x|^2
                        const float t1 = fmaf(r0.w, c, t0);            // + C[parent] / len
                        sc[j] = fmaf(r0.x, __uint_as_float(v[j]) * qv.x, t1);
                        // an ineligible row leaves its slot alone: a slot no eligible row reaches keeps its fill
                        // (0x80 bytes, about -3.4e38), so the threshold drops to -inf when fewer than m slots are reached
                        if (MODE == EPI_TAU) { if (elig) smax[j] = fmaxf(smax[j], sc[j]); }
                        else if (elig && fmaf(e1, qv.z, sc[j]) >= tau) hit |= 1u << j;
                    }
                    if (MODE == EPI_FILTER) {
                        // rows past the set are tile padding (only in the last tile)
                        const long long left = (long long)epi.n_rows - (n0 + cb * BW);
                        if (left < BW) hit &= left <= 0 ? 0u : (1u << left) - 1u;
                        if (live && hit) {
                            // one counter update per thread and batch: a returning atomic per hit would put an L2
                            // round trip between the rows
                            int at = atomicAdd(epi.cnt + q, __popc(hit));
#pragma unroll
                            for (int j = 0; j < BW; j++) {
                                if (hit >> j & 1) {
                                    if (at < epi.cap) {
                                        epi.cand_val[q * epi.cap + at] = sc[j];
                                        epi.cand_row[q * epi.cap + at] = (int)(n0 + cb * BW + j);
                                    }
                                    at++;
                                }
                            }
                        }
                    }
                    if (MODE == EPI_TAU && (HALF ? b == 7 : (b & 3) == 3)) {
                        // this query half is done: publish the slot maxima that beat what the slots already hold
                        if (live) {
                            int *sl = epi.slots + q * 32 + (sub & 1) * BW;
#pragma unroll
                            for (int j4 = 0; j4 < BW / 4; j4++) {
                                const int4 cur4 = __ldcg(reinterpret_cast<const int4 *>(sl) + j4);
                                const int k0 = float_key(smax[4 * j4]), k1 = float_key(smax[4 * j4 + 1]);
                                const int k2 = float_key(smax[4 * j4 + 2]), k3 = float_key(smax[4 * j4 + 3]);
                                if (k0 > cur4.x) atomicMax(sl + 4 * j4, k0);
                                if (k1 > cur4.y) atomicMax(sl + 4 * j4 + 1, k1);
                                if (k2 > cur4.z) atomicMax(sl + 4 * j4 + 2, k2);
                                if (k3 > cur4.w) atomicMax(sl + 4 * j4 + 3, k3);
                            }
                        }
#pragma unroll
                        for (int j = 0; j < BW; j++) smax[j] = -__int_as_float(0x7f800000);
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acce);
            aphase ^= 1;
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(K::TMEM_COLS) : "memory");
    }
}

// ------------------------------------------------------------------ operand builders
__device__ __forceinline__ double warp_sum(double v) {
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
    for (int off = 16; off > 0; off >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, off));
    return v;
}
// power-of-two scale that puts a row maximum into [2^14, 2^15): the fp16 range is used to its top, elements down to
// 2^-29 of the row maximum keep all 11 bits
__device__ __forceinline__ int scale_exp(float rowmax) {
    if (!(rowmax > 0.0f) || !isfinite(rowmax)) return 0;
    int e = 14 - ilogbf(rowmax);
    return e < -100 ? -100 : (e > 100 ? 100 : e);
}
// eight scaled values -> one 16-byte chunk of the hi image and (optionally) of the lo image
__device__ __forceinline__ void store_chunk(unsigned char *hi_img, unsigned char *lo_img, int off, const float (&v)[8]) {
    __align__(16) __half h[8], l[8];
#pragma unroll
    for (int e = 0; e < 8; e++) {
        h[e] = __float2half_rn(v[e]);
        l[e] = __float2half_rn(v[e] - __half2float(h[e]));
    }
    *reinterpret_cast<uint4 *>(hi_img + off) = *reinterpret_cast<const uint4 *>(h);
    if (lo_img) *reinterpret_cast<uint4 *>(lo_img + off) = *reinterpret_cast<const uint4 *>(l);
}

// Queries: one warp per query row (rows past nq are zero padding of the last tile).  Writes qv and both operand
// sets: A_int (layout F2, hi + lo) if present and A_leaf (leaf layout, hi only).
__global__ void __launch_bounds__(256)
hq_build_kernel(const float *__restrict__ Q, long long nq, long long n_rows_pad, int D, int leaf_layout, unsigned char *A_int,
                unsigned char *A_leaf, float4 *qv) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * 8 + warp;
    if (row >= n_rows_pad) return;
    const bool valid = row < nq;
    const float *x = Q + row * D;
    float mx = 0.0f;
    double xx = 0.0, x4 = 0.0;
    if (valid) {
        for (int d = lane; d < D; d += 32) {
            const float v = x[d];
            mx = fmaxf(mx, fabsf(v));
            const double v2 = (double)v * (double)v;
            xx += v2;
            x4 += v2 * v2;
        }
    }
    mx = warp_max(mx);
    xx = warp_sum(xx);
    x4 = warp_sum(x4);
    const float max_f2 = fmaxf(mx, mx * mx);
    const int s_int = scale_exp(max_f2), s_leaf = scale_exp(leaf_layout == CW_H_F1 ? mx : max_f2);
    const float mul_int = ldexpf(1.0f, s_int), mul_leaf = ldexpf(1.0f, s_leaf);
    if (lane == 0) {
        const double nrm = leaf_layout == CW_H_F1 ? sqrt(xx) : sqrt(xx + x4);
        qv[row] = valid ? make_float4(ldexpf(1.0f, -s_leaf), (float)xx, (float)(nrm * (1.0 + 1e-6)), ldexpf(1.0f, -s_int))
                        : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    }
    const long long qt = row / TQ;
    const int r = (int)(row % TQ), c = lane & 3;
    auto emit = [&](unsigned char *Aset, int layout, int nprod, float mul) {
        const int n_sl = slabs_of(D, layout), n_sl_pad = nprod == 3 ? n_sl : (n_sl + 1) & ~1;
        for (int slab = lane >> 2; slab < n_sl_pad; slab += 8) {
            float v[8];
#pragma unroll
            for (int e = 0; e < 8; e++) {
                const int d = layout == CW_H_F1 ? slab * 32 + c * 8 + e : slab * 16 + (c & 1) * 8 + e;
                float t = (valid && slab < n_sl && d < D) ? x[d] : 0.0f;
                if (layout == CW_H_F2 && c < 2) t = t * t;
                v[e] = t * mul;
            }
            unsigned char *hi = nprod == 3 ? Aset + ((size_t)(qt * n_sl + slab) * 2) * IMG : Aset + (size_t)(qt * n_sl_pad + slab) * IMG;
            store_chunk(hi, nprod == 3 ? hi + IMG : nullptr, swz_off(r, c), v);
        }
    };
    if (A_int) emit(A_int, CW_H_F2, 3, mul_int);
    emit(A_leaf, leaf_layout, 1, mul_leaf);
}

__device__ __forceinline__ float var_at(const cw_store &s, int node, float cnt, int d) {
    if (!(cnt > 0.0f)) return s.prior_var;
    const float v = s.m2[(size_t)node * s.D + d] / cnt;  // CobwebTorchTree.compute_var
    return (s.flags & CW_ACUITY_CUTOFF) ? (v < s.prior_var ? s.prior_var : v) : v + s.prior_var;
}

// Index rows: one warp per row of the operand set (rows past n_rows are zero padding of the last tile).
// Internal rows (int_par given) hold their path sums B'_n = sum_{j in path(n)} w_j B_j, h'_n = sum_j w_j h_j, summed in
// binary64 walking int_par up from the row, so that the score kernel's s = h' - 0.5 acc IS the ancestor sum
// C[n] = sum_j w_j s_j.  Walking up needs no scratch (a level-by-level build would need a binary64 [n_int, 2D] buffer).
// int_par[n] < n: the internal rows are ordered by depth.
constexpr double C1 = 0.0009765625 * 1.002;  // 2^-10 + 2^-22 (two fp16 roundings per product), with slack for the fp32 conversions
__global__ void __launch_bounds__(256)
hn_build_kernel(cw_store s, const int *__restrict__ order, const int *__restrict__ rows, const float *__restrict__ sumlog,
                cw_h_set hs, const int *__restrict__ int_par, const float *__restrict__ int_w, const float *__restrict__ leaf_w,
                const float *__restrict__ leaf_il, const int *__restrict__ leaf_par, const int *__restrict__ leaf_len) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + warp;
    if (row >= hs.n_ntiles * TN) return;
    const bool valid = row < hs.n_rows;
    const int D = s.D, layout = hs.layout, nprod = hs.nprod;
    int node = 0, brow = 0;
    float cnt = 0.0f;
    if (valid) { brow = rows[row]; node = order[brow]; cnt = s.count[node]; }
    // the rows whose operands make up this row's: the path for an internal row (weights int_w), the row itself (weight 1)
    // for a leaf row.  A parent that is not an earlier row breaks the depth order the walk relies on: trap (the launch
    // fails with an error) rather than return truncated sums.
    auto up = [&](int j) {
        if (!int_par) return -1;
        const int p = int_par[j];
        if (p >= j) __trap();
        return p;
    };
    auto weight = [&](int j) { return int_par ? (double)int_w[j] : 1.0; };
    float mx = 0.0f;
    double b2 = 0.0, hsum = 0.0;
    if (valid) {
        for (int d = lane; d < D; d += 32) {
            // w = 1 (a leaf row, one step) multiplies and adds to 0 exactly: the row's own operands bit for bit
            double iv = 0.0, m = 0.0;
            for (int j = row; j >= 0; j = up(j)) {
                const int nj = order[rows[j]];
                const double w = weight(j), ivj = 1.0 / (double)var_at(s, nj, s.count[nj], d);
                const double mu = (double)s.mean[(size_t)nj * D + d];
                iv += w * ivj;
                m += w * (-2.0 * mu * ivj);
                hsum += w * mu * mu * ivj;
            }
            mx = fmaxf(mx, (float)fabs(m) * (1.0f + 1e-6f));
            b2 += m * m;
            if (layout == CW_H_F2) { mx = fmaxf(mx, (float)fabs(iv) * (1.0f + 1e-6f)); b2 += iv * iv; }
        }
    }
    mx = warp_max(mx);
    b2 = warp_sum(b2);
    hsum = warp_sum(hsum);
    const int sb = scale_exp(mx);
    const double mul = ldexp(1.0, sb);
    const int tile = row / TN, r = row % TN, c = lane & 3;
    const int n_sl = slabs_of(D, layout), n_sl_pad = nprod == 3 ? n_sl : (n_sl + 1) & ~1;
    unsigned char *Bset = reinterpret_cast<unsigned char *>(hs.B);
    for (int slab = lane >> 2; slab < n_sl_pad; slab += 8) {
        double t[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        if (valid && slab < n_sl) {
            for (int j = row; j >= 0; j = up(j)) {
                const int nj = order[rows[j]];
                const float cj = s.count[nj];
                const double w = weight(j);
#pragma unroll
                for (int e = 0; e < 8; e++) {
                    const int d = layout == CW_H_F1 ? slab * 32 + c * 8 + e : slab * 16 + (c & 1) * 8 + e;
                    if (d < D) {
                        const double ivj = 1.0 / (double)var_at(s, nj, cj, d);
                        t[e] += (layout == CW_H_F2 && c < 2) ? w * ivj : w * (-2.0 * (double)s.mean[(size_t)nj * D + d] * ivj);
                    }
                }
            }
        }
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; e++) v[e] = (float)(t[e] * mul);
        unsigned char *hi = nprod == 3 ? Bset + ((size_t)(tile * n_sl + slab) * 2) * IMG : Bset + (size_t)(tile * n_sl_pad + slab) * IMG;
        store_chunk(hi, nprod == 3 ? hi + IMG : nullptr, swz_off(r, c), v);
    }
    if (lane == 0) {
        double lsum = 0.0;  // sum_j w_j sumlog_j
        if (valid)
            for (int j = row; j >= 0; j = up(j)) lsum += weight(j) * (double)sumlog[rows[j]];
        const double h = valid ? -0.5 * (lsum + hsum) : 0.0;
        if (nprod == 3) {
            reinterpret_cast<float2 *>(hs.rc)[row] = make_float2((float)h, valid ? (float)(-0.5 * ldexp(1.0, -sb)) : 0.0f);
        } else {
            float4 r0 = make_float4(0.0f, -__int_as_float(0x7f800000), 0.0f, 0.0f);  // padding rows score -inf
            float4 r1 = make_float4(0.0f, __int_as_float(-1), 0.0f, __int_as_float(1));
            if (valid) {
                const double w = (double)leaf_w[row], il = (double)leaf_il[row];
                const double iv0 = 1.0 / (double)var_at(s, node, cnt, 0);
                r0.x = (float)(-0.5 * w * il * ldexp(1.0, -sb));
                r0.y = (float)(w * il * h);
                r0.z = layout == CW_H_F1 ? (float)(-0.5 * w * il * iv0) : 0.0f;
                r0.w = (float)il;
                r1.x = (float)(fabs(w) * il * 0.5 * C1 * sqrt(b2) * (1.0 + 1e-6));
                r1.y = __int_as_float(leaf_par[row]);
                r1.z = leaf_w[row];
                r1.w = __int_as_float(leaf_len[row]);
            }
            reinterpret_cast<float4 *>(hs.rc)[row * 2] = r0;
            reinterpret_cast<float4 *>(hs.rc)[row * 2 + 1] = r1;
        }
    }
}

// flag = 0 if some row has attributes with different variances
__global__ void __launch_bounds__(256)
h_iso_kernel(cw_store s, const int *__restrict__ order, const int *__restrict__ rows, int n_rows, int *flag) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + warp;
    if (row >= n_rows) return;
    const int node = order[rows[row]];
    const float cnt = s.count[node];
    const float v0 = var_at(s, node, cnt, 0);
    bool same = true;
    for (int d = lane; d < s.D; d += 32) same = same && var_at(s, node, cnt, d) == v0;
    if (!__all_sync(0xffffffffu, same) && lane == 0) atomicExch(flag, 0);
}

// ------------------------------------------------------------------ filter threshold
// eps: bound of |a3 - exact| for a leaf score of the query, a3 = the leaf score with exact leaf term and the fp16x3
// ancestor sums (statistical: operand term eps_scale * T plus (4 + 3 sqrt(max_len)) ulps of the score magnitude, as
// measured for the split-TF32 form whose precision the fp16 split equals; audited in production by
// DenseIndex.audit_fraction)
__device__ __forceinline__ float eps_of(float xx, float inv_prior, float hmax, float lmax, float wfac, float eps_scale, int max_len) {
    const float tq = 2.0f * (xx * inv_prior + hmax);
    return wfac * (eps_scale * tq + 1.1920929e-07f * (4.0f + 3.0f * sqrtf((float)max_len)) * 0.5f * (lmax + hmax + tq));
}
// tau[q] = (m-th largest of the 32 slot maxima) - margin; a heuristic for speed only: the finish stage verifies
// on the device that nothing below the threshold could have mattered.
__global__ void __launch_bounds__(128)
h_tau_kernel(const int *__restrict__ slots, const float4 *__restrict__ qv, long long nq, int m, float e1max, float inv_prior,
             float hmax, float lmax, float wfac, float eps_scale, int max_len, float *tau) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    float v[32];
#pragma unroll
    for (int j4 = 0; j4 < 8; j4++) {
        const int4 k = reinterpret_cast<const int4 *>(slots + q * 32)[j4];
        v[4 * j4] = key_float(k.x); v[4 * j4 + 1] = key_float(k.y); v[4 * j4 + 2] = key_float(k.z); v[4 * j4 + 3] = key_float(k.w);
    }
    float last = __int_as_float(0x7f800000);
    for (int it = 0; it < m; it++) {  // m-th largest: repeated maximum below the previous one (ties collapse: conservative)
        float best = -__int_as_float(0x7f800000);
#pragma unroll
        for (int j = 0; j < 32; j++)
            if (v[j] < last && v[j] > best) best = v[j];
        last = best;
    }
    float t = last;
    if (!(last > -1e38f)) t = -__int_as_float(0x7f800000);  // fewer than m sampled rows: no threshold
    tau[q] = t;
}
__global__ void h_fill_kernel(float *p, long long n, float v) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// ------------------------------------------------------------------ finish: select, exact pair scores, line test, top-k
// Five launches instead of one CTA per query, so that dozens of warps per SM keep row loads in flight and no warp waits
// at a block barrier for another warp's FMA chain:
//   fn_select_kernel  one warp per query: interval pruning of the candidates, the refine list, eps, U
//   fn_exact_kernel   one warp per query: exact node scores of a list of index rows (the refine list, then the ancestors)
//   fn_line_kernel    one warp per query: a3, the line test, the survivors and their distinct ancestors
//   fn_exact_kernel   (ancestors)
//   fn_topk_kernel    one warp per query: exact path sums of the survivors, top-k sentences
// The per-query lists live in global scratch behind the flag words (cw_fused_flag_words).
constexpr int FQ_WARPS = 8;  // queries per CTA of the per-query kernels
constexpr int KC1 = CW_FUSED_KC1, MS = CW_FUSED_MSURV, MAXS = CW_FUSED_MAX_SENT;
// meta words per query; the survivors (indices into the refine list) follow at FM_SURV
enum { FM_NSEL, FM_NANC, FM_M, FM_EPS, FM_U, FM_FAIL, FM_SURV = 8, FM_STRIDE = FM_SURV + MS };

__host__ __device__ inline long long fin_words(long long cap_q, int ml) { return cap_q * (FM_STRIDE + 3 * KC1 + 3LL * MS * ml); }

struct FinArgs {
    cw_index ix;
    const float2 *RM;  // [nn, D] {r, mb}
    const float *Q;
    long long nq;
    int k, cap;
    const int *cnt;
    const float *cand_val;
    const int *cand_row;
    const float *tau;
    const float4 *qv;
    const float4 *leaf_rc;   // 2 per leaf row
    const int *leaf_row_b, *leaf_pos, *sent_off, *sent_ids;
    const float *C;
    long long ldq;
    float inv_prior, hmax, lmax, wfac, eps_scale;
    int *out_sid;
    float *out_val;
    int *flag;   // [0] count, [4..] queries
    int *stats;
    // scratch (fin_carve)
    int em;          // MS * max_len: ancestor entries per query
    int *meta;       // [nq, FM_STRIDE]
    int *ref_row;    // [nq, KC1] leaf rows of the refined candidates
    int *ref_b;      // [nq, KC1] their index rows
    float *ref_s;    // [nq, KC1] their exact node scores
    int *anc_b;      // [nq, em] distinct ancestor index rows of the survivors
    float *anc_s;    // [nq, em] their exact node scores
    int *anc_slot;   // [nq, em] (survivor, level) -> entry of anc_b
    // tagged form (cw_fused_predict_tagged): the queries' masks and the sentences' tags
    const unsigned *qtags, *sent_tags;
};

static void fin_carve(FinArgs &a, int *p, long long cap_q, int ml) {
    a.em = MS * ml;
    a.meta = p; p += cap_q * FM_STRIDE;
    a.ref_row = p; p += cap_q * KC1;
    a.ref_b = p; p += cap_q * KC1;
    a.ref_s = reinterpret_cast<float *>(p); p += cap_q * KC1;
    a.anc_b = p; p += cap_q * a.em;
    a.anc_s = reinterpret_cast<float *>(p); p += cap_q * a.em;
    a.anc_slot = p;
}

__device__ __forceinline__ int warp_sum(int v) {
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}
// candidate order: a1 descending, leaf row ascending (one 64-bit key, larger = better; -0 and +0 are one a1)
__device__ __forceinline__ unsigned long long cand_key(float v, int row) {
    return (unsigned long long)((unsigned)float_key(v == 0.0f ? 0.0f : v) ^ 0x80000000u) << 32 | (unsigned)~row;
}

// Which candidates need the exact leaf term.  Every candidate has the interval [a1 - E, a1 + E] (E = e1[row] *
// ||a_q||, the filter's derived bound) around its leaf score with exact leaf term; L_k = the smallest lower end among
// the k best candidates by a1 is a lower bound of the k-th best such score (k different leaves reach it), so a
// candidate whose upper end stays 3 eps below L_k cannot reach the line drawn later and is dropped unrefined.  The
// rest -- the best KC1 of them by a1 -- is refined.  U = the largest upper end among everything left unrefined
// (dropped or cut here, or rejected by the filter: below tau).  Also adds the filter's candidate count to the stats.
__global__ void __launch_bounds__(FQ_WARPS * 32)
fn_select_kernel(const FinArgs a) {
    extern __shared__ __align__(16) unsigned char fs_smem[];
    __shared__ unsigned long long cand_sum;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, cap = a.cap;
    float *cv = reinterpret_cast<float *>(fs_smem) + (size_t)warp * cap * 3;  // [cap] a1
    int *cr = reinterpret_cast<int *>(cv + cap);                              // [cap] leaf row
    float *ce = cv + 2 * cap;                                                 // [cap] E
    const float NEG_INF = -__int_as_float(0x7f800000);
    if (threadIdx.x == 0) cand_sum = 0;
    __syncthreads();
    const long long q = (long long)blockIdx.x * FQ_WARPS + warp;
    if (q < a.nq) {
        const int n_all = a.cnt[q], n = min(n_all, cap);
        const float4 qq = a.qv[q];
        const float eps = eps_of(qq.y, a.inv_prior, a.hmax, a.lmax, a.wfac, a.eps_scale, a.ix.max_len);
        for (int i = lane; i < n; i += 32) {
            const int row = a.cand_row[q * cap + i];
            cv[i] = a.cand_val[q * cap + i];
            cr[i] = row;
            ce[i] = __fmul_rn(a.leaf_rc[row * 2 + 1].x, qq.z);
        }
        __syncwarp();
        // L_k: the k-th best key by k rounds of a warp-wide maximum below the previous one; the k best are the keys >= it
        float Lk = NEG_INF;
        if (n >= a.k) {
            unsigned long long last = ~0ull;
            for (int it = 0; it < a.k; it++) {
                unsigned long long best = 0;
                for (int i = lane; i < n; i += 32) {
                    const unsigned long long key = cand_key(cv[i], cr[i]);
                    if (key < last && key > best) best = key;
                }
                for (int off = 16; off > 0; off >>= 1) {
                    const unsigned long long o = __shfl_xor_sync(0xffffffffu, best, off);
                    best = o > best ? o : best;
                }
                last = best;
            }
            int lo = 0x7fffffff;
            for (int i = lane; i < n; i += 32)
                if (cand_key(cv[i], cr[i]) >= last) lo = min(lo, float_key(__fsub_rn(__fsub_rn(cv[i], ce[i]), eps)));
            for (int off = 16; off > 0; off >>= 1) lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, off));
            Lk = key_float(lo);
        }
        int count = 0;
        for (int i = lane; i < n; i += 32) count += __fmaf_rn(3.0f, eps, __fadd_rn(cv[i], ce[i])) >= Lk;
        count = warp_sum(count);
        // refine list: every kept candidate, or the best KC1 of them by a1 when more are kept
        int* const rrow = a.ref_row + q * KC1;
        int* const rb = a.ref_b + q * KC1;
        float umax = NEG_INF;
        int pos0 = 0;
        for (int base = 0; base < n; base += 32) {
            const int i = base + lane;
            const bool keep = i < n && __fmaf_rn(3.0f, eps, __fadd_rn(cv[i], ce[i])) >= Lk;
            int pos;
            if (count <= KC1) {
                pos = pos0 + __popc(__ballot_sync(0xffffffffu, keep) & ((1u << lane) - 1u));
                pos0 += __popc(__ballot_sync(0xffffffffu, keep));
            } else {
                pos = 0;
                if (keep) {
                    const unsigned long long key = cand_key(cv[i], cr[i]);
                    for (int j = 0; j < n; j++)
                        pos += cand_key(cv[j], cr[j]) > key && __fmaf_rn(3.0f, eps, __fadd_rn(cv[j], ce[j])) >= Lk;
                }
            }
            if (keep && pos < KC1) {
                rrow[pos] = cr[i];
                rb[pos] = a.leaf_row_b[cr[i]];
            } else if (i < n) {
                umax = fmaxf(umax, __fadd_rn(cv[i], ce[i]));  // left unrefined
            }
        }
        umax = warp_max(umax);
        if (lane == 0) {
            int *m = a.meta + q * FM_STRIDE;
            m[FM_NSEL] = min(count, KC1);
            m[FM_EPS] = __float_as_int(eps);
            m[FM_U] = __float_as_int(fmaxf(a.tau[q], umax));
            m[FM_FAIL] = n_all > cap ? 1 : 0;  // candidate-buffer overflow
            atomicAdd(&cand_sum, (unsigned long long)(unsigned)n_all);
        }
    }
    __syncthreads();
    // candidates appended by the filter (64-bit total in words 5, 6), queries in word 7
    if (threadIdx.x == 0 && cand_sum) atomicAdd(reinterpret_cast<unsigned long long *>(a.stats + 6), cand_sum);
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(a.stats + 5, (int)a.nq);
}

__device__ __forceinline__ void cp_async4(void *dst, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
// adds to the transaction count of the barrier's current phase without arriving
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}

// The exact chain over 32 attributes of a row segment in shared memory: rv = the segment's {r, mb} pairs, xs = the
// query's 32 attributes.  The whole piece is read into registers first (16-byte reads; an ODD row starts 8 bytes off
// that alignment and is read by float2), then the chain runs in ascending d.
template <bool ODD>
__device__ __forceinline__ float exact_chain32(const float2 *rv, const float *xs, float acc) {
    float4 rr[16], xv[8];
#pragma unroll
    for (int j = 0; j < 16; j++) {
        if (ODD) {
            const float2 u = rv[2 * j], v = rv[2 * j + 1];
            rr[j] = make_float4(u.x, u.y, v.x, v.y);
        } else {
            rr[j] = reinterpret_cast<const float4 *>(rv)[j];  // {r, mb} of 2 attributes
        }
    }
#pragma unroll
    for (int j = 0; j < 8; j++) xv[j] = reinterpret_cast<const float4 *>(xs)[j];
#pragma unroll
    for (int j = 0; j < 16; j++) {
        const float x0 = (j & 1) ? xv[j >> 1].z : xv[j >> 1].x, x1 = (j & 1) ? xv[j >> 1].w : xv[j >> 1].y;
        const float t0 = __fmaf_rn(x0, rr[j].x, rr[j].y);
        acc = __fmaf_rn(t0, t0, acc);
        const float t1 = __fmaf_rn(x1, rr[j].z, rr[j].w);
        acc = __fmaf_rn(t1, t1, acc);
    }
    return acc;
}

// Exact node scores with the FP32 path's arithmetic: out[q * stride + i] = -0.5 (sumlog[b] + sum_d (x_qd r_bd + mb_bd)^2)
// for b = list[q * stride + i], i < n = meta[q * meta_stride + n_word].  One warp per (query, row block): blockIdx.y
// takes rows [y * per, (y + 1) * per) with per = max(EX_R, ceil(n / gridDim.y)), so a long list is spread over several
// warps (gridDim.y = 1: one warp takes the whole list); a warp's rows go in rounds of at most EX_R.  Lane = row: every
// lane runs its row's FMA chain in ascending d from 0, so the result is bit-identical to dense_score_kernel.
// The rows arrive by bulk copies (cp.async.bulk, completion counted in bytes on an mbarrier), EX_SEG attributes (512
// bytes) of a row per copy, into a ring of EX_STAGES slots, EX_STAGES - 1 segments ahead of the arithmetic; each lane
// copies its own row's segment.  One warp per CTA, so a warp slot is handed to the next work item as soon as its list
// is done rather than when the CTA's longest list is; 12 such CTAs (17 KB each) fit an SM.  This geometry was chosen
// by timing the cfg3 launches against others (DESIGN §5).  A bulk copy needs 16-byte-aligned ends; a row of the
// [nn, D, 2] buffer (16-byte aligned: the entry points check it) starts 8 bytes off when b * D is odd, so a copy takes
// the aligned-down span (at most EX_SEG * 8 + 16 bytes: the slot pitch EX_RS) and the lane reads its segment from that
// offset.  No copy reads past the buffer's last byte: where that byte ends 8 bytes into a 16-byte unit, the copy stops
// short and the lane reads the buffer's last {r, mb} pair from global memory.  The pitch of EX_SEG + 2 float2 puts
// consecutive rows 4 banks apart, so the 16-byte reads by row are conflict-free.  The query's slice of a segment comes
// with 4-byte cp.async copies, one commit group per segment.
constexpr int EX_WARPS = 1, EX_R = 16, EX_SEG = 64, EX_STAGES = 2, EX_RS = EX_SEG + 2;
// per warp: the ring [EX_STAGES][EX_R][EX_RS] float2, the query slices [EX_STAGES][EX_SEG], one mbarrier per slot
constexpr int EX_WARP_BYTES = (EX_STAGES * EX_R * EX_RS * 8 + EX_STAGES * EX_SEG * 4 + EX_STAGES * 8 + 15) / 16 * 16;
static_assert(EX_SEG % 32 == 0 && EX_RS * 8 % 16 == 0, "ring geometry");
__global__ void __launch_bounds__(EX_WARPS * 32)
fn_exact_kernel(const cw_index ix, const float2 *__restrict__ RM, const float *__restrict__ Q, long long nq,
                const int *__restrict__ list, const int *__restrict__ meta, int meta_stride, int n_word, int stride,
                float *out) {
    extern __shared__ __align__(16) unsigned char ex_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, D = ix.D;
    float2 *ring = reinterpret_cast<float2 *>(ex_smem + (size_t)warp * EX_WARP_BYTES);  // [EX_STAGES][EX_R][EX_RS]
    float *xr = reinterpret_cast<float *>(ring + EX_STAGES * EX_R * EX_RS);             // [EX_STAGES][EX_SEG]
    const uint32_t bar0 = smem_u32(xr + EX_STAGES * EX_SEG);                             // [EX_STAGES] mbarriers
    const long long q = (long long)blockIdx.x * EX_WARPS + warp;
    if (q >= nq) return;
    const int n_all = meta[q * meta_stride + n_word];
    const int per = max(EX_R, (n_all + (int)gridDim.y - 1) / (int)gridDim.y), first = (int)blockIdx.y * per;
    if (first >= n_all) return;
    const int n = min(n_all, first + per);  // rows [first, n)
    if (lane == 0) {
        for (int s = 0; s < EX_STAGES; s++) mbar_init(bar0 + 8 * s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    const float *xq = Q + q * D;
    const int n_seg = (D + EX_SEG - 1) / EX_SEG;
    const long long lim = (long long)ix.nn * D * 8 & ~15ll;  // the buffer's last 16-byte boundary
    unsigned parity = 0;  // bit s: the phase of slot s's barrier that the next wait on it expects
    const int n_rounds = (n - first + EX_R - 1) / EX_R, rpr = (n - first + n_rounds - 1) / n_rounds;  // rows per round <= EX_R
    for (int lo = first; lo < n; lo += rpr) {
        const int cnt = min(rpr, n - lo);
        const int b = lane < cnt ? list[q * stride + lo + lane] : 0;
        const long long rb = (long long)b * D * 8;  // byte offset of the lane's row
        const int odd = (int)(rb & 8);              // 8 when the row starts off 16-byte alignment
        auto issue = [&](int seg) {
            if (seg < n_seg) {
                const int s = seg % EX_STAGES, d0 = seg * EX_SEG;
                const uint32_t bar = bar0 + 8 * s;
                if (lane < cnt) {
                    const long long from = rb + d0 * 8 - odd;
                    long long to = (rb + (long long)min(D, d0 + EX_SEG) * 8 + 15) & ~15ll;
                    if (to > lim) to -= 16;
                    if (to > from) {
                        mbar_expect_tx(bar, (uint32_t)(to - from));
                        bulk_g2s(smem_u32(ring + (s * EX_R + lane) * EX_RS), reinterpret_cast<const char *>(RM) + from,
                                 (uint32_t)(to - from), bar);
                    }
                }
#pragma unroll
                for (int i = lane; i < EX_SEG; i += 32)
                    if (d0 + i < D) cp_async4(xr + s * EX_SEG + i, xq + d0 + i);
                __syncwarp();  // every lane's expected bytes are on the barrier before it can complete
                if (lane == 0) mbar_arrive(bar);
            }
            asm volatile("cp.async.commit_group;" ::: "memory");  // one group per segment, empty past the end
        };
#pragma unroll
        for (int p = 0; p < EX_STAGES - 1; p++) issue(p);
        float acc = 0.0f;
        for (int seg = 0; seg < n_seg; seg++) {
            issue(seg + EX_STAGES - 1);
            const int s = seg % EX_STAGES, d0 = seg * EX_SEG;
            asm volatile("cp.async.wait_group %0;" ::"n"(EX_STAGES - 1) : "memory");
            mbar_wait(bar0 + 8 * s, (parity >> s) & 1u);
            parity ^= 1u << s;
            __syncwarp();  // the query slice: every lane's copies
            const float2 *rv = ring + (s * EX_R + lane) * EX_RS + (odd >> 3);
            const float *xs = xr + s * EX_SEG;
            if (lane < cnt) {
#pragma unroll
                for (int c = 0; c < EX_SEG; c += 32) {
                    if (d0 + c + 32 <= D) {
                        acc = odd ? exact_chain32<true>(rv + c, xs + c, acc) : exact_chain32<false>(rv + c, xs + c, acc);
                    } else {
                        for (int j = c; j < D - d0; j++) {
                            const float2 v = rb + (d0 + j + 1) * 8 > lim ? RM[(size_t)b * D + d0 + j] : rv[j];
                            const float t = __fmaf_rn(xs[j], v.x, v.y);
                            acc = __fmaf_rn(t, t, acc);
                        }
                        break;
                    }
                }
            }
            __syncwarp();  // the slot is refilled by the next issue
        }
        if (lane < cnt) out[q * stride + lo + lane] = __fmul_rn(-0.5f, __fadd_rn(ix.sumlog[b], acc));
    }
}

// a3 = (C[parent] + w_leaf s) / len of the refined leaves, the k-th best sentence score A_k over them, the line
// thr = A_k - 2 eps and its test against U, the survivors (a3 >= thr), and the distinct index rows on their paths
// (the leaf itself is already scored).  A query that fails is flagged here for the exact small-batch path.
// TAGGED: a leaf counts its eligible sentences only.  Every candidate leaf holds at least one, and counting the others
// would let A_k rise above the k-th best eligible score and drop leaves of the answer.
__device__ __forceinline__ int eligible_sentences(const FinArgs &a, int row, unsigned qtag) {
    int n = 0;
    for (int i = a.sent_off[row]; i < a.sent_off[row + 1]; i++) n += (a.sent_tags[a.sent_ids[i]] & qtag) != 0u;
    return n;
}
template <bool TAGGED>
__global__ void __launch_bounds__(FQ_WARPS * 32)
fn_line_kernel(const FinArgs a) {
    __shared__ float sa3_s[FQ_WARPS][KC1];
    __shared__ int sns_s[FQ_WARPS][KC1];
    __shared__ int spos_s[FQ_WARPS][MS], slen_s[FQ_WARPS][MS];
    __shared__ int counts[2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, ML = a.ix.max_len;
    float *sa3 = sa3_s[warp];
    int *sns = sns_s[warp], *spos = spos_s[warp], *slen = slen_s[warp];
    const float NEG_INF = -__int_as_float(0x7f800000);
    if (threadIdx.x < 2) counts[threadIdx.x] = 0;
    __syncthreads();
    const long long q = (long long)blockIdx.x * FQ_WARPS + warp;
    if (q < a.nq) {
        int *meta = a.meta + q * FM_STRIDE;
        const int nsel = meta[FM_NSEL];
        const float eps = __int_as_float(meta[FM_EPS]), U = __int_as_float(meta[FM_U]);
        int fail = meta[FM_FAIL];
        const int *rrow = a.ref_row + q * KC1;
        const unsigned qtag = TAGGED ? a.qtags[q] : 0u;
        for (int i = lane; i < nsel; i += 32) {
            const int row = rrow[i];
            const float4 r0 = a.leaf_rc[row * 2], r1 = a.leaf_rc[row * 2 + 1];
            const int par = __float_as_int(r1.y);
            const float c = par >= 0 ? a.C[(long long)par * a.ldq + q] : 0.0f;
            sa3[i] = __fmul_rn(__fmaf_rn(r1.z, a.ref_s[q * KC1 + i], c), r0.w);
            sns[i] = TAGGED ? eligible_sentences(a, row, qtag) : a.sent_off[row + 1] - a.sent_off[row];
        }
        __syncwarp();
        // A_k: the a3 of the leaf that holds the k-th sentence in (a3 desc, list position asc) order
        bool found = false;
        float Ak = 0.0f;
        for (int i = lane; i < nsel; i += 32) {
            const float v = sa3[i];
            int before = 0;
            for (int c = 0; c < nsel; c++)
                if (sa3[c] > v || (sa3[c] == v && c < i)) before += sns[c];
            if (before < a.k && before + sns[i] >= a.k) found = true, Ak = v;
        }
        const unsigned fm = __ballot_sync(0xffffffffu, found);
        const float thr = fm ? __shfl_sync(0xffffffffu, Ak, __ffs(fm) - 1) - 2.0f * eps : NEG_INF;
        // Everything unrefined scores (exactly) at most U + 2 eps, the k-th best exact score is at least A_k - eps: the
        // answer is complete if U + 3 eps < A_k.  With fewer than k sentences among the refined leaves every one of
        // them is needed and nothing may be left out (U = -inf).
        if (!(thr - eps > U) && !(U == NEG_INF)) fail = fail ? fail : 2;
        // survivors: refined leaves at or above the line, in list order
        int m = 0, n_sent = 0;
        for (int base = 0; base < nsel; base += 32) {
            const int i = base + lane;
            const bool surv = i < nsel && sa3[i] >= thr;
            const unsigned mask = __ballot_sync(0xffffffffu, surv);
            const int at = m + __popc(mask & ((1u << lane) - 1u));
            if (surv) {
                n_sent += sns[i];
                if (at < MS) {
                    meta[FM_SURV + at] = i;
                    const int row = rrow[i];
                    spos[at] = a.leaf_pos[row];
                    slen[at] = __float_as_int(a.leaf_rc[row * 2 + 1].w);
                }
            }
            m += __popc(mask);
        }
        n_sent = warp_sum(n_sent);
        if (m > MS || n_sent > MAXS) fail = fail ? fail : 3;
        if (lane == 0) { atomicAdd(&counts[0], nsel); atomicAdd(&counts[1], m); }
        int nanc = 0;
        if (fail) {  // flagged: the exact small-batch path answers this query
            if (lane == 0) {
                const int at = atomicAdd(a.flag, 1);
                a.flag[4 + at] = (int)q;
                a.out_sid[q * a.k] = CW_SID_UNRESOLVED;
                atomicAdd(a.stats + 0, 1);
                atomicAdd(a.stats + 1 + fail, 1);
            }
            m = -1;
        } else {
            // (survivor, level) -> index row of the ancestor; the first survivor through a node gives it an entry
            __syncwarp();
            int *ab = a.anc_b + q * a.em, *slot = a.anc_slot + q * a.em;
            const int *pidx = a.ix.path_idx;
            auto node = [&](int c, int j) { return j < slen[c] - 1 ? pidx[(size_t)spos[c] * ML + j] : -1; };
            const int E = m * ML;
            for (int base = 0; base < E; base += 32) {
                const int e = base + lane;
                int b = -1, f = 0, c = 0, j = 0;
                if (e < E) {
                    c = e / ML, j = e - c * ML;
                    b = node(c, j);
                    if (b >= 0)
                        while (node(f, j) != b) f++;  // first survivor through this node (f <= c)
                }
                const bool first = b >= 0 && f == c;
                const unsigned mask = __ballot_sync(0xffffffffu, first);
                if (first) {
                    const int sl = nanc + __popc(mask & ((1u << lane) - 1u));
                    ab[sl] = b;
                    slot[e] = sl;
                } else if (b >= 0) {
                    slot[e] = -2 - (f * ML + j);  // resolved below, once every first entry has its slot
                }
                nanc += __popc(mask);
            }
            __syncwarp();
            for (int e = lane; e < E; e += 32) {
                const int v = slot[e];
                if (v <= -2) slot[e] = slot[-2 - v];
            }
        }
        if (lane == 0) { meta[FM_NANC] = nanc; meta[FM_M] = m; }
    }
    __syncthreads();
    // leaves refined and leaves re-scored, flagged queries included
    if (threadIdx.x == 0 && (counts[0] | counts[1])) { atomicAdd(a.stats + 10, counts[0]); atomicAdd(a.stats + 11, counts[1]); }
}

// exact leaf scores of the survivors: sequential FMA along the path, root first, the leaf last (cw_dense_paths_topk's
// order); their sentences ranked by (score desc, sentence id asc).  TAGGED: their eligible sentences only.
template <bool TAGGED>
__global__ void __launch_bounds__(FQ_WARPS * 32)
fn_topk_kernel(const FinArgs a) {
    __shared__ int lsid_s[FQ_WARPS][MAXS];
    __shared__ float lval_s[FQ_WARPS][MAXS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, ML = a.ix.max_len;
    const long long q = (long long)blockIdx.x * FQ_WARPS + warp;
    if (q >= a.nq) return;
    const int *meta = a.meta + q * FM_STRIDE;
    const int m = meta[FM_M];
    if (m < 0) return;  // flagged
    int *lsid = lsid_s[warp];
    float *lval = lval_s[warp];
    const float NEG_INF = -__int_as_float(0x7f800000);
    int row = 0, ns = 0;
    float mex = 0.0f;
    const unsigned qtag = TAGGED ? a.qtags[q] : 0u;
    if (lane < m) {  // m <= MS = 32
        const int sel = meta[FM_SURV + lane];
        row = a.ref_row[q * KC1 + sel];
        const int len = __float_as_int(a.leaf_rc[row * 2 + 1].w);
        const int *slot = a.anc_slot + q * a.em + lane * ML;
        const float *as = a.anc_s + q * a.em;
        float acc = 0.0f;
#pragma unroll 1
        for (int j = 0; j < len - 1; j++) acc = __fmaf_rn((float)(a.ix.level_w[j] / (double)len), as[slot[j]], acc);
        mex = __fmaf_rn((float)(a.ix.level_w[len - 1] / (double)len), a.ref_s[q * KC1 + sel], acc);
        ns = TAGGED ? eligible_sentences(a, row, qtag) : a.sent_off[row + 1] - a.sent_off[row];
    }
    int off = ns;  // inclusive prefix sum of the sentence counts
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, off, d);
        if (lane >= d) off += o;
    }
    const int ns_tot = __shfl_sync(0xffffffffu, off, 31);
    off -= ns;
    for (int c = 0; c < m; c++) {
        const int s0 = __shfl_sync(0xffffffffu, row, c), cntc = __shfl_sync(0xffffffffu, ns, c),
                  o = __shfl_sync(0xffffffffu, off, c);
        const float v = __shfl_sync(0xffffffffu, mex, c);
        const int first = a.sent_off[s0];
        if (!TAGGED) {
            for (int i = lane; i < cntc; i += 32) { lsid[o + i] = a.sent_ids[first + i]; lval[o + i] = v; }
        } else {
            const int n_all = a.sent_off[s0 + 1] - first;
            int at = o;
            for (int base = 0; base < n_all; base += 32) {
                const int sid = base + lane < n_all ? a.sent_ids[first + base + lane] : -1;
                const bool ok = sid >= 0 && (a.sent_tags[sid] & qtag) != 0u;
                const unsigned mask = __ballot_sync(0xffffffffu, ok);
                if (ok) { const int i = at + __popc(mask & ((1u << lane) - 1u)); lsid[i] = sid; lval[i] = v; }
                at += __popc(mask);
            }
        }
    }
    __syncwarp();
    for (int i = lane; i < ns_tot; i += 32) {
        const float v = lval[i];
        const int sid = lsid[i];
        int rank = 0;
        for (int j = 0; j < ns_tot; j++) rank += lval[j] > v || (lval[j] == v && lsid[j] < sid);
        if (rank < a.k) { a.out_sid[q * a.k + rank] = sid; a.out_val[q * a.k + rank] = v; }
    }
    for (int r = ns_tot + lane; r < a.k; r += 32) {  // fewer than k sentences in the index
        a.out_sid[q * a.k + r] = -1;
        a.out_val[q * a.k + r] = NEG_INF;
    }
}

__global__ void h_unresolved_kernel(const int *flag, int capacity, int *stats) {
    if (flag[0] > capacity) atomicAdd(stats + 1, flag[0] - capacity);
}
// always-on audit: queries phase, phase + every, ... (at most n_a) are answered again by the exact path and compared
__global__ void h_audit_pick_kernel(int *which, int n_a, int every, int phase, long long nq) {
    const int i = threadIdx.x;
    if (i < n_a) {
        long long q = (long long)i * every + phase;
        which[i] = (int)(q < nq ? q : nq - 1);
    }
}
__global__ void h_audit_cmp_kernel(const int *__restrict__ which, int n_a, int k, const int *__restrict__ ex_sid,
                                   const float *__restrict__ ex_val, const int *__restrict__ out_sid,
                                   const float *__restrict__ out_val, int *stats) {
    const int i = threadIdx.x;
    if (i >= n_a) return;
    const long long q = which[i];
    bool same = true;
    for (int j = 0; j < k; j++)
        same = same && ex_sid[i * k + j] == out_sid[q * k + j] &&
               __float_as_int(ex_val[i * k + j]) == __float_as_int(out_val[q * k + j]);
    atomicAdd(stats + 8, 1);
    if (!same && out_sid[q * k] != CW_SID_UNRESOLVED) atomicAdd(stats + 9, 1);
}

// leaf_tags[r] = OR of the tags of leaf row r's sentences (torch has no scatter-OR)
__global__ void leaf_tags_kernel(const int *__restrict__ sent_off, const int *__restrict__ sent_ids, int n_leaf,
                                 const unsigned *__restrict__ sent_tags, unsigned *leaf_tags) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_leaf) return;
    unsigned t = 0u;
    for (int i = sent_off[r]; i < sent_off[r + 1]; i++) t |= sent_tags[sent_ids[i]];
    leaf_tags[r] = t;
}

}  // namespace cwh

using namespace cwh;

extern "C" int cw_leaf_tags(const int32_t *sent_off, const int32_t *sent_ids, int32_t n_leaf, const uint32_t *sent_tags,
                            uint32_t *leaf_tags, void *stream) {
    if (!sent_off || !sent_ids || !sent_tags || !leaf_tags || n_leaf < 0) {
        cw_set_error("cw_leaf_tags: bad argument");
        return CW_E_ARG;
    }
    if (n_leaf == 0) return 0;
    leaf_tags_kernel<<<(n_leaf + 255) / 256, 256, 0, (cudaStream_t)stream>>>(sent_off, sent_ids, n_leaf, sent_tags, leaf_tags);
    return cw_check_cuda(cudaGetLastError(), "cw_leaf_tags");
}

// fn_exact_kernel for other translation units (cw_pairs.cu); the attributes are per device, so they are set per call
int cw_exact_rows_attr() {
    int rc = cw_check_cuda(cudaFuncSetAttribute(fn_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                EX_WARPS * EX_WARP_BYTES), "cw_exact_rows: smem attribute");
    if (!rc)
        rc = cw_check_cuda(cudaFuncSetAttribute(fn_exact_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                                cudaSharedmemCarveoutMaxShared), "cw_exact_rows: carveout attribute");
    return rc;
}
void cw_exact_rows_launch(const cw_index &ix, const float2 *RM, const float *Q, long long nq, const int *list,
                          const int *meta, int meta_stride, int n_word, int stride, float *out, int row_blocks,
                          cudaStream_t st) {
    const dim3 grid((unsigned)((nq + EX_WARPS - 1) / EX_WARPS), (unsigned)row_blocks);
    fn_exact_kernel<<<grid, EX_WARPS * 32, EX_WARPS * EX_WARP_BYTES, st>>>(ix, RM, Q, nq, list, meta, meta_stride, n_word,
                                                                          stride, out);
}

extern "C" int64_t cw_fused_flag_words(int64_t cap_q, int32_t max_len) { return 4 + cap_q + CW_SMALL_Q + fin_words(cap_q, max_len); }
extern "C" int cw_h_stages(int32_t D, int32_t layout, int32_t nprod) { return stages_of(D, layout, nprod); }
extern "C" int64_t cw_h_b_bytes(int32_t n_rows, int32_t D, int32_t layout, int32_t nprod) {
    return (int64_t)((n_rows + TN - 1) / TN) * stages_of(D, layout, nprod) * SIDE;
}
extern "C" int64_t cw_h_a_bytes(int64_t nq, int32_t D, int32_t layout, int32_t nprod) {
    return ((nq + TQ - 1) / TQ) * (int64_t)stages_of(D, layout, nprod) * SIDE;
}

static bool set_ok(const cw_h_set *hs, int D) {
    return hs && hs->n_rows >= 1 && hs->n_ntiles == (hs->n_rows + TN - 1) / TN && (hs->nprod == 1 || hs->nprod == 3) &&
           (hs->layout == CW_H_F1 || hs->layout == CW_H_F2) && hs->n_stages == stages_of(D, hs->layout, hs->nprod) && hs->B && hs->rc;
}

extern "C" int cw_h_set_build(const cw_store *s, const int32_t *order, const int32_t *rows, const float *sumlog, const cw_h_set *hs,
                              const int32_t *int_parent, const float *int_w, const float *leaf_w, const float *leaf_inv_len,
                              const int32_t *leaf_parent, const int32_t *leaf_len, void *stream) {
    if (!s || !order || !rows || !sumlog || !set_ok(hs, s->D) ||
        (hs->nprod == 3 && (!int_parent || !int_w)) ||
        (hs->nprod == 1 && (int_parent || int_w || !leaf_w || !leaf_inv_len || !leaf_parent || !leaf_len))) {
        cw_set_error("cw_h_set_build: bad argument / inconsistent header");
        return CW_E_ARG;
    }
    const int n_pad = hs->n_ntiles * TN;
    hn_build_kernel<<<(n_pad + 7) / 8, 256, 0, (cudaStream_t)stream>>>(*s, order, rows, sumlog, *hs, int_parent, int_w, leaf_w,
                                                                      leaf_inv_len, leaf_parent, leaf_len);
    return cw_check_cuda(cudaGetLastError(), "cw_h_set_build");
}

extern "C" int cw_h_rows_isotropic(const cw_store *s, const int32_t *order, const int32_t *rows, int32_t n_rows, int32_t *flag_dev,
                                   void *stream) {
    if (!s || !order || !rows || !flag_dev || n_rows < 1) {
        cw_set_error("cw_h_rows_isotropic: bad argument");
        return -1;
    }
    cudaStream_t st = (cudaStream_t)stream;
    int one = 1, out = 0;
    if (cw_check_cuda(cudaMemcpyAsync(flag_dev, &one, sizeof(int), cudaMemcpyHostToDevice, st), "cw_h_rows_isotropic")) return -1;
    h_iso_kernel<<<(n_rows + 7) / 8, 256, 0, st>>>(*s, order, rows, n_rows, flag_dev);
    if (cw_check_cuda(cudaMemcpyAsync(&out, flag_dev, sizeof(int), cudaMemcpyDeviceToHost, st), "cw_h_rows_isotropic")) return -1;
    if (cw_check_cuda(cudaStreamSynchronize(st), "cw_h_rows_isotropic")) return -1;
    return out;
}

template <int NPROD, int MODE, bool HALF, bool TAGGED>
static int h_launch_t(const cw_h_set *hs, const void *A, int64_t nq, int nt_begin, int nt_count, const HEpi &epi, cudaStream_t st,
                      const cw_tag_filter *tf) {
    using K = KCfg<HALF>;
    const int n_qtiles = (int)((nq + K::TQK - 1) / K::TQK);
    auto kern = h_score_kernel<NPROD, MODE, HALF, TAGGED>;
    int rc = cw_check_cuda(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, K::SMEM), "cw_h: smem attribute");
    if (rc) return rc;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long n_tiles = (long long)n_qtiles * nt_count;
    if (n_tiles == 0) return 0;
    const int grid = (int)(n_tiles < (long long)sms * K::CTAS ? n_tiles : sms * K::CTAS);
    // query-tile panels: the panel's query operands should sit in L2 (~40 MB of it) while the row operands stream
    const long long a_tile = (long long)hs->n_stages * K::A_SIDE;
    int pq_max = (int)((40ll << 20) / a_tile);
    if (pq_max < 1) pq_max = 1;
    const int n_panels = (n_qtiles + pq_max - 1) / pq_max;
    const int pq = (n_qtiles + n_panels - 1) / n_panels;
    kern<<<grid, K::THR, K::SMEM, st>>>(reinterpret_cast<const unsigned char *>(A), reinterpret_cast<const unsigned char *>(hs->B),
                                        epi, n_qtiles, nt_begin, nt_count, hs->n_stages, pq, tf ? tf->query_tags : nullptr,
                                        tf ? tf->leaf_tags : nullptr);
    return cw_check_cuda(cudaGetLastError(), "cw_h: score kernel");
}
// the one-product kernels take half tiles (two CTAs per SM) unless COBWEB_B200_FULL_TILE=1 asks for the full ones;
// tf (leaf-row modes only): the tagged instantiation
template <int NPROD, int MODE>
static int h_launch(const cw_h_set *hs, const void *A, int64_t nq, int nt_begin, int nt_count, const HEpi &epi, cudaStream_t st,
                    const cw_tag_filter *tf = nullptr) {
    static const bool full_tile = getenv("COBWEB_B200_FULL_TILE") && atoi(getenv("COBWEB_B200_FULL_TILE")) != 0;
    if constexpr (MODE != EPI_NODE) {
        if (tf) {
            if (NPROD == 1 && !full_tile) return h_launch_t<NPROD, MODE, true, true>(hs, A, nq, nt_begin, nt_count, epi, st, tf);
            return h_launch_t<NPROD, MODE, false, true>(hs, A, nq, nt_begin, nt_count, epi, st, tf);
        }
    }
    if (NPROD == 1 && !full_tile) return h_launch_t<NPROD, MODE, true, false>(hs, A, nq, nt_begin, nt_count, epi, st, nullptr);
    return h_launch_t<NPROD, MODE, false, false>(hs, A, nq, nt_begin, nt_count, epi, st, nullptr);
}

int cw_small_predict_impl(const cw_index *ix, const float *Q, int64_t nq, const int32_t *which, const int32_t *n_dev,
                          int32_t which_off, int scatter, int k, float *sm_Q, float *sm_scores, int32_t *sm_scratch, int32_t *sm_sid,
                          float *sm_val, int32_t *sm_n, int32_t *out_sid, float *out_val, cudaStream_t st,
                          const cw_tag_filter *tf);

// one chunk of at most w->cap_q queries, all on the device
// ev (optional): CW_FUSED_STAGES + 1 events recorded at the stage boundaries (cw_fused_profile)
// tf (optional): the tagged form, tf->query_tags indexed like this chunk's Q
static int fused_chunk(const cw_fused_index *fi, const cw_fused_work *w, const float *Q, int64_t nq, int k, int32_t *out_sid,
                       float *out_val, cudaStream_t st, cudaEvent_t *ev = nullptr, const cw_tag_filter *tf = nullptr) {
    CwRange range("cw_fused_chunk");
    static const char *const stage_names[CW_FUSED_STAGES] = {"query_operands", "internal_scores", "cumulative_sums", "sample_threshold",
                                                              "leaf_filter", "finish", "fallback_audit"};
    int open_stage = -1;
    auto mark = [&](int i) {
        if (ev) cudaEventRecord(ev[i], st);
        if (open_stage >= 0) nvtxRangePop();
        open_stage = i < CW_FUSED_STAGES ? i : -1;
        if (open_stage >= 0) nvtxRangePushA(stage_names[i]);
    };
    struct StageCloser { int &s; ~StageCloser() { if (s >= 0) nvtxRangePop(); } } closer{open_stage};
    mark(0);
    const int D = fi->ix.D;
    const long long ldq = w->ldq;
    const long long n_pad = (nq + TQ - 1) / TQ * TQ;
    int rc;
    if ((rc = cw_check_cuda(cudaMemsetAsync(w->cnt, 0, (size_t)nq * sizeof(int), st), "cw_fused: memset"))) return rc;
    if ((rc = cw_check_cuda(cudaMemsetAsync(w->flag, 0, 4 * sizeof(int), st), "cw_fused: memset"))) return rc;
    float4 *qv = reinterpret_cast<float4 *>(w->qv);
    hq_build_kernel<<<(unsigned)((n_pad + 7) / 8), 256, 0, st>>>(Q, nq, n_pad, D, fi->leaves.layout,
                                                                fi->n_int ? reinterpret_cast<unsigned char *>(w->A_int) : nullptr,
                                                                reinterpret_cast<unsigned char *>(w->A_leaf), qv);
    mark(1);
    HEpi epi;
    epi.out = w->S;
    epi.ldq = ldq;
    epi.qv = qv;
    epi.C = w->S;
    epi.nq = nq;
    epi.slots = w->slots;
    epi.tau = w->tau;
    epi.cap = w->cap;
    epi.cnt = w->cnt;
    epi.cand_val = w->cand_val;
    epi.cand_row = w->cand_row;
    if (fi->n_int) {
        epi.rc = fi->internal.rc;
        epi.n_rows = fi->internal.n_rows;
        if ((rc = h_launch<3, EPI_NODE>(&fi->internal, w->A_int, nq, 0, fi->internal.n_ntiles, epi, st))) return rc;
    }
    mark(2);  // the internal operands are path sums: S holds the ancestor sums C already, this stage is empty
    mark(3);
    epi.rc = fi->leaves.rc;
    epi.n_rows = fi->leaves.n_rows;
    const float inv_prior = 1.0f / fi->prior_var;
    if (fi->n_sample_tiles > 0) {
        if ((rc = cw_check_cuda(cudaMemsetAsync(w->slots, 0x80, (size_t)nq * 32 * sizeof(int), st), "cw_fused: memset"))) return rc;
        if ((rc = h_launch<1, EPI_TAU>(&fi->leaves, w->A_leaf, nq, 0, fi->n_sample_tiles, epi, st, tf))) return rc;
        const int m = k + 2 < 32 ? k + 2 : 32;
        h_tau_kernel<<<(unsigned)((nq + 127) / 128), 128, 0, st>>>(w->slots, qv, nq, m, fi->e1max, inv_prior, fi->hmax, fi->lmax,
                                                                  fi->wfac, fi->eps_scale, fi->ix.max_len, w->tau);
    } else {
        h_fill_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, st>>>(w->tau, nq, -INFINITY);
    }
    mark(4);
    if ((rc = h_launch<1, EPI_FILTER>(&fi->leaves, w->A_leaf, nq, 0, fi->leaves.n_ntiles, epi, st, tf))) return rc;
    mark(5);
    FinArgs a;
    a.ix = fi->ix;
    a.RM = reinterpret_cast<const float2 *>(fi->rows);
    a.Q = Q;
    a.nq = nq;
    a.k = k;
    a.cap = w->cap;
    a.cnt = w->cnt;
    a.cand_val = w->cand_val;
    a.cand_row = w->cand_row;
    a.tau = w->tau;
    a.qv = qv;
    a.leaf_rc = reinterpret_cast<const float4 *>(fi->leaves.rc);
    a.leaf_row_b = fi->leaf_row_b;
    a.leaf_pos = fi->leaf_pos;
    a.sent_off = fi->sent_off;
    a.sent_ids = fi->sent_ids;
    a.C = w->S;
    a.ldq = ldq;
    a.inv_prior = inv_prior;
    a.hmax = fi->hmax;
    a.lmax = fi->lmax;
    a.wfac = fi->wfac;
    a.eps_scale = fi->eps_scale;
    a.out_sid = out_sid;
    a.out_val = out_val;
    a.flag = w->flag;
    a.stats = w->stats;
    a.qtags = tf ? tf->query_tags : nullptr;
    a.sent_tags = tf ? tf->sent_tags : nullptr;
    fin_carve(a, w->flag + 4 + w->cap_q + CW_SMALL_Q, w->cap_q, w->fin_ml);
    // the candidates of a select warp sit in shared memory: at most FQ_WARPS x 2048 x 12 bytes (fused_args_ok bounds cap)
    const int sel_smem = FQ_WARPS * w->cap * 12;
    if ((rc = cw_check_cuda(cudaFuncSetAttribute(fn_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, sel_smem),
                            "cw_fused: smem attribute")) ||
        (rc = cw_exact_rows_attr()))
        return rc;
    const unsigned gq = (unsigned)((nq + FQ_WARPS - 1) / FQ_WARPS);
    fn_select_kernel<<<gq, FQ_WARPS * 32, sel_smem, st>>>(a);
    cw_exact_rows_launch(a.ix, a.RM, Q, nq, a.ref_b, a.meta, FM_STRIDE, FM_NSEL, KC1, a.ref_s, 1, st);
    (tf ? fn_line_kernel<true> : fn_line_kernel<false>)<<<gq, FQ_WARPS * 32, 0, st>>>(a);
    cw_exact_rows_launch(a.ix, a.RM, Q, nq, a.anc_b, a.meta, FM_STRIDE, FM_NANC, a.em, a.anc_s, 1, st);
    (tf ? fn_topk_kernel<true> : fn_topk_kernel<false>)<<<gq, FQ_WARPS * 32, 0, st>>>(a);
    if ((rc = cw_check_cuda(cudaGetLastError(), "cw_fused_predict"))) return rc;
    mark(6);
    // flagged queries: exact small-batch path, driven by the device-side count
    for (int r = 0; r < CW_FUSED_FB_ROUNDS; r++) {
        if ((rc = cw_small_predict_impl(&fi->ix, Q, CW_SMALL_Q, w->flag + 4, w->flag, r * CW_SMALL_Q, 1, k, w->sm_Q, w->sm_scores,
                                        w->sm_scratch, w->sm_sid, w->sm_val, w->sm_n, out_sid, out_val, st, tf)))
            return rc;
    }
    h_unresolved_kernel<<<1, 1, 0, st>>>(w->flag, CW_FUSED_FB_ROUNDS * CW_SMALL_Q, w->stats);
    // The exact answer of even one query streams all node operands once, so the audit runs in one call out of
    // CW_FUSED_AUDIT_STRIDE with that many times the queries: the same audited fraction at a quarter of the cost.
    if (w->audit_every > 0 && w->audit_phase % CW_FUSED_AUDIT_STRIDE == 0) {
        // the audited queries' exact answers land in sm_sid / sm_val; their list sits behind the flagged queries
        long long every = w->audit_every / CW_FUSED_AUDIT_STRIDE;
        if (every < 1) every = 1;
        long long n_a = (nq + every - 1) / every;
        if (n_a > CW_SMALL_Q) n_a = CW_SMALL_Q;
        int *which = w->flag + 4 + w->cap_q;
        h_audit_pick_kernel<<<1, CW_SMALL_Q, 0, st>>>(which, (int)n_a, (int)every, (int)((w->audit_phase / CW_FUSED_AUDIT_STRIDE) % every), nq);
        if ((rc = cw_small_predict_impl(&fi->ix, Q, n_a, which, nullptr, 0, 0, k, w->sm_Q, w->sm_scores, w->sm_scratch, w->sm_sid,
                                        w->sm_val, w->sm_n, out_sid, out_val, st, tf)))
            return rc;
        h_audit_cmp_kernel<<<1, CW_SMALL_Q, 0, st>>>(which, (int)n_a, k, w->sm_sid, w->sm_val, out_sid, out_val, w->stats);
    }
    mark(7);
    return cw_check_cuda(cudaGetLastError(), "cw_fused_predict: tail");
}

static bool fused_args_ok(const cw_fused_index *fi, const cw_fused_work *w, int k) {
    if (!fi || !w || k < 1 || k > CW_FUSED_MAX_K || fi->n_leaf < 1 || fi->ix.n_pos < 1 || !fi->ix.path_idx || !fi->ix.level_w ||
        !fi->ix.sumlog || !fi->rows || !fi->leaf_row_b || !fi->leaf_pos || !fi->sent_off || !fi->sent_ids)
        return false;
    if (reinterpret_cast<uintptr_t>(fi->rows) % 16) return false;  // fn_exact_kernel's bulk copies
    if (!set_ok(&fi->leaves, fi->ix.D) || fi->leaves.nprod != 1 || fi->leaves.n_rows != fi->n_leaf) return false;
    if (fi->n_int && (!set_ok(&fi->internal, fi->ix.D) || fi->internal.nprod != 3 || fi->internal.layout != CW_H_F2 ||
                      fi->internal.n_rows != fi->n_int))
        return false;
    if (fi->n_sample_tiles < 0 || fi->n_sample_tiles > fi->leaves.n_ntiles) return false;
    if (w->cap_q < TQ || (w->cap_q % TQ) || w->ldq != w->cap_q || !w->A_leaf || (fi->n_int && (!w->A_int || !w->S)) || !w->qv ||
        !w->slots || !w->tau || w->cap < 4 || w->cap > 2048 || (w->cap & 3) || !w->cnt || !w->cand_val || !w->cand_row || !w->flag || !w->sm_Q ||
        !w->sm_scores || !w->sm_scratch || !w->sm_sid || !w->sm_val || !w->sm_n || !w->stats ||
        w->fin_ml < fi->ix.max_len)
        return false;
    return true;
}

extern "C" int cw_fused_predict(const cw_fused_index *fi, const cw_fused_work *w, const float *Q, int64_t nq, int k,
                                int32_t *out_sid, float *out_val, void *stream) {
    if (!fused_args_ok(fi, w, k) || !Q || !out_sid || !out_val || nq < 0) {
        cw_set_error("cw_fused_predict: bad argument (k=%d, 1..%d)", k, CW_FUSED_MAX_K);
        return CW_E_ARG;
    }
    for (int64_t lo = 0; lo < nq; lo += w->cap_q) {
        const int64_t n = nq - lo < w->cap_q ? nq - lo : w->cap_q;
        int rc = fused_chunk(fi, w, Q + lo * fi->ix.D, n, k, out_sid + lo * k, out_val + lo * k, (cudaStream_t)stream);
        if (rc) return rc;
    }
    return 0;
}

// Tagged form: the chunks take their slice of the query masks; flagged and audited queries run the tagged small path
extern "C" int cw_fused_predict_tagged(const cw_fused_index *fi, const cw_fused_work *w, const cw_tag_filter *tf, const float *Q,
                                       int64_t nq, int k, int32_t *out_sid, float *out_val, void *stream) {
    if (!fused_args_ok(fi, w, k) || !tf || !tf->query_tags || !tf->pos_tags || !tf->leaf_tags || !tf->sent_tags || !Q || !out_sid ||
        !out_val || nq < 0) {
        cw_set_error("cw_fused_predict_tagged: bad argument (k=%d, 1..%d; every tag array is needed)", k, CW_FUSED_MAX_K);
        return CW_E_ARG;
    }
    for (int64_t lo = 0; lo < nq; lo += w->cap_q) {
        const int64_t n = nq - lo < w->cap_q ? nq - lo : w->cap_q;
        cw_tag_filter t = *tf;
        t.query_tags = tf->query_tags + lo;
        int rc = fused_chunk(fi, w, Q + lo * fi->ix.D, n, k, out_sid + lo * k, out_val + lo * k, (cudaStream_t)stream, nullptr, &t);
        if (rc) return rc;
    }
    return 0;
}

extern "C" int cw_fused_predict_host(const cw_fused_index *fi, const cw_fused_work *w, const float *Q_host, int64_t nq, int k,
                                     int32_t *out_sid_host, float *out_val_host, int32_t *stats_host, void *stream) {
    if (!fused_args_ok(fi, w, k) || !Q_host || !out_sid_host || !out_val_host || nq < 0 || !w->Q_dev || !w->out_sid_dev ||
        !w->out_val_dev) {
        cw_set_error("cw_fused_predict_host: bad argument (k=%d, 1..%d)", k, CW_FUSED_MAX_K);
        return CW_E_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int D = fi->ix.D;
    int rc = cw_check_cuda(cudaMemsetAsync(w->stats, 0, CW_FUSED_STATS * sizeof(int), st), "cw_fused_predict_host: memset");
    if (rc) return rc;
    int32_t stats[CW_FUSED_STATS] = {0};
    for (int64_t lo = 0; lo < nq; lo += w->cap_q) {
        const int64_t n = nq - lo < w->cap_q ? nq - lo : w->cap_q;
        if ((rc = cw_check_cuda(cudaMemcpyAsync(w->Q_dev, Q_host + lo * D, (size_t)n * D * sizeof(float), cudaMemcpyHostToDevice, st),
                                "cw_fused_predict_host: H2D")))
            return rc;
        if ((rc = fused_chunk(fi, w, w->Q_dev, n, k, w->out_sid_dev, w->out_val_dev, st))) return rc;
        int32_t n_flag = 0;
        const bool last = lo + w->cap_q >= nq;
        if ((rc = cw_check_cuda(cudaMemcpyAsync(out_sid_host + lo * k, w->out_sid_dev, (size_t)n * k * sizeof(int32_t),
                                                cudaMemcpyDeviceToHost, st), "cw_fused_predict_host: D2H ids")))
            return rc;
        if ((rc = cw_check_cuda(cudaMemcpyAsync(out_val_host + lo * k, w->out_val_dev, (size_t)n * k * sizeof(float),
                                                cudaMemcpyDeviceToHost, st), "cw_fused_predict_host: D2H scores")))
            return rc;
        if ((rc = cw_check_cuda(cudaMemcpyAsync(&n_flag, w->flag, sizeof(int32_t), cudaMemcpyDeviceToHost, st),
                                "cw_fused_predict_host: D2H flag count")))
            return rc;
        if (last && (rc = cw_check_cuda(cudaMemcpyAsync(stats, w->stats, sizeof(stats), cudaMemcpyDeviceToHost, st),
                                        "cw_fused_predict_host: D2H stats")))
            return rc;
        // the work buffers are re-used by the next chunk, so every chunk ends with the one synchronisation
        if ((rc = cw_check_cuda(cudaStreamSynchronize(st), "cw_fused_predict_host: sync"))) return rc;
        if (n_flag > CW_FUSED_FB_ROUNDS * CW_SMALL_Q) {  // more flagged queries than the device-side rounds take: finish them now
            for (int off = CW_FUSED_FB_ROUNDS * CW_SMALL_Q; off < n_flag; off += CW_SMALL_Q)
                if ((rc = cw_small_predict_impl(&fi->ix, w->Q_dev, CW_SMALL_Q, w->flag + 4, w->flag, off, 1, k, w->sm_Q, w->sm_scores,
                                                w->sm_scratch, w->sm_sid, w->sm_val, w->sm_n, w->out_sid_dev, w->out_val_dev, st,
                                                nullptr)))
                    return rc;
            cudaMemcpyAsync(out_sid_host + lo * k, w->out_sid_dev, (size_t)n * k * sizeof(int32_t), cudaMemcpyDeviceToHost, st);
            cudaMemcpyAsync(out_val_host + lo * k, w->out_val_dev, (size_t)n * k * sizeof(float), cudaMemcpyDeviceToHost, st);
            if ((rc = cw_check_cuda(cudaStreamSynchronize(st), "cw_fused_predict_host: fallback sync"))) return rc;
        }
    }
    if (stats_host)
        for (int i = 0; i < CW_FUSED_STATS; i++) stats_host[i] = stats[i];
    return 0;
}

// One chunk with CUDA events at the stage boundaries; synchronises.  stage_ms[CW_FUSED_STAGES]: query operands,
// internal-row scores (fp16 x3, the ancestor sums), cumulative sums (empty: kept so the stage list stays the same),
// sampled tiles + threshold, leaf filter (fp16 x1), finish (select /
// refine / line test / exact re-score / top-k), tail (device-side fallback rounds, audit).
extern "C" int cw_fused_profile(const cw_fused_index *fi, const cw_fused_work *w, const float *Q, int64_t nq, int k,
                                int32_t *out_sid, float *out_val, float *stage_ms_host, void *stream) {
    if (!fused_args_ok(fi, w, k) || !Q || !out_sid || !out_val || !stage_ms_host || nq < 1 || nq > w->cap_q) {
        cw_set_error("cw_fused_profile: bad argument (one chunk: nq <= cap_q)");
        return CW_E_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    cudaEvent_t ev[CW_FUSED_STAGES + 1];
    for (auto &e : ev) cudaEventCreate(&e);
    int rc = fused_chunk(fi, w, Q, nq, k, out_sid, out_val, st, ev);
    if (!rc) rc = cw_check_cuda(cudaStreamSynchronize(st), "cw_fused_profile: sync");
    for (int i = 0; i < CW_FUSED_STAGES && !rc; i++) cudaEventElapsedTime(stage_ms_host + i, ev[i], ev[i + 1]);
    for (auto &e : ev) cudaEventDestroy(e);
    return rc;
}
