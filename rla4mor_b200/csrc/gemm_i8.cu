// gemm_i8.cu -- dense embeddings of FLOAT64 blocks on the int8 tensor cores (Ozaki scheme I):
//   Y(m, k) = U(m, n) * Theta(k, n)^T,  U float64, Theta (kinds 0 and 2) generated in the kernel.
//
// FP64 has no tcgen05 kind; kind::i8 accumulates in int32, exactly.  Both operands are split into
// IS = 8 signed int8 slices of 7 bits, and the products of slice pairs (i, j) with i + j < IS are
// summed exactly on the tensor cores (36 MMAs per step instead of one DMMA-equivalent).
//
// Slicing.  U is cut into exponent blocks of IL = 2^14 consecutive columns (b = j / IL, counted from
// the first column of the block handed in).  For row c and block b, e = e(c, b) is the smallest
// integer with max_j |U[c, j]| < 2^e (e = 0 for an all-zero block); x = U 2^-e is in (-1, 1).  Theta
// entries are FP32 values with |theta| < 8 (Box-Muller with u1 >= 2^-33: r <= 6.8), so t = theta / 8
// is in (-1, 1) with one fixed exponent.  A value v in (-1, 1) is written as the truncation of
// |v| 2^56 to an integer M < 2^56, whose 7-bit digits d_s = (M >> 7 (7 - s)) & 127 carry the sign
// of v: v = sum_s d_s 2^-7(s+1) + r_8(v), |r_k(v)| < 2^-7k (residual after k digits).  The slices of
// U are written by a pre-pass (slice_u_kernel: one read of U, 8 bytes per element of workspace,
// plus e(c, b)); those of Theta are made by the producer warps from the one draw of each entry.
//
// Accumulators.  All pairs of one level l = i + j have the weight 2^(e + 3 - 7 (l + 2)), so they share
// one int32 accumulator in TMEM: IS levels x 64 sketch columns = 512 columns (all of TMEM).  Level l
// holds at most 8 pairs, |d_i d_j| <= 127^2, and a block has at most IL terms:
//   8 * 127^2 * 2^14 = 2 114 060 288 < 2^31 - 1   (no overflow).
// At the end of each exponent block the flush warps read the IS levels of their lane (lane = row c
// of U, so e(c, b) is a per-thread scalar), form t = D_0 + 2^-7 (D_1 + 2^-7 (... D_7)) with one FMA per
// level (FP64), and add ldexp(t, e - 11) into FP64 registers; blocks in order, then the split-n
// partials in chunk order (gemm_reduce_kernel of gemm.cu).  No atomics: bit-identical run to run.
//
// Accuracy contract (every element y_ci = sum_j U[c, j] Theta[i, j]; L = min(IL, n), n_b blocks):
//   For one term with x = u 2^-e, t = theta / 8, the kept product P = sum_{i+j<8} x_i t_j satisfies
//   x t - P = r_8(x) t + sum_{i=0..7} x_i r_{8-i}(t), with |x_0| <= |x| and |x_i| < 2^-7i, so
//   |x t - P| < 2^-56 (|t| + |x| + 7)  and  |u theta - 2^(e+3) P| < 2^(e-53) (|theta| / 8 + |u| 2^-e + 7).
//   Summed over a block with 2^e <= 2 max|u| <= 2 ||u_b||_2 and Cauchy-Schwarz (sum |theta| <= sqrt(L)
//   ||theta_b||, sum |u| <= sqrt(L) ||u_b||), then over the blocks (sum_b ||u_b|| <= sqrt(n_b) ||u||):
//     |yhat - y| <= 2^-53 sqrt(L) ||u_c||_2 (||theta_i||_2 / 4 + 15 sqrt(n))
//                   + (n_b + 10) 2^-52 ||u_c||_2 ||theta_i||_2 + 2^-1073 n_b
//   (second term: the FP64 roundings of the flush, the block sum and the chunk sum; third: one
//   rounding per block when ldexp(t, e - 11) is subnormal).  For a Gaussian Theta ||theta_i|| ~ sqrt(n),
//   so the first term is ~ 2^-49 sqrt(L) ||u|| ||theta||, i.e. C ~ 2 against 2^-50 sqrt(L) ||u|| ||theta||,
//   whatever the dynamic range of U.  The DMMA path satisfies the classical componentwise bound
//   |yhat - y| <= gamma_n sum_j |u_j| |theta_j| (gamma_n = n 2^-53 / (1 - n 2^-53)), normwise
//   gamma_n ||u|| ||theta||; at the n of a sketch (n >= 15 sqrt(L) ~ 2 000) the bound above is the
//   tighter of the two normwise bounds.  What is NOT kept: the componentwise bound in sum |theta| |u|
//   -- an entry far below the maximum of its block loses its low bits.
// Blocks with a non-finite entry or an entry >= 2^900 are not sliced: the pre-pass raises a flag
// and the caller (rla_embed_apply_rng_f64) runs the DMMA path, so NaN / Inf semantics are those of
// FP64 arithmetic.
//
// One CTA per SM, 128 x 64 tile of Y over one chunk of whole exponent blocks, 16 warps:
//   warps 0..7   flush: tcgen05.ld of the 8 levels (x16 per step), FP64 accumulation (32 columns each)
//   warps 8..13  producers: the 64 x 32 Theta tile of the stage (Philox + Box-Muller, rng.cuh), its
//                8 slices written straight into the 32-byte-swizzled K-major layout
//   warp 14      bulk copy of the 8 U slices of the stage (32 KB, contiguous in the workspace)
//   warp 15      MMA: one thread issues the 36 slice products of a stage as 12 tcgen05.mma.kind::i8
//                (M = 128, K = 32, N = 64 (8 - i) split at 256: U slice i against B slices 0 .. 7 - i)
// Cluster pairs along m share the Theta tile as in gemm32.cu: each CTA generates 32 of its 64 rows and
// pushes their slices to the peer (DSMEM bulk copies that signal the peer's full barrier).
// Measured on one B200 (1000 W limit), C2 shape (2^22 x 512, k = 2000): 146 ms per step (this kernel
// 126 ms), the board at its power cap (sw_power_cap, ~995 W) -- FP64 DMMA: 240 ms.  The same products
// as 36 MMAs of N = 64 took 160 ms per step: the MMAs cost per instruction, about 60 cycles for one of
// 128 x 64 x 32 (tools/micro/i8_probe.cu).  Dead ends: U slices read with a 3-D TMA box of 32-byte
// rows, 390 ms (hence the pre-pass writes each stage's 32 KB contiguously); clusters of four CTAs
// sharing Theta (16 rows each), 174 ms; the 36 MMAs with A-collector reuse and the pair as one 2-CTA
// MMA (M = 256, no DSMEM push), 157 ms.
#include "common.cuh"
#include "rng.cuh"
#include <algorithm>

namespace rla {

constexpr int IS = 8;                         // slices per operand = accumulator levels
constexpr int IL = 1 << 14;                   // exponent block = flush period (columns of U)
constexpr int IK = 32;                        // int8 per row per stage (32 bytes = swizzle span = MMA K)
constexpr int IBM = 128, IBN = 64;
constexpr int ISTAGES = 4;
constexpr int IFLUSH = 8, IPROD = 6;          // warps
constexpr int ITHREADS = (IFLUSH + IPROD + 2) * 32;
constexpr int IA_SLICE = IBM * IK, IB_SLICE = IBN * IK;
constexpr int IA_BYTES = IS * IA_SLICE, IB_BYTES = IS * IB_SLICE;
constexpr int ISTAGE_BYTES = IA_BYTES + IB_BYTES;          // 48 KB
constexpr int ISPB = IL / IK;                              // stages per exponent block
constexpr int I_TMEM_COLS = IS * IBN;                      // 512
constexpr int IE_MAX = 900;                                // blocks with max |u| >= 2^IE_MAX go to DMMA
static_assert((int64_t)8 * 127 * 127 * IL < (int64_t(1) << 31), "int32 accumulator overflow");
static_assert(I_TMEM_COLS <= 512, "TMEM");

namespace {

__device__ __forceinline__ uint32_t s32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(s32(bar)), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void bulk_load(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(s32(dst)), "l"(src), "r"(bytes), "r"(s32(bar)) : "memory");
}
// K-major operand tile in the canonical 32-byte-swizzle layout: rows of 32 bytes whose two 16-byte
// halves swap places in rows 4..7 of every 8 (byte address bit 4 ^= bit 7), groups of 8 rows 256 bytes
// apart (cute::UMMA::SmemDescriptor, version 1, layout 6)
__device__ __forceinline__ uint64_t desc_sw32(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (uint64_t(1) << 16) | (uint64_t(256 >> 4) << 32) |
           (uint64_t(1) << 46) | (uint64_t(6) << 61);
}
// D (int32, TMEM) (+)= A (s8, smem) * B (s8, smem)^T.  COLL, the A collector: 0 A read from shared
// memory; 1 read and kept (fill); 3 the kept A, for the last time (lastuse)
#define RLA_UMMA_I8(QUAL)                                                                              \
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::i8" QUAL " [%0], %1, %2, %3, p;\n\t}" \
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory")
template <int COLL>
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    static_assert(COLL == 0 || COLL == 1 || COLL == 3, "collector mode");
    if constexpr (COLL == 0) RLA_UMMA_I8("");
    else if constexpr (COLL == 1) RLA_UMMA_I8(".collector::a::fill");
    else RLA_UMMA_I8(".collector::a::lastuse");
}
#undef RLA_UMMA_I8
// The 36 slice products of one stage as 12 MMAs.  The products A_i B_j (j = 0 .. IS - 1 - i) go to
// levels i .. IS - 1, which are consecutive 64-column groups of TMEM, and the B slices B_j are
// consecutive 64-row groups of one K-major tile; so one MMA with N = 64 (IS - i) does them all, split
// at the N <= 256 of the instruction (a second part reuses A from the collector).  Every level is first
// written at i = 0.  The sums per level are exact int32 sums: the order does not change the result.
template <int I = 0>
__device__ __forceinline__ void stage_mmas(uint32_t tmem_base, uint32_t a_addr, uint32_t b_addr, bool first) {
    if constexpr (I < IS) {
        constexpr int NS = IS - I;                       // B slices this U slice meets
        constexpr int N0 = NS < 4 ? NS : 4, N1 = NS - N0;    // slices per MMA (N = 64 per slice, <= 256)
        // kind::i8, int32 accumulate, A and B signed and K-major, M = 128 (cute::UMMA::InstrDescriptor)
        constexpr uint32_t id_base = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(IBM >> 4) << 24);
        constexpr uint32_t id0 = id_base | ((uint32_t)(N0 * IBN >> 3) << 17), id1 = id_base | ((uint32_t)(N1 * IBN >> 3) << 17);
        const uint32_t acc = (first && I == 0) ? 0u : 1u;
        const uint64_t adesc = desc_sw32(a_addr + I * IA_SLICE);
        umma_i8<N1 ? 1 : 0>(tmem_base + (uint32_t)(I * IBN), adesc, desc_sw32(b_addr), id0, acc);
        if constexpr (N1 > 0)
            umma_i8<3>(tmem_base + (uint32_t)((I + N0) * IBN), adesc, desc_sw32(b_addr + N0 * IB_SLICE), id1, acc);
        stage_mmas<I + 1>(tmem_base, a_addr, b_addr, first);
    }
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s32(bar)) : "memory");
}
// the same arrive on the barrier at this offset in every CTA of the cluster (mask of ranks)
__device__ __forceinline__ void umma_commit_all(uint64_t *bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(s32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ uint32_t mapa(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void dsmem_push(uint32_t dst_cluster_addr, uint32_t src_cta_addr, uint32_t bytes, uint32_t bar_cluster_addr) {
    asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst_cluster_addr), "r"(src_cta_addr), "r"(bytes), "r"(bar_cluster_addr) : "memory");
}
__device__ __forceinline__ uint32_t ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// trunc(|v| 2^(56 - e)) for a float64 v with |v| < 2^e
__device__ __forceinline__ uint64_t fix56_f64(double v, int e) {
    const uint64_t b = (uint64_t)__double_as_longlong(v);
    int ex = (int)((b >> 52) & 0x7ff);
    uint64_t mant = b & ((uint64_t(1) << 52) - 1);
    if (ex == 0) ex = 1; else mant |= uint64_t(1) << 52;
    const int sh = ex - 1019 - e;                              // |v| = mant 2^(ex - 1075)
    return sh >= 0 ? mant << sh : (sh > -64 ? mant >> -sh : 0);
}
// trunc(|theta| 2^53) = trunc(|theta / 8| 2^56) for an FP32 theta with |theta| < 8
__device__ __forceinline__ uint64_t fix56_theta(float v) {
    const uint32_t b = __float_as_uint(v);
    int ex = (int)((b >> 23) & 0xff);
    uint64_t mant = b & 0x7fffffu;
    if (ex == 0) ex = 1; else mant |= 0x800000u;
    const int sh = ex - 97;                                    // |v| = mant 2^(ex - 150)
    return sh >= 0 ? mant << sh : (sh > -64 ? mant >> -sh : 0);
}
// digit s (7 bits, s = 0 most significant) of M as a signed byte with the sign of the value
__device__ __forceinline__ uint32_t digit(uint64_t M, int s, uint32_t neg) {
    const uint32_t d = (uint32_t)(M >> (7 * (IS - 1 - s))) & 127u;
    return ((d ^ neg) - neg) & 0xffu;                          // neg = 0 or 0xffffffff
}

}  // namespace

struct GemmI8Args {
    int64_t m, k, n;
    int64_t bpc;              // exponent blocks per chunk
    int64_t nb;               // exponent blocks of n
    int mtiles, ntiles;
    double *ws;               // [nchunks][m][k] partial sketches
    const int *expo;          // [m][nb] e(c, b)
    const unsigned char *slices;   // U slices, layout of slice_u_kernel
    uint64_t seed;
    int64_t row0, col0;
};

// one CTA per (row c, exponent block b): e(c, b) and the IS slices of U[c, b IL .. + IL)
// slices: [m tile][stage][IS][128 rows][32 bytes], each row 32-byte swizzled: the 32 KB a stage of the
// GEMM needs are one contiguous bulk copy (a 3-D TMA box of 32-byte rows ran at a fraction of the
// rate).  Columns from n to the end of the last stage are zero; rows of the last m tile beyond m are
// never written (they only feed sketch rows that are not stored).
// A non-finite entry or max |u| >= 2^IE_MAX sets *flag.
__global__ void __launch_bounds__(256) slice_u_kernel(const double *__restrict__ u, int64_t ldu, int64_t m, int64_t n,
                                                      int64_t nb, int64_t nst, uint32_t *__restrict__ slices,
                                                      int *__restrict__ expo, int *__restrict__ flag) {
    const int64_t c = blockIdx.x / nb, b = blockIdx.x % nb;
    const int64_t j0 = b * IL, j1 = min(n, j0 + IL);
    const double *row = u + c * ldu;
    unsigned long long mx = 0;
    for (int64_t j = j0 + threadIdx.x; j < j1; j += 256)
        mx = max(mx, (unsigned long long)__double_as_longlong(row[j]) & 0x7fffffffffffffffull);
#pragma unroll
    for (int o = 16; o; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    __shared__ unsigned long long red[8];
    __shared__ int e_s;
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) mx = max(mx, red[w]);
        int e = 0;
        if (mx != 0) {
            const int ex = (int)(mx >> 52);
            const unsigned long long sig = ex ? ((mx & ((1ull << 52) - 1)) | (1ull << 52)) : mx;
            e = (64 - __clzll((long long)sig)) + max(ex, 1) - 1075;   // smallest e with max < 2^e
        }
        if (mx >= 0x7ff0000000000000ull || e > IE_MAX) *flag = 1;
        expo[c * nb + b] = e;
        e_s = e;
    }
    __syncthreads();
    const int e = e_s;
    // four consecutive columns per thread and step: one 32-bit word of 4 digits per slice
    const int64_t jend = min(nst * IK, j0 + IL);
    const int r = (int)(c % IBM);
    uint32_t *tile = slices + (c / IBM) * nst * (IS * IA_SLICE / 4) + r * (IK / 4);
    for (int64_t j = j0 + 4 * (int64_t)threadIdx.x; j < jend; j += 4 * 256) {
        uint32_t w[IS];
#pragma unroll
        for (int s = 0; s < IS; ++s) w[s] = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const double v = (j + q < j1) ? row[j + q] : 0.0;
            const uint64_t M = fix56_f64(v, e);
            const uint32_t neg = (__double_as_longlong(v) < 0) ? 0xffffffffu : 0u;
#pragma unroll
            for (int s = 0; s < IS; ++s) w[s] |= digit(M, s, neg) << (8 * q);
        }
#pragma unroll
        for (int s = 0; s < IS; ++s)
            tile[(j / IK) * (IS * IA_SLICE / 4) + s * (IA_SLICE / 4) + (((int)(j % IK) >> 4) ^ ((r >> 2) & 1)) * 4 + ((j & 15) >> 2)] = w[s];
    }
}

template <int KIND, int CL>
__global__ void __launch_bounds__(ITHREADS, 1)
sketch_gemm_i8_kernel(const GemmI8Args a) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    __shared__ __align__(8) uint64_t full[ISTAGES], empty[ISTAGES], tmem_full, tmem_empty;
    __shared__ uint32_t tmem_base_s;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // blockIdx.x = rank + CL * (ntile + ntiles * (mgroup + mgroups * chunk))
    const uint32_t rank = (CL > 1) ? ctarank() : 0u;
    int64_t bx = blockIdx.x / CL;
    const int ntile = (int)(bx % a.ntiles); bx /= a.ntiles;
    const int mgrp = a.mtiles / CL;
    const int mtile = (int)(bx % mgrp) * CL + (int)rank; bx /= mgrp;
    const int64_t chunk = bx;
    const int64_t blk0 = chunk * a.bpc;                          // first exponent block of the chunk
    const int64_t kb0 = blk0 * ISPB;                             // first stage
    const int64_t nst = (a.n + IK - 1) / IK;
    const int64_t kb1 = (kb0 + a.bpc * ISPB < nst) ? kb0 + a.bpc * ISPB : nst;
    const int iters = (int)(kb1 - kb0);
    const int nblk = (iters + ISPB - 1) / ISPB;
    const int m0 = mtile * IBM, n0 = ntile * IBN;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < ISTAGES; ++s) {
            mbar_init(&full[s], 2 + (CL > 1 ? 1 : 0));    // U bulk copy expect_tx + producers + expect_tx of the peer's rows
            mbar_init(&empty[s], CL);                     // the MMA warps of every CTA of the cluster
        }
        mbar_init(&tmem_full, 1);
        mbar_init(&tmem_empty, IFLUSH);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(&tmem_base_s)), "r"(I_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_before();
    if (CL > 1) cluster_sync(); else __syncthreads();
    fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (warp < IFLUSH) {
        // ------------------------------------------------------------ flush warps
        asm volatile("setmaxnreg.inc.sync.aligned.u32 176;");
        const int q = warp & 3, h = warp >> 2;            // TMEM lane quarter (= warp % 4), 32-column half
        const int64_t row = m0 + 32 * q + lane;
        double acc[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[j] = 0.0;
        for (int bi = 0; bi < nblk; ++bi) {
            const int sc = (row < a.m ? a.expo[row * a.nb + blk0 + bi] : 0) - 11;   // weight of level 0: 2^(e + 3 - 14)
            mbar_wait(&tmem_full, (uint32_t)bi & 1u);
            fence_after();
            double t[2][16];
#pragma unroll
            for (int g = 0; g < 2; ++g) {
#pragma unroll
                for (int l = IS - 1; l >= 0; --l) {
                    uint32_t v[16];
                    const uint32_t taddr = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(l * IBN + 32 * h + 16 * g);
                    asm volatile(
                        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                        : "r"(taddr) : "memory");
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        t[g][j] = (l == IS - 1) ? (double)(int)v[j] : fma(t[g][j], 0x1p-7, (double)(int)v[j]);
                }
            }
            // every level is in registers: the accumulators can take the MMAs of the next block
            fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty);
#pragma unroll
            for (int g = 0; g < 2; ++g)
#pragma unroll
                for (int j = 0; j < 16; ++j) acc[16 * g + j] += ldexp(t[g][j], sc);
        }
        if (row < a.m) {
            double *wsp = a.ws + (chunk * a.m + row) * a.k;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int64_t col = n0 + 32 * h + j;
                if (col < a.k) wsp[col] = acc[j];
            }
        }
    } else if (warp < IFLUSH + IPROD) {
        // ------------------------------------------------------------ producers
        asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
        const int p = tid - IFLUSH * 32;
        constexpr int NPT = IPROD * 32;                    // a multiple of 8: an item's quad is p & 7 for every j
        // Theta tile: 64 rows x 8 quads of four entries; this CTA generates rows [rank ROWS, + ROWS)
        constexpr int ROWS = IBN / CL;
        constexpr int NJ = (ROWS * 8 + NPT - 1) / NPT;
        const int c = p & 7;
        uint64_t qv = ((uint64_t)(a.col0 + kb0 * IK) >> 2) + (uint64_t)c;
        for (int it = 0; it < iters; ++it, qv += IK / 4) {
            const int s = it % ISTAGES;
            if (it >= ISTAGES) mbar_wait(&empty[s], (uint32_t)((it / ISTAGES) - 1) & 1u);
            unsigned char *stb = smem + s * ISTAGE_BYTES + IA_BYTES;
            if (CL > 1 && p == 0) mbar_expect_tx(&full[s], (CL - 1) * IS * ROWS * IK);
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                const int rl = (p + NPT * j) >> 3;
                const int r = (int)rank * ROWS + rl;       // row inside the tile
                if (rl < ROWS && n0 + r < a.k) {
                    float f[4];
                    theta4f<KIND>(a.seed, (uint32_t)(a.row0 + n0 + r), qv, f);
                    uint32_t w[IS];
#pragma unroll
                    for (int sl = 0; sl < IS; ++sl) w[sl] = 0;
#pragma unroll
                    for (int e4 = 0; e4 < 4; ++e4) {
                        const uint64_t M = fix56_theta(f[e4]);
                        const uint32_t neg = (__float_as_uint(f[e4]) >> 31) ? 0xffffffffu : 0u;
#pragma unroll
                        for (int sl = 0; sl < IS; ++sl) w[sl] |= digit(M, sl, neg) << (8 * e4);
                    }
                    const int off = r * IK + (((c >> 2) ^ ((r >> 2) & 1)) << 4) + (c & 3) * 4;   // 32-byte swizzle
#pragma unroll
                    for (int sl = 0; sl < IS; ++sl) *reinterpret_cast<uint32_t *>(stb + sl * IB_SLICE + off) = w[sl];
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");    // generic writes -> async proxy
            asm volatile("bar.sync 1, %0;" ::"n"(NPT) : "memory");
            if (CL > 1 && p < IS * (CL - 1)) {
                // thread p pushes slice p % IS of this CTA's rows to the (p / IS + 1)-th next rank
                const uint32_t dst = (rank + 1u + (uint32_t)(p / IS)) % CL;
                const uint32_t off = (uint32_t)(s * ISTAGE_BYTES + IA_BYTES + (p % IS) * IB_SLICE + (int)rank * ROWS * IK);
                dsmem_push(mapa(s32(smem) + off, dst), s32(smem) + off, (uint32_t)(ROWS * IK), mapa(s32(&full[s]), dst));
            }
            if (p == 0) mbar_arrive(&full[s]);
        }
    } else if (warp == IFLUSH + IPROD) {
        // ------------------------------------------------------------ TMA
        asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
        if (lane == 0) {
            for (int it = 0; it < iters; ++it) {
                const int s = it % ISTAGES;
                if (it >= ISTAGES) mbar_wait(&empty[s], (uint32_t)((it / ISTAGES) - 1) & 1u);
                mbar_expect_tx(&full[s], IA_BYTES);
                bulk_load(smem + s * ISTAGE_BYTES, a.slices + ((int64_t)mtile * nst + kb0 + it) * IA_BYTES, IA_BYTES, &full[s]);
            }
        }
    } else {
        // ------------------------------------------------------------ MMA issue
        asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
        if (lane == 0) {
            const uint32_t sbase = s32(smem);
            for (int it = 0; it < iters; ++it) {
                const int s = it % ISTAGES;
                const int bi = it / ISPB;
                const bool first = (it % ISPB) == 0;
                if (first && bi >= 1) {
                    mbar_wait(&tmem_empty, (uint32_t)(bi - 1) & 1u);
                    fence_after();
                }
                mbar_wait(&full[s], (uint32_t)(it / ISTAGES) & 1u);
                fence_after();
                const uint32_t st = sbase + (uint32_t)(s * ISTAGE_BYTES);
                stage_mmas(tmem_base, st, st + IA_BYTES, first);
                if (CL > 1) umma_commit_all(&empty[s], (uint16_t)((1u << CL) - 1)); else umma_commit(&empty[s]);
                if ((it % ISPB) == ISPB - 1 || it == iters - 1) umma_commit(&tmem_full);
            }
        }
    }
    fence_before();
    // no CTA of a cluster may exit while a peer can still push into its shared memory or signal its barriers
    if (CL > 1) cluster_sync(); else __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(I_TMEM_COLS) : "memory");
    }
}

struct GemmI8Plan {
    int mtiles, ntiles;
    int64_t nb, bpc, nchunks, nst;
    size_t ws_partials, ws_slices, ws_expo, ws_total;
};

static GemmI8Plan plan_gemm_i8(int64_t m, int64_t k, int64_t n) {
    GemmI8Plan p;
    p.mtiles = (int)((m + IBM - 1) / IBM);
    p.ntiles = (int)((k + IBN - 1) / IBN);
    p.nb = (n + IL - 1) / IL;
    const int64_t tiles = (int64_t)p.mtiles * p.ntiles, sms = sm_count();
    // chunk counts up to one block each; the count whose grid fills its last wave best (one CTA per
    // SM), fewer chunks (less workspace) among near-equal fills
    int64_t chunks = 1;
    double best = -1.0;
    for (int64_t c = 1; c <= p.nb; ++c) {
        const int64_t bpc = (p.nb + c - 1) / c, nc = (p.nb + bpc - 1) / bpc;
        const int64_t waves = (nc * tiles + sms - 1) / sms;
        const double eff = (double)p.nb * tiles / ((double)waves * sms * bpc);
        if (eff > best + 2e-3) { best = eff; chunks = c; }
    }
    p.bpc = (p.nb + chunks - 1) / chunks;
    p.nchunks = (p.nb + p.bpc - 1) / p.bpc;
    p.nst = (n + IK - 1) / IK;
    p.ws_partials = ((size_t)p.nchunks * m * k * sizeof(double) + 255) / 256 * 256;   // the slices are bulk-copied: aligned
    p.ws_slices = (size_t)p.mtiles * p.nst * IA_BYTES;
    p.ws_expo = ((size_t)m * p.nb * sizeof(int) + 255) / 256 * 256;
    p.ws_total = p.ws_partials + p.ws_slices + p.ws_expo + 256;
    return p;
}

size_t gemm_i8_workspace_bytes(int64_t m, int64_t k, int64_t n) {
    if (m <= 0 || k <= 0 || n <= 0) return 0;
    return plan_gemm_i8(m, k, n).ws_total;
}

// Slices U, then -- unless a block holds a non-finite entry or one >= 2^IE_MAX (*ran = false: the
// caller takes the DMMA path) -- writes the partial sketches [nchunks][m][k] at the start of ws.
// Synchronises the stream once (the routing flag).
int sketch_gemm_i8(int kind, uint64_t seed, int64_t row0, int64_t col0, const double *u, int64_t m, int64_t ldu,
                   int64_t k, int64_t n, void *ws, size_t ws_bytes, cudaStream_t st, int64_t *nchunks, bool *ran) {
    *ran = false;
    const GemmI8Plan p = plan_gemm_i8(m, k, n);
    if (ws_bytes < p.ws_total) return fail(RLA_ERR_WORKSPACE, "sketch gemm i8: workspace %zu < %zu bytes", ws_bytes, p.ws_total);
    unsigned char *wb = static_cast<unsigned char *>(ws);
    uint32_t *slices = reinterpret_cast<uint32_t *>(wb + p.ws_partials);
    int *expo = reinterpret_cast<int *>(wb + p.ws_partials + p.ws_slices);
    int *flag = reinterpret_cast<int *>(wb + p.ws_partials + p.ws_slices + p.ws_expo);
    RLA_REQUIRE(m * p.nb < (int64_t(1) << 31), "sketch gemm i8: grid too large");
    RLA_CUDA_CHECK(cudaMemsetAsync(flag, 0, sizeof(int), st));
    slice_u_kernel<<<(unsigned)(m * p.nb), 256, 0, st>>>(u, ldu, m, n, p.nb, p.nst, slices, expo, flag);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    int hflag = 0;
    RLA_CUDA_CHECK(cudaMemcpyAsync(&hflag, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    RLA_CUDA_CHECK(cudaStreamSynchronize(st));
    if (hflag) return RLA_OK;

    GemmI8Args a;
    a.m = m; a.k = k; a.n = n; a.bpc = p.bpc; a.nb = p.nb; a.mtiles = p.mtiles; a.ntiles = p.ntiles;
    a.ws = static_cast<double *>(ws); a.expo = expo; a.slices = reinterpret_cast<const unsigned char *>(slices); a.seed = seed; a.row0 = row0; a.col0 = col0;
    const int64_t grid = (int64_t)p.mtiles * p.ntiles * p.nchunks;
    RLA_REQUIRE(grid < (int64_t(1) << 31), "sketch gemm i8: grid too large");
    const int smem = ISTAGES * ISTAGE_BYTES + 1024;
    const int cl = (p.mtiles % 2 == 0) ? 2 : 1;
    const void *fn = kind == 0 ? (cl == 2 ? (const void *)sketch_gemm_i8_kernel<0, 2> : (const void *)sketch_gemm_i8_kernel<0, 1>)
                               : (cl == 2 ? (const void *)sketch_gemm_i8_kernel<2, 2> : (const void *)sketch_gemm_i8_kernel<2, 1>);
    RLA_CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid, 1, 1);
    cfg.blockDim = dim3(ITHREADS, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cl; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = cl > 1 ? 1 : 0;
    void *kargs[] = {(void *)&a};
    RLA_CUDA_CHECK(cudaLaunchKernelExC(&cfg, fn, kargs));
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    *nchunks = p.nchunks;
    *ran = true;
    return RLA_OK;
}

}  // namespace rla
