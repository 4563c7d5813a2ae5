// gemm.cu -- dense embeddings:  Y(m, k) = U(m, n) * Theta(k, n)^T  in FP64 on the
// tensor pipe (DMMA), fed by TMA, with Theta either resident in HBM (explicit) or
// generated on the fly in registers from the counter-based RNG of rng.cuh.
//
// Replaces NumpyMatrixOperator(Theta).apply(Q U) = (Theta @ (QU)^T)^T of
//   GaussianEmbedding.apply            rla/embeddings.py:250-254
//   BlockGaussianEmbedding.apply       rla/embeddings.py:425-434 (one call per row block)
//
// Structure (one CTA per SM, 8 consumer warps):
//   * CTA tile  BM x BN  of Y over one chunk of the reduction dimension n (split-n:
//     the k x m sketch is far too small to fill 148 SMs); per-chunk partial tiles go to
//     a workspace and are summed in chunk order by a reduce kernel (deterministic).
//   * U (and Theta when explicit) stream through a 4-stage shared-memory ring of
//     [rows x 16 doubles] boxes written by TMA (cp.async.bulk.tensor, 128-byte swizzle,
//     out-of-range rows/columns zero-filled by the TMA unit: ragged m, k, n for free).
//   * 8 consumer warps, warp tile 64 x 32 (64 accumulator doubles per thread), issue
//     mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4).  Fragments are held per 8-wide half of the 16-wide
//     k block, double buffered: in half h a thread owns k = 4t + 2h + {0,1} of every row, i.e.
//     one conflict-free ld.shared.v2.f64 per row and half (the k permutation inside a block is
//     free as long as A and B fragments agree).  Full warp tiles run with no predicate or
//     branch between the DMMAs.
//   * 4 producer warps: lane 0 of the first issues the TMA loads; with on-the-fly Theta all
//     128 producer threads generate the [BN x 16] Theta tile of the stage (one sketch row each,
//     four Philox blocks -> Box-Muller) straight into the swizzled layout the consumers read.
//     Theta is never in memory; rla_theta_materialize_f64 exports the same values for parity.
//   * setmaxnreg: consumers 232 registers, producers 40.
#include "common.cuh"
#include "rng.cuh"
#include <cuda.h>
#include <cudaTypedefs.h>
#include <algorithm>

namespace rla {

constexpr int GK = 16;                 // doubles per row per stage (128 bytes = swizzle span)
constexpr int GSTAGES = 4;
constexpr int GWARPS = 8;
constexpr int GTHREADS = GWARPS * 32;   // consumer threads
constexpr int GPRODUCERS = 128;           // producer threads (one warpgroup)

// ------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return done;
}
// cluster pairs: the Theta tile of a stage is written by the producers of BOTH CTAs of a pair
// (each generates half of the rows into its own shared memory and pushes that slice to its
// peer with a DSMEM bulk copy that signals the peer's full barrier through complete_tx).
// Barrier operations on a peer use the default .release.cta form, as TMA-multicast pipelines
// do: the explicit .cluster scope costs MEMBAR.ALL.GPU / CCTL.IVALL per stage (measured: the
// pair ran 5 % slower than no pair at all).
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void dsmem_push(uint32_t dst_cluster_addr, uint32_t src_cta_addr, uint32_t bytes, uint32_t bar_cluster_addr) {
    asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst_cluster_addr), "r"(src_cta_addr), "r"(bytes), "r"(bar_cluster_addr) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, uint64_t *bar, int x, int y) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__device__ __forceinline__ void lds_f64x2(uint32_t addr, double2 &v) {
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
}
struct GemmArgs {
    int64_t m, k, n;          // Y is m x k, reduction over n
    int64_t kc0, kc1;         // sketch columns [kc0, kc1) handled by this launch
    int64_t kper;             // 16-wide k blocks per chunk
    int64_t nchunks;
    int mtiles, ntiles;       // tiles along m and along the sketch dimension
    double *ws;               // [nchunks][m][k] partial sketches
    uint64_t seed;            // RNG modes
    int64_t row0, col0;       // offsets of this block inside the virtual Theta
};

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// MODE 0: Theta explicit (second tensor map); 1: Philox normal; 2: Philox Rademacher; 3: Philox normal rounded to TF32
// NG: 8-wide column groups per consumer warp (warp tile 64 x 8 NG; CTA tile BM x BN = 64 WM x 8 NG WN)
// CL: CTAs per cluster along m (RNG modes): the pair works on the same Theta tile, each
//     CTA's producers generate BN / CL of its rows per stage and store them into the shared
//     memory of every CTA of the cluster (st.shared::cluster), so a Theta entry is generated
//     once per CL * BM rows of U.  Measured (tools/micro/gemm_probe.cu): every instruction the
//     producer warp of a sub-partition issues costs the DMMA pipe ~0.3 cycles, so the
//     generator's instruction count is what separates this mode from the explicit one.
//
// Warp roles: warps 0..7 are DMMA consumers (2 per SM sub-partition, free-running: they
// only meet through the per-stage full/empty mbarriers, so one warp's shared-memory
// bubble is covered by the other's DMMAs); warps 8..11 are producers: lane 0 of warp 8
// issues the TMA loads, and in the RNG modes all 128 producer threads generate Theta
// (one Philox block = four consecutive entries of a row per item) straight into the
// swizzled shared-memory layout the consumers read.
template <int WM, int WN, int NG, int MODE, int CL>
__global__ void __launch_bounds__(GTHREADS + GPRODUCERS, 1)
sketch_gemm_kernel(const __grid_constant__ CUtensorMap mapU, const __grid_constant__ CUtensorMap mapT, const GemmArgs a) {
    constexpr int BM = WM * 64, BN = WN * NG * 8;
    static_assert(WM * WN == GWARPS, "8 consumer warps");
    static_assert(MODE != 0 || CL == 1, "explicit Theta: no cluster");
    constexpr int A_BYTES = BM * GK * 8;
    constexpr int B_BYTES = BN * GK * 8;
    constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    constexpr uint32_t TX_BYTES = (MODE == 0) ? STAGE_BYTES : A_BYTES;
    constexpr int NPW = (MODE == 0) ? 1 : GPRODUCERS / 32;     // producer warps that do work
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    __shared__ __align__(8) uint64_t full_bar[GSTAGES];
    __shared__ __align__(8) uint64_t empty_bar[GSTAGES];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // blockIdx.x = rank + CL * (ntile + ntiles * (mgroup + mgroups * chunk)): the CTAs of a
    // cluster are consecutive, CTAs sharing a U chunk are adjacent
    const uint32_t rank = (CL > 1) ? cluster_ctarank() : 0u;
    int64_t b = blockIdx.x / CL;
    const int ntile = (int)(b % a.ntiles); b /= a.ntiles;
    const int mgrp = a.mtiles / CL;
    const int mtile = (int)(b % mgrp) * CL + (int)rank; b /= mgrp;
    const int64_t chunk = b;
    const int64_t kb0 = chunk * a.kper;
    const int64_t nk16 = (a.n + GK - 1) / GK;
    const int64_t kb1 = (kb0 + a.kper < nk16) ? kb0 + a.kper : nk16;
    const int iters = (int)(kb1 - kb0);
    const int m0 = mtile * BM, n0 = (int)a.kc0 + ntile * BN;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < GSTAGES; ++s) {
            mbar_init(&full_bar[s], MODE == 0 ? 1 : 1 + NPW);
            mbar_init(&empty_bar[s], GWARPS * CL);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (CL > 1) cluster_sync_all(); else __syncthreads();

    if (warp >= GWARPS) {
        // ------------------------------------------------------------ producers
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
        if (warp < GWARPS + NPW) {
            const int p = tid - GTHREADS;                  // 0..127
            const int pw = warp - GWARPS;                  // producer warp
            // RNG modes: warp pw owns RPW consecutive rows of this CTA's slice
            // [rank * BN / CL, (rank + 1) * BN / CL) of the Theta tile; a thread's items of a stage
            // are (row, quad) = (RPW pw + 8 j + lane / 4, lane & 3): one Philox block each
            constexpr int ROWS_PER_CTA = BN / CL;
            constexpr int NITEM = (ROWS_PER_CTA + 31) / 32;
            constexpr int RPW = 8 * NITEM;
            const int c = lane & 3;
            const int wrow0 = (int)rank * ROWS_PER_CTA + RPW * pw;              // first row of this warp inside the tile
            const int wrows = min(max(ROWS_PER_CTA - RPW * pw, 0), RPW);      // rows this warp owns (multiple of 8)
            const uint32_t smem_b = smem_u32(smem) + A_BYTES;
            uint32_t peer_b = 0, peer_full = 0;
            if (CL > 1) {
                peer_b = mapa_u32(smem_b, rank ^ 1u);
                peer_full = mapa_u32(smem_u32(&full_bar[0]), rank ^ 1u);
            }
            uint64_t q = ((uint64_t)(a.col0 + kb0 * GK) >> 2) + (uint64_t)c;
            for (int it = 0; it < iters; ++it, q += GK / 4) {
                const int s = it % GSTAGES;
                if (it >= GSTAGES) mbar_wait(&empty_bar[s], ((it / GSTAGES) - 1) & 1);
                unsigned char *st = smem + s * STAGE_BYTES;
                if (p == 0) {
                    mbar_expect_tx(&full_bar[s], TX_BYTES + (CL - 1) * ROWS_PER_CTA * 128);
                    const int x = (int)((kb0 + it) * GK);
                    tma_load_2d(st, &mapU, &full_bar[s], x, m0);
                    if (MODE == 0) tma_load_2d(st + A_BYTES, &mapT, &full_bar[s], x, n0);
                }
                if (MODE != 0) {
#pragma unroll
                    for (int j = 0; j < NITEM; ++j) {
                        const int rl = 8 * j + (lane >> 2);
                        const int r = wrow0 + rl;                                   // row inside the tile
                        if (rl < wrows && n0 + r < a.kc1) {
                            double v[4];
                            theta4<MODE - 1>(a.seed, (uint32_t)(a.row0 + n0 + r), q, v);   // MODE 1, 2, 3 = kind 0, 1, 2
                            unsigned char *rowp = st + A_BYTES + r * 128;
                            *reinterpret_cast<double2 *>(rowp + (((2 * c) ^ (r & 7)) << 4)) = make_double2(v[0], v[1]);
                            *reinterpret_cast<double2 *>(rowp + (((2 * c + 1) ^ (r & 7)) << 4)) = make_double2(v[2], v[3]);
                        }
                    }
                    if (CL > 1) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) {
                        if (CL > 1 && wrows > 0) {
                            const uint32_t off = (uint32_t)(s * STAGE_BYTES + wrow0 * 128);
                            dsmem_push(peer_b + off, smem_b + off, (uint32_t)wrows * 128u, peer_full + (uint32_t)s * 8u);
                        }
                        mbar_arrive(&full_bar[s]);
                    }
                }
            }
        }
    } else {
    // ---------------------------------------------------------------- consumers
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp / WN, wn = warp % WN;
    double acc[8][NG][2];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < NG; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

    // 8-wide column groups of this warp that fall inside the sketch (ragged k), row groups inside m
    const int64_t ng64 = (a.kc1 - (n0 + wn * NG * 8) + 7) / 8;
    const int ngroups = ng64 < 0 ? 0 : (ng64 > NG ? NG : (int)ng64);
    const int64_t mg64 = (a.m - (m0 + wm * 64) + 7) / 8;
    const int mgroups = mg64 < 0 ? 0 : (mg64 > 8 ? 8 : (int)mg64);

    // empty barriers of every CTA of the cluster (lane r signals CTA r)
    uint32_t empty_addr = smem_u32(&empty_bar[0]);
    if (CL > 1) empty_addr = mapa_u32(empty_addr, (uint32_t)(lane < CL ? lane : 0));

    // Fragments are held per 8-wide half of the 16-wide k block.  In half h a thread owns
    // k = 4t + 2h + {0, 1} of every row: the 16-byte chunk 2t + h, XOR-swizzled with
    // (row & 7) = g for every row this thread touches.  The B fragments (Theta, used by every
    // row group) are double buffered; an A fragment is reloaded for the next half right after
    // the 4 NG DMMAs of its pair of row groups, so only one set of A fragments is live
    // (192 + 16 NG registers of tile state instead of 224 + ...: no spills at 232).
    double2 a8[8], b8[2][NG];
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t row_off = (uint32_t)g * 128u;
    const uint32_t off0 = row_off + ((uint32_t)((2 * t) ^ g) << 4);
    const uint32_t off1 = row_off + ((uint32_t)((2 * t + 1) ^ g) << 4);
    const uint32_t a_warp = smem_base + (uint32_t)(wm * 64) * 128u, b_warp = smem_base + (uint32_t)A_BYTES + (uint32_t)(wn * NG * 8) * 128u;
#define LOAD_A(I, STAGE, OFF) lds_f64x2(a_warp + (OFF) + (STAGE) * STAGE_BYTES + (I) * 1024, a8[I])
#define LOAD_B(BUF, STAGE, OFF)                                                                  \
    {                                                                                            \
        const uint32_t sb_ = b_warp + (OFF) + (STAGE) * STAGE_BYTES;                             \
        _Pragma("unroll") for (int j = 0; j < NG; ++j) lds_f64x2(sb_ + j * 1024, b8[BUF][j]);    \
    }
    // row groups I, I + 1 against the NG column groups: both k4 steps of the half; an
    // accumulator is touched again after 2 NG DMMAs
#define MMA_PAIR(I, BUF)                                                                         \
    {                                                                                            \
        _Pragma("unroll") for (int ii = (I); ii < (I) + 2; ++ii)                                 \
            _Pragma("unroll") for (int j = 0; j < NG; ++j)                                       \
                dmma884(acc[ii][j][0], acc[ii][j][1], a8[ii].x, b8[BUF][j].x);                   \
        _Pragma("unroll") for (int ii = (I); ii < (I) + 2; ++ii)                                 \
            _Pragma("unroll") for (int j = 0; j < NG; ++j)                                       \
                dmma884(acc[ii][j][0], acc[ii][j][1], a8[ii].y, b8[BUF][j].y);                   \
    }
#define FULL_TRY(BAR, PAR) mbar_try_wait(BAR, PAR)
#define RELEASE_STAGE(S)                                                                         \
    {                                                                                            \
        __syncwarp();                                                                            \
        if (CL > 1) { if (lane < CL) mbar_arrive_remote(empty_addr + (uint32_t)(S) * 8u); }      \
        else if (lane == 0) mbar_arrive(&empty_bar[S]);                                          \
    }

    // A warp with any row and column group inside the sketch runs the whole warp tile
    // without predicates or branches between the DMMAs: rows beyond m are zero-filled by TMA
    // and columns beyond k are computed but never stored.  Warps entirely outside only keep
    // the pipeline barriers moving.
    if (mgroups > 0 && ngroups > 0) {
        if (iters > 0) {
            while (!FULL_TRY(&full_bar[0], 0)) {}
#pragma unroll
            for (int i = 0; i < 8; ++i) LOAD_A(i, 0, off0);
            LOAD_B(0, 0, off0);
        }
        // the ring is unrolled so that stage offsets and barrier addresses are immediates
        uint32_t ph = 0;                                   // parity of the ring pass of iteration it0
        for (int it0 = 0; it0 < iters; it0 += GSTAGES, ph ^= 1u) {
#pragma unroll
            for (int s = 0; s < GSTAGES; ++s) {
                const int it = it0 + s;
                if (it >= iters) break;
                const bool more = it + 1 < iters;
                const int sn = (s + 1) % GSTAGES;
                const uint32_t pn = (s + 1 == GSTAGES) ? (ph ^ 1u) : ph;
                LOAD_B(1, s, off1);
                uint32_t ready = 1;
                if (more) ready = FULL_TRY(&full_bar[sn], pn);   /* polled early, used after the DMMAs */
#pragma unroll
                for (int ip = 0; ip < 4; ++ip) {
                    MMA_PAIR(2 * ip, 0);
                    LOAD_A(2 * ip, s, off1);
                    LOAD_A(2 * ip + 1, s, off1);
                }
                if (more) { while (!ready) ready = FULL_TRY(&full_bar[sn], pn); }
                /* after the last iteration these loads fetch stale (harmless) data */
                LOAD_B(0, sn, off0);
#pragma unroll
                for (int ip = 0; ip < 4; ++ip) {
                    MMA_PAIR(2 * ip, 1);
                    LOAD_A(2 * ip, sn, off0);
                    LOAD_A(2 * ip + 1, sn, off0);
                }
                /* every shared-memory read of stage s was issued before the second half and has
                   completed (its data fed the DMMAs above) */
                RELEASE_STAGE(s);
            }
        }
    } else {
        for (int it = 0; it < iters; ++it) {
            const int s = it % GSTAGES;
            while (!FULL_TRY(&full_bar[s], (it / GSTAGES) & 1)) {}
            RELEASE_STAGE(s);
        }
    }
#undef LOAD_A
#undef LOAD_B
#undef MMA_PAIR
#undef FULL_TRY
#undef RELEASE_STAGE

    // partial tile -> workspace [chunk][m][k]
    double *wsp = a.ws + chunk * a.m * a.k;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int64_t row = m0 + wm * 64 + 8 * i + g;
        if (row >= a.m) continue;
#pragma unroll
        for (int j = 0; j < NG; ++j) {
            const int64_t col = n0 + wn * NG * 8 + 8 * j + 2 * t;
            if (col < a.kc1) wsp[row * a.k + col] = acc[i][j][0];
            if (col + 1 < a.kc1) wsp[row * a.k + col + 1] = acc[i][j][1];
        }
    }
    }
    // no CTA of a cluster may exit while a peer can still store into its shared memory or
    // signal its barriers
    if (CL > 1) cluster_sync_all();
}

// y[c, i] = (accumulate ? y[c, i] : 0) + scale * sum_chunks ws[chunk][c][i]; columns below ksplit
// were produced in nchunks0 partial sketches, the others in nchunks1
__global__ void gemm_reduce_kernel(const double *__restrict__ ws, int64_t nchunks0, int64_t nchunks1, int64_t ksplit,
                                   int64_t m, int64_t k, double scale, double *__restrict__ y, int64_t ldy, int accumulate) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= m * k) return;
    const int64_t row = idx / k, col = idx % k;
    const int64_t nchunks = col < ksplit ? nchunks0 : nchunks1;
    double s = 0.0;
    for (int64_t c = 0; c < nchunks; ++c) s += ws[c * m * k + idx];
    double *dst = y + row * ldy + col;
    *dst = accumulate ? (*dst + scale * s) : scale * s;
}

template <int KIND>
__global__ void theta_materialize_kernel(uint64_t seed, double scale, int64_t row0, int64_t rows, int64_t col0,
                                         int64_t cols, double *__restrict__ out, int64_t ldo) {
    // one thread per aligned group of 4 columns
    const int64_t q0 = col0 >> 2, q1 = (col0 + cols + 3) >> 2;
    const int64_t nq = q1 - q0;
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= rows * nq) return;
    const int64_t r = idx / nq, q = q0 + idx % nq;
    double v[4];
    theta4<KIND>(seed, (uint32_t)(row0 + r), (uint64_t)q, v);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int64_t c = 4 * q + j - col0;
        if (c >= 0 && c < cols) out[r * ldo + c] = scale * v[j];
    }
}

// ---- fallback for operands TMA cannot address (odd leading dimension / unaligned base):
// plain FP64 FMA, one thread per output element, coalesced along n via warp reduction.
__global__ void gemm_fallback_kernel(const double *__restrict__ u, int64_t ldu, const double *__restrict__ th,
                                     int64_t ldt, int64_t m, int64_t k, int64_t n, double *__restrict__ y,
                                     int64_t ldy) {
    const int64_t o = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
    if (o >= m * k) return;
    const int64_t row = o / k, col = o % k;
    const int lane = threadIdx.x & 31;
    double s = 0.0;
    for (int64_t j = lane; j < n; j += 32) s = fma(u[row * ldu + j], th[col * ldt + j], s);
#pragma unroll
    for (int off = 16; off; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if (lane == 0) y[row * ldy + col] = s;
}

// back-to-back independent DMMAs: the FP64 tensor-pipe issue peak of this device
__global__ void dmma_peak_kernel(double *out, int iters) {
    double a = threadIdx.x * 1e-3 + 1.0, b = threadIdx.x * 1e-4 + 0.5;
    double c[16][2];
#pragma unroll
    for (int j = 0; j < 16; ++j) { c[j][0] = 0.0; c[j][1] = 0.0; }
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int j = 0; j < 16; ++j) dmma884(c[j][0], c[j][1], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < 16; ++j) s += c[j][0] + c[j][1];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

static PFN_cuTensorMapEncodeTiled get_encode() {
    static PFN_cuTensorMapEncodeTiled fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(p);
    }
    return fn;
}

// tensor map over a row-major (rows x cols) FP64 matrix with row stride ld, box [box_rows x 16]
static int make_map(CUtensorMap *map, const double *base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
    PFN_cuTensorMapEncodeTiled enc = get_encode();
    if (!enc) return fail(RLA_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t gstr[1] = {(cuuint64_t)ld * 8};
    cuuint32_t box[2] = {(cuuint32_t)GK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double *>(base), gdim, gstr, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(RLA_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return RLA_OK;
}

static bool tma_ok(const double *p, int64_t ld) {
    return (reinterpret_cast<uintptr_t>(p) % 16 == 0) && (ld % 2 == 0);
}

struct GemmPlan {
    int wm, wn, ng, cl, bm, bn;
    int mtiles, ntiles;
    int64_t kper, nchunks;
};

static int env_int(const char *name, int dflt) {
    const char *e = getenv(name);
    return e ? atoi(e) : dflt;
}

// CTA tile rows / 64 for an (m, n) block.  Measured on C2 shapes (m = 512, k = 2048, Theta
// generated in the kernel): 256 x 64 tiles in cluster pairs 35.9 TFLOP/s (a Theta entry is
// generated once per 512 rows of U), 128 x 128 in pairs 35.2, 256 x 64 alone 35.3, 128 x 128
// alone 33.8; with Theta explicit 128 x 128 reaches 36.2.  Fewest padded rows first.
static int choose_wm(int64_t m, bool rng) {
    static const int wm_env = env_int("RLA_GEMM_WM", 0);
    if (wm_env == 1 || wm_env == 2 || wm_env == 4) return wm_env;
    if (m <= 64) return 1;
    const int64_t pad2 = (m + 127) / 128 * 128, pad4 = (m + 255) / 256 * 256;
    if (!rng || pad2 < pad4) return 2;
    const bool pair4 = (pad4 / 256) % 2 == 0, pair2 = (pad2 / 128) % 2 == 0;
    return (pair4 || !pair2) ? 4 : 2;
}

// plan of one range of kcols sketch columns with ng column groups per consumer warp
// rng: Theta generated in the kernel (cluster pairs along m share the generation)
static GemmPlan plan_range(int64_t m, int64_t kcols, int64_t n, bool rng, int ng, bool pairs) {
    GemmPlan p;
    static const int cl_env = env_int("RLA_GEMM_CL", 0), waves_env = env_int("RLA_GEMM_WAVES", 24);
    p.wm = choose_wm(m, rng);
    p.wn = GWARPS / p.wm;
    p.bm = p.wm * 64;
    p.ng = p.wm == 1 ? 4 : ng;
    p.bn = p.wn * p.ng * 8;
    p.mtiles = (int)((m + p.bm - 1) / p.bm);
    p.ntiles = (int)((kcols + p.bn - 1) / p.bn);
    p.cl = (rng && pairs && p.wm >= 2 && p.mtiles % 2 == 0) ? 2 : 1;
    if (cl_env == 1) p.cl = 1;
    const int64_t nk16 = (n + GK - 1) / GK;
    const int64_t tiles = (int64_t)p.mtiles * p.ntiles;
    const int64_t sms = sm_count();
    const int64_t target = sms * waves_env;
    // chunk counts up to target / tiles; keep every chunk >= 32 k-blocks unless the problem is
    // tiny, and pick the count whose grid fills its last wave best (one CTA per SM), preferring
    // fewer chunks (less workspace) among near-equal fills
    const int64_t cmax = std::max<int64_t>(1, std::min<int64_t>(std::max<int64_t>(1, nk16 / 32), (target + tiles - 1) / tiles));
    const int64_t cmin = std::max<int64_t>(1, cmax / 4);
    int64_t chunks = cmax;
    double best = -1.0;
    for (int64_t c = cmin; c <= cmax; ++c) {
        const int64_t kper = (nk16 + c - 1) / c;
        const int64_t nc = (nk16 + kper - 1) / kper;
        const int64_t grid = nc * tiles;
        const int64_t waves = (grid + sms - 1) / sms;
        // useful work / occupied SM time (chunks are kper blocks long, the last may be shorter)
        const double eff = (double)nk16 * tiles / ((double)waves * sms * kper);
        if (eff > best + 2e-3) { best = eff; chunks = c; }
    }
    p.kper = (nk16 + chunks - 1) / chunks;
    p.nchunks = (nk16 + p.kper - 1) / p.kper;
    return p;
}

// The sketch columns are covered by up to two launches: full tiles (4 column groups per
// warp), then the ragged rest with the narrowest tile (1..3 groups per warp) that holds it
// (k = 2000 with 64-wide tiles: 31 x 64 + one 16-wide tile instead of 32 x 64 = 2048 computed columns).
struct GemmRanges {
    int count;
    int64_t kc0[2], kc1[2];
    GemmPlan plan[2];
    int64_t max_chunks() const { return count == 2 ? std::max(plan[0].nchunks, plan[1].nchunks) : plan[0].nchunks; }
};

static GemmRanges plan_gemm(int64_t m, int64_t k, int64_t n, bool rng) {
    GemmRanges r;
    static const int split_env = env_int("RLA_GEMM_SPLIT", 1);
    const GemmPlan whole = plan_range(m, k, n, rng, 4, true);
    const int64_t kmain = k / whole.bn * whole.bn, ktail = k - kmain;
    const int ngt = (int)((ktail + whole.wn * 8 - 1) / (whole.wn * 8));        // groups per warp the tail needs
    const bool split = split_env && whole.wm >= 2 && kmain > 0 && ktail > 0 && ngt < 4;
    if (!split) {
        r.count = 1; r.kc0[0] = 0; r.kc1[0] = k; r.plan[0] = whole;
        return r;
    }
    r.count = 2;
    r.kc0[0] = 0; r.kc1[0] = kmain; r.plan[0] = plan_range(m, kmain, n, rng, 4, true);
    r.kc0[1] = kmain; r.kc1[1] = k; r.plan[1] = plan_range(m, ktail, n, rng, ngt, false);
    return r;
}

template <int WM, int WN, int NG, int MODE, int CL>
static int launch_gemm(const CUtensorMap &mu, const CUtensorMap &mt, const GemmArgs &a, int64_t grid, cudaStream_t st) {
    auto kern = sketch_gemm_kernel<WM, WN, NG, MODE, CL>;
    constexpr int BM = WM * 64, BN = WN * NG * 8;
    constexpr int stage = BM * GK * 8 + BN * GK * 8;
    const int smem = GSTAGES * stage + 1024;
    RLA_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid, 1, 1);
    cfg.blockDim = dim3(GTHREADS + GPRODUCERS, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = CL > 1 ? 1 : 0;
    RLA_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, mu, mt, a));
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

template <int MODE>
static int dispatch_gemm(const GemmPlan &p, const CUtensorMap &mu, const CUtensorMap &mt, const GemmArgs &a, int64_t grid,
                         cudaStream_t st) {
    constexpr int CLR = MODE == 0 ? 1 : 2;     // cluster pairs only when Theta is generated
    if (p.wm == 1) return launch_gemm<1, 8, 4, MODE, 1>(mu, mt, a, grid, st);
    if (p.wm == 4) {
        if (p.ng == 1) return launch_gemm<4, 2, 1, MODE, 1>(mu, mt, a, grid, st);
        if (p.ng == 2) return launch_gemm<4, 2, 2, MODE, 1>(mu, mt, a, grid, st);
        if (p.ng == 3) return launch_gemm<4, 2, 3, MODE, 1>(mu, mt, a, grid, st);
        return p.cl == 2 ? launch_gemm<4, 2, 4, MODE, CLR>(mu, mt, a, grid, st) : launch_gemm<4, 2, 4, MODE, 1>(mu, mt, a, grid, st);
    }
    if (p.ng == 1) return launch_gemm<2, 4, 1, MODE, 1>(mu, mt, a, grid, st);
    if (p.ng == 2) return launch_gemm<2, 4, 2, MODE, 1>(mu, mt, a, grid, st);
    if (p.ng == 3) return launch_gemm<2, 4, 3, MODE, 1>(mu, mt, a, grid, st);
    return p.cl == 2 ? launch_gemm<2, 4, 4, MODE, CLR>(mu, mt, a, grid, st) : launch_gemm<2, 4, 4, MODE, 1>(mu, mt, a, grid, st);
}

// mode 0 explicit / 1 normal / 2 rademacher
static int sketch_gemm(int mode, const double *theta, int64_t ldt, uint64_t seed, double scale, int64_t row0,
                       int64_t col0, const double *u, int64_t m, int64_t ldu, int64_t k, int64_t n, double *y,
                       int64_t ldy, int accumulate, void *ws, size_t ws_bytes, cudaStream_t st) {
    if (m == 0 || k == 0) return RLA_OK;
    const GemmRanges rg = plan_gemm(m, k, n, mode != 0);
    const size_t need = (size_t)rg.max_chunks() * m * k * sizeof(double);
    if (ws_bytes < need) return fail(RLA_ERR_WORKSPACE, "sketch gemm: workspace %zu < %zu bytes", ws_bytes, need);
    for (int ri = 0; ri < rg.count; ++ri) {
        const GemmPlan &p = rg.plan[ri];
        CUtensorMap mu, mt;
        int rc = make_map(&mu, u, m, n, ldu, p.bm);
        if (rc != RLA_OK) return rc;
        if (mode == 0) {
            // rows [kc0, kc1) of Theta: the map starts at row 0, the kernel offsets by kc0
            rc = make_map(&mt, theta, rg.kc1[ri], n, ldt, p.bn);
            if (rc != RLA_OK) return rc;
        } else {
            mt = mu;
        }
        GemmArgs a;
        a.m = m; a.k = k; a.n = n; a.kc0 = rg.kc0[ri]; a.kc1 = rg.kc1[ri];
        a.kper = p.kper; a.nchunks = p.nchunks; a.mtiles = p.mtiles; a.ntiles = p.ntiles;
        a.ws = static_cast<double *>(ws); a.seed = seed; a.row0 = row0; a.col0 = col0;
        const int64_t grid = (int64_t)p.mtiles * p.ntiles * p.nchunks;
        RLA_REQUIRE(grid < (int64_t(1) << 31), "sketch gemm: grid too large");
        rc = mode == 0 ? dispatch_gemm<0>(p, mu, mt, a, grid, st)
           : mode == 1 ? dispatch_gemm<1>(p, mu, mt, a, grid, st)
           : mode == 2 ? dispatch_gemm<2>(p, mu, mt, a, grid, st) : dispatch_gemm<3>(p, mu, mt, a, grid, st);
        if (rc != RLA_OK) return rc;
    }
    const int64_t tot = m * k;
    gemm_reduce_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(
        static_cast<double *>(ws), rg.plan[0].nchunks, rg.count == 2 ? rg.plan[1].nchunks : 0, rg.kc1[0], m, k, scale, y, ldy,
        accumulate);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

// gemm_i8.cu: kinds 0 and 2 on the int8 tensor cores
size_t gemm_i8_workspace_bytes(int64_t m, int64_t k, int64_t n);
int sketch_gemm_i8(int kind, uint64_t seed, int64_t row0, int64_t col0, const double *u, int64_t m, int64_t ldu,
                   int64_t k, int64_t n, void *ws, size_t ws_bytes, cudaStream_t st, int64_t *nchunks, bool *ran);

}  // namespace rla

using namespace rla;

// Measured FP64 tensor-pipe peak (TFLOP/s) of the current device: 8 warps per SM issuing
// independent mma.sync.m8n8k4.f64 back to back.  scratch_dev: >= 1 MiB.  Synchronises.
extern "C" int rla_dmma_peak_tflops(double *tflops, void *scratch_dev, void *stream) {
    RLA_REQUIRE(tflops && scratch_dev, "rla_dmma_peak_tflops: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const int sms = sm_count();
    RLA_REQUIRE(sms * 256 * 8 <= 1024 * 1024, "rla_dmma_peak_tflops: scratch too small");
    cudaEvent_t e0, e1;
    RLA_CUDA_CHECK(cudaEventCreate(&e0));
    RLA_CUDA_CHECK(cudaEventCreate(&e1));
    const int iters = 20000;
    dmma_peak_kernel<<<sms, 256, 0, st>>>(static_cast<double *>(scratch_dev), 200);
    RLA_CUDA_CHECK(cudaEventRecord(e0, st));
    dmma_peak_kernel<<<sms, 256, 0, st>>>(static_cast<double *>(scratch_dev), iters);
    RLA_CUDA_CHECK(cudaEventRecord(e1, st));
    RLA_CUDA_CHECK(cudaEventSynchronize(e1));
    float ms = 0.f;
    RLA_CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    const double flop = 2.0 * 8 * 8 * 4 * 16.0 * iters * 8.0 * sms;
    *tflops = flop / (ms * 1e-3) / 1e12;
    return RLA_OK;
}

namespace rla {
__global__ void philox_kat_kernel(const uint32_t *__restrict__ in, int64_t count, uint32_t *__restrict__ out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    const PhiloxOut p = philox4x32_10(in[6 * i], in[6 * i + 1], in[6 * i + 2], in[6 * i + 3], in[6 * i + 4], in[6 * i + 5]);
    out[4 * i] = p.x; out[4 * i + 1] = p.y; out[4 * i + 2] = p.z; out[4 * i + 3] = p.w;
}
}  // namespace rla

extern "C" int rla_philox4x32_10_host(const uint32_t *in, int64_t count, uint32_t *out) {
    RLA_REQUIRE(count >= 0 && (count == 0 || (in && out)), "rla_philox4x32_10_host: bad arguments");
    for (int64_t i = 0; i < count; ++i) {
        const PhiloxOut p = philox4x32_10(in[6 * i], in[6 * i + 1], in[6 * i + 2], in[6 * i + 3], in[6 * i + 4], in[6 * i + 5]);
        out[4 * i] = p.x; out[4 * i + 1] = p.y; out[4 * i + 2] = p.z; out[4 * i + 3] = p.w;
    }
    return RLA_OK;
}

extern "C" int rla_philox4x32_10_device(const uint32_t *in, int64_t count, uint32_t *out, void *stream) {
    RLA_REQUIRE(count >= 0 && (count == 0 || (in && out)), "rla_philox4x32_10_device: bad arguments");
    if (count == 0) return RLA_OK;
    philox_kat_kernel<<<(unsigned)((count + 127) / 128), 128, 0, (cudaStream_t)stream>>>(in, count, out);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

extern "C" size_t rla_gemm_workspace_bytes(int64_t m, int64_t k, int64_t n) {
    if (m <= 0 || k <= 0 || n <= 0) return 0;
    // the larger of the two modes' plans (they differ only in the cluster width today)
    const GemmRanges p = plan_gemm(m, k, n, true), q = plan_gemm(m, k, n, false);
    return (size_t)std::max(p.max_chunks(), q.max_chunks()) * m * k * sizeof(double);
}

// kinds 0 and 2 try the int8 path first (gemm_i8.cu) and fall back to DMMA in the same workspace
extern "C" size_t rla_gemm_rng_workspace_bytes(int64_t m, int64_t k, int64_t n) {
    return std::max(rla_gemm_workspace_bytes(m, k, n), gemm_i8_workspace_bytes(m, k, n));
}

extern "C" int rla_gauss_apply_explicit_f64(const double *theta, int64_t k, int64_t n, int64_t ldt, const double *u,
                                            int64_t m, int64_t ldu, double *y, int64_t ldy, void *ws,
                                            size_t ws_bytes, void *stream) {
    RLA_REQUIRE(k >= 0 && n >= 1 && m >= 0 && ldt >= n && ldu >= n && ldy >= k, "rla_gauss_apply_explicit_f64: bad sizes");
    if (m == 0 || k == 0) return RLA_OK;
    RLA_REQUIRE(theta && u && y, "rla_gauss_apply_explicit_f64: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (!tma_ok(theta, ldt) || !tma_ok(u, ldu)) {
        const int64_t outs = m * k;
        gemm_fallback_kernel<<<(unsigned)((outs + 7) / 8), 256, 0, st>>>(u, ldu, theta, ldt, m, k, n, y, ldy);
        count_launch();
        RLA_CUDA_CHECK(cudaGetLastError());
        return RLA_OK;
    }
    RLA_REQUIRE(ws, "rla_gauss_apply_explicit_f64: null workspace");
    return sketch_gemm(0, theta, ldt, 0, 1.0, 0, 0, u, m, ldu, k, n, y, ldy, 0, ws, ws_bytes, st);
}

extern "C" int rla_embed_apply_rng_f64(uint64_t seed, int kind, double scale, int64_t row0, int64_t k_blk,
                                       int64_t col0, int64_t n, const double *u, int64_t m, int64_t ldu, double *y,
                                       int64_t ldy, int accumulate, void *ws, size_t ws_bytes, void *stream) {
    RLA_REQUIRE(kind >= 0 && kind <= 2, "rla_embed_apply_rng_f64: kind must be 0 (normal), 1 (rademacher) or 2 (normal rounded to TF32)");
    RLA_REQUIRE(k_blk >= 0 && n >= 1 && m >= 0 && ldu >= n && ldy >= k_blk && row0 >= 0 && col0 >= 0,
                "rla_embed_apply_rng_f64: bad sizes");
    RLA_REQUIRE(col0 % 16 == 0, "rla_embed_apply_rng_f64: col0 must be a multiple of 16");
    RLA_REQUIRE(row0 + k_blk <= (int64_t(1) << 32), "rla_embed_apply_rng_f64: more than 2^32 sketch rows");
    if (m == 0 || k_blk == 0) return RLA_OK;
    RLA_REQUIRE(u && y && ws, "rla_embed_apply_rng_f64: null pointer");
    RLA_REQUIRE(tma_ok(u, ldu), "rla_embed_apply_rng_f64: u must be 16-byte aligned with an even leading dimension");
    if (kind != 1) {
        // Theta of kinds 0 and 2 is FP32: Ozaki slices on the int8 tensor cores, unless a block holds a
        // non-finite entry or one near the FP64 overflow limit (then DMMA, FP64 semantics)
        cudaStream_t st = (cudaStream_t)stream;
        int64_t nchunks = 0;
        bool ran = false;
        const int rc = sketch_gemm_i8(kind, seed, row0, col0, u, m, ldu, k_blk, n, ws, ws_bytes, st, &nchunks, &ran);
        if (rc != RLA_OK) return rc;
        if (ran) {
            const int64_t tot = m * k_blk;
            gemm_reduce_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(
                static_cast<double *>(ws), nchunks, 0, k_blk, m, k_blk, scale, y, ldy, accumulate);
            count_launch();
            RLA_CUDA_CHECK(cudaGetLastError());
            return RLA_OK;
        }
    }
    return sketch_gemm(kind + 1, nullptr, 0, seed, scale, row0, col0, u, m, ldu, k_blk, n, y, ldy,
                       accumulate, ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" int rla_theta_materialize_f64(uint64_t seed, int kind, double scale, int64_t row0, int64_t rows,
                                         int64_t col0, int64_t cols, double *out, int64_t ldo, void *stream) {
    RLA_REQUIRE(kind >= 0 && kind <= 2, "rla_theta_materialize_f64: kind must be 0, 1 or 2");
    RLA_REQUIRE(rows >= 0 && cols >= 0 && row0 >= 0 && col0 >= 0 && ldo >= cols, "rla_theta_materialize_f64: bad sizes");
    if (rows == 0 || cols == 0) return RLA_OK;
    RLA_REQUIRE(out, "rla_theta_materialize_f64: null pointer");
    const int64_t nq = ((col0 + cols + 3) >> 2) - (col0 >> 2);
    const int64_t tot = rows * nq;
    const unsigned grid = (unsigned)((tot + 255) / 256);
    if (kind == 0) theta_materialize_kernel<0><<<grid, 256, 0, (cudaStream_t)stream>>>(seed, scale, row0, rows, col0, cols, out, ldo);
    else if (kind == 1) theta_materialize_kernel<1><<<grid, 256, 0, (cudaStream_t)stream>>>(seed, scale, row0, rows, col0, cols, out, ldo);
    else theta_materialize_kernel<2><<<grid, 256, 0, (cudaStream_t)stream>>>(seed, scale, row0, rows, col0, cols, out, ldo);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}
