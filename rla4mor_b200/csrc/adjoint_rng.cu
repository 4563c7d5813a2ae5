// adjoint_rng.cu -- the adjoint of the Gaussian / block-Gaussian embeddings with Theta generated in
// the kernel:  out(m, n) = V(m, k) * Theta(k, n), all row-major, Theta never in memory.
//
// Replaces pyMOR's adjoint of the explicit matrix, V @ get_matrix(), of
//   GaussianEmbedding        rla/embeddings.py:214-270
//   BlockGaussianEmbedding   rla/embeddings.py:373-467
// Theta is the stack of `nblocks` blocks: block b holds rows [row_start[b], row_start[b+1]) of the
// stack, which are rows 0 .. size_b - 1 of the virtual matrix scale * g(seeds[b], row, col) of
// rng.cuh (kind 0, 1 or 2).  A GaussianEmbedding is one block; all blocks of a
// BlockGaussianEmbedding go in one launch, so `out` is written once.
//
// Structure (one CTA per SM, 12 warps):
//   * 8 consumer warps run mma.sync.m8n8k4.f64 on the CTA tile (WM*WTM) x (WN*32) of `out` with the
//     fragment layout of lincomb_mma_kernel (lincomb.cu): a = V[i0 + g][k0 + t], b = Theta[k0 + t][j0 + g].
//   * 4 producer warps fill a 4-stage shared-memory ring, one 16-wide chunk of the reduction dimension
//     per stage: they copy the V chunk [BM x 16] with cp.async (8-byte pieces when V's rows are not
//     16-byte aligned; zero-filled outside m x k) and generate the Theta chunk [16 x BN] with
//     theta4f, each entry formed as fl(scale * (double)g) exactly as theta_materialize_kernel forms it.
//     Full barrier: one arrive per producer warp plus the cp.async completions of every producer
//     thread (cp.async.mbarrier.arrive); empty barrier: one arrive per consumer warp.
//
// Bit-identity with gemm_nn(V, Theta materialised) on its tensor-pipe path: every output element is
// one register chain over k in ascending order, four terms per DMMA, chunks of 16 with zero-filled
// tails -- the DMMA sequence lincomb_mma_kernel issues for the same element.  There is deliberately
// no split over k (it would change the chain), so a short n underfills the GPU.
//
// An m-tile holds up to 128 rows of V; for m > 128 every m-tile generates Theta again.
#include "common.cuh"
#include "rng.cuh"

namespace rla {
namespace {

constexpr int AR_BK = 16;                  // reduction chunk: the chunk of lincomb_mma_kernel
constexpr int AR_STAGES = 4;
constexpr int AR_LDV = AR_BK + 4;          // V chunk row stride (doubles): conflict-free fragment loads
constexpr int AR_CONSUMERS = 256;
constexpr int AR_PRODUCERS = 128;
constexpr int AR_PWARPS = AR_PRODUCERS / 32;

__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void bar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}
// the barrier's current phase also waits for every cp.async this thread has issued so far
__device__ __forceinline__ void bar_arrive_cp_async(uint64_t *bar) {
    asm volatile("cp.async.mbarrier.arrive.shared::cta.b64 [%0];" ::"r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void bar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(smem_addr(bar)), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void cp16_zfill(void *smem, const void *gmem, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_addr(smem)), "l"(gmem), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp8_zfill(void *smem, const void *gmem, int src_bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(smem_addr(smem)), "l"(gmem), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void dmma(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

template <int KIND, int WTM, int WM>
__global__ void __launch_bounds__(AR_CONSUMERS + AR_PRODUCERS, 1)
adjoint_rng_kernel(const uint64_t *__restrict__ seeds, const int64_t *__restrict__ row_start, int64_t nblocks,
                   double scale, const double *__restrict__ v, int64_t ldv, int64_t m, int64_t n,
                   double *__restrict__ out, int64_t ldo, int mtiles, int vec_v, int vec_out) {
    constexpr int WN = 8 / WM, BM = WM * WTM, BN = WN * 32, LDX = BN + 4;
    constexpr int MI = WTM / 8;                            // 8-row groups per warp tile
    constexpr int XS = AR_BK * LDX, VS = BM * AR_LDV;      // doubles per stage
    constexpr int RPW = AR_BK / AR_PWARPS;                 // Theta rows per producer warp and stage
    constexpr int QPL = BN / 128;                          // Philox quads per producer lane and row
    extern __shared__ __align__(16) unsigned char ar_smem[];
    double *sx = reinterpret_cast<double *>(ar_smem);
    double *sv = sx + AR_STAGES * XS;
    __shared__ __align__(8) uint64_t full_bar[AR_STAGES];
    __shared__ __align__(8) uint64_t empty_bar[AR_STAGES];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t n0 = (int64_t)(blockIdx.x / mtiles) * BN;
    const int64_t m0 = (int64_t)(blockIdx.x % mtiles) * BM;
    const int64_t k = row_start[nblocks];
    const int64_t nchunks = (k + AR_BK - 1) / AR_BK;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < AR_STAGES; ++s) {
            bar_init(&full_bar[s], AR_PWARPS);
            bar_init(&empty_bar[s], AR_CONSUMERS / 32);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp >= AR_CONSUMERS / 32) {
        // ------------------------------------------------------------------ producers
        const int p = tid - AR_CONSUMERS, pw = warp - AR_CONSUMERS / 32;
        // warp pw generates rows RPW pw .. RPW pw + RPW - 1 of every chunk; lane l the quads
        // l + 32 j of a row.  The block of each row is found by a cursor that only moves forward.
        int64_t blk[RPW];
#pragma unroll
        for (int i = 0; i < RPW; ++i) blk[i] = 0;
        for (int64_t c = 0; c < nchunks; ++c) {
            const int s = (int)(c % AR_STAGES);
            if (c >= AR_STAGES) bar_wait(&empty_bar[s], (uint32_t)((c / AR_STAGES) - 1) & 1u);
            const int64_t k0 = c * AR_BK;
            double *dv = sv + s * VS;
            if (vec_v) {
                for (int id = p; id < BM * (AR_BK / 2); id += AR_PRODUCERS) {
                    const int r = id / (AR_BK / 2), cc = (id % (AR_BK / 2)) * 2;
                    const int64_t row = m0 + r, col = k0 + cc;
                    const int bytes = (row < m && col < k) ? (col + 1 < k ? 16 : 8) : 0;
                    cp16_zfill(dv + r * AR_LDV + cc, bytes ? v + row * ldv + col : v, bytes);
                }
            } else {
                for (int id = p; id < BM * AR_BK; id += AR_PRODUCERS) {
                    const int r = id / AR_BK, cc = id % AR_BK;
                    const int64_t row = m0 + r, col = k0 + cc;
                    const int bytes = (row < m && col < k) ? 8 : 0;
                    cp8_zfill(dv + r * AR_LDV + cc, bytes ? v + row * ldv + col : v, bytes);
                }
            }
            bar_arrive_cp_async(&full_bar[s]);
            // block of each row first (rows beyond k take the last row's block), then the RPW * QPL
            // items of the chunk without a branch, so that their latency chains overlap: entries
            // outside k x n are generated and replaced by zero
            uint64_t seed[RPW];
            uint32_t lrow[RPW];
#pragma unroll
            for (int i = 0; i < RPW; ++i) {
                const int64_t r = min(k0 + RPW * pw + i, k - 1);
                while (blk[i] + 1 < nblocks && __ldg(row_start + blk[i] + 1) <= r) ++blk[i];
                seed[i] = __ldg(seeds + blk[i]);
                lrow[i] = (uint32_t)(r - __ldg(row_start + blk[i]));
            }
            double *dx = sx + s * XS;
#pragma unroll
            for (int i = 0; i < RPW; ++i) {
                const int kk = RPW * pw + i;
#pragma unroll
                for (int j = 0; j < QPL; ++j) {
                    const int qc = lane + 32 * j;
                    const int64_t col = n0 + 4 * qc;
                    float f[4];
                    theta4f<KIND>(seed[i], lrow[i], (uint64_t)col >> 2, f);
                    const bool live = k0 + kk < k && col < n;
                    double2 *dst = reinterpret_cast<double2 *>(dx + kk * LDX + 4 * qc);
                    dst[0] = live ? make_double2(scale * (double)f[0], scale * (double)f[1]) : make_double2(0.0, 0.0);
                    dst[1] = live ? make_double2(scale * (double)f[2], scale * (double)f[3]) : make_double2(0.0, 0.0);
                }
            }
            __syncwarp();
            if (lane == 0) bar_arrive(&full_bar[s]);
        }
    } else {
        // ------------------------------------------------------------------ consumers
        const int g = lane >> 2, t = lane & 3;
        const int wm = warp / WN, wn = warp % WN;
        double acc[MI][4][2];
#pragma unroll
        for (int i = 0; i < MI; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }
        for (int64_t c = 0; c < nchunks; ++c) {
            const int s = (int)(c % AR_STAGES);
            bar_wait(&full_bar[s], (uint32_t)(c / AR_STAGES) & 1u);
            const double *px = sx + s * XS + wn * 32 + g;
            const double *pv = sv + s * VS + (wm * WTM + g) * AR_LDV + t;
#pragma unroll
            for (int ks = 0; ks < AR_BK / 4; ++ks) {
                double a[MI], b[4];
#pragma unroll
                for (int i = 0; i < MI; ++i) a[i] = pv[i * 8 * AR_LDV + ks * 4];
#pragma unroll
                for (int j = 0; j < 4; ++j) b[j] = px[(ks * 4 + t) * LDX + j * 8];
#pragma unroll
                for (int i = 0; i < MI; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) dmma(acc[i][j][0], acc[i][j][1], a[i], b[j]);
            }
            __syncwarp();
            if (lane == 0) bar_arrive(&empty_bar[s]);
        }
#pragma unroll
        for (int i = 0; i < MI; ++i) {
            const int64_t row = m0 + wm * WTM + 8 * i + g;
            if (row >= m) continue;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int64_t col = n0 + wn * 32 + 8 * j + 2 * t;
                double *dst = out + row * ldo + col;
                if (vec_out && col + 1 < n) {
                    *reinterpret_cast<double2 *>(dst) = make_double2(acc[i][j][0], acc[i][j][1]);
                } else {
                    if (col < n) dst[0] = acc[i][j][0];
                    if (col + 1 < n) dst[1] = acc[i][j][1];
                }
            }
        }
    }
}

template <int KIND, int WTM, int WM>
int adjoint_rng_launch(const uint64_t *seeds, const int64_t *row_start, int64_t nblocks, double scale, int64_t n,
                       const double *v, int64_t m, int64_t ldv, double *out, int64_t ldo, cudaStream_t st) {
    constexpr int WN = 8 / WM, BM = WM * WTM, BN = WN * 32;
    const int64_t gx = (n + BN - 1) / BN, gy = (m + BM - 1) / BM;
    RLA_REQUIRE(gx * gy < (int64_t(1) << 31), "rla_embed_adjoint_rng_f64: problem too large");
    const int smem = (int)(AR_STAGES * (AR_BK * (BN + 4) + BM * AR_LDV) * sizeof(double));
    const int vec_v = (reinterpret_cast<uintptr_t>(v) % 16 == 0) && (m == 1 || ldv % 2 == 0);
    const int vec_out = (reinterpret_cast<uintptr_t>(out) % 16 == 0) && (m == 1 || ldo % 2 == 0);
    auto kern = adjoint_rng_kernel<KIND, WTM, WM>;
    RLA_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kern<<<(unsigned)(gx * gy), AR_CONSUMERS + AR_PRODUCERS, smem, st>>>(seeds, row_start, nblocks, scale, v, ldv, m, n,
                                                                       out, ldo, (int)gy, vec_v, vec_out);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

// the tiles of lincomb_launch: 128 x 128 for m > 64, 64 x 256 and 32 x 256 below
template <int KIND>
int adjoint_rng_dispatch(const uint64_t *seeds, const int64_t *row_start, int64_t nblocks, double scale, int64_t n,
                         const double *v, int64_t m, int64_t ldv, double *out, int64_t ldo, cudaStream_t st) {
    if (m > 64) return adjoint_rng_launch<KIND, 64, 2>(seeds, row_start, nblocks, scale, n, v, m, ldv, out, ldo, st);
    if (m > 32) return adjoint_rng_launch<KIND, 64, 1>(seeds, row_start, nblocks, scale, n, v, m, ldv, out, ldo, st);
    return adjoint_rng_launch<KIND, 32, 1>(seeds, row_start, nblocks, scale, n, v, m, ldv, out, ldo, st);
}

}  // namespace
}  // namespace rla

using namespace rla;

extern "C" int rla_embed_adjoint_rng_f64(int kind, double scale, const uint64_t *seeds_dev, const int64_t *row_start_dev,
                                         int64_t nblocks, int64_t n, const double *v_dev, int64_t m, int64_t ldv,
                                         double *out_dev, int64_t ldo, void *stream) {
    RLA_REQUIRE(kind >= 0 && kind <= 2, "rla_embed_adjoint_rng_f64: kind must be 0 (normal), 1 (rademacher) or 2 (normal rounded to TF32)");
    RLA_REQUIRE(nblocks >= 1 && n >= 0 && m >= 0 && ldv >= 1 && ldo >= n, "rla_embed_adjoint_rng_f64: bad sizes");
    if (m == 0 || n == 0) return RLA_OK;
    RLA_REQUIRE(seeds_dev && row_start_dev && v_dev && out_dev, "rla_embed_adjoint_rng_f64: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (kind == 0) return adjoint_rng_dispatch<0>(seeds_dev, row_start_dev, nblocks, scale, n, v_dev, m, ldv, out_dev, ldo, st);
    if (kind == 1) return adjoint_rng_dispatch<1>(seeds_dev, row_start_dev, nblocks, scale, n, v_dev, m, ldv, out_dev, ldo, st);
    return adjoint_rng_dispatch<2>(seeds_dev, row_start_dev, nblocks, scale, n, v_dev, m, ldv, out_dev, ldo, st);
}
