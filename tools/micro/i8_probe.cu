// i8_probe.cu -- developer probe: where does the stage time of sketch_gemm_i8_kernel (csrc/gemm_i8.cu)
// go?  It runs the kernel's pipeline at the C2 grid (4 m tiles x 32 n tiles x 128 chunks of bpc = 2
// exponent blocks = 16 384 CTAs in cluster pairs, 1024 stages each, with the kernel's flush warps and
// TMEM hand-over) with parts switched on at compile time:
//   1  36 MMAs per stage on operands resident in shared memory, level-major (the order of the 36-MMA kernel)
//   2  the same, A-slice-major with A-collector reuse
//   3  the same with the pair's MMAs as one cta_group::2 MMA (M = 256; 40 KB stages, five)
//   4  + the U-slice bulk copies (32 KB per stage from a 16 GB workspace) and the full / empty barriers
//   5  + the Theta producers (Philox + Box-Muller + slicing of this CTA's 32 rows)
//   5p like 5 with one-CTA MMAs in level-major order, each CTA generating all 64 rows (the pipeline
//      of the 36-MMA kernel, without the DSMEM push of the pair's rows)
//   2w / 4w / 5w  like 2 / 4 / 5p with the 12 wide one-CTA MMAs per stage of the kernel (N = 64 (8 - i),
//      split at 256): the products of one U slice with B slices 0 .. 7 - i as one tall B tile
// The full kernel (6) is timed through the library by tools/i8_probe.py.  Timing only: the operands
// are random bytes and the results are meaningless.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a tools/micro/i8_probe.cu -o tools/micro/i8_probe
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
#include "../../rla4mor_b200/csrc/rng.cuh"

constexpr int IS = 8, IK = 32, IBM = 128, IBN = 64, ISPB = 512, BPC = 2;
constexpr int IFLUSH = 8, IPROD = 6, ITHREADS = (IFLUSH + IPROD + 2) * 32;
constexpr int IA_SLICE = IBM * IK, IA_BYTES = IS * IA_SLICE;
constexpr int MT = 4, NT = 32, CHUNKS = 128;          // C2: m = 512, k = 2000, n = 2^22

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
__device__ __forceinline__ void mbar_arrive_remote(uint32_t addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(s32(bar)), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ uint32_t mapa(uint32_t a, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
    return r;
}
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint64_t desc_sw32(uint32_t a) {
    return (uint64_t)((a & 0x3FFFFu) >> 4) | (uint64_t(1) << 16) | (uint64_t(256 >> 4) << 32) | (uint64_t(1) << 46) | (uint64_t(6) << 61);
}
#define UMMA(QUAL)                                                                                     \
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma." QUAL " [%0], %1, %2, %3, p;\n\t}" \
                 ::"r"(d), "l"(a), "l"(b), "r"(id), "r"(acc) : "memory")
template <int CG, int COLL>
__device__ __forceinline__ void umma(uint32_t d, uint64_t a, uint64_t b, uint32_t id, uint32_t acc) {
    if constexpr (CG == 1 && COLL == 0) UMMA("cta_group::1.kind::i8");
    else if constexpr (CG == 1 && COLL == 1) UMMA("cta_group::1.kind::i8.collector::a::fill");
    else if constexpr (CG == 1 && COLL == 2) UMMA("cta_group::1.kind::i8.collector::a::use");
    else if constexpr (CG == 1) UMMA("cta_group::1.kind::i8.collector::a::lastuse");
    else if constexpr (COLL == 0) UMMA("cta_group::2.kind::i8");
    else if constexpr (COLL == 1) UMMA("cta_group::2.kind::i8.collector::a::fill");
    else if constexpr (COLL == 2) UMMA("cta_group::2.kind::i8.collector::a::use");
    else UMMA("cta_group::2.kind::i8.collector::a::lastuse");
}
template <int CG>
__device__ __forceinline__ void commit(uint64_t *bar) {
    if constexpr (CG == 1)
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s32(bar)) : "memory");
    else
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                     ::"r"(s32(bar)), "h"((uint16_t)3) : "memory");
}
template <int CG, int I = 0, int J = 0>
__device__ __forceinline__ void mmas_a_major(uint32_t tm, uint32_t a, uint32_t b, uint32_t bs, uint32_t id, bool first) {
    if constexpr (I < IS) {
        constexpr int COLL = (I == IS - 1) ? 0 : (J == 0) ? 1 : (J == IS - 1 - I) ? 3 : 2;
        umma<CG, COLL>(tm + (I + J) * IBN, desc_sw32(a + I * IA_SLICE), desc_sw32(b + J * bs), id, (first && I == 0) ? 0u : 1u);
        if constexpr (J == IS - 1 - I) mmas_a_major<CG, I + 1, 0>(tm, a, b, bs, id, first);
        else mmas_a_major<CG, I, J + 1>(tm, a, b, bs, id, first);
    }
}
// 12 MMAs of N = 64 (IS - i) (split at 256) instead of 36 of N = 64: the order of csrc/gemm_i8.cu
template <int I = 0>
__device__ __forceinline__ void mmas_wide(uint32_t tm, uint32_t a, uint32_t b, bool first) {
    if constexpr (I < IS) {
        constexpr int NS = IS - I, N0 = NS < 4 ? NS : 4, N1 = NS - N0;
        constexpr uint32_t idb = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(IBM >> 4) << 24);
        const uint32_t acc = (first && I == 0) ? 0u : 1u;
        umma<1, N1 ? 1 : 0>(tm + I * IBN, desc_sw32(a + I * IA_SLICE), desc_sw32(b), idb | ((uint32_t)(N0 * IBN >> 3) << 17), acc);
        if constexpr (N1 > 0)
            umma<1, 3>(tm + (I + N0) * IBN, desc_sw32(a + I * IA_SLICE), desc_sw32(b + N0 * IBN * IK), idb | ((uint32_t)(N1 * IBN >> 3) << 17), acc);
        mmas_wide<I + 1>(tm, a, b, first);
    }
}
__device__ __forceinline__ uint64_t fix56_theta(float v) {
    const uint32_t b = __float_as_uint(v);
    int ex = (int)((b >> 23) & 0xff);
    uint64_t mant = b & 0x7fffffu;
    if (ex == 0) ex = 1; else mant |= 0x800000u;
    const int sh = ex - 97;
    return sh >= 0 ? mant << sh : (sh > -64 ? mant >> -sh : 0);
}

// ORDER 0: level-major, 1: A-slice-major with the collector, 2: 12 wide MMAs (CG = 1 only).  CG: MMA CTA group.  UCOPY: U slices by bulk
// copy (else resident, no full / empty waits).  PROD: Theta generated per stage.
template <int ORDER, int CG, bool UCOPY, bool PROD>
__global__ void __launch_bounds__(ITHREADS, 1) probe(const unsigned char *slices, double *out, uint64_t seed) {
    constexpr int ROWS = IBN / CG, B_SLICE = ROWS * IK, STAGE = IA_BYTES + IS * B_SLICE, NS = CG == 2 ? 5 : 4;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    __shared__ __align__(8) uint64_t full[5], empty[5], tmem_full, tmem_empty;
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    const int64_t bx = blockIdx.x / 2;
    const int ntile = (int)(bx % NT), mtile = (int)((bx / NT) % (MT / 2)) * 2 + (int)rank;
    const int64_t chunk = bx / (NT * MT / 2);
    const int iters = BPC * ISPB;
    const int64_t nst = (int64_t)CHUNKS * iters;
    constexpr bool waits = UCOPY || PROD;
    for (int i = tid; i < NS * STAGE / 4; i += ITHREADS)     // resident operands: random bytes
        reinterpret_cast<uint32_t *>(smem)[i] = (uint32_t)i * 2654435761u ^ (uint32_t)blockIdx.x * 40503u;
    if (tid == 0) {
        for (int s = 0; s < NS; ++s) {
            mbar_init(&full[s], waits ? (UCOPY ? 1 : 0) + (PROD ? 1 : 0) + (CG == 2 && rank == 0 ? 1 : 0) : 1);   // unused without waits
            mbar_init(&empty[s], 1);
        }
        mbar_init(&tmem_full, 1);
        mbar_init(&tmem_empty, CG * IFLUSH);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 0) {
        if constexpr (CG == 2) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(s32(&tmem_base_s)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(s32(&tmem_base_s)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    cluster_sync();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_s;

    if (warp < IFLUSH) {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 176;");
        const int q = warp & 3, h = warp >> 2;
        double acc[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[j] = 0.0;
        for (int bi = 0; bi < BPC; ++bi) {
            mbar_wait(&tmem_full, (uint32_t)bi & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            double t[2][16];
#pragma unroll
            for (int g = 0; g < 2; ++g)
#pragma unroll
                for (int l = IS - 1; l >= 0; --l) {
                    uint32_t v[16];
                    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                                 : "r"(tmem + ((uint32_t)(32 * q) << 16) + (uint32_t)(l * IBN + 32 * h + 16 * g)) : "memory");
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 16; ++j) t[g][j] = (l == IS - 1) ? (double)(int)v[j] : fma(t[g][j], 0x1p-7, (double)(int)v[j]);
                }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) {
                if (CG == 2 && rank != 0) mbar_arrive_remote(mapa(s32(&tmem_empty), 0));
                else mbar_arrive(&tmem_empty);
            }
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[j] += ldexp(t[j >> 4][j & 15], -11);
        }
        double sum = 0.0;
#pragma unroll
        for (int j = 0; j < 32; ++j) sum += acc[j];
        out[(int64_t)blockIdx.x * 256 + tid] = sum;
    } else if (warp < IFLUSH + IPROD) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
        if constexpr (PROD) {
            const int p = tid - IFLUSH * 32;
            constexpr int NPT = IPROD * 32, NJ = (ROWS * 8 + NPT - 1) / NPT;
            const int c = p & 7;
            uint64_t qv = ((uint64_t)(chunk * iters * IK) >> 2) + (uint64_t)c;
            for (int it = 0; it < iters; ++it, qv += IK / 4) {
                const int s = it % NS;
                if (it >= NS) mbar_wait(&empty[s], (uint32_t)((it / NS) - 1) & 1u);
                unsigned char *stb = smem + s * STAGE + IA_BYTES;
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    const int rl = (p + NPT * j) >> 3;
                    if (rl < ROWS) {
                        float f[4];
                        rla::theta4f<0>(seed, (uint32_t)(ntile * IBN + (int)rank * ROWS + rl), qv, f);
                        uint32_t w[IS];
#pragma unroll
                        for (int sl = 0; sl < IS; ++sl) w[sl] = 0;
#pragma unroll
                        for (int e4 = 0; e4 < 4; ++e4) {
                            const uint64_t M = fix56_theta(f[e4]);
                            const uint32_t neg = (__float_as_uint(f[e4]) >> 31) ? 0xffffffffu : 0u;
#pragma unroll
                            for (int sl = 0; sl < IS; ++sl) w[sl] |= ((((uint32_t)(M >> (7 * (IS - 1 - sl))) & 127u) ^ neg) - neg & 0xffu) << (8 * e4);
                        }
                        const int off = rl * IK + (((c >> 2) ^ ((rl >> 2) & 1)) << 4) + (c & 3) * 4;
#pragma unroll
                        for (int sl = 0; sl < IS; ++sl) *reinterpret_cast<uint32_t *>(stb + sl * B_SLICE + off) = w[sl];
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("bar.sync 1, %0;" ::"n"(NPT) : "memory");
                if (p == 0) mbar_arrive(&full[s]);
            }
        }
    } else if (warp == IFLUSH + IPROD) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
        if (UCOPY && lane == 0) {
            for (int it = 0; it < iters; ++it) {
                const int s = it % NS;
                if (it >= NS) mbar_wait(&empty[s], (uint32_t)((it / NS) - 1) & 1u);
                mbar_expect_tx(&full[s], IA_BYTES);
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(s32(smem + s * STAGE)), "l"(slices + ((int64_t)mtile * nst + chunk * iters + it) * IA_BYTES),
                               "r"(IA_BYTES), "r"(s32(&full[s])) : "memory");
            }
        }
    } else {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
        if (lane == 0 && CG == 2 && rank != 0) {
            if (waits)
                for (int it = 0; it < iters; ++it) {
                    mbar_wait(&full[it % NS], (uint32_t)(it / NS) & 1u);
                    mbar_arrive_remote(mapa(s32(&full[it % NS]), 0));
                }
        } else if (lane == 0) {
            constexpr uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(IBN >> 3) << 17) | ((uint32_t)(CG * IBM >> 4) << 24);
            const uint32_t sbase = s32(smem);
            for (int it = 0; it < iters; ++it) {
                const int s = it % NS, bi = it / ISPB;
                const bool first = (it % ISPB) == 0;
                if (first && bi >= 1) {
                    mbar_wait(&tmem_empty, (uint32_t)(bi - 1) & 1u);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                }
                if (waits) {
                    mbar_wait(&full[s], (uint32_t)(it / NS) & 1u);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                }
                const uint32_t st = sbase + (uint32_t)(s * STAGE);
                if constexpr (ORDER == 2) {
                    mmas_wide(tmem, st, st + IA_BYTES, first);
                } else if constexpr (ORDER == 1) {
                    mmas_a_major<CG>(tmem, st, st + IA_BYTES, B_SLICE, idesc, first);
                } else {
#pragma unroll
                    for (int l = 0; l < IS; ++l)
#pragma unroll
                        for (int i = 0; i <= l; ++i)
                            umma<CG, 0>(tmem + l * IBN, desc_sw32(st + i * IA_SLICE), desc_sw32(st + IA_BYTES + (l - i) * B_SLICE), idesc,
                                        (first && i == 0) ? 0u : 1u);
                }
                commit<CG>(&empty[s]);
                if (it % ISPB == ISPB - 1) commit<CG>(&tmem_full);
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    cluster_sync();
    if (warp == 0) {
        if constexpr (CG == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
    }
}

__global__ void fill_random(uint32_t *p, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        p[i] = (uint32_t)i * 2654435761u ^ (uint32_t)(i >> 32) * 40503u ^ 0x5bd1e995u * (uint32_t)(i >> 7);
}

template <int ORDER, int CG, bool UCOPY, bool PROD>
static void run(const char *name, const unsigned char *slices, double *out) {
    auto k = probe<ORDER, CG, UCOPY, PROD>;
    const int smem = (CG == 2 ? 5 * (IA_BYTES + IS * 32 * IK) : 4 * (IA_BYTES + IS * 64 * IK)) + 1024;
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(MT * NT * CHUNKS); cfg.blockDim = dim3(ITHREADS); cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    uint64_t seed = 1234;
    cudaLaunchKernelEx(&cfg, k, slices, out, seed);               // warm-up
    float best = 1e30f;
    for (int rep = 0; rep < 3; ++rep) {
        cudaEventRecord(e0);
        cudaLaunchKernelEx(&cfg, k, slices, out, seed);
        cudaEventRecord(e1); cudaEventSynchronize(e1);
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    const double macs = 36.0 * IBM * IBN * IK * (double)BPC * ISPB * MT * NT * CHUNKS;
    printf("%-66s %8.2f ms  %6.0f T int8 MAC/s  (%s)\n", name, best, macs / best / 1e9, cudaGetErrorString(cudaGetLastError()));
    fflush(stdout);
}

int main() {
    const int64_t bytes = (int64_t)MT * CHUNKS * BPC * ISPB * IA_BYTES;    // U slices of the C2 block: 16 GB
    unsigned char *slices; double *out;
    if (cudaMalloc(&slices, bytes) != cudaSuccess || cudaMalloc(&out, (size_t)MT * NT * CHUNKS * 256 * 8) != cudaSuccess) {
        printf("allocation failed\n");
        return 1;
    }
    fill_random<<<1024, 256>>>(reinterpret_cast<uint32_t *>(slices), bytes / 4);
    run<0, 1, false, false>("1: 36 MMAs, resident operands, level-major", slices, out);
    run<1, 1, false, false>("2: + A-slice-major, A collector", slices, out);
    run<1, 2, false, false>("3: + cta_group::2 pair MMA (M = 256)", slices, out);
    run<1, 2, true, false>("4: + U-slice bulk copies, full / empty barriers", slices, out);
    run<1, 2, true, true>("5: + Theta producers (32 rows per CTA)", slices, out);
    run<0, 1, true, true>("5p: one-CTA level-major MMAs, U copies, producers of 64 rows", slices, out);
    run<2, 1, false, false>("2w: 12 MMAs of N = 64 (8 - i) <= 256, resident operands", slices, out);
    run<2, 1, true, false>("4w: 2w + U-slice bulk copies, full / empty barriers", slices, out);
    run<2, 1, true, true>("5w: 4w + Theta producers of 64 rows", slices, out);
    cudaFree(slices); cudaFree(out);
    return 0;
}
