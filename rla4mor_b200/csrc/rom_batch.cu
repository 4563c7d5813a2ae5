// rom_batch.cu -- the online half of the sketched ROM over a whole parameter set: the reduced
// Galerkin solve and the sketched residual norm for P parameter values in one launch each.
// Replaces, per mu_p, the StationaryModel solve and ResidualErrorEstimator.estimate_error of
// mor/sketched_reductor.py:165-166,210-219 (SketchedRom.solve / estimate_error).
//
// rom_solve_batch_kernel: one CTA per mu (grid-stride loop over mu), the augmented system
// [A_p | b_p] (r x (r + 1), row-major) in shared memory:
//   * A_p = sum_q th[p, q] A_q and b_p = sum_j tf[p, j] f_j, terms in ascending q / j, one fma each;
//   * LU with partial pivoting: the pivot is the largest |.| of the column, ties to the smallest row
//     (LAPACK's idamax rule); rows are swapped whole, b included, and the elimination updates b
//     with the trailing block (the forward solve);
//   * back substitution on the column of b.
// info[p] = 0, or i > 0 when U(i, i) (1-based) is exactly zero, LAPACK's convention; such a
// column is skipped as dgetf2 skips it and the row a_p is written as NaN.  Largest r: the
// augmented system must fit the 227 KB of shared memory of one CTA, r (r + 1) 8 bytes:
// RB_MAX_R = 169.  Threads per CTA from r: 32 up to r = 32, 128 up to 64, 256 beyond.
//
// rom_lstsq_batch_kernel: the least-squares (minres) ROM, mor/sketched_reductor.py:170-187 (LsOperator,
// utilities/other_operators.py:12-39):  a_p = argmin_a || sum_q th[p, q] M_q a - sum_j tf[p, j] g_j ||_2
// with M_q: k_eff x r, g_j: k_eff, read from the row-major stack W = [M_0^T; ...; g_0^T; ...] (N x k_eff,
// the residual kernel's layout).  One CTA per mu (grid-stride loop), TSQR in one CTA:
//   * R (r x r) and the transformed right-hand side d stay in shared memory as [R | d], zero at first;
//   * rows of [M(mu) | b(mu)] are assembled in panels of c rows straight from W (terms in ascending
//     q / j, one fma each; W is shared by every mu and stays in L2);
//   * each panel is folded into [R d; panel] by Householder reflections in LAPACK's dlarfg convention
//     (beta = -sign(alpha) ||(alpha, x)||, tau = 0 for a zero column), but ||(alpha, x)|| is the plain
//     sqrt(alpha^2 + sum x_i^2), without dnrm2 / dlapy2 scaling or dlarfg's safmin rescaling: columns
//     with entries below ~1e-154 underflow (tau = 0, R(j, j) may become an exact zero) and entries
//     above ~1e154 overflow.  Reflector j touches row j of R and the panel's rows only.  Column k
//     belongs to the group of G lanes k % (threads / G), whose lanes hold rows lg, lg + G, ...: dot
//     products are a fixed fma chain per lane and a fixed shuffle tree, and one barrier per
//     reflector suffices;
//   * back substitution on d by one warp.
// Every sum runs in a fixed order and there are no atomics; the configuration depends on r only, so a
// mu's result depends on its own inputs only (P = 1 and P = 10^5 give the same bits).  info[p] = 0,
// or the first 1-based i with R(i, i) exactly zero (dtrtrs' convention), and a_p is then NaN.
// Launch rule (rl_config; threads {64 .. 512} x G {2, 4, 8} x c {32, 64, 128} timed at P = 10^5 on a
// B200 by tools/sweep_rom_lstsq.py, profiles/rom_lstsq_sweep.jsonl: the fastest at r = 64 and 128,
// within 12 % of the fastest, 64 threads and G = 8, at r = 16): c = 64 rows per panel; up to r = 32, 64 threads and G = 4; up to 64, 256 threads and G = 8; beyond, 512 threads
// and G = 8.  Largest r: [R | d] and the panel,
// r (r + 1) + (r + 1)(c + G) doubles, in 227 KB: RL_MAX_R = 137.  k_eff and Q are limited only by
// 64-bit indexing.
//
// residual_norm_batch_kernel:  est[p] = || sum_q th[p, q] S_q a_p - sum_j tf[p, j] g_j ||_2
// as one product R(P, k') = X(P, N) W(N, k'), N = Q r + Pf, with
//   W = [S_0^T; ...; S_{Q-1}^T; g_0^T; ...]   (the ROM's (r, k') row blocks and (k',) vectors)
//   X[p, q r + i] = th[p, q] a[p, i],  X[p, Q r + j] = -tf[p, j]   (formed in the kernel).
// The CTA tile and the DMMA fragment layout are lincomb_mma_kernel's 128 x 128 (lincomb.cu): W
// streams through a 3-stage cp.async ring; each thread loads its 8 entries of the X chunk two
// chunks ahead into registers and writes their products to the ring after the chunk's MMAs.  R is
// never stored: the tile squares its entries and sums them per row (fixed order in a thread, a fixed
// shuffle tree over the 4 lanes of a row, the 4 column warps in order) into ws[tile_n][p]; a second
// kernel adds the ceil(k' / 128) partial sums of each row in tile order and takes sqrt.  No atomics:
// results are bit-identical from run to run.
#include "common.cuh"
#include <algorithm>
#include <math.h>

namespace rla {
namespace {

constexpr int RB_MAX_R = 169;

__global__ void rom_solve_batch_kernel(const double *__restrict__ lhs, int Q, int r, const double *__restrict__ rhs,
                                       int Pf, const double *__restrict__ th, int64_t ldth,
                                       const double *__restrict__ tf, int64_t ldtf, int64_t P,
                                       double *__restrict__ a, int64_t lda, int32_t *__restrict__ info) {
    extern __shared__ __align__(16) double rs_smem[];
    __shared__ int s_piv;
    const int ld = r + 1, tid = threadIdx.x, nt = blockDim.x;
    double *M = rs_smem;                                              // r x (r + 1): [A | b]
    for (int64_t p = blockIdx.x; p < P; p += gridDim.x) {
        const double *thp = th + p * ldth, *tfp = tf + p * ldtf;
        for (int e = tid; e < r * r; e += nt) {
            double s = 0.0;
            for (int q = 0; q < Q; ++q) s = fma(__ldg(thp + q), __ldg(lhs + (int64_t)q * r * r + e), s);
            M[(e / r) * ld + e % r] = s;
        }
        for (int i = tid; i < r; i += nt) {
            double s = 0.0;
            for (int j = 0; j < Pf; ++j) s = fma(__ldg(tfp + j), __ldg(rhs + (int64_t)j * r + i), s);
            M[i * ld + r] = s;
        }
        int inf = 0;                                                  // the same value in every thread
        __syncthreads();
        for (int k = 0; k < r; ++k) {
            if (tid < 32) {
                double best = -1.0;
                int bi = r;
                for (int i = k + tid; i < r; i += 32) {
                    const double v = fabs(M[i * ld + k]);
                    if (v > best) { best = v; bi = i; }
                }
#pragma unroll
                for (int off = 16; off; off >>= 1) {
                    const double ob = __shfl_xor_sync(0xffffffffu, best, off);
                    const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
                    if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
                }
                // all-NaN column: no row compares greater, keep row k (the NaN propagates)
                if (tid == 0) s_piv = best == 0.0 ? -1 : (bi < r ? bi : k);
            }
            __syncthreads();
            const int pv = s_piv;
            if (pv < 0) {                                            // U(k, k) == 0: dgetf2 skips the column
                if (inf == 0) inf = k + 1;
                __syncthreads();
                continue;
            }
            if (pv != k)
                for (int j = tid; j <= r; j += nt) {
                    const double t = M[k * ld + j];
                    M[k * ld + j] = M[pv * ld + j];
                    M[pv * ld + j] = t;
                }
            __syncthreads();
            const double piv = M[k * ld + k];
            for (int i = k + 1 + tid; i < r; i += nt) M[i * ld + k] /= piv;
            __syncthreads();
            const int w = r - k;                                     // trailing columns k+1 .. r (b included)
            const int n = (r - k - 1) * w;
            for (int e = tid; e < n; e += nt) {
                const int i = k + 1 + e / w, j = k + 1 + e % w;
                M[i * ld + j] = fma(-M[i * ld + k], M[k * ld + j], M[i * ld + j]);
            }
            __syncthreads();
        }
        double *ap = a + p * lda;
        if (inf != 0) {
            for (int i = tid; i < r; i += nt) ap[i] = __longlong_as_double(0x7ff8000000000000LL);
        } else {
            for (int k = r - 1; k >= 0; --k) {
                const double x = M[k * ld + r] / M[k * ld + k];
                if (tid == 0) ap[k] = x;
                for (int i = tid; i < k; i += nt) M[i * ld + r] = fma(-M[i * ld + k], x, M[i * ld + r]);
                __syncthreads();
            }
        }
        if (tid == 0) info[p] = inf;
        __syncthreads();                                             // M is reused by the next mu
    }
}

// ------------------------------------------------------------------ least-squares solve
// Shared memory of one CTA: [R | d] (r x (r + 1), row-major) and the panel [Y | y] column-major,
// column k at Y + k ldy with ldy = c + G (a multiple of 16 plus G: the G-lane groups of a warp
// read different columns without bank conflicts).
__host__ __device__ constexpr int64_t rl_smem_doubles(int r, int c, int G) {
    return (int64_t)r * (r + 1) + (int64_t)(r + 1) * (c + G);
}

__global__ void __launch_bounds__(512, 2)
rom_lstsq_batch_kernel(const double *__restrict__ W, int64_t ldw, int Q, int r, int Pf, int64_t ke,
                       const double *__restrict__ th, int64_t ldth, const double *__restrict__ tf, int64_t ldtf,
                       int64_t P, double *__restrict__ a, int64_t lda, int32_t *__restrict__ info, int G, int c) {
    extern __shared__ __align__(16) double rl_smem[];
    __shared__ double s_tau[2];
    const int ld = r + 1, ldy = c + G, tid = threadIdx.x, nt = blockDim.x;
    const int lg = tid & (G - 1), grp = tid / G, ng = nt / G;     // G lanes per column, ng column groups
    const unsigned gmask = G == 32 ? 0xffffffffu : ((1u << G) - 1u) << ((tid & 31) & ~(G - 1));
    double *R = rl_smem;                                              // [R | d]
    double *Y = rl_smem + r * ld;                                     // [Y | y], c x (r + 1)
    for (int64_t p = blockIdx.x; p < P; p += gridDim.x) {
        const double *thp = th + p * ldth, *tfp = tf + p * ldtf;
        for (int e = tid; e < r * ld; e += nt) R[e] = 0.0;
        for (int64_t i0 = 0; i0 < ke; i0 += c) {
            // rows i0 .. i0 + cl - 1 of [M(mu) | b(mu)]; consecutive threads read consecutive columns of W
            const int cl = ke - i0 < c ? (int)(ke - i0) : c;
            for (int e = tid; e < ld * cl; e += nt) {
                const int k = e / cl, i = e - k * cl;
                double s = 0.0;
                if (k < r)
                    for (int q = 0; q < Q; ++q) s = fma(__ldg(thp + q), __ldg(W + ((int64_t)q * r + k) * ldw + i0 + i), s);
                else
                    for (int j = 0; j < Pf; ++j) s = fma(__ldg(tfp + j), __ldg(W + ((int64_t)Q * r + j) * ldw + i0 + i), s);
                Y[k * ldy + i] = s;
            }
            __syncthreads();
            // Householder QR of [R d; Y y]: reflector j touches row j of R and the cl panel rows.  Column
            // k is owned by group k % ng, whose lane lg holds rows lg, lg + G, ...; the group that owns
            // column j forms reflector j after it has applied reflector j - 1 to it, so one barrier
            // per reflector orders everything (tau is double-buffered).
            for (int j = 0; j < r; ++j) {
                if (grp == j % ng) {                                  // dlarfg on (R(j, j), Y(:, j))
                    double *v = Y + j * ldy;
                    double ss = 0.0;
                    for (int i = lg; i < cl; i += G) ss = fma(v[i], v[i], ss);
                    for (int off = G >> 1; off; off >>= 1) ss += __shfl_xor_sync(gmask, ss, off);
                    double tau = 0.0;                                 // zero column: H = I
                    if (ss != 0.0) {
                        const double alpha = R[j * ld + j];
                        const double h = sqrt(fma(alpha, alpha, ss));
                        const double beta = alpha >= 0.0 ? -h : h;    // beta = -sign(alpha) ||(alpha, x)||
                        tau = (beta - alpha) / beta;
                        const double sc = 1.0 / (alpha - beta);
                        for (int i = lg; i < cl; i += G) v[i] *= sc;
                        __syncwarp(gmask);                            // every lane has read alpha
                        if (lg == 0) R[j * ld + j] = beta;
                    }
                    if (lg == 0) s_tau[j & 1] = tau;
                }
                __syncthreads();
                const double tau = s_tau[j & 1];
                if (tau != 0.0) {
                    const double *v = Y + j * ldy;
                    for (int k = j + 1 + ((grp - (j + 1) % ng) + ng) % ng; k <= r; k += ng) {
                        double *y = Y + k * ldy;
                        const double rjk = R[j * ld + k];
                        double s = 0.0;
                        for (int i = lg; i < cl; i += G) s = fma(v[i], y[i], s);
                        for (int off = G >> 1; off; off >>= 1) s += __shfl_xor_sync(gmask, s, off);
                        const double w = tau * (rjk + s);
                        for (int i = lg; i < cl; i += G) y[i] = fma(-w, v[i], y[i]);
                        __syncwarp(gmask);                            // every lane has read R(j, k)
                        if (lg == 0) R[j * ld + k] = rjk - w;
                    }
                }
            }
            __syncthreads();                                          // the next panel overwrites Y
        }
        if (tid < 32) {                                               // info, then back substitution
            int bad = r;
            for (int i = tid; i < r; i += 32)
                if (R[i * ld + i] == 0.0) { bad = i; break; }
#pragma unroll
            for (int off = 16; off; off >>= 1) bad = min(bad, __shfl_xor_sync(0xffffffffu, bad, off));
            double *ap = a + p * lda;
            if (bad < r) {
                for (int i = tid; i < r; i += 32) ap[i] = __longlong_as_double(0x7ff8000000000000LL);
            } else {
                for (int k = r - 1; k >= 0; --k) {
                    const double x = R[k * ld + r] / R[k * ld + k];
                    if (tid == 0) ap[k] = x;
                    for (int i = tid; i < k; i += 32) R[i * ld + r] = fma(-R[i * ld + k], x, R[i * ld + r]);
                    __syncwarp();
                }
            }
            if (tid == 0) info[p] = bad < r ? bad + 1 : 0;
        }
        __syncthreads();                                              // R is reused by the next mu
    }
}

// ------------------------------------------------------------------ residual norm
constexpr int RN_BM = 128, RN_BN = 128, RN_BK = 16, RN_STAGES = 3;
constexpr int RN_LDW = RN_BN + 4, RN_LDX = RN_BK + 4;               // 4 (mod 16): conflict-free fragments
constexpr int RN_THREADS = 256;

__device__ __forceinline__ void rn_cp16(void *smem, const void *gmem, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;"
                 ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void rn_cp8(void *smem, const void *gmem, int src_bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;"
                 ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void rn_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void rn_wait1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }
__device__ __forceinline__ void rn_dmma(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(RN_THREADS, 1)
residual_norm_batch_kernel(const double *__restrict__ W, int64_t ldw, int64_t Q, int64_t r, int64_t Pf, int64_t kp,
                           const double *__restrict__ th, int64_t ldth, const double *__restrict__ tf, int64_t ldtf,
                           const double *__restrict__ a, int64_t lda, int64_t P, double *__restrict__ ws,
                           int ntiles, int vec_w) {
    constexpr int WTM = 64, WN = 4, MI = WTM / 8;                    // 2 x 4 warps of 64 x 32
    constexpr int WS = RN_BK * RN_LDW, XS = RN_BM * RN_LDX;          // doubles per stage
    extern __shared__ __align__(16) unsigned char rn_smem[];
    double *sw = reinterpret_cast<double *>(rn_smem);
    double *sx = sw + RN_STAGES * WS;
    __shared__ double red[WN][RN_BM];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const int wm = warp / WN, wn = warp % WN;
    // the n tiles of one m tile are adjacent in launch order: the rows of a and th are re-read from L2
    const int64_t n0 = (int64_t)(blockIdx.x % ntiles) * RN_BN;
    const int64_t m0 = (int64_t)(blockIdx.x / ntiles) * RN_BM;
    const int64_t QR = Q * r, N = QR + Pf;
    const int nchunks = (int)((N + RN_BK - 1) / RN_BK);

    auto load_w = [&](int st, int c) {
        const int64_t k0 = (int64_t)c * RN_BK;
        double *dw = sw + st * WS;
        if (vec_w) {
            for (int id = tid; id < RN_BK * (RN_BN / 2); id += RN_THREADS) {
                const int kk = id / (RN_BN / 2), cc = (id % (RN_BN / 2)) * 2;
                const int64_t row = k0 + kk, col = n0 + cc;
                const int bytes = (row < N && col < kp) ? (col + 1 < kp ? 16 : 8) : 0;
                rn_cp16(dw + kk * RN_LDW + cc, bytes ? W + row * ldw + col : W, bytes);
            }
        } else {
            for (int id = tid; id < RN_BK * RN_BN; id += RN_THREADS) {
                const int kk = id / RN_BN, cc = id % RN_BN;
                const int64_t row = k0 + kk, col = n0 + cc;
                const int bytes = (row < N && col < kp) ? 8 : 0;
                rn_cp8(dw + kk * RN_LDW + cc, bytes ? W + row * ldw + col : W, bytes);
            }
        }
    };
    // thread tid owns the X entries (rows tid / 16 + 16 e, e = 0..7; column tid % 16) of every chunk
    const int xc = tid % RN_BK, xr = tid / RN_BK;
    double xa[8], xt[8];
    auto fetch_x = [&](int c) {
        const int col = c * RN_BK + xc;                          // N < 2^31: 32-bit division
        const bool lhs_col = col < QR, rhs_col = !lhs_col && col < N;
        const int q = lhs_col ? col / (int)r : 0, i = lhs_col ? col - q * (int)r : 0, j = (int)(col - QR);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int64_t row = m0 + xr + 16 * e;
            const bool live = row < P;
            xa[e] = (live && lhs_col) ? __ldg(a + row * lda + i) : 0.0;
            xt[e] = (live && lhs_col) ? __ldg(th + row * ldth + q) : ((live && rhs_col) ? -__ldg(tf + row * ldtf + j) : 0.0);
        }
        return lhs_col;
    };
    auto store_x = [&](int st, bool lhs_col) {
        double *dx = sx + st * XS;
#pragma unroll
        for (int e = 0; e < 8; ++e) dx[(xr + 16 * e) * RN_LDX + xc] = lhs_col ? xt[e] * xa[e] : xt[e];
    };

    double acc[MI][4][2];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

#pragma unroll
    for (int s = 0; s < RN_STAGES - 1; ++s) {
        if (s < nchunks) {
            load_w(s, s);
            store_x(s, fetch_x(s));
        }
        rn_commit();
    }
    for (int c = 0; c < nchunks; ++c) {
        rn_wait1();
        __syncthreads();                                 // chunk c has landed; everyone is done with chunk c - 1
        const int nxt = c + RN_STAGES - 1;
        bool nxt_lhs = false;
        if (nxt < nchunks) {
            load_w(nxt % RN_STAGES, nxt);
            nxt_lhs = fetch_x(nxt);                      // consumed after this chunk's MMAs
        }
        rn_commit();
        const double *pw = sw + (c % RN_STAGES) * WS + wn * 32 + g;
        const double *px = sx + (c % RN_STAGES) * XS + (wm * WTM + g) * RN_LDX + t;
#pragma unroll
        for (int ks = 0; ks < RN_BK / 4; ++ks) {
            double fa[MI], fb[4];
#pragma unroll
            for (int i = 0; i < MI; ++i) fa[i] = px[i * 8 * RN_LDX + ks * 4];
#pragma unroll
            for (int j = 0; j < 4; ++j) fb[j] = pw[(ks * 4 + t) * RN_LDW + j * 8];
#pragma unroll
            for (int i = 0; i < MI; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) rn_dmma(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
        }
        if (nxt < nchunks) store_x(nxt % RN_STAGES, nxt_lhs);
    }
    // fused norm epilogue: entries outside P x k' are exact zeros (zero-filled W columns, zero X rows)
#pragma unroll
    for (int i = 0; i < MI; ++i) {
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            s = fma(acc[i][j][0], acc[i][j][0], s);
            s = fma(acc[i][j][1], acc[i][j][1], s);
        }
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        if (t == 0) red[wn][wm * WTM + 8 * i + g] = s;
    }
    __syncthreads();
    if (tid < RN_BM && m0 + tid < P) {
        double s = red[0][tid];
#pragma unroll
        for (int w = 1; w < WN; ++w) s += red[w][tid];
        ws[(int64_t)(blockIdx.x % ntiles) * P + m0 + tid] = s;
    }
}

__global__ void residual_norm_batch_reduce_kernel(const double *__restrict__ ws, int ntiles, int64_t P,
                                                  double *__restrict__ est) {
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= P) return;
    double s = 0.0;
    for (int n = 0; n < ntiles; ++n) s += ws[(int64_t)n * P + p];
    est[p] = sqrt(s);
}

int64_t rn_tiles(int64_t kp) { return (kp + RN_BN - 1) / RN_BN; }

struct RlConfig {
    int threads, G, c;
};
constexpr RlConfig rl_config(int r) {
    return r <= 32 ? RlConfig{64, 4, 64} : (r <= 64 ? RlConfig{256, 8, 64} : RlConfig{512, 8, 64});
}
constexpr int64_t RL_SMEM_LIMIT = 227 * 1024 - 2 * sizeof(double);   // less the static s_tau
constexpr int rl_max_r() {
    int r = 1;
    while (rl_smem_doubles(r + 1, rl_config(r + 1).c, rl_config(r + 1).G) * 8 <= RL_SMEM_LIMIT) ++r;
    return r;
}
constexpr int RL_MAX_R = rl_max_r();
static_assert(RL_MAX_R >= 128, "the least-squares batch must hold r = 128");

}  // namespace
}  // namespace rla

using namespace rla;

extern "C" int rla_rom_solve_batch_max_r(void) { return RB_MAX_R; }

extern "C" int rla_rom_solve_batch_f64(const double *lhs_dev, int64_t Q, int64_t r, const double *rhs_dev, int64_t Pf,
                                       const double *th_dev, int64_t ldth, const double *tf_dev, int64_t ldtf, int64_t P,
                                       double *a_dev, int64_t lda, int32_t *info_dev, void *stream) {
    RLA_REQUIRE(Q >= 0 && Pf >= 0 && P >= 0 && r >= 1 && ldth >= Q && ldtf >= Pf && lda >= r,
                "rla_rom_solve_batch_f64: bad sizes");
    RLA_REQUIRE(r <= RB_MAX_R, "rla_rom_solve_batch_f64: r=%lld exceeds the largest supported r=%d",
                (long long)r, RB_MAX_R);
    RLA_REQUIRE(Q < (1 << 30) && Pf < (1 << 30), "rla_rom_solve_batch_f64: too many affine terms");
    if (P == 0) return RLA_OK;
    RLA_REQUIRE(a_dev && info_dev && (Q == 0 || (lhs_dev && th_dev)) && (Pf == 0 || (rhs_dev && tf_dev)),
                "rla_rom_solve_batch_f64: null pointer");
    const int threads = r <= 32 ? 32 : (r <= 64 ? 128 : 256);
    const int smem = (int)(r * (r + 1) * sizeof(double));
    RLA_CUDA_CHECK(cudaFuncSetAttribute(rom_solve_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int per_sm = 0;
    RLA_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rom_solve_batch_kernel, threads, smem));
    const int64_t grid = std::min<int64_t>(P, (int64_t)std::max(per_sm, 1) * sm_count());
    rom_solve_batch_kernel<<<(unsigned)grid, threads, smem, (cudaStream_t)stream>>>(
        lhs_dev, (int)Q, (int)r, rhs_dev, (int)Pf, th_dev, ldth, tf_dev, ldtf, P, a_dev, lda, info_dev);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

extern "C" int rla_rom_lstsq_batch_max_r(void) { return RL_MAX_R; }

extern "C" int rla_rom_lstsq_batch_f64(const double *W_dev, int64_t ldw, int64_t Q, int64_t r, int64_t Pf, int64_t ke,
                                       const double *th_dev, int64_t ldth, const double *tf_dev, int64_t ldtf, int64_t P,
                                       double *a_dev, int64_t lda, int32_t *info_dev, void *stream) {
    RLA_REQUIRE(Q >= 0 && Pf >= 0 && P >= 0 && r >= 1 && ke >= 1 && ldw >= ke && ldth >= Q && ldtf >= Pf && lda >= r,
                "rla_rom_lstsq_batch_f64: bad sizes");
    RLA_REQUIRE(r <= RL_MAX_R, "rla_rom_lstsq_batch_f64: r=%lld exceeds the largest supported r=%d",
                (long long)r, RL_MAX_R);
    RLA_REQUIRE(ke >= r, "rla_rom_lstsq_batch_f64: k_eff=%lld < r=%lld: the system is underdetermined",
                (long long)ke, (long long)r);
    RLA_REQUIRE(Q < (1 << 30) && Pf < (1 << 30), "rla_rom_lstsq_batch_f64: too many affine terms");
    if (P == 0) return RLA_OK;
    RLA_REQUIRE(a_dev && info_dev && W_dev && (Q == 0 || th_dev) && (Pf == 0 || tf_dev),
                "rla_rom_lstsq_batch_f64: null pointer");
    const RlConfig cfg = rl_config((int)r);
    const int smem = (int)(rl_smem_doubles((int)r, cfg.c, cfg.G) * sizeof(double));
    RLA_CUDA_CHECK(cudaFuncSetAttribute(rom_lstsq_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int per_sm = 0;
    RLA_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rom_lstsq_batch_kernel, cfg.threads, smem));
    const int64_t grid = std::min<int64_t>(P, (int64_t)std::max(per_sm, 1) * sm_count());
    rom_lstsq_batch_kernel<<<(unsigned)grid, cfg.threads, smem, (cudaStream_t)stream>>>(
        W_dev, ldw, (int)Q, (int)r, (int)Pf, ke, th_dev, ldth, tf_dev, ldtf, P, a_dev, lda, info_dev, cfg.G, cfg.c);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

extern "C" size_t rla_residual_norm_batch_workspace_bytes(int64_t P, int64_t kp) {
    if (P <= 0 || kp <= 0) return 0;
    return (size_t)(rn_tiles(kp) * P) * sizeof(double);
}

extern "C" int rla_residual_norm_batch_f64(const double *W_dev, int64_t ldw, int64_t Q, int64_t r, int64_t Pf,
                                           int64_t kp, const double *th_dev, int64_t ldth, const double *tf_dev,
                                           int64_t ldtf, const double *a_dev, int64_t lda, int64_t P,
                                           double *est_dev, void *ws_dev, size_t ws_bytes, void *stream) {
    RLA_REQUIRE(Q >= 0 && r >= 0 && Pf >= 0 && kp >= 1 && P >= 0 && ldw >= kp && ldth >= Q && ldtf >= Pf &&
                lda >= r, "rla_residual_norm_batch_f64: bad sizes");
    if (P == 0) return RLA_OK;
    RLA_REQUIRE(est_dev && ws_dev && (Q * r + Pf == 0 || W_dev) && (Q * r == 0 || (th_dev && a_dev)) &&
                (Pf == 0 || tf_dev), "rla_residual_norm_batch_f64: null pointer");
    RLA_REQUIRE(ws_bytes >= rla_residual_norm_batch_workspace_bytes(P, kp),
                "rla_residual_norm_batch_f64: workspace of %zu bytes, %zu needed", ws_bytes,
                rla_residual_norm_batch_workspace_bytes(P, kp));
    const int64_t ntiles = rn_tiles(kp), mtiles = (P + RN_BM - 1) / RN_BM;
    RLA_REQUIRE(ntiles * mtiles < (int64_t(1) << 31) && Q * r + Pf < (int64_t(1) << 30),
                "rla_residual_norm_batch_f64: problem too large");
    cudaStream_t st = (cudaStream_t)stream;
    const int vec_w = (reinterpret_cast<uintptr_t>(W_dev) % 16 == 0) && (ldw % 2 == 0);
    const int smem = (int)(RN_STAGES * (RN_BK * RN_LDW + RN_BM * RN_LDX) * sizeof(double));
    RLA_CUDA_CHECK(cudaFuncSetAttribute(residual_norm_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    double *ws = static_cast<double *>(ws_dev);
    residual_norm_batch_kernel<<<(unsigned)(ntiles * mtiles), RN_THREADS, smem, st>>>(
        W_dev, ldw, Q, r, Pf, kp, th_dev, ldth, tf_dev, ldtf, a_dev, lda, P, ws, (int)ntiles, vec_w);
    count_launch();
    residual_norm_batch_reduce_kernel<<<(unsigned)((P + 255) / 256), 256, 0, st>>>(ws, (int)ntiles, P, est_dev);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}
