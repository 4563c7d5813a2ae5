// affine_cg.cu -- block preconditioned CG for the affine full-order model
//   A(mu_p) x_p = b_p,   A(mu_p) = sum_q th[p, q] A_q   (symmetric positive definite),
// one row p of every (P, n) block per parameter value mu_p (pyMOR's StationaryModel.solve ->
// apply_inverse over a block of mu; fom_solve.py drives the iteration).  The preconditioner
// z = R^-1 r (the sparse LU of the inner product, sptrsv.cu) runs between these kernels.
//
// Every inner product <a_p, b_p> is written as one partial sum per tile of ACG_TILE consecutive
// entries (ws[p * ntiles + tile]) and the partials of a row are added in tile order by one CTA per
// row.  No atomics, and the tiles depend on n only: a row's result does not depend on P or on which
// other rows are still iterating, and two runs give the same bits.
#include "common.cuh"
#include <algorithm>

namespace rla {
namespace {

constexpr int ACG_TILE = 256;        // operator rows per CTA of the SpMM = entries per partial sum
constexpr int ACG_WARPS = ACG_TILE / 32;
constexpr int ACG_MAX_Q = 32;

// istate rows (int32, P each): iterations, info, mode.  mode: what the next vector kernels do with row p
enum : int32_t { CG_IDLE = 0, CG_LAST = 1, CG_LIVE = 2 };
// state rows (double, P each)
enum { S_RHO = 0, S_RHOB = 1, S_ALPHA = 2, S_BETA = 3, S_RESID = 4 };
enum { I_ITERS = 0, I_INFO = 1, I_MODE = 2 };

__host__ __device__ inline int64_t acg_tiles(int64_t n) { return (n + ACG_TILE - 1) / ACG_TILE; }

// Deterministic sum of VB values over the CTA: a fixed xor-shuffle tree inside each warp (every lane
// ends with the same bits), then the warp partials in warp order.  Thread v < VB writes row c0 + v.
template <int VB>
__device__ __forceinline__ void tile_sums(double (&d)[VB], double (*red)[VB], double *__restrict__ ws, int64_t nt,
                                          int64_t tile, int64_t c0, unsigned live) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int v = 0; v < VB; ++v) {
#pragma unroll
        for (int off = 16; off; off >>= 1) d[v] += __shfl_xor_sync(0xffffffffu, d[v], off);
    }
    if (lane == 0) {
#pragma unroll
        for (int v = 0; v < VB; ++v) red[warp][v] = d[v];
    }
    __syncthreads();
    if (threadIdx.x < VB && ((live >> threadIdx.x) & 1u)) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < ACG_WARPS; ++w) s += red[w][threadIdx.x];
        ws[(c0 + threadIdx.x) * nt + tile] = s;
    }
    __syncthreads();
}

template <int VB>
__device__ __forceinline__ unsigned live_rows(int64_t c0, int64_t P, const int32_t *__restrict__ mode) {
    unsigned live = 0;
#pragma unroll
    for (int v = 0; v < VB; ++v)
        if (c0 + v < P && (!mode || mode[c0 + v] == CG_LIVE)) live |= 1u << v;
    return live;
}

// ------------------------------------------------------------------ affine SpMM
// y[p, i] = sum_e (sum_q th[p, q] val[q, e]) x[p, col[e]] over the union pattern of the Q terms.
// Thread = operator row i, CTA = a tile of ACG_TILE rows for ACG_VB rows p of the block.  The CTAs of
// one tile are adjacent in launch order (blockIdx.x walks the rows of the block), so the tile's
// pattern and values come from HBM once and from L2 for the others.  The coefficients of the CTA's
// rows sit in shared memory as [q][v] (broadcast 16-byte reads), and two entries of a row are
// gathered at once (the x loads depend on the col loads).  Optional epilogue (ws != NULL): the tile's
// partial sums of <x_p, y_p>.  Rows whose mode is not CG_LIVE (mode != NULL) are skipped.
constexpr int ACG_VB = 8;

__global__ void __launch_bounds__(ACG_TILE, 2)
affine_spmm_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col, const double *__restrict__ val,
                   int64_t nnz, int Q, int64_t n, const double *__restrict__ th, int64_t ldth,
                   const double *__restrict__ x, int64_t ldx, int64_t P, double *__restrict__ y, int64_t ldy,
                   const int32_t *__restrict__ mode, double *__restrict__ ws) {
    constexpr int VB = ACG_VB;
    extern __shared__ double2 sth2[];                                // [Q][VB / 2]
    __shared__ double red[ACG_WARPS][VB];
    const int64_t c0 = (int64_t)blockIdx.x * VB;
    const unsigned live = live_rows<VB>(c0, P, mode);
    if (!live) return;                                               // uniform over the CTA
    double *sth = reinterpret_cast<double *>(sth2);
    for (int k = threadIdx.x; k < Q * VB; k += blockDim.x) {
        const int q = k / VB, v = k % VB;
        sth[k] = ((live >> v) & 1u) ? __ldg(th + (c0 + v) * ldth + q) : 0.0;
    }
    __syncthreads();
    const int64_t nt = acg_tiles(n);
    for (int64_t tile = blockIdx.y; tile < nt; tile += gridDim.y) {
        const int64_t i = tile * ACG_TILE + threadIdx.x;
        const bool row = i < n;
        const int64_t e0 = row ? __ldg(rowptr + i) : 0, e1 = row ? __ldg(rowptr + i + 1) : 0;
        double acc[VB];
#pragma unroll
        for (int v = 0; v < VB; ++v) acc[v] = 0.0;
#pragma unroll 2
        for (int64_t e = e0; e < e1; ++e) {
            const int64_t j = __ldg(col + e);
            double a[VB];
#pragma unroll
            for (int v = 0; v < VB; ++v) a[v] = 0.0;
            for (int q = 0; q < Q; ++q) {
                const double w = __ldg(val + q * nnz + e);
#pragma unroll
                for (int v2 = 0; v2 < VB / 2; ++v2) {
                    const double2 c = sth2[q * (VB / 2) + v2];
                    a[2 * v2] = fma(c.x, w, a[2 * v2]);
                    a[2 * v2 + 1] = fma(c.y, w, a[2 * v2 + 1]);
                }
            }
#pragma unroll
            for (int v = 0; v < VB; ++v)
                if ((live >> v) & 1u) acc[v] = fma(a[v], __ldg(x + (c0 + v) * ldx + j), acc[v]);
        }
        double d[VB];
#pragma unroll
        for (int v = 0; v < VB; ++v) {
            d[v] = 0.0;
            if (row && ((live >> v) & 1u)) {
                y[(c0 + v) * ldy + i] = acc[v];
                if (ws) d[v] = x[(c0 + v) * ldx + i] * acc[v];
            }
        }
        if (ws) tile_sums<VB>(d, red, ws, nt, tile, c0, live);
    }
}

// ------------------------------------------------------- per-tile row dot products
// ws[p * ntiles + tile] = sum over the tile of a[p, i] b[p, i]   (rows with mode CG_LIVE, or all)
template <int VB>
__global__ void __launch_bounds__(ACG_TILE)
row_dot_kernel(const double *__restrict__ a, int64_t lda, const double *__restrict__ b, int64_t ldb, int64_t n,
               int64_t P, const int32_t *__restrict__ mode, double *__restrict__ ws) {
    __shared__ double red[ACG_WARPS][VB];
    const int64_t nt = acg_tiles(n);
    for (int64_t tile = blockIdx.x; tile < nt; tile += gridDim.x) {
        const int64_t i = tile * ACG_TILE + threadIdx.x;
        for (int64_t c0 = 0; c0 < P; c0 += VB) {
            const unsigned live = live_rows<VB>(c0, P, mode);
            if (!live) continue;
            double d[VB];
#pragma unroll
            for (int v = 0; v < VB; ++v)
                d[v] = (i < n && ((live >> v) & 1u)) ? ldg_stream_f64(a + (c0 + v) * lda + i) *
                                                           ldg_stream_f64(b + (c0 + v) * ldb + i) : 0.0;
            tile_sums<VB>(d, red, ws, nt, tile, c0, live);
        }
    }
}

// ------------------------------------------------ second stage: one CTA per row
__device__ __forceinline__ double row_total(const double *__restrict__ ws, int64_t nt, int64_t p) {
    __shared__ double red[ACG_WARPS];
    double s = 0.0;
    for (int64_t t = threadIdx.x; t < nt; t += ACG_TILE) s += ws[p * nt + t];
#pragma unroll
    for (int off = 16; off; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    __syncthreads();                                                 // red is reused by the next row
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    double tot = 0.0;
#pragma unroll
    for (int w = 0; w < ACG_WARPS; ++w) tot += red[w];
    return tot;
}

__global__ void __launch_bounds__(ACG_TILE)
row_sum_kernel(const double *__restrict__ ws, int64_t nt, int64_t P, double *__restrict__ out) {
    for (int64_t p = blockIdx.x; p < P; p += gridDim.x) {
        const double s = row_total(ws, nt, p);
        if (threadIdx.x == 0) out[p] = s;
    }
}

// rho_0 = <r_0, R^-1 r_0>, rho_b = <b, R^-1 b>: a row with b = 0 is solved (x = 0) in 0 iterations,
// a row already within tol needs none; a negative (or NaN) dual norm is a breakdown
__global__ void __launch_bounds__(ACG_TILE)
cg_start_kernel(const double *__restrict__ ws_r, const double *__restrict__ ws_b, int64_t nt, int64_t P, double tol2,
                int64_t maxiter, double *__restrict__ st, int32_t *__restrict__ ist) {
    for (int64_t p = blockIdx.x; p < P; p += gridDim.x) {
        const double rho = row_total(ws_r, nt, p);
        const double rhob = ws_b == ws_r ? rho : row_total(ws_b, nt, p);
        if (threadIdx.x) continue;
        int32_t info = 0, mode = CG_IDLE;
        double resid = 0.0;
        if (!(rho >= 0.0) || !(rhob >= 0.0)) {
            info = 2;
            resid = __longlong_as_double(0x7ff8000000000000LL);
        } else if (rhob > 0.0) {
            resid = sqrt(rho / rhob);
            if (!(rho <= tol2 * rhob)) {
                if (maxiter > 0) mode = CG_LIVE;
                else info = 1;
            }
        }
        st[S_RHO * P + p] = rho;
        st[S_RHOB * P + p] = rhob;
        st[S_RESID * P + p] = resid;
        ist[I_ITERS * P + p] = 0;
        ist[I_INFO * P + p] = info;
        ist[I_MODE * P + p] = mode;
    }
}

// gamma = <p, A p>: alpha = rho / gamma, or a breakdown when gamma <= 0 (A(mu) not SPD)
__global__ void __launch_bounds__(ACG_TILE)
cg_alpha_kernel(const double *__restrict__ ws, int64_t nt, int64_t P, double *__restrict__ st, int32_t *__restrict__ ist) {
    for (int64_t p = blockIdx.x; p < P; p += gridDim.x) {
        if (ist[I_MODE * P + p] != CG_LIVE) continue;                // uniform over the CTA
        const double gamma = row_total(ws, nt, p);
        if (threadIdx.x) continue;
        if (gamma > 0.0) {
            st[S_ALPHA * P + p] = st[S_RHO * P + p] / gamma;
        } else {
            ist[I_INFO * P + p] = 2;
            ist[I_MODE * P + p] = CG_IDLE;
            st[S_RESID * P + p] = __longlong_as_double(0x7ff8000000000000LL);
        }
    }
}

// rho' = <r, R^-1 r> = ||r||^2 in the dual norm: converged (x takes its last step), out of
// iterations (likewise), breakdown (rho' < 0: the preconditioner is not SPD) or beta = rho' / rho.
// A row that took its last step in the previous iteration goes idle here.
__global__ void __launch_bounds__(ACG_TILE)
cg_beta_kernel(const double *__restrict__ ws, int64_t nt, int64_t P, double tol2, int64_t maxiter,
               double *__restrict__ st, int32_t *__restrict__ ist) {
    for (int64_t p = blockIdx.x; p < P; p += gridDim.x) {
        const int32_t mode = ist[I_MODE * P + p];
        if (mode != CG_LIVE) {
            if (mode == CG_LAST && threadIdx.x == 0) ist[I_MODE * P + p] = CG_IDLE;
            continue;
        }
        const double rho = row_total(ws, nt, p);
        if (threadIdx.x) continue;
        const int32_t it = ist[I_ITERS * P + p] + 1;
        ist[I_ITERS * P + p] = it;
        if (!(rho >= 0.0)) {
            ist[I_INFO * P + p] = 2;
            ist[I_MODE * P + p] = CG_IDLE;
            st[S_RESID * P + p] = __longlong_as_double(0x7ff8000000000000LL);
            continue;
        }
        const double rhob = st[S_RHOB * P + p];
        st[S_RESID * P + p] = sqrt(rho / rhob);
        if (rho <= tol2 * rhob) {
            ist[I_MODE * P + p] = CG_LAST;
        } else if (it >= maxiter) {
            ist[I_INFO * P + p] = 1;
            ist[I_MODE * P + p] = CG_LAST;
        } else {
            st[S_BETA * P + p] = rho / st[S_RHO * P + p];
            st[S_RHO * P + p] = rho;
        }
    }
}

// ------------------------------------------------------------ vector updates
// blockIdx.y walks the rows, blockIdx.x the entries of a row; a row that is not iterating costs one
// read of its mode per CTA
constexpr int ACG_UPD_BLOCKS = 512;

__global__ void __launch_bounds__(256)
cg_update_r_kernel(double *__restrict__ r, int64_t ldr, const double *__restrict__ q, int64_t ldq, int64_t n, int64_t P,
                   const double *__restrict__ st, const int32_t *__restrict__ ist) {
    for (int64_t p = blockIdx.y; p < P; p += gridDim.y) {
        if (ist[I_MODE * P + p] != CG_LIVE) continue;
        const double alpha = st[S_ALPHA * P + p];
        double *rp = r + p * ldr;
        const double *qp = q + p * ldq;
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
            rp[i] = fma(-alpha, ldg_stream_f64(qp + i), rp[i]);
    }
}

// x += alpha p for rows that took a step this iteration (CG_LIVE, CG_LAST); p = z + beta p for CG_LIVE
__global__ void __launch_bounds__(256)
cg_update_xp_kernel(double *__restrict__ x, int64_t ldx, double *__restrict__ pv, int64_t ldp,
                    const double *__restrict__ z, int64_t ldz, int64_t n, int64_t P,
                    const double *__restrict__ st, const int32_t *__restrict__ ist) {
    for (int64_t p = blockIdx.y; p < P; p += gridDim.y) {
        const int32_t mode = ist[I_MODE * P + p];
        if (mode == CG_IDLE) continue;
        const double alpha = st[S_ALPHA * P + p], beta = st[S_BETA * P + p];
        double *xp = x + p * ldx, *pp = pv + p * ldp;
        const double *zp = z + p * ldz;
        const int64_t i0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
        if (mode == CG_LIVE) {
            for (int64_t i = i0; i < n; i += stride) {
                const double pi = pp[i];
                xp[i] = fma(alpha, pi, xp[i]);
                pp[i] = fma(beta, pi, ldg_stream_f64(zp + i));
            }
        } else {
            for (int64_t i = i0; i < n; i += stride) xp[i] = fma(alpha, pp[i], xp[i]);
        }
    }
}

dim3 update_grid(int64_t n, int64_t P) {
    return dim3((unsigned)std::min<int64_t>((n + 255) / 256, ACG_UPD_BLOCKS), (unsigned)std::min<int64_t>(P, 65535));
}

unsigned row_grid(int64_t P) { return (unsigned)std::min<int64_t>(P, 65535); }

unsigned tile_grid(int64_t n) { return (unsigned)std::min<int64_t>(acg_tiles(n), INT32_MAX); }

}  // namespace
}  // namespace rla

using namespace rla;

#define ACG_WS_CHECK(what, n, P)                                                                                   \
    RLA_REQUIRE(ws && ws_bytes >= (size_t)(P) * acg_tiles(n) * sizeof(double),                                   \
                what ": workspace of %zu bytes, %zu needed", ws_bytes, (size_t)(P) * acg_tiles(n) * sizeof(double))

extern "C" size_t rla_affine_cg_workspace_bytes(int64_t n, int64_t P) {
    if (n <= 0 || P <= 0) return 0;
    return (size_t)P * (size_t)acg_tiles(n) * sizeof(double);
}

extern "C" int rla_affine_spmm_f64(const int64_t *rowptr, const int32_t *col, const double *val, int64_t nnz, int64_t Q,
                                   int64_t n, const double *th, int64_t ldth, const double *x, int64_t ldx, int64_t P,
                                   double *y, int64_t ldy, const int32_t *mode, void *ws, size_t ws_bytes,
                                   void *stream) {
    RLA_REQUIRE(n >= 0 && nnz >= 0 && P >= 0 && Q >= 1 && ldth >= Q && ldx >= n && ldy >= n,
                "rla_affine_spmm_f64: bad sizes");
    RLA_REQUIRE(Q <= ACG_MAX_Q, "rla_affine_spmm_f64: Q=%lld affine terms, at most %d supported", (long long)Q,
                ACG_MAX_Q);
    if (n == 0 || P == 0) return RLA_OK;
    RLA_REQUIRE(rowptr && th && x && y && (nnz == 0 || (col && val)), "rla_affine_spmm_f64: null pointer");
    if (ws) ACG_WS_CHECK("rla_affine_spmm_f64", n, P);
    cudaStream_t st = (cudaStream_t)stream;
    double *w = (double *)ws;
    dim3 grid((unsigned)((P + ACG_VB - 1) / ACG_VB), (unsigned)std::min<int64_t>(acg_tiles(n), 65535));
    affine_spmm_kernel<<<grid, ACG_TILE, Q * ACG_VB * sizeof(double), st>>>(rowptr, col, val, nnz, (int)Q, n, th, ldth,
                                                                           x, ldx, P, y, ldy, mode, w);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

extern "C" int rla_row_dot_partials_f64(const double *a, int64_t lda, const double *b, int64_t ldb, int64_t n, int64_t P,
                                        const int32_t *mode, void *ws, size_t ws_bytes, void *stream) {
    RLA_REQUIRE(n >= 0 && P >= 0 && lda >= n && ldb >= n, "rla_row_dot_partials_f64: bad sizes");
    if (n == 0 || P == 0) return RLA_OK;
    RLA_REQUIRE(a && b, "rla_row_dot_partials_f64: null pointer");
    ACG_WS_CHECK("rla_row_dot_partials_f64", n, P);
    row_dot_kernel<8><<<tile_grid(n), ACG_TILE, 0, (cudaStream_t)stream>>>(a, lda, b, ldb, n, P, mode, (double *)ws);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

extern "C" int rla_row_dot_sum_f64(const void *ws, size_t ws_bytes, int64_t n, int64_t P, double *out, void *stream) {
    RLA_REQUIRE(n >= 1 && P >= 0, "rla_row_dot_sum_f64: bad sizes");
    if (P == 0) return RLA_OK;
    RLA_REQUIRE(out, "rla_row_dot_sum_f64: null pointer");
    ACG_WS_CHECK("rla_row_dot_sum_f64", n, P);
    row_sum_kernel<<<row_grid(P), ACG_TILE, 0, (cudaStream_t)stream>>>((const double *)ws, acg_tiles(n), P, out);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

extern "C" int rla_affine_cg_start_f64(const void *ws_r, const void *ws_b, size_t ws_bytes, int64_t n, int64_t P,
                                       double tol, int64_t maxiter, double *state, int32_t *istate, void *stream) {
    RLA_REQUIRE(n >= 1 && P >= 0 && maxiter >= 0 && tol >= 0.0, "rla_affine_cg_start_f64: bad arguments");
    if (P == 0) return RLA_OK;
    RLA_REQUIRE(ws_b && state && istate, "rla_affine_cg_start_f64: null pointer");
    const void *ws = ws_r;
    ACG_WS_CHECK("rla_affine_cg_start_f64", n, P);
    cg_start_kernel<<<row_grid(P), ACG_TILE, 0, (cudaStream_t)stream>>>((const double *)ws_r, (const double *)ws_b,
                                                                         acg_tiles(n), P, tol * tol, maxiter, state,
                                                                         istate);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

extern "C" int rla_affine_cg_alpha_f64(const void *ws, size_t ws_bytes, int64_t n, int64_t P, double *state,
                                       int32_t *istate, void *stream) {
    RLA_REQUIRE(n >= 1 && P >= 0, "rla_affine_cg_alpha_f64: bad sizes");
    if (P == 0) return RLA_OK;
    RLA_REQUIRE(state && istate, "rla_affine_cg_alpha_f64: null pointer");
    ACG_WS_CHECK("rla_affine_cg_alpha_f64", n, P);
    cg_alpha_kernel<<<row_grid(P), ACG_TILE, 0, (cudaStream_t)stream>>>((const double *)ws, acg_tiles(n), P, state,
                                                                         istate);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

extern "C" int rla_affine_cg_beta_f64(const void *ws, size_t ws_bytes, int64_t n, int64_t P, double tol, int64_t maxiter,
                                      double *state, int32_t *istate, void *stream) {
    RLA_REQUIRE(n >= 1 && P >= 0 && maxiter >= 0 && tol >= 0.0, "rla_affine_cg_beta_f64: bad arguments");
    if (P == 0) return RLA_OK;
    RLA_REQUIRE(state && istate, "rla_affine_cg_beta_f64: null pointer");
    ACG_WS_CHECK("rla_affine_cg_beta_f64", n, P);
    cg_beta_kernel<<<row_grid(P), ACG_TILE, 0, (cudaStream_t)stream>>>((const double *)ws, acg_tiles(n), P, tol * tol,
                                                                        maxiter, state, istate);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

extern "C" int rla_affine_cg_update_r_f64(double *r, int64_t ldr, const double *q, int64_t ldq, int64_t n, int64_t P,
                                          const double *state, const int32_t *istate, void *stream) {
    RLA_REQUIRE(n >= 0 && P >= 0 && ldr >= n && ldq >= n, "rla_affine_cg_update_r_f64: bad sizes");
    if (n == 0 || P == 0) return RLA_OK;
    RLA_REQUIRE(r && q && state && istate, "rla_affine_cg_update_r_f64: null pointer");
    cg_update_r_kernel<<<update_grid(n, P), 256, 0, (cudaStream_t)stream>>>(r, ldr, q, ldq, n, P, state, istate);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

extern "C" int rla_affine_cg_update_xp_f64(double *x, int64_t ldx, double *p, int64_t ldp, const double *z, int64_t ldz,
                                           int64_t n, int64_t P, const double *state, const int32_t *istate,
                                           void *stream) {
    RLA_REQUIRE(n >= 0 && P >= 0 && ldx >= n && ldp >= n && ldz >= n, "rla_affine_cg_update_xp_f64: bad sizes");
    if (n == 0 || P == 0) return RLA_OK;
    RLA_REQUIRE(x && p && z && state && istate, "rla_affine_cg_update_xp_f64: null pointer");
    cg_update_xp_kernel<<<update_grid(n, P), 256, 0, (cudaStream_t)stream>>>(x, ldx, p, ldp, z, ldz, n, P, state,
                                                                             istate);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}
