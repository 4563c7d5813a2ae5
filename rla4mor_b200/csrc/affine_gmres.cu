// affine_gmres.cu -- restarted GMRES(m) for the affine full-order model
//   A(mu_p) x_p = b_p,   A(mu_p) = sum_q th[p, q] A_q   (any square, nonsingular A(mu)),
// left-preconditioned by R^-1 and orthogonalised in the R inner product, so that every row minimises
// ||b - A x||_{R^-1} over its Krylov space (fom_solve.affine_gmres drives the iteration).  R is never
// applied: each row keeps a primal basis v_i and a dual basis w_i = R v_i, and <z, v_i>_R = <z, w_i>.
//
// Storage (row-major, P rows of length n each): V and W are (P, m, n), row p's basis contiguous;
// z = R^-1 y and y (P, n) are the vector being orthogonalised and its dual; U (P, n) is what the next
// affine SpMM multiplies (v_j while a row is in a cycle, x when it restarts).  The per-row scalars
// (Hessenberg matrix, rotations, g, the triangle's solution) live in `hess` on the device.
//
// Reductions follow affine_cg.cu: one partial sum per 256-entry tile, the partials of a row added in
// tile order by rla_row_dot_sum_f64.  No atomics, a row's arithmetic reads its own data only, so its
// iterates do not depend on P or on the other rows, and two runs give the same bits.
#include "common.cuh"
#include <algorithm>

namespace rla {
namespace {

constexpr int GM_TILE = 256;                  // entries per partial sum (= ACG_TILE of affine_cg.cu)
constexpr int GM_WARPS = GM_TILE / 32;
constexpr int GM_CHUNK = 32;                  // inner products reduced per shared-memory round
constexpr int GM_ROWS = 128;                  // threads per CTA of the per-row scalar kernels

// istate rows (int32, P each).  mode: what the row does in the current step.  The flag rows hold 2
// ("yes") or 0; they are the masks the vector kernels and the affine SpMM test.
enum : int32_t { G_IDLE = 0, G_ARNOLDI = 1, G_RESTART = 2 };
enum { I_ITERS = 0, I_INFO = 1, I_MODE = 2, I_NCOL = 3, I_CYCLES = 4,
       F_ACT = 5, F_ARN = 6, F_REORTH = 7, F_RESTART = 8, F_END = 9, GM_IROWS = 10 };
// state rows (double, P each)
enum { S_BN2 = 0, S_RESID = 1, S_SCALE = 2, S_NZ2 = 3, S_NZP2 = 4, GM_SROWS = 5 };
constexpr int32_t YES = 2;

__host__ __device__ inline int64_t gm_tiles(int64_t n) { return (n + GM_TILE - 1) / GM_TILE; }

// hess of one row: H (m + 1, m) row-major, g (m + 1), cos (m), sin (m), y (m)
__host__ __device__ inline int64_t hess_per_row(int64_t m) { return (m + 1) * m + (m + 1) + 3 * m; }

struct Hess {
    double *H, *g, *c, *s, *y;
    int64_t m;
    __device__ Hess(double *hess, int64_t m_, int64_t p) : m(m_) {
        H = hess + p * hess_per_row(m);
        g = H + (m + 1) * m;
        c = g + m + 1;
        s = c + m;
        y = s + m;
    }
    __device__ double &h(int64_t i, int64_t j) { return H[i * m + j]; }
};

__device__ __forceinline__ double gm_nan() { return __longlong_as_double(0x7ff8000000000000LL); }

// the row is done for good: every mask cleared
__device__ void gm_stop(int32_t *ist, int64_t P, int64_t p, int32_t info) {
    ist[I_INFO * P + p] = info;
    ist[I_MODE * P + p] = G_IDLE;
    ist[F_ACT * P + p] = 0;
    ist[F_ARN * P + p] = 0;
    ist[F_REORTH * P + p] = 0;
    ist[F_RESTART * P + p] = 0;
    ist[F_END * P + p] = 0;
}

__device__ void gm_breakdown(double *st, int32_t *ist, int64_t P, int64_t p) {
    gm_stop(ist, P, p, 2);
    st[S_RESID * P + p] = gm_nan();
}

// Warp sum by a fixed xor tree (every lane ends with the same bits); lane 0 stores it.
__device__ __forceinline__ void warp_store(double d, double *dst) {
#pragma unroll
    for (int off = 16; off; off >>= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
    if ((threadIdx.x & 31) == 0) *dst = d;
}

// ------------------------------------------------------------------ multi-dot
// Rows with mask[p] == 2: ws[(p J + k) nt + tile] = tile's part of <z_p, w_{p,k}> for k < c and of
// <z_p, y_p> for k = c, where J = m + 2 and c = ncol[p] in a cycle, 0 at a restart (then the only
// product is <R^-1 r, r>).  z and y are read once; the c + 1 sums of a tile are reduced GM_CHUNK
// at a time through shared memory, warp partials added in warp order.
__global__ void __launch_bounds__(GM_TILE)
gmres_dots_kernel(const double *__restrict__ z, const double *__restrict__ y, const double *__restrict__ W,
                  int64_t n, int64_t m, int64_t P, const int32_t *__restrict__ ist, const int32_t *__restrict__ mask,
                  double *__restrict__ ws) {
    __shared__ double red[GM_WARPS][GM_CHUNK];
    const int64_t nt = gm_tiles(n), J = m + 2;
    const int warp = threadIdx.x >> 5;
    for (int64_t p = blockIdx.y; p < P; p += gridDim.y) {
        if (mask[p] != YES) continue;                                     // uniform over the CTA
        const int64_t c = ist[I_MODE * P + p] == G_ARNOLDI ? ist[I_NCOL * P + p] : 0;
        const double *Wp = W + p * m * n;
        for (int64_t tile = blockIdx.x; tile < nt; tile += gridDim.x) {
            const int64_t i = tile * GM_TILE + threadIdx.x;
            const bool in = i < n;
            const double zi = in ? ldg_stream_f64(z + p * n + i) : 0.0;
            for (int64_t k0 = 0; k0 <= c; k0 += GM_CHUNK) {
                const int kn = (int)(c + 1 - k0 < GM_CHUNK ? c + 1 - k0 : GM_CHUNK);
#pragma unroll 4
                for (int kk = 0; kk < kn; ++kk) {
                    const int64_t k = k0 + kk;
                    const double *src = k < c ? Wp + k * n : y + p * n;
                    warp_store(in ? zi * ldg_stream_f64(src + i) : 0.0, &red[warp][kk]);
                }
                __syncthreads();
                if ((int)threadIdx.x < kn) {
                    double s = 0.0;
#pragma unroll
                    for (int w = 0; w < GM_WARPS; ++w) s += red[w][threadIdx.x];
                    ws[(p * J + k0 + threadIdx.x) * nt + tile] = s;
                }
                __syncthreads();
            }
        }
    }
}

// ------------------------------------------------------- orthogonalisation update
// Rows with mask[p] == 2 (in a cycle): z -= sum_{k<c} h_k v_k, y -= sum_{k<c} h_k w_k with
// h_k = hb[p J + k], then the tile's part of <z', y'> in ws[p nt + tile].
__global__ void __launch_bounds__(GM_TILE)
gmres_orth_kernel(double *__restrict__ z, double *__restrict__ y, const double *__restrict__ V,
                  const double *__restrict__ W, const double *__restrict__ hb, int64_t n, int64_t m, int64_t P,
                  const int32_t *__restrict__ ist, const int32_t *__restrict__ mask, double *__restrict__ ws) {
    __shared__ double red[GM_WARPS];
    const int64_t nt = gm_tiles(n), J = m + 2;
    for (int64_t p = blockIdx.y; p < P; p += gridDim.y) {
        if (mask[p] != YES) continue;
        const int64_t c = ist[I_NCOL * P + p];
        const double *Vp = V + p * m * n, *Wp = W + p * m * n, *h = hb + p * J;
        for (int64_t tile = blockIdx.x; tile < nt; tile += gridDim.x) {
            const int64_t i = tile * GM_TILE + threadIdx.x;
            double d = 0.0;
            if (i < n) {
                double zi = z[p * n + i], yi = y[p * n + i];
#pragma unroll 4
                for (int64_t k = 0; k < c; ++k) {
                    const double hk = __ldg(h + k);
                    zi = fma(-hk, ldg_stream_f64(Vp + k * n + i), zi);
                    yi = fma(-hk, ldg_stream_f64(Wp + k * n + i), yi);
                }
                z[p * n + i] = zi;
                y[p * n + i] = yi;
                d = zi * yi;
            }
            warp_store(d, &red[threadIdx.x >> 5]);
            __syncthreads();
            if (threadIdx.x == 0) {
                double s = 0.0;
#pragma unroll
                for (int w = 0; w < GM_WARPS; ++w) s += red[w];
                ws[p * nt + tile] = s;
            }
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------- per-row scalars
// After the first Gram-Schmidt pass: column j = c - 1 of H from the pass's coefficients, ||z||_R^2
// before and ||z'||_R^2 after it, and the DGKS decision (a second pass when ||z'||_R < ||z||_R / sqrt 2).
__global__ void __launch_bounds__(GM_ROWS)
gmres_dgks_kernel(const double *__restrict__ hb, const double *__restrict__ hb2, int64_t m, int64_t P,
                  double *__restrict__ st, int32_t *__restrict__ ist, double *__restrict__ hess) {
    const int64_t p = blockIdx.x * (int64_t)GM_ROWS + threadIdx.x;
    if (p >= P || ist[F_ARN * P + p] != YES) return;
    const int64_t c = ist[I_NCOL * P + p], j = c - 1, J = m + 2;
    Hess R(hess, m, p);
    bool ok = true;
    for (int64_t k = 0; k < c; ++k) {
        const double h = hb[p * J + k];
        ok &= isfinite(h);
        R.h(k, j) = h;
    }
    const double nz2 = hb[p * J + c], nzp2 = hb2[p];
    if (!ok || !(nz2 >= 0.0) || !isfinite(nz2) || !isfinite(nzp2)) {
        gm_breakdown(st, ist, P, p);
        return;
    }
    st[S_NZ2 * P + p] = nz2;
    st[S_NZP2 * P + p] = nzp2;
    ist[F_REORTH * P + p] = nzp2 < 0.5 * nz2 ? YES : 0;
}

// Cycle start (mode G_RESTART, from <R^-1 r, r>): converged, out of iterations, breakdown, or
// v_0 = z / beta, w_0 = r / beta, g = beta e_0.
__device__ void gmres_start_row(const double *hb, int64_t m, int64_t P, int64_t p, double tol2, int64_t maxiter,
                                double *st, int32_t *ist, double *hess) {
    const double beta2 = hb[p * (m + 2)], bn2 = st[S_BN2 * P + p];
    ist[F_END * P + p] = 0;
    if (!(bn2 >= 0.0) || !isfinite(bn2)) {
        gm_breakdown(st, ist, P, p);
        return;
    }
    if (bn2 == 0.0) {                                                  // b = 0: x = 0 (set by the host)
        st[S_RESID * P + p] = 0.0;
        gm_stop(ist, P, p, 0);
        return;
    }
    if (!(beta2 >= 0.0) || !isfinite(beta2)) {
        gm_breakdown(st, ist, P, p);
        return;
    }
    st[S_RESID * P + p] = sqrt(beta2 / bn2);
    if (beta2 <= tol2 * bn2) {
        gm_stop(ist, P, p, 0);
        return;
    }
    if (ist[I_ITERS * P + p] >= maxiter) {
        gm_stop(ist, P, p, 1);
        return;
    }
    Hess R(hess, m, p);
    const double beta = sqrt(beta2);
    R.g[0] = beta;
    for (int64_t k = 1; k <= m; ++k) R.g[k] = 0.0;
    st[S_SCALE * P + p] = 1.0 / beta;
    ist[I_MODE * P + p] = G_ARNOLDI;
    ist[I_NCOL * P + p] = 1;
    ist[I_CYCLES * P + p] += 1;
    ist[F_ARN * P + p] = YES;
    ist[F_RESTART * P + p] = 0;
}

// Arnoldi step j = c - 1 ends: h_{j+1,j} = ||z'||_R, the row's rotations applied to column j, a new
// rotation, g updated.  The cycle ends at j + 1 = m, when |g_{j+1}| <= tol ||b||_{R^-1}, on a happy
// breakdown (h_{j+1,j} = 0) or when the iterations run out: then H(0:c, 0:c) y = g(0:c) is solved
// and the row restarts (x += V y in the update kernel, the true residual in the next step).
__device__ void gmres_arnoldi_row(const double *hb, const double *hb2, int64_t m, int64_t P, int64_t p,
                                  double tol2, int64_t maxiter, double *st, int32_t *ist, double *hess) {
    const int64_t c = ist[I_NCOL * P + p], j = c - 1, J = m + 2;
    Hess R(hess, m, p);
    double nzp2 = st[S_NZP2 * P + p];
    bool ok = true;
    if (ist[F_REORTH * P + p] == YES) {
        for (int64_t k = 0; k < c; ++k) {
            const double h = hb[p * J + k];
            ok &= isfinite(h);
            R.h(k, j) += h;
        }
        nzp2 = hb2[p];
        ist[F_REORTH * P + p] = 0;
    }
    // after two passes a negative ||z'||_R^2 of rounding size is an exact invariant subspace
    if (nzp2 < 0.0 && -nzp2 <= 2.220446049250313e-16 * st[S_NZ2 * P + p]) nzp2 = 0.0;
    if (!ok || !(nzp2 >= 0.0) || !isfinite(nzp2)) {
        gm_breakdown(st, ist, P, p);
        return;
    }
    const double hn = sqrt(nzp2);
    for (int64_t k = 0; k < j; ++k) {
        const double a = R.h(k, j), b = R.h(k + 1, j);
        R.h(k, j) = R.c[k] * a + R.s[k] * b;
        R.h(k + 1, j) = -R.s[k] * a + R.c[k] * b;
    }
    const double a = R.h(j, j), r = hypot(a, hn);
    if (!(r > 0.0) || !isfinite(r)) {                                  // singular A(mu) on the Krylov space
        gm_breakdown(st, ist, P, p);
        return;
    }
    R.c[j] = a / r;
    R.s[j] = hn / r;
    R.h(j, j) = r;
    R.h(j + 1, j) = 0.0;
    R.g[j + 1] = -R.s[j] * R.g[j];
    R.g[j] = R.c[j] * R.g[j];
    const int32_t it = ist[I_ITERS * P + p] + 1;
    ist[I_ITERS * P + p] = it;
    const double gj1 = R.g[j + 1];
    if (c == m || gj1 * gj1 <= tol2 * st[S_BN2 * P + p] || hn == 0.0 || it >= maxiter) {
        for (int64_t k = j; k >= 0; --k) {                            // back substitution
            double t = R.g[k];
            for (int64_t l = k + 1; l <= j; ++l) t = fma(-R.h(k, l), R.y[l], t);
            R.y[k] = t / R.h(k, k);
        }
        ist[I_MODE * P + p] = G_RESTART;
        ist[F_ARN * P + p] = 0;
        ist[F_RESTART * P + p] = YES;
        ist[F_END * P + p] = YES;
    } else {
        st[S_SCALE * P + p] = 1.0 / hn;
        ist[I_NCOL * P + p] = c + 1;
    }
}

__global__ void __launch_bounds__(GM_ROWS)
gmres_step_kernel(const double *__restrict__ hb, const double *__restrict__ hb2, int64_t m, int64_t P, double tol2,
                  int64_t maxiter, double *__restrict__ st, int32_t *__restrict__ ist, double *__restrict__ hess) {
    const int64_t p = blockIdx.x * (int64_t)GM_ROWS + threadIdx.x;
    if (p >= P) return;
    if (ist[F_ARN * P + p] == YES) gmres_arnoldi_row(hb, hb2, m, P, p, tol2, maxiter, st, ist, hess);
    else if (ist[F_RESTART * P + p] == YES)
        gmres_start_row(hb, m, P, p, tol2, maxiter, st, ist, hess);
}

// ------------------------------------------------------------ vector passes
// blockIdx.y walks the rows, blockIdx.x the entries; a row outside the mask costs one flag read per CTA
constexpr int GM_UPD_BLOCKS = 512;

// y <- b - y at a restart (y = A x from the affine SpMM)
__global__ void __launch_bounds__(256)
gmres_residual_kernel(double *__restrict__ y, const double *__restrict__ b, int64_t n, int64_t P,
                      const int32_t *__restrict__ ist) {
    for (int64_t p = blockIdx.y; p < P; p += gridDim.y) {
        if (ist[F_RESTART * P + p] != YES) continue;
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
            y[p * n + i] = ldg_stream_f64(b + p * n + i) - y[p * n + i];
    }
}

// v_{c-1} = z' / h, w_{c-1} = y' / h and U = v_{c-1} on rows that continue a cycle (or start one)
__global__ void __launch_bounds__(256)
gmres_normalize_kernel(const double *__restrict__ z, const double *__restrict__ y, double *__restrict__ V,
                       double *__restrict__ W, double *__restrict__ U, int64_t n, int64_t m, int64_t P,
                       const double *__restrict__ st, const int32_t *__restrict__ ist) {
    for (int64_t p = blockIdx.y; p < P; p += gridDim.y) {
        if (ist[F_ARN * P + p] != YES) continue;
        const double sc = st[S_SCALE * P + p];
        const int64_t k = ist[I_NCOL * P + p] - 1;
        double *Vk = V + (p * m + k) * n, *Wk = W + (p * m + k) * n;
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
            const double v = ldg_stream_f64(z + p * n + i) * sc;
            Vk[i] = v;
            Wk[i] = ldg_stream_f64(y + p * n + i) * sc;
            U[p * n + i] = v;
        }
    }
}

// cycle end: x += sum_{k<c} y_k v_k, and U = x for the true residual of the next step
__global__ void __launch_bounds__(256)
gmres_update_kernel(double *__restrict__ x, double *__restrict__ U, const double *__restrict__ V, int64_t n, int64_t m,
                    int64_t P, const int32_t *__restrict__ ist, const double *__restrict__ hess) {
    for (int64_t p = blockIdx.y; p < P; p += gridDim.y) {
        if (ist[F_END * P + p] != YES) continue;
        const int64_t c = ist[I_NCOL * P + p];
        const double *yc = hess + p * hess_per_row(m) + (m + 1) * m + (m + 1) + 2 * m;
        const double *Vp = V + p * m * n;
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
            double xi = x[p * n + i];
#pragma unroll 4
            for (int64_t k = 0; k < c; ++k) xi = fma(__ldg(yc + k), ldg_stream_f64(Vp + k * n + i), xi);
            x[p * n + i] = xi;
            U[p * n + i] = xi;
        }
    }
}

dim3 vec_grid(int64_t n, int64_t P) {
    return dim3((unsigned)std::min<int64_t>((n + 255) / 256, GM_UPD_BLOCKS), (unsigned)std::min<int64_t>(P, 65535));
}

dim3 tile_rows_grid(int64_t n, int64_t P) {
    return dim3((unsigned)std::min<int64_t>(gm_tiles(n), INT32_MAX), (unsigned)std::min<int64_t>(P, 65535));
}

unsigned scalar_grid(int64_t P) { return (unsigned)((P + GM_ROWS - 1) / GM_ROWS); }

}  // namespace
}  // namespace rla

using namespace rla;

#define GM_LAUNCHED()                                                                                              \
    do {                                                                                                           \
        count_launch();                                                                                            \
        RLA_CUDA_CHECK(cudaGetLastError());                                                                        \
        return RLA_OK;                                                                                             \
    } while (0)

extern "C" size_t rla_affine_gmres_workspace_bytes(int64_t n, int64_t m, int64_t P) {
    if (n <= 0 || m <= 0 || P <= 0) return 0;
    return (size_t)P * (size_t)(m + 2) * (size_t)gm_tiles(n) * sizeof(double);
}

extern "C" size_t rla_affine_gmres_hess_bytes(int64_t m, int64_t P) {
    if (m <= 0 || P <= 0) return 0;
    return (size_t)P * (size_t)hess_per_row(m) * sizeof(double);
}

extern "C" int rla_affine_gmres_dots_f64(const double *z, const double *y, const double *W, int64_t n, int64_t m,
                                         int64_t P, const int32_t *istate, const int32_t *mask, void *ws,
                                         size_t ws_bytes, void *stream) {
    RLA_REQUIRE(n >= 1 && m >= 1 && P >= 0, "rla_affine_gmres_dots_f64: bad sizes");
    if (P == 0) return RLA_OK;
    RLA_REQUIRE(z && y && W && istate && mask && ws, "rla_affine_gmres_dots_f64: null pointer");
    RLA_REQUIRE(ws_bytes >= rla_affine_gmres_workspace_bytes(n, m, P),
                "rla_affine_gmres_dots_f64: workspace of %zu bytes, %zu needed", ws_bytes,
                rla_affine_gmres_workspace_bytes(n, m, P));
    gmres_dots_kernel<<<tile_rows_grid(n, P), GM_TILE, 0, (cudaStream_t)stream>>>(z, y, W, n, m, P, istate, mask,
                                                                                (double *)ws);
    GM_LAUNCHED();
}

extern "C" int rla_affine_gmres_orth_f64(double *z, double *y, const double *V, const double *W, const double *hb,
                                         int64_t n, int64_t m, int64_t P, const int32_t *istate, const int32_t *mask,
                                         void *ws, size_t ws_bytes, void *stream) {
    RLA_REQUIRE(n >= 1 && m >= 1 && P >= 0, "rla_affine_gmres_orth_f64: bad sizes");
    if (P == 0) return RLA_OK;
    RLA_REQUIRE(z && y && V && W && hb && istate && mask && ws, "rla_affine_gmres_orth_f64: null pointer");
    RLA_REQUIRE(ws_bytes >= (size_t)P * gm_tiles(n) * sizeof(double),
                "rla_affine_gmres_orth_f64: workspace of %zu bytes, %zu needed", ws_bytes,
                (size_t)P * gm_tiles(n) * sizeof(double));
    gmres_orth_kernel<<<tile_rows_grid(n, P), GM_TILE, 0, (cudaStream_t)stream>>>(z, y, V, W, hb, n, m, P, istate,
                                                                                mask, (double *)ws);
    GM_LAUNCHED();
}

extern "C" int rla_affine_gmres_dgks_f64(const double *hb, const double *hb2, int64_t m, int64_t P, double *state,
                                         int32_t *istate, double *hess, void *stream) {
    RLA_REQUIRE(m >= 1 && P >= 0, "rla_affine_gmres_dgks_f64: bad sizes");
    if (P == 0) return RLA_OK;
    RLA_REQUIRE(hb && hb2 && state && istate && hess, "rla_affine_gmres_dgks_f64: null pointer");
    gmres_dgks_kernel<<<scalar_grid(P), GM_ROWS, 0, (cudaStream_t)stream>>>(hb, hb2, m, P, state, istate, hess);
    GM_LAUNCHED();
}

extern "C" int rla_affine_gmres_step_f64(const double *hb, const double *hb2, int64_t m, int64_t P, double tol,
                                         int64_t maxiter, double *state, int32_t *istate, double *hess, void *stream) {
    RLA_REQUIRE(m >= 1 && P >= 0 && maxiter >= 0 && tol >= 0.0, "rla_affine_gmres_step_f64: bad arguments");
    if (P == 0) return RLA_OK;
    RLA_REQUIRE(hb && hb2 && state && istate && hess, "rla_affine_gmres_step_f64: null pointer");
    gmres_step_kernel<<<scalar_grid(P), GM_ROWS, 0, (cudaStream_t)stream>>>(hb, hb2, m, P, tol * tol, maxiter, state,
                                                                          istate, hess);
    GM_LAUNCHED();
}

extern "C" int rla_affine_gmres_residual_f64(double *y, const double *b, int64_t n, int64_t P, const int32_t *istate,
                                             void *stream) {
    RLA_REQUIRE(n >= 0 && P >= 0, "rla_affine_gmres_residual_f64: bad sizes");
    if (n == 0 || P == 0) return RLA_OK;
    RLA_REQUIRE(y && b && istate, "rla_affine_gmres_residual_f64: null pointer");
    gmres_residual_kernel<<<vec_grid(n, P), 256, 0, (cudaStream_t)stream>>>(y, b, n, P, istate);
    GM_LAUNCHED();
}

extern "C" int rla_affine_gmres_normalize_f64(const double *z, const double *y, double *V, double *W, double *U,
                                              int64_t n, int64_t m, int64_t P, const double *state,
                                              const int32_t *istate, void *stream) {
    RLA_REQUIRE(n >= 0 && m >= 1 && P >= 0, "rla_affine_gmres_normalize_f64: bad sizes");
    if (n == 0 || P == 0) return RLA_OK;
    RLA_REQUIRE(z && y && V && W && U && state && istate, "rla_affine_gmres_normalize_f64: null pointer");
    gmres_normalize_kernel<<<vec_grid(n, P), 256, 0, (cudaStream_t)stream>>>(z, y, V, W, U, n, m, P, state, istate);
    GM_LAUNCHED();
}

extern "C" int rla_affine_gmres_update_f64(double *x, double *U, const double *V, int64_t n, int64_t m, int64_t P,
                                           const int32_t *istate, const double *hess, void *stream) {
    RLA_REQUIRE(n >= 0 && m >= 1 && P >= 0, "rla_affine_gmres_update_f64: bad sizes");
    if (n == 0 || P == 0) return RLA_OK;
    RLA_REQUIRE(x && U && V && istate && hess, "rla_affine_gmres_update_f64: null pointer");
    gmres_update_kernel<<<vec_grid(n, P), 256, 0, (cudaStream_t)stream>>>(x, U, V, n, m, P, istate, hess);
    GM_LAUNCHED();
}
