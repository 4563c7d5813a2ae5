// sptrsv.cu -- sparse triangular solves with a block of right-hand sides: the device side of
// InverseLuOperator.apply (utilities/factorization.py:118-124: `slu.solve(V.T).T`), i.e. the
// `inverse_product` R^-1 applied in front of every sketch (mor/sketched_reductor.py:69,73;
// SURVEY.md section 8f rank 1).  The sparse LU factorisation itself stays on the host (SciPy
// SuperLU, as in the reference); its factors  Pr A Pc = L U  are uploaded once as CSR.
//
// Layout: the block (m, n) of the reference (one vector per row) is transposed ON THE WAY IN to
// X (n, ldx) with the m right-hand sides contiguous, with the row permutation applied by the same
// kernel; the solves run in place on X; the way out transposes back and applies the column
// permutation.  A row of a factor then reads, for every off-diagonal entry (i, j), the 8*m
// contiguous bytes X[j, :] (one 512-byte request per warp at m = 64): HBM/L2-bound.
//
// Scheduling (host, rla_sptrsv_plan_host): rows are collected into GROUPS -- chains of up to 128
// rows that depend on each other (the supernodes of the factor) -- and the groups, together with
// the remaining single rows, are sorted into the levels of the GROUP dependency graph (a 2-D FEM
// factor with 5161 row levels has ~50-70 group levels).  One group level = up to three launches:
//   * kind 1 / kind 0: every row of the level subtracts its EXTERNAL entries (columns solved in
//     earlier levels) from its right-hand sides: one CTA of 16 warps per long row, one warp per
//     short row; a single row also divides by its diagonal and is finished;
//   * kind 2: one CTA per group multiplies the group's rows by the INVERSE of the group's dense
//     triangular block (computed once on the host, rla_sptrsv_group_inverses_host): the chain of
//     up to 128 dependent rows is resolved by one small dense product instead of 128 sequential
//     steps -- no tickets, no fences, no partial sums through global memory.
// Deterministic: every sum has a fixed order.
#include "common.cuh"
#include <algorithm>
#include <utility>
#include <vector>

namespace rla {

constexpr int TRSV_RHS = 64;                          // right-hand sides per chunk (2 per lane)

__device__ __forceinline__ double2 ldcg2(const double *p) { return __ldcg(reinterpret_cast<const double2 *>(p)); }

// X[dest(i), c] = B[c, i]   (dest = perm[i] or i)
__global__ void trsv_in_kernel(const double *__restrict__ B, int64_t m, int64_t n, int64_t ldb,
                               const int32_t *__restrict__ perm, double *__restrict__ X, int64_t ldx) {
    __shared__ double tile[32][33];
    const int64_t i0 = (int64_t)blockIdx.x * 32, c0 = (int64_t)blockIdx.y * 32;
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        const int64_t c = c0 + y, i = i0 + threadIdx.x;
        tile[y][threadIdx.x] = (c < m && i < n) ? B[c * ldb + i] : 0.0;
    }
    __syncthreads();
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        const int64_t i = i0 + y, c = c0 + threadIdx.x;
        if (i < n && c < ldx) X[(int64_t)(perm ? perm[i] : i) * ldx + c] = tile[threadIdx.x][y];
    }
}

// out[c, i] = X[src(i), c]   (src = perm[i] or i)
__global__ void trsv_out_kernel(const double *__restrict__ X, int64_t m, int64_t n, int64_t ldx,
                                const int32_t *__restrict__ perm, double *__restrict__ out, int64_t ldo) {
    __shared__ double tile[32][33];
    const int64_t i0 = (int64_t)blockIdx.x * 32, c0 = (int64_t)blockIdx.y * 32;
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        const int64_t i = i0 + y, c = c0 + threadIdx.x;
        tile[y][threadIdx.x] = (i < n && c < m) ? X[(int64_t)(perm ? perm[i] : i) * ldx + c] : 0.0;
    }
    __syncthreads();
    for (int y = threadIdx.y; y < 32; y += blockDim.y) {
        const int64_t c = c0 + y, i = i0 + threadIdx.x;
        if (c < m && i < n) out[c * ldo + i] = tile[threadIdx.x][y];
    }
}

// Everything the kernels touch is stored IN SCHEDULE ORDER: row p of X, rowptr, split, diag is the
// p-th row of the processing order, and external column indices are positions too -- no
// order / inverse-order indirection on the critical path of a launch.
// out[p, :] = in[map[p], :]  (re-ordering of the block between the L and the U schedule)
__global__ void trsv_permute_rows_kernel(const double *__restrict__ in, const int32_t *__restrict__ map,
                                         double *__restrict__ out, int64_t n, int64_t ldx) {
    const int64_t w2 = ldx / 2;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n * w2; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p = t / w2, c = 2 * (t - p * w2);
        *reinterpret_cast<double2 *>(out + p * ldx + c) =
            *reinterpret_cast<const double2 *>(in + (int64_t)map[p] * ldx + c);
    }
}

struct TrsvArgs {
    const int64_t *rowptr;      // CSR of the strictly triangular part, rows and columns renumbered by
    const int32_t *col;         //   schedule position, entries of a row sorted by column
    const double *val;
    const double *diag;         // divisor by position (1.0 for the rows of a group), or null: no division
    const int64_t *split;       // per row: end of its external entries (the rest refers to its own group)
    double *X;
    int64_t ldx, m;
};

constexpr int TRSV_GROUP = 128;                       // rows per group (chain of dependent rows resolved by one CTA)

constexpr int TRSV_WARPS = 16;                        // warps of a CTA that owns one (long) row
constexpr int TRSV_WARPS_SMALL = 4;                   // ... in steps of many short rows

// -sum_e val[e] * X[col[e], c..c+1] over the entries [e0, e1) of one row, for warp `w` of `nw`
// warps sharing the row.  A warp takes 32 consecutive entries at a time: (col, val) come in with
// ONE coalesced load per lane and are broadcast by shuffles; the X rows are fetched 8 at a time
// (8 independent 16-byte loads in flight per lane).  Every lane of the warp must call this.
template <int INFLIGHT>
__device__ __forceinline__ double2 row_sum_warp(const TrsvArgs &a, int64_t e0, int64_t e1, int64_t c, bool live,
                                                int w, int nw) {
    const int lane = threadIdx.x & 31;
    double2 acc = make_double2(0.0, 0.0);
    int64_t base = e0 + 32 * (int64_t)w;
    int32_t jn = 0;
    double vn = 0.0;
    if (base + lane < e1) { jn = a.col[base + lane]; vn = a.val[base + lane]; }
    for (; base < e1; base += 32 * (int64_t)nw) {
        const int32_t jc = jn;
        const double vc = vn;
        // prefetch the (col, val) of this warp's next 32 entries while the X rows of these are fetched
        const int64_t nb = base + 32 * (int64_t)nw + lane;
        jn = 0; vn = 0.0;
        if (nb < e1) { jn = a.col[nb]; vn = a.val[nb]; }
        const int cnt = (int)min((int64_t)32, e1 - base);
        for (int t0 = 0; t0 < cnt; t0 += INFLIGHT) {    // INFLIGHT independent 16-byte loads in flight per lane
            int32_t j[INFLIGHT];
            double v[INFLIGHT];
            double2 x[INFLIGHT];
#pragma unroll
            for (int u = 0; u < INFLIGHT; ++u) {
                j[u] = __shfl_sync(0xffffffffu, jc, (t0 + u) & 31);
                v[u] = __shfl_sync(0xffffffffu, vc, (t0 + u) & 31);
            }
#pragma unroll
            for (int u = 0; u < INFLIGHT; ++u)
                x[u] = (live && t0 + u < cnt) ? ldcg2(a.X + (int64_t)j[u] * a.ldx + c) : make_double2(0.0, 0.0);
#pragma unroll
            for (int u = 0; u < INFLIGHT; ++u) {
                if (t0 + u < cnt) { acc.x = fma(-v[u], x[u].x, acc.x); acc.y = fma(-v[u], x[u].y, acc.y); }
            }
        }
    }
    return acc;
}

// kind 0: warp = one row x one chunk of 64 right-hand sides; external entries [rowptr, split)
__global__ void __launch_bounds__(256)
trsv_rows_warp_kernel(const TrsvArgs a, int64_t lo, int64_t hi) {
    const int lane = threadIdx.x & 31;
    const int64_t idx = lo + (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (idx >= hi) return;                             // whole warp
    const int64_t c = (int64_t)blockIdx.y * TRSV_RHS + 2 * lane;
    const bool live = c < a.ldx;
    const int64_t i = idx;
    // the row's own right-hand sides and divisor do not depend on the sum: fetch them first
    double *xi = a.X + i * a.ldx + c;
    const double2 b = live ? ldcg2(xi) : make_double2(0.0, 0.0);
    const double d = a.diag ? a.diag[i] : 1.0;
    double2 acc = row_sum_warp<8>(a, a.rowptr[i], a.split[i], c, live, 0, 1);
    if (live) {
        acc.x += b.x; acc.y += b.y;
        if (a.diag) { acc.x /= d; acc.y /= d; }
        *reinterpret_cast<double2 *>(xi) = acc;
    }
}

// the same sum with the row split over the NW warps of the CTA, combined in warp order;
// result valid in warp 0
template <int NW>
__device__ __forceinline__ double2 row_sum_cta(const TrsvArgs &a, int64_t e0, int64_t e1, int64_t c, bool live,
                                               double2 (*part)[32]) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double2 acc = row_sum_warp<(NW >= 16 ? 16 : 8)>(a, e0, e1, c, live, warp, NW);
    part[warp][lane] = acc;
    __syncthreads();
    if (warp == 0) {
        acc = part[0][lane];
#pragma unroll
        for (int w = 1; w < NW; ++w) { acc.x += part[w][lane].x; acc.y += part[w][lane].y; }
    }
    return acc;
}

// kind 1: one CTA = one LONG row (more than 64 external entries, up to thousands near the root of the
// elimination tree) x one chunk of right-hand sides.  NW = 16 warps with 16 loads in flight each
// when the step has few rows (all the parallelism must come from inside the row), 8 warps x 8
// loads and four CTAs per SM when it has many.
template <int NW>
__global__ void __launch_bounds__(32 * NW, NW >= 16 ? 1 : 4)
trsv_rows_cta_kernel(const TrsvArgs a, int64_t lo) {
    __shared__ double2 part[NW][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t i = lo + blockIdx.x;
    const int64_t c = (int64_t)blockIdx.y * TRSV_RHS + 2 * lane;
    const bool live = c < a.ldx;
    double *xi = a.X + i * a.ldx + c;
    double2 b = make_double2(0.0, 0.0);
    double d = 1.0;
    if (warp == 0) {
        if (live) b = ldcg2(xi);
        if (a.diag) d = a.diag[i];
    }
    double2 acc = row_sum_cta<NW>(a, a.rowptr[i], a.split[i], c, live, part);
    if (warp == 0 && live) {
        acc.x += b.x; acc.y += b.y;
        if (a.diag) { acc.x /= d; acc.y /= d; }
        *reinterpret_cast<double2 *>(xi) = acc;
    }
}

// kind 2: P CTAs per group and chunk of right-hand sides.  The rows of the group hold
// y = b - (external sums); x = Dinv y with the inverse of the group's triangular block (row-major
// nrows x nrows at dinv + dinv_ptr[g], lower triangle).  y is staged in shared memory (lanes =
// pairs of right-hand sides); row r belongs to CTA r % P, warp (r / P) % 16 of it.  The entries
// of a row of Dinv come in with one coalesced load per 32 (zero beyond the diagonal) and are
// broadcast by shuffles; a 32-entry piece is fully unrolled over four independent accumulator
// pairs, so neither the shuffle nor the FP64 latency is on the critical path (the round-2a
// kernel walked `cnt` entries with one accumulator: 32 us for ONE group, and a 2-D FEM factor
// has ~150 group levels of one to a few groups each).  P = 4 when a step has few groups: the
// step then lasts as long as a quarter of the chain's rows.
template <int P>
__global__ void __launch_bounds__(32 * TRSV_WARPS, 2)
trsv_resolve_kernel(double *__restrict__ X, int64_t ldx, const int64_t *__restrict__ grp_start,
                    const int32_t *__restrict__ grp_rows, const int64_t *__restrict__ dinv_ptr,
                    const double *__restrict__ dinv, int64_t g_first) {
    extern __shared__ __align__(16) double2 ys[];      // [TRSV_GROUP][32]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t gid = g_first + blockIdx.x / P;
    const int part = blockIdx.x % P;
    const int nrows = grp_rows[gid];
    const int64_t g0 = grp_start[gid];
    const double *Dg = dinv + dinv_ptr[gid];
    const int64_t c = (int64_t)blockIdx.y * TRSV_RHS + 2 * lane;
    const bool live = c < ldx;
    // rows up to the last 32-entry piece any row of this group touches; beyond nrows: zeros
    const int npad = (nrows + 31) & ~31;
    for (int q = warp; q < npad; q += TRSV_WARPS)
        ys[q * 32 + lane] = (live && q < nrows) ? ldcg2(X + (g0 + q) * ldx + c) : make_double2(0.0, 0.0);
    constexpr int NP = TRSV_GROUP / 32;
    auto fetch = [&](int r, double (&dv)[NP]) {
#pragma unroll
        for (int k = 0; k < NP; ++k) {
            const int q = 32 * k + lane;
            dv[k] = (r >= 0 && q <= r) ? __ldg(Dg + (int64_t)r * nrows + q) : 0.0;
        }
    };
    // this warp's rows: r = part + P * (warp + 16 j), longest first
    const int stride = P * TRSV_WARPS;
    const int rfirst = part + P * warp;
    int r = nrows - 1 >= rfirst ? rfirst + ((nrows - 1 - rfirst) / stride) * stride : -1;
    double dv[NP], dn[NP];
    fetch(r, dv);
    __syncthreads();
    for (; r >= 0; r -= stride) {
        fetch(r - stride, dn);
        double2 a0 = make_double2(0.0, 0.0), a1 = a0, a2 = a0, a3 = a0;
#pragma unroll
        for (int k = 0; k < NP; ++k) {
            if (32 * k <= r) {
                const double2 *yk = ys + (32 * k) * 32 + lane;
#pragma unroll
                for (int u = 0; u < 32; u += 4) {
                    const double v0 = __shfl_sync(0xffffffffu, dv[k], u), v1 = __shfl_sync(0xffffffffu, dv[k], u + 1);
                    const double v2 = __shfl_sync(0xffffffffu, dv[k], u + 2), v3 = __shfl_sync(0xffffffffu, dv[k], u + 3);
                    const double2 y0 = yk[u * 32], y1 = yk[(u + 1) * 32], y2 = yk[(u + 2) * 32], y3 = yk[(u + 3) * 32];
                    a0.x = fma(v0, y0.x, a0.x); a0.y = fma(v0, y0.y, a0.y);
                    a1.x = fma(v1, y1.x, a1.x); a1.y = fma(v1, y1.y, a1.y);
                    a2.x = fma(v2, y2.x, a2.x); a2.y = fma(v2, y2.y, a2.y);
                    a3.x = fma(v3, y3.x, a3.x); a3.y = fma(v3, y3.y, a3.y);
                }
            }
        }
        if (live) *reinterpret_cast<double2 *>(X + (g0 + r) * ldx + c) =
            make_double2((a0.x + a1.x) + (a2.x + a3.x), (a0.y + a1.y) + (a2.y + a3.y));
#pragma unroll
        for (int k = 0; k < NP; ++k) dv[k] = dn[k];
    }
}

}  // namespace rla

using namespace rla;

// Host-side analysis of one triangular CSR factor (HOST arrays in, HOST arrays out; plain C++):
//   level_out[i]   longest dependency chain ending in row i (lower != 0: deps j < i, else j > i)
//   order_out      the processing order of the rows, pos_out its inverse
//   rowptr2/col2/val2  the strictly triangular part, entries of each row sorted by pos[col]
//   diag_out       the diagonal (1.0 where absent)
//   groups         group g = order positions [grp_start[g], grp_start[g] + grp_rows[g]), <= group_rows rows
//   groups         MULTI-ROW groups only: group g = order positions [grp_start[g], + grp_rows[g])
//   steps          kind 0 / kind 1: order positions [step_lo, step_hi): every row subtracts its external
//                  entries (one warp / one CTA of 16 warps per row) and, if it is a single row, divides
//                  by its diagonal; kind 2: groups [step_lo, step_hi) are resolved (x = Dinv y).
//                  Up to three steps per level of the GROUP dependency graph; step_mid = step_hi.
//   split_out[i]   first entry of row i that refers to a row of its own group (row end when there is
//                  none); for those entries col2 holds the slot of the column inside the group.
// Groups are CHAINS of up to `group_rows` dependent rows (see the grouping loop below); at most
// max_multi multi-row groups per step (they need scratch).  Arrays of n entries each.
extern "C" int rla_sptrsv_plan_host(int64_t n, const int64_t *rowptr, const int32_t *col, const double *val,
                                    int lower, int wide_min, int group_rows, int max_multi,
                                    int32_t *level_out, int32_t *order_out, int32_t *pos_out,
                                    int64_t *rowptr2, int32_t *col2, double *val2, double *diag_out,
                                    int64_t *split_out, int64_t *grp_start, int32_t *grp_rows, int64_t *ngroups_out,
                                    int64_t *step_lo, int64_t *step_mid, int64_t *step_hi, int32_t *step_kind,
                                    int64_t *nsteps_out, int32_t *nlevels_out) {
    RLA_REQUIRE(n >= 0 && rowptr && level_out && order_out && pos_out && rowptr2 && diag_out && split_out &&
                grp_start && grp_rows && ngroups_out && step_lo && step_mid && step_hi && step_kind && nsteps_out &&
                nlevels_out, "rla_sptrsv_plan_host: null pointer");
    RLA_REQUIRE(wide_min >= 1 && group_rows >= 1 && group_rows <= TRSV_GROUP && max_multi >= 1,
                "rla_sptrsv_plan_host: bad parameters");
    int32_t nl = 0;
    for (int64_t t = 0; t < n; ++t) {
        const int64_t i = lower ? t : n - 1 - t;
        int32_t l = 0;
        for (int64_t e = rowptr[i]; e < rowptr[i + 1]; ++e) {
            const int32_t j = col[e];
            RLA_REQUIRE(j >= 0 && j < n && (lower ? j <= i : j >= i),
                        "rla_sptrsv_plan_host: entry (%lld, %d) on the wrong side of the diagonal", (long long)i, j);
            if (j != i) l = std::max(l, level_out[j] + 1);
        }
        level_out[i] = l;
        nl = std::max(nl, l + 1);
    }
    *nlevels_out = nl;
    // counting sort by level
    std::vector<int64_t> lvlptr((size_t)nl + 1, 0);
    for (int64_t i = 0; i < n; ++i) ++lvlptr[(size_t)level_out[i] + 1];
    for (int32_t l = 0; l < nl; ++l) lvlptr[(size_t)l + 1] += lvlptr[l];
    {
        std::vector<int64_t> fill(lvlptr.begin(), lvlptr.end() - 1);
        for (int64_t i = 0; i < n; ++i) {
            const int64_t p = fill[level_out[i]]++;
            order_out[p] = (int32_t)i;
            pos_out[i] = (int32_t)p;
        }
    }
    // ---- groups: CHAINS instead of global bands of levels.
    // Rows are visited in level order.  Row i joins the group G of its deepest dependency when G has
    // room and every other dependency outside G lies strictly below G's first level; else it opens a
    // group of its own.  All external dependencies of a group then have a level below the group's
    // first level, so (a) groups sorted by first level are in topological order and (b) the group
    // DAG has its own levels `glevel`: one STEP per group level instead of one per band of row
    // levels.  A chain of 32 dependent rows (a supernode of the factor) is ONE group whatever the
    // rest of the matrix looks like at those levels: the critical path of a 2-D FEM factor drops
    // from ~800 steps (bands cut short by unrelated components) to levels / 32.
    // Rows of wide levels (> wide_min rows: the leaves of the elimination tree) stay single and closed.
    std::vector<int64_t> gstart_of_pos((size_t)n, -1);  // start position of the group of the row at a position
    std::vector<int32_t> gid((size_t)n, -1), gsize, gminlevel;
    std::vector<char> gclosed;
    std::vector<int32_t> ord0(order_out, order_out + n);               // level order
    auto new_group = [&](int64_t i, bool closed) {
        gid[i] = (int32_t)gsize.size();
        gsize.push_back(1); gminlevel.push_back(level_out[i]); gclosed.push_back(closed ? 1 : 0);
    };
    for (int64_t q = 0; q < n; ++q) {
        const int64_t i = ord0[q];
        const int32_t li = level_out[i];
        if (lvlptr[(size_t)li + 1] - lvlptr[li] > wide_min) { new_group(i, true); continue; }
        int64_t best = -1;
        for (int64_t e = rowptr[i]; e < rowptr[i + 1]; ++e) {
            const int32_t j = col[e];
            if (j != i && (best < 0 || level_out[j] > level_out[best])) best = j;
        }
        if (best < 0) { new_group(i, false); continue; }
        const int32_t g = gid[best];
        bool ok = !gclosed[g] && gsize[g] < group_rows;
        for (int64_t e = rowptr[i]; ok && e < rowptr[i + 1]; ++e) {
            const int32_t j = col[e];
            if (j != i && gid[j] != g && level_out[j] >= gminlevel[g]) ok = false;
        }
        if (ok) { gid[i] = g; ++gsize[g]; } else new_group(i, false);
    }
    const int64_t ngr = (int64_t)gsize.size();
    // rows of every group, in level order (= a topological order of the group's internal dependencies)
    std::vector<int64_t> gptr((size_t)ngr + 1, 0);
    for (int64_t g = 0; g < ngr; ++g) gptr[(size_t)g + 1] = gptr[g] + gsize[g];
    std::vector<int32_t> grow((size_t)n);
    {
        std::vector<int64_t> fill(gptr.begin(), gptr.end() - 1);
        for (int64_t q = 0; q < n; ++q) { const int64_t i = ord0[q]; grow[fill[gid[i]]++] = (int32_t)i; }
    }
    // group levels: groups were created in level order of their first row = topological order
    std::vector<int32_t> glevel((size_t)ngr, 0);
    std::vector<int64_t> gmaxlen((size_t)ngr, 0), gext((size_t)ngr, 0);
    int32_t ngl = 0;
    for (int64_t g = 0; g < ngr; ++g) {
        int32_t gl = 0;
        for (int64_t t = gptr[g]; t < gptr[(size_t)g + 1]; ++t) {
            const int64_t i = grow[t];
            gmaxlen[g] = std::max<int64_t>(gmaxlen[g], rowptr[i + 1] - rowptr[i]);
            for (int64_t e = rowptr[i]; e < rowptr[i + 1]; ++e) {
                const int32_t j = col[e];
                if (j != i && gid[j] != g) { gl = std::max(gl, glevel[gid[j]] + 1); ++gext[g]; }
            }
        }
        glevel[g] = gl;
        ngl = std::max(ngl, gl + 1);
    }
    // bucket the groups by group level
    std::vector<int64_t> glptr((size_t)ngl + 1, 0);
    for (int64_t g = 0; g < ngr; ++g) ++glptr[(size_t)glevel[g] + 1];
    for (int32_t l = 0; l < ngl; ++l) glptr[(size_t)l + 1] += glptr[l];
    std::vector<int32_t> gsorted((size_t)ngr);
    {
        std::vector<int64_t> fill(glptr.begin(), glptr.end() - 1);
        for (int64_t g = 0; g < ngr; ++g) gsorted[fill[glevel[g]]++] = (int32_t)g;
    }
    int64_t ns = 0, ng = 0, p = 0;
    std::vector<int32_t> multi, single;
    auto place_group = [&](int32_t g) {                 // rows of group g take the next positions of the order
        grp_start[ng] = p; grp_rows[ng] = gsize[g];
        for (int64_t t = gptr[g]; t < gptr[(size_t)g + 1]; ++t) {
            const int32_t i = grow[t];
            order_out[p] = i; pos_out[i] = (int32_t)p; gstart_of_pos[p] = grp_start[ng];
            ++p;
        }
        ++ng;
    };
    // One group level = up to three steps: kind 1 (CTA of 16 warps per row) over the rows of the groups /
    // single rows whose longest row exceeds LONG_ROW entries, kind 0 (warp per row) over the others, then
    // kind 2 (one CTA per group) over the level's multi-row groups.  A 1500-entry row summed by ONE warp
    // would cost ~190 us of dependent 512-byte loads and hold up its whole level (a warp keeps 8 loads in flight).
    constexpr int64_t LONG_ROW = 64;
    std::vector<int32_t> multi_s, single_s;
    (void)max_multi;
    for (int32_t gl = 0; gl < ngl; ++gl) {
        multi.clear(); single.clear(); multi_s.clear(); single_s.clear();
        for (int64_t t = glptr[gl]; t < glptr[(size_t)gl + 1]; ++t) {
            const int32_t g = gsorted[t];
            const bool lng = gmaxlen[g] > LONG_ROW;
            (gsize[g] > 1 ? (lng ? multi : multi_s) : (lng ? single : single_s)).push_back(g);
        }
        // longest rows first: a step ends with its slowest CTA
        auto by_len = [&](int32_t x, int32_t y) { return gmaxlen[x] > gmaxlen[y]; };
        std::stable_sort(multi.begin(), multi.end(), by_len);
        std::stable_sort(single.begin(), single.end(), by_len);
        const int64_t g_lo = ng;
        auto place_single = [&](int32_t g) {
            const int32_t i = grow[gptr[g]];
            order_out[p] = i; pos_out[i] = (int32_t)p; gstart_of_pos[p] = -1;
            ++p;
        };
        auto emit_rows = [&](int kind, const std::vector<int32_t> &mg, const std::vector<int32_t> &sg) {
            if (mg.empty() && sg.empty()) return;
            step_kind[ns] = kind;
            step_lo[ns] = p;
            for (int32_t g : mg) place_group(g);
            for (int32_t g : sg) place_single(g);
            step_mid[ns] = p; step_hi[ns] = p;
            ++ns;
        };
        emit_rows(1, multi, single);
        emit_rows(0, multi_s, single_s);
        if (ng > g_lo) {
            step_kind[ns] = 2;
            step_lo[ns] = g_lo; step_mid[ns] = ng; step_hi[ns] = ng;
            ++ns;
        }
    }
    *nsteps_out = ns;
    *ngroups_out = ng;
    // strictly triangular CSR IN SCHEDULE ORDER: row p = row order[p], external columns = positions
    std::vector<std::pair<int32_t, int64_t>> tmp;
    int64_t w = 0;
    for (int64_t p = 0; p < n; ++p) {
        const int64_t i = order_out[p];
        rowptr2[p] = w;
        diag_out[p] = 1.0;
        tmp.clear();
        for (int64_t e = rowptr[i]; e < rowptr[i + 1]; ++e) {
            if (col[e] == i) { diag_out[p] = val[e]; continue; }
            tmp.emplace_back(pos_out[col[e]], e);
        }
        std::sort(tmp.begin(), tmp.end());
        const int64_t gs = gstart_of_pos[p];
        int64_t sp = -1;
        for (const auto &pe : tmp) {
            if (sp < 0 && gs >= 0 && pe.first >= gs) sp = w;
            col2[w] = sp >= 0 ? (int32_t)(pe.first - gs) : pe.first;   // internal: slot inside the group
            val2[w] = val[pe.second];
            ++w;
        }
        split_out[p] = sp < 0 ? w : sp;
    }
    rowptr2[n] = w;
    return RLA_OK;
}

extern "C" int rla_sptrsv_transpose_in_f64(const double *b_dev, int64_t m, int64_t n, int64_t ldb,
                                           const int32_t *perm_dev, double *x_dev, int64_t ldx, void *stream) {
    RLA_REQUIRE(m >= 0 && n >= 0 && ldb >= n && ldx >= m && (ldx & 1) == 0, "rla_sptrsv_transpose_in_f64: bad sizes");
    if (m == 0 || n == 0) return RLA_OK;
    RLA_REQUIRE(b_dev && x_dev, "rla_sptrsv_transpose_in_f64: null pointer");
    dim3 grid((unsigned)((n + 31) / 32), (unsigned)((ldx + 31) / 32));
    RLA_REQUIRE(grid.y <= 65535, "rla_sptrsv_transpose_in_f64: too many right-hand sides");
    trsv_in_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(b_dev, m, n, ldb, perm_dev, x_dev, ldx);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

extern "C" int rla_sptrsv_transpose_out_f64(const double *x_dev, int64_t m, int64_t n, int64_t ldx,
                                            const int32_t *perm_dev, double *out_dev, int64_t ldo, void *stream) {
    RLA_REQUIRE(m >= 0 && n >= 0 && ldo >= n && ldx >= m, "rla_sptrsv_transpose_out_f64: bad sizes");
    if (m == 0 || n == 0) return RLA_OK;
    RLA_REQUIRE(x_dev && out_dev, "rla_sptrsv_transpose_out_f64: null pointer");
    dim3 grid((unsigned)((n + 31) / 32), (unsigned)((m + 31) / 32));
    RLA_REQUIRE(grid.y <= 65535, "rla_sptrsv_transpose_out_f64: too many right-hand sides");
    trsv_out_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(x_dev, m, n, ldx, perm_dev, out_dev, ldo);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

// Inverses of the groups' triangular blocks (HOST, once per factor).  Group g holds the rows at
// positions [grp_start[g], + grp_rows[g]); its block D has diag_in[p] on the diagonal and the row's
// internal entries (col2 = slot inside the group) below it.  dinv_out + dinv_ptr[g] receives
// D^-1 row-major (nrows x nrows, upper triangle zero) by forward substitution, column by column;
// diag_eff_out[p] = 1.0 for the rows of a group (their division is inside D^-1), diag_in[p] else.
extern "C" int rla_sptrsv_group_inverses_host(int64_t n, const int64_t *rowptr2, const int32_t *col2, const double *val2,
                                              const double *diag_in, const int64_t *split, int64_t ngroups,
                                              const int64_t *grp_start, const int32_t *grp_rows,
                                              const int64_t *dinv_ptr, double *dinv_out, double *diag_eff_out) {
    RLA_REQUIRE(n >= 0 && ngroups >= 0 && rowptr2 && diag_in && split && diag_eff_out &&
                (ngroups == 0 || (grp_start && grp_rows && dinv_ptr && dinv_out)), "rla_sptrsv_group_inverses_host: null pointer");
    for (int64_t q = 0; q < n; ++q) diag_eff_out[q] = diag_in[q];
    std::vector<double> D;
    for (int64_t g = 0; g < ngroups; ++g) {
        const int64_t g0 = grp_start[g];
        const int nr = grp_rows[g];
        RLA_REQUIRE(nr >= 1 && nr <= TRSV_GROUP && g0 >= 0 && g0 + nr <= n, "rla_sptrsv_group_inverses_host: bad group %lld", (long long)g);
        D.assign((size_t)nr * nr, 0.0);
        for (int r = 0; r < nr; ++r) {
            const int64_t q = g0 + r;
            D[(size_t)r * nr + r] = diag_in[q];
            RLA_REQUIRE(diag_in[q] != 0.0, "rla_sptrsv_group_inverses_host: zero diagonal at position %lld", (long long)q);
            for (int64_t e = split[q]; e < rowptr2[q + 1]; ++e) {
                RLA_REQUIRE(col2[e] >= 0 && col2[e] < r, "rla_sptrsv_group_inverses_host: internal entry outside the group");
                D[(size_t)r * nr + col2[e]] = val2[e];
            }
            diag_eff_out[q] = 1.0;
        }
        double *W = dinv_out + dinv_ptr[g];
        for (int c = 0; c < nr; ++c) {                  // column c of the inverse: D w = e_c
            for (int r = 0; r < c; ++r) W[(size_t)r * nr + c] = 0.0;
            for (int r = c; r < nr; ++r) {
                double acc = r == c ? 1.0 : 0.0;
                const double *Dr = D.data() + (size_t)r * nr;
                for (int k = c; k < r; ++k) acc -= Dr[k] * W[(size_t)k * nr + c];
                W[(size_t)r * nr + c] = acc / Dr[r];
            }
        }
    }
    return RLA_OK;
}

// In-place triangular solve T X = X on the (n, ldx) block (right-hand sides contiguous, rows in
// schedule order), driven by the step list of rla_sptrsv_plan_host (HOST arrays step_*); all other
// arrays on the device.  diag_eff_dev: divisor per position (rla_sptrsv_group_inverses_host), or NULL
// when every divisor is 1 (unit-diagonal factor).
extern "C" int rla_sptrsv_solve_f64(const int64_t *rowptr_dev, const int32_t *col_dev, const double *val_dev,
                                    const double *diag_eff_dev, const int64_t *split_dev,
                                    const int64_t *grp_start_dev, const int32_t *grp_rows_dev,
                                    const int64_t *dinv_ptr_dev, const double *dinv_dev,
                                    const int64_t *step_lo, const int64_t *step_hi, const int32_t *step_kind,
                                    int64_t nsteps, double *x_dev, int64_t m, int64_t ldx, void *stream) {
    RLA_REQUIRE(nsteps >= 0 && m >= 0 && ldx >= m && (ldx & 1) == 0, "rla_sptrsv_solve_f64: bad sizes");
    if (nsteps == 0 || m == 0) return RLA_OK;
    RLA_REQUIRE(rowptr_dev && col_dev && val_dev && split_dev && step_lo && step_hi && step_kind && x_dev,
                "rla_sptrsv_solve_f64: null pointer");
    RLA_REQUIRE(((uintptr_t)x_dev & 15) == 0, "rla_sptrsv_solve_f64: X must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    TrsvArgs a = {rowptr_dev, col_dev, val_dev, diag_eff_dev, split_dev, x_dev, ldx, m};
    const unsigned chunks = (unsigned)((ldx + TRSV_RHS - 1) / TRSV_RHS);
    RLA_REQUIRE(chunks <= 65535, "rla_sptrsv_solve_f64: too many right-hand sides");
    // the opt-in to 64 KB of dynamic shared memory holds for the current device only: made once per
    // device, as a process may solve on several.  SparseLU.solve runs a shape eagerly before it
    // captures it into a graph, so on its path the opt-in is never made during a capture.
    static bool attr_set[64] = {};
    int dev = 0;
    RLA_CUDA_CHECK(cudaGetDevice(&dev));
    const int resolve_smem = TRSV_GROUP * 32 * (int)sizeof(double2);
    if (dev < 0 || dev >= 64 || !attr_set[dev]) {
        RLA_CUDA_CHECK(cudaFuncSetAttribute(trsv_resolve_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, resolve_smem));
        RLA_CUDA_CHECK(cudaFuncSetAttribute(trsv_resolve_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, resolve_smem));
        if (dev >= 0 && dev < 64) attr_set[dev] = true;
    }
    for (int64_t s = 0; s < nsteps; ++s) {
        const int64_t cnt = step_hi[s] - step_lo[s];
        RLA_REQUIRE(cnt >= 1, "rla_sptrsv_solve_f64: empty step %lld", (long long)s);
        if (step_kind[s] == 0) {
            dim3 grid((unsigned)((cnt + 7) / 8), chunks);
            trsv_rows_warp_kernel<<<grid, 256, 0, st>>>(a, step_lo[s], step_hi[s]);
        } else if (step_kind[s] == 1) {
            RLA_REQUIRE(cnt < (int64_t(1) << 31), "rla_sptrsv_solve_f64: step too large");
            dim3 grid((unsigned)cnt, chunks);
            if (cnt * chunks <= 2 * (int64_t)sm_count()) trsv_rows_cta_kernel<16><<<grid, 32 * 16, 0, st>>>(a, step_lo[s]);
            else trsv_rows_cta_kernel<8><<<grid, 32 * 8, 0, st>>>(a, step_lo[s]);
        } else if (step_kind[s] == 2) {
            RLA_REQUIRE(grp_start_dev && grp_rows_dev && dinv_ptr_dev && dinv_dev && cnt < (int64_t(1) << 31),
                        "rla_sptrsv_solve_f64: group arrays missing");
            // few groups in the step: four CTAs per group (a quarter of the chain's rows each)
            if (cnt * chunks * 4 <= 2 * (int64_t)sm_count()) {
                dim3 grid((unsigned)cnt * 4, chunks);
                trsv_resolve_kernel<4><<<grid, 32 * TRSV_WARPS, resolve_smem, st>>>(x_dev, ldx, grp_start_dev, grp_rows_dev,
                                                                                   dinv_ptr_dev, dinv_dev, step_lo[s]);
            } else {
                dim3 grid((unsigned)cnt, chunks);
                trsv_resolve_kernel<1><<<grid, 32 * TRSV_WARPS, resolve_smem, st>>>(x_dev, ldx, grp_start_dev, grp_rows_dev,
                                                                                   dinv_ptr_dev, dinv_dev, step_lo[s]);
            }
        } else {
            return fail(RLA_ERR_INVALID, "rla_sptrsv_solve_f64: unknown step kind %d", step_kind[s]);
        }
        count_launch();
    }
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}

// out[p, :] = in[map[p], :] on (n, ldx) blocks: the re-ordering between the schedules of L and U
extern "C" int rla_sptrsv_permute_rows_f64(const double *in_dev, const int32_t *map_dev, double *out_dev, int64_t n,
                                           int64_t ldx, void *stream) {
    RLA_REQUIRE(n >= 0 && ldx >= 0 && (ldx & 1) == 0, "rla_sptrsv_permute_rows_f64: bad sizes");
    if (n == 0 || ldx == 0) return RLA_OK;
    RLA_REQUIRE(in_dev && map_dev && out_dev && in_dev != out_dev, "rla_sptrsv_permute_rows_f64: bad pointers");
    const int64_t work = n * (ldx / 2);
    const unsigned blocks = (unsigned)std::min<int64_t>((work + 255) / 256, (int64_t)sm_count() * 16);
    trsv_permute_rows_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(in_dev, map_dev, out_dev, n, ldx);
    count_launch();
    RLA_CUDA_CHECK(cudaGetLastError());
    return RLA_OK;
}
