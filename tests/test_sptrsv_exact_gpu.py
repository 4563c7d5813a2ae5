"""The device's sparse LU solves (csrc/sptrsv.cu through factorization.SparseLU) against an
extended-precision reference, at the edges where the kernels could go subtly wrong.

A normwise comparison with SuperLU at 1e-12 cannot tell a right kernel from one that drops a small
external term or divides a row twice: on benign inputs both stay near 1e-14.  The checks here are
sharper:
  * every factor on its own (`TriangularFactor.solve_inplace`): each entry of the residual
    b - T x, computed exactly, against the componentwise bound of the schedule's arithmetic
    (`componentwise_bound`, derivation there), with a factor of 2 of slack;
  * the whole solve (`InverseLuOperator.apply` / `apply_adjoint`): per right-hand side, the
    forward error against the exact solution with the same factors is at most 4x SuperLU's own
    (on ill-conditioned group blocks: 4x the larger of SuperLU's and the NumPy replay's, see
    EXPLICIT_INVERSE_LOSS);
  * the CUDA-graph replay of `SparseLU.solve` is bit-identical to the eager launches, through
    replays, eviction and re-capture, on a side stream, and counts the same launches;
  * a second device.
The cases are chosen so that, forward and adjoint, they reach all five launch variants of
`rla_sptrsv_solve_f64` and the schedule shapes listed in `REQUIRED_SHAPES` (checked by
`test_cases_cover_every_launch_variant_and_shape`).
The reference, the residual and the bound run on the CPU; tests/test_sptrsv_exact_cpu.py runs them
on the NumPy replay of the schedule and shows that the bound rejects a subtly wrong kernel.
"""
import functools

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.linalg import splu

from exact_ref import U_ROUND, gamma, require_longdouble, two_product
from rla4mor_b200.factorization import plan_triangular, splu_symetric
from test_sptrsv_plan import _replay

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------- extended-precision reference

def substitute(T, B, lower):
    """T X = B by substitution over the CSR rows of T in np.longdouble (64-bit mantissa), all
    right-hand sides (columns of B) at once.  Every row must hold its diagonal."""
    require_longdouble()
    T = T.tocsr()
    T.sort_indices()
    n = T.shape[0]
    ptr, ind, val = T.indptr, T.indices, T.data.astype(np.longdouble)
    X = np.array(B, dtype=np.longdouble).reshape(n, -1)
    for i in (range(n) if lower else range(n - 1, -1, -1)):
        c, v = ind[ptr[i]:ptr[i + 1]], val[ptr[i]:ptr[i + 1]]
        on = c == i
        assert on.sum() == 1, f"row {i} has no diagonal entry"
        off = ~on
        X[i] = (X[i] - v[off] @ X[c[off]]) / v[on][0]
    return X


def exact_lu_solve(factorization, B, adjoint=False):
    """The solve of SparseLU.solve with the same L, U, perm_r and perm_c (Pr A Pc = L U), in
    np.longdouble: B is the (m, n) block, one right-hand side per row; returns (m, n) longdouble.
    A x = b:    L U z = Pr b,        x = Pc z      (z[perm_c[i]] -> x[i])
    A^T x = b:  U^T L^T w = Pc^T b,  x = Pr^T w    (w[perm_r[i]] -> x[i])"""
    f = factorization
    B = np.asarray(B, dtype=np.float64)
    n = B.shape[1]
    L, U = f.L.tocsr(), f.U.tocsr()
    p_in, p_out = (f.perm_c, f.perm_r) if adjoint else (f.perm_r, f.perm_c)
    Y = np.empty((n, B.shape[0]), dtype=np.longdouble)
    Y[p_in] = B.T
    if adjoint:
        Z = substitute(L.T.tocsr(), substitute(U.T.tocsr(), Y, True), False)
    else:
        Z = substitute(U, substitute(L, Y, True), False)
    return Z[p_out].T


def exact_residual(T, X, B):
    """R = B - T X for float64 T (sparse), X and B (n, m), with every product T_ij X_jc split
    exactly into two doubles and the row sums taken in np.longdouble: the error of R is at most
    ~ w * 2^-64 * (|B| + |T||X|) for a row of w entries, far below float64's unit roundoff."""
    require_longdouble()
    T = T.tocsr()
    n = T.shape[0]
    X = np.asarray(X, dtype=np.float64).reshape(n, -1)
    R = np.array(B, dtype=np.longdouble).reshape(n, -1)
    ptr, ind, val = T.indptr, T.indices, T.data
    m = X.shape[1]
    # exactness of TwoProduct: no overflow in the split, no underflow of the error term
    big = max(np.abs(val).max(initial=0.0), np.abs(X).max(initial=0.0))
    assert big < 2.0 ** 995, "values too large for an exact split"
    step = max(1, (1 << 22) // max(m, 1))                # entries x right-hand sides per chunk
    r0 = 0
    while r0 < n:
        r1 = int(np.searchsorted(ptr, ptr[r0] + step, side="right")) - 1
        r1 = min(n, max(r1, r0 + 1))
        e0, e1 = ptr[r0], ptr[r1]
        if e1 > e0:
            p, e = two_product(val[e0:e1, None], X[ind[e0:e1]])
            tiny = (p != 0) & (np.abs(p) < 2.0 ** -960)
            assert not tiny.any(), "products too small for an exact TwoProduct"
            terms = p.astype(np.longdouble) + e.astype(np.longdouble)
            cnt = np.diff(ptr[r0:r1 + 1])
            nz = cnt > 0
            sums = np.add.reduceat(terms, (ptr[r0:r1] - e0)[nz], axis=0)
            R[r0:r1][nz] -= sums
        r0 = r1
    return R


def componentwise_bound(T, lower, X, B, plan=None):
    """Bound on |B - T X| entry by entry for X computed from B by the schedule of plan_triangular
    (the arithmetic of rla_sptrsv_solve_f64), with u = 2^-53 and gamma_k = k u / (1 - k u).

    A row i that is not in a group has w off-diagonal entries and is finished by one kind-0 or
    kind-1 launch: s = fl(b_i - sum_j T_ij x_j) over the w products (fused multiply-adds, one warp
    or 8-16 warps combined in warp order: every term goes through at most w + 1 roundings
    including the addition of b_i; partial sums of empty warps are zeros, added exactly), then
    x_i = fl(s / d_i).  Hence (Higham, Accuracy and Stability, section 8.1)
        |r_i| <= gamma_{w+2} (|b_i| + sum_j |T_ij| |x_j|)           (the diagonal term included).
    A row of a group g of nr rows (block D of the group, Dinv = W, the host's inverse of D in
    the plan) first gets y_i = fl(b_i - sum_{j outside g} T_ij x_j) with the same error term,
    y_i = b_i - sum_ext T_ij x_j + eta_i, |eta_i| <= gamma_{w+2} (|b_i| + sum_ext |T_ij||x_j|),
    and then x_g = fl(W y_g) = (W + dW) y_g with |dW| <= gamma_nr |W| (dot products of at most nr
    terms).  W was computed column by column by forward substitution, D w_c = e_c, so
    D W = I + E with |E| <= gamma_nr |D| |W|.  Therefore
        (b - T x)_i = -eta_i - (E y_g + D dW y_g)_i
        |r_i| <= gamma_{w+2} (|b_i| + sum_j |T_ij||x_j|) + 2 gamma_nr (|D| |W| |y_g|)_i.
    |y_g| is taken as the float64 value of b - T_ext x plus the bound on its rounding error.
    The returned array is this bound; the tests allow a factor of 2 above it and no more."""
    T = T.tocsr()
    n = T.shape[0]
    X = np.asarray(X, dtype=np.float64).reshape(n, -1)
    B = np.asarray(B, dtype=np.float64).reshape(n, -1)
    if plan is None:
        plan = plan_triangular(T, lower)
    A = abs(T)
    w = np.diff(T.indptr) - 1                            # off-diagonal entries per row
    bound = gamma(w + 2)[:, None] * (np.abs(B) + A @ np.abs(X))
    order = plan["order"]
    grp = np.full(n, -1, dtype=np.int64)
    for g in range(plan["ngroups"]):
        g0, nr = int(plan["grp_start"][g]), int(plan["grp_rows"][g])
        grp[order[g0:g0 + nr]] = g
    if plan["ngroups"] == 0:
        return bound
    C = T.tocoo()
    ext = (C.row != C.col) & ((grp[C.row] < 0) | (grp[C.row] != grp[C.col]))
    Text = sp.csr_matrix((C.data[ext], (C.row[ext], C.col[ext])), shape=T.shape)
    Aext = abs(Text)
    Y = np.abs(B - Text @ X) + gamma(w + 2)[:, None] * (np.abs(B) + Aext @ np.abs(X))
    for g in range(plan["ngroups"]):
        g0, nr = int(plan["grp_start"][g]), int(plan["grp_rows"][g])
        rows = order[g0:g0 + nr]                         # slots of the group = schedule order
        D = np.abs(T[rows][:, rows].toarray())
        W = np.abs(plan["dinv"][plan["dinv_ptr"][g]:plan["dinv_ptr"][g + 1]].reshape(nr, nr))
        bound[rows] += 2.0 * gamma(nr) * (D @ (W @ Y[rows]))
    return bound


def assert_within_bound(T, lower, X, B, plan=None, slack=2.0, what=""):
    """Every entry of the exact residual within `slack` times componentwise_bound."""
    R = np.abs(exact_residual(T, X, B)).astype(np.float64)
    bnd = componentwise_bound(T, lower, X, B, plan)
    ratio = np.divide(R, bnd, out=np.zeros_like(R), where=bnd > 0)
    assert np.all(R[bnd == 0] == 0), f"{what}: nonzero residual where the bound is zero"
    worst = np.unravel_index(np.argmax(ratio), ratio.shape) if ratio.size else None
    assert ratio.max(initial=0.0) <= slack, \
        f"{what}: residual {ratio.max():.3g} x its componentwise bound at (row, rhs) {worst}"
    return float(ratio.max(initial=0.0))


# ---------------------------------------------------------------- launch variants and schedule shapes

VARIANTS = ("rows_warp", "rows_cta<16>", "rows_cta<8>", "resolve<4>", "resolve<1>")
REQUIRED_SHAPES = ("level wider than 4096 rows", "group of 128 rows", "group of 2 rows",
                   "row of more than 64 entries in a multi-row group")


def launch_variants(plan, m, sms):
    """The kernels rla_sptrsv_solve_f64 launches for this schedule and m right-hand sides on a
    device of `sms` SMs (the same selection as the host code there)."""
    chunks = (m + (m & 1) + 63) // 64
    cnt = plan["step_hi"] - plan["step_lo"]
    kind = plan["step_kind"]
    hit = {
        "rows_warp": kind == 0,
        "rows_cta<16>": (kind == 1) & (cnt * chunks <= 2 * sms),
        "rows_cta<8>": (kind == 1) & (cnt * chunks > 2 * sms),
        "resolve<4>": (kind == 2) & (cnt * chunks * 4 <= 2 * sms),
        "resolve<1>": (kind == 2) & (cnt * chunks * 4 > 2 * sms),
    }
    return {v for v in VARIANTS if hit[v].any()}


def schedule_shapes(plan, wide_min=4096):
    sizes = plan["grp_rows"][:plan["ngroups"]]
    out = set()
    if np.bincount(plan["level"]).max(initial=0) > wide_min:
        out.add("level wider than 4096 rows")
    if (sizes == 128).any():
        out.add("group of 128 rows")
    if (sizes == 2).any():
        out.add("group of 2 rows")
    long_row = np.diff(plan["rowptr"]) > 64
    for lo, hi, kind in zip(plan["step_lo"], plan["step_hi"], plan["step_kind"]):
        if kind == 1:
            in_group = np.zeros(plan["n"], dtype=bool)
            for g0, nr in zip(plan["grp_start"][:plan["ngroups"]], sizes):
                if lo <= g0 < hi:
                    in_group[g0:g0 + nr] = True
            if (long_row & in_group).any():
                out.add("row of more than 64 entries in a multi-row group")
    return out


def factors(f, adjoint):
    """(T, lower, unit diagonal) of the two triangular solves of SparseLU, in launch order."""
    if adjoint:
        return ((f.U.T.tocsr(), True, False), (f.L.T.tocsr(), False, True))
    return ((f.L.tocsr(), True, True), (f.U.tocsr(), False, False))


# ---------------------------------------------------------------- cases

def _lap1(nx, coef=None):
    c = np.ones(nx + 1) if coef is None else coef
    return sp.diags([-c[1:-1], c[:-1] + c[1:], -c[1:-1]], [-1, 0, 1])


def _fem(nx, shift=0.1):
    T = _lap1(nx)
    return (sp.kron(sp.eye(nx), T) + sp.kron(T, sp.eye(nx)) + shift * sp.eye(nx * nx)).tocsc()


def _convection_diffusion(nx, peclet):
    """-Laplace u + b . grad u on the unit square, central differences, cell Peclet number
    |b_x| h / 1 = peclet along x and peclet / 2 along y: off-diagonals -1 -+ Pe/2 (not
    diagonally dominant, so SuperLU's partial pivoting swaps rows)."""
    ex = np.ones(nx)
    Tx = sp.diags([(-1 - peclet / 2) * ex[:-1], 2 * ex, (-1 + peclet / 2) * ex[:-1]], [-1, 0, 1])
    Ty = sp.diags([(-1 - peclet / 4) * ex[:-1], 2 * ex, (-1 + peclet / 4) * ex[:-1]], [-1, 0, 1])
    return (sp.kron(sp.eye(nx), Tx) + sp.kron(Ty, sp.eye(nx))).tocsc()


def _red_black_1d(n_half):
    """1-D diffusion with random coefficients, red-black ordered (even points first), factored
    without column reordering: the n_half red rows of L are one level (wider than 4096 rows), the
    black rows one chain (groups of 128 rows)."""
    n = 2 * n_half
    coef = np.exp(np.random.RandomState(7).uniform(-1.0, 1.0, n + 1))
    A = (_lap1(n, coef) + 0.01 * sp.eye(n)).tocsr()
    p = np.concatenate([np.arange(0, n, 2), np.arange(1, n, 2)])
    return A[p][:, p].tocsc()


def _scaled_fem(nx):
    """S K S with K a 2-D Laplacian and S random powers of ten in 1e-50..1e50: diagonals of A and
    of U spanning about 1e-100..1e100, rows and columns of every magnitude next to each other.
    Factored in symmetric mode, the factors are S L S^-1 and S U S: as well conditioned as K's
    (row pivoting on such a matrix would make SuperLU's own solve meaningless)."""
    s = 10.0 ** np.random.RandomState(5).uniform(-50.0, 50.0, nx * nx)
    return (sp.diags(s) @ _fem(nx) @ sp.diags(s)).tocsc()


# name -> (matrix, factorisation, numbers of right-hand sides).  Together (forward and adjoint)
# the cases reach every launch variant and every entry of REQUIRED_SHAPES, and the m cover 1 to 4
# chunks of 64 right-hand sides with and without the odd padding.
CASES = {
    # a 2-D FEM Laplacian (n = 6400), general splu: every variant in both directions, dense
    # supernodes near the root (rows of up to ~480 entries inside groups), groups of 2 and 128
    "fem80": (lambda: _fem(80), splu, (200, 1)),
    # non-symmetric convection-diffusion, cell Peclet 10, partial pivoting active: badly
    # conditioned triangular blocks
    "convection_diffusion_pe10": (lambda: _convection_diffusion(60, 10.0), splu, (129, 63)),
    # symmetric indefinite (shifted Laplacian with eigenvalues of both signs) in the reference's
    # symmetric mode (diag_pivot_thresh=0): no pivoting, small pivots
    "symmetric_indefinite": (lambda: _fem(50, -1.3), splu_symetric, (127, 2)),
    # diagonals spanning 1e-100..1e100
    "scaled_1e100": (lambda: _scaled_fem(50), splu_symetric, (64, 65)),
    # a level of 4200 rows and a 4200-row chain
    "red_black_wide_level": (lambda: _red_black_1d(4200), lambda A: splu(A, permc_spec="NATURAL"), (65, 1)),
}
RHS_COUNTS = {1, 2, 63, 64, 65, 127, 129, 200}


@functools.lru_cache(maxsize=None)
def case(name):
    make, factorize, ms = CASES[name]
    A = make()
    return A, factorize(A), ms


def _rhs(name, m, n, salt):
    seed = (sum(map(ord, name)) * 1009 + 31 * m + salt) % (2 ** 31)
    return np.random.RandomState(seed).standard_normal((m, n))


@pytest.fixture(scope="module")
def rb():
    import rla4mor_b200
    rla4mor_b200.lib()
    return rla4mor_b200


@pytest.fixture(scope="module")
def sms(rb):
    import torch
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# ---------------------------------------------------------------- tests

@pytest.mark.parametrize("adjoint", [False, True], ids=["forward", "adjoint"])
@pytest.mark.parametrize("name", list(CASES))
def test_each_factor_within_componentwise_bound(rb, name, adjoint):
    """TriangularFactor.solve_inplace on the block in schedule order (as SparseLU lays it out:
    (n, ldx) with ldx = m rounded up to even, the padding column zero), every entry of the exact
    residual within twice the bound of componentwise_bound."""
    import torch
    from rla4mor_b200.factorization import TriangularFactor
    A, f, ms = case(name)
    n = A.shape[0]
    for which, (T, lower, unit) in enumerate(factors(f, adjoint)):
        plan = plan_triangular(T, lower)
        tf = TriangularFactor(T, lower, unit, "cuda")
        assert np.array_equal(tf.order_host, plan["order"])
        for m in ms:
            B = _rhs(name, m, n, 17 + 2 * which + adjoint).T                 # (n, m), row i = row i of T
            ldx = m + (m & 1)
            X = torch.zeros((n, ldx), dtype=torch.float64, device="cuda")
            X[:, :m] = torch.from_numpy(B[plan["order"]]).cuda()
            tf.solve_inplace(X, m)
            Xs = X.cpu().numpy()
            assert not Xs[:, m:].any(), "the padding column picked up a value"
            x = np.empty((n, m))
            x[plan["order"]] = Xs[:, :m]
            assert_within_bound(T, lower, x, B, plan, what=f"{name} factor {which} m={m}")


def replay_lu_solve(factorization, B, adjoint=False):
    """The solve of SparseLU.solve with the NumPy replay of the device schedule (`_replay` of
    tests/test_sptrsv_plan.py: each group resolved as x = Dinv y with the plan's explicit inverse),
    in float64: the accuracy the schedule's algorithm has, whatever the order of the kernels' sums."""
    f = factorization
    n = B.shape[1]
    (T1, l1, u1), (T2, l2, u2) = factors(f, adjoint)
    p_in, p_out = (f.perm_c, f.perm_r) if adjoint else (f.perm_r, f.perm_c)
    Y = np.empty((n, B.shape[0]))
    Y[p_in] = B.T
    Z = _replay(plan_triangular(T2, l2), _replay(plan_triangular(T1, l1), Y, u1), u2)
    return Z[p_out].T


def group_block_condition(T, plan):
    """max over the groups of the plan of || |Dinv| |D| ||_inf, D the group's triangular block:
    the factor by which x = Dinv y can lose accuracy against substitution in the group."""
    worst = 1.0
    for g in range(plan["ngroups"]):
        g0, nr = int(plan["grp_start"][g]), int(plan["grp_rows"][g])
        rows = plan["order"][g0:g0 + nr]
        D = np.abs(T[rows][:, rows].toarray())
        W = np.abs(plan["dinv"][plan["dinv_ptr"][g]:plan["dinv_ptr"][g + 1]].reshape(nr, nr))
        worst = max(worst, float((W @ D).sum(axis=1).max()))
    return worst


# Cases whose group blocks are ill-conditioned: there the explicit inverse of the group resolve
# (x = Dinv y) is less accurate than SuperLU's substitution, and the whole solve is held to the
# NumPy replay of the same schedule as well (test_sptrsv_exact_cpu.py measures the loss).
EXPLICIT_INVERSE_LOSS = {"symmetric_indefinite"}


@pytest.mark.parametrize("name", list(CASES))
def test_whole_solve_forward_error_within_4x_superlu(rb, name):
    """InverseLuOperator.apply / apply_adjoint: per right-hand side, the 2-norm error against the
    exact solution with the same factors is at most 4x that of SuperLU's solve with those
    factors, or 8 u ||x||.  On the cases of EXPLICIT_INVERSE_LOSS (group blocks with
    || |Dinv| |D| || above 1e3) the yardstick is the larger of SuperLU's error and that of the
    NumPy replay of the schedule, which resolves the groups with the same explicit inverses."""
    from rla4mor_b200.factorization import InverseLuOperator
    A, f, ms = case(name)
    n = A.shape[0]
    if name in EXPLICIT_INVERSE_LOSS:
        assert max(group_block_condition(T, plan_triangular(T, lower))
                   for adj in (False, True) for T, lower, _ in factors(f, adj)) > 1e3
    op = rb.MatrixOperator(A)
    inv = InverseLuOperator(op, factorization=f)
    for m in ms:
        for adjoint in (False, True):
            V = _rhs(name, m, n, 1 + adjoint)
            U = op.source.from_numpy(V)
            got = (inv.apply_adjoint(U) if adjoint else inv.apply(U)).to_numpy()
            slu = f.solve(np.ascontiguousarray(V.T), trans="T" if adjoint else "N").T
            ex = exact_lu_solve(f, V, adjoint)
            err_gpu = np.linalg.norm((got - ex).astype(np.float64), axis=1)
            err_ref = np.linalg.norm((slu - ex).astype(np.float64), axis=1)
            if name in EXPLICIT_INVERSE_LOSS:
                err_ref = np.maximum(err_ref, np.linalg.norm((replay_lu_solve(f, V, adjoint) - ex).astype(np.float64), axis=1))
            floor = 8 * U_ROUND * np.linalg.norm(ex.astype(np.float64), axis=1)
            bad = err_gpu > np.maximum(4 * err_ref, floor)
            assert not bad.any(), (f"{name} m={m} adjoint={adjoint}: rhs {np.flatnonzero(bad)[:5]}: "
                                   f"error {err_gpu[bad][:3]} vs reference solve {err_ref[bad][:3]}")


def test_strided_block(rb):
    """A block whose rows are not adjacent (row stride 2 (n + 3)) and a column-strided view go
    through the same solve as the contiguous copy, bit for bit, and meet the forward-error test."""
    import torch
    from rla4mor_b200.factorization import SparseLU
    A, f, _ = case("convection_diffusion_pe10")
    n, m = A.shape[0], 33
    lu = SparseLU(f)
    big = torch.from_numpy(np.random.RandomState(11).standard_normal((2 * m, n + 3))).cuda()
    Bv = big[::2, :n]
    assert Bv.stride() == (2 * (n + 3), 1)
    for adjoint in (False, True):
        got = lu.solve(Bv, adjoint=adjoint)
        assert torch.equal(got, lu.solve(Bv.contiguous(), adjoint=adjoint))
        Bt = Bv.contiguous().t().contiguous().t()                              # stride (1, m)
        assert torch.equal(got, lu.solve(Bt, adjoint=adjoint))
        V = Bv.cpu().numpy()
        ex = exact_lu_solve(f, V, adjoint).astype(np.float64)
        slu = f.solve(np.ascontiguousarray(V.T), trans="T" if adjoint else "N").T
        err_gpu = np.linalg.norm(got.cpu().numpy() - ex, axis=1)
        err_slu = np.linalg.norm(slu - ex, axis=1)
        assert np.all(err_gpu <= np.maximum(4 * err_slu, 8 * U_ROUND * np.linalg.norm(ex, axis=1)))


def test_cases_cover_every_launch_variant_and_shape(rb, sms):
    """The five launch variants in each direction, the schedule shapes of REQUIRED_SHAPES and the
    matrices and right-hand side counts the cases are meant to have."""
    seen = {False: set(), True: set()}
    shapes = set()
    for name in CASES:
        A, f, ms = case(name)
        for adjoint in (False, True):
            for T, lower, _ in factors(f, adjoint):
                plan = plan_triangular(T, lower)
                shapes |= schedule_shapes(plan)
                for m in ms:
                    seen[adjoint] |= launch_variants(plan, m, sms)
    assert seen[False] == set(VARIANTS), f"forward solves miss {set(VARIANTS) - seen[False]}"
    assert seen[True] == set(VARIANTS), f"adjoint solves miss {set(VARIANTS) - seen[True]}"
    assert shapes >= set(REQUIRED_SHAPES), f"no case has {set(REQUIRED_SHAPES) - shapes}"
    assert set().union(*(case(c)[2] for c in CASES)) == RHS_COUNTS
    _, f, _ = case("convection_diffusion_pe10")
    assert (f.perm_r != np.arange(f.shape[0])).mean() > 0.5                  # pivoting active
    A, f, _ = case("symmetric_indefinite")
    d = f.U.diagonal()
    assert (d > 0).any() and (d < 0).any()
    A, f, _ = case("scaled_1e100")
    d = np.abs(f.U.diagonal())
    assert d.min() < 1e-90 and d.max() > 1e90


def test_graph_replay_is_bit_identical_to_eager(rb, monkeypatch):
    """SparseLU.solve with CUDA graphs against SparseLU.solve with RLA_SPTRSV_GRAPH=0 (eager
    launches), through the sequence  m1, m2, m1 (replay), adjoint m1, m3, m4 (evicts m1: at most
    four shapes are kept, the oldest first out), m5, m1 (captured again); fresh right-hand sides
    every time.  The same kernels run, so every result is the same bit for bit, also for a replay
    issued on a side stream and for two identical calls; a replay counts the launches of an eager
    call."""
    import torch
    from rla4mor_b200.factorization import SparseLU
    A, f, _ = case("fem80")
    n = A.shape[0]
    monkeypatch.delenv("RLA_SPTRSV_GRAPH", raising=False)
    lu_g = SparseLU(f)
    monkeypatch.setenv("RLA_SPTRSV_GRAPH", "0")
    lu_e = SparseLU(f)
    assert lu_g.use_graph and not lu_e.use_graph
    m1, m2, m3, m4, m5 = 65, 1, 64, 2, 129
    seq = [(m1, False), (m2, False), (m1, False), (m1, True), (m3, False), (m4, False), (m5, False), (m1, False)]
    rs = np.random.RandomState(23)
    first_graph = None

    def run(lu, B, adjoint):
        n0 = rb.lib().rla_launch_count()
        out = lu.solve(B, adjoint=adjoint)
        torch.cuda.synchronize()
        return out, rb.lib().rla_launch_count() - n0

    for t, (m, adjoint) in enumerate(seq):
        key = (adjoint, m)
        replay = key in lu_g._graphs
        assert replay == (t == 2), f"call {t}: cached shapes {list(lu_g._graphs)}"
        B = torch.from_numpy(rs.standard_normal((m, n))).cuda()
        got, d_g = run(lu_g, B, adjoint)
        ref, d_e = run(lu_e, B, adjoint)
        assert torch.equal(got, ref), f"call {t} (m={m}, adjoint={adjoint}) differs from the eager solve"
        assert d_g == d_e, f"call {t}: {d_g} launches counted with the graph, {d_e} eager"
        assert key in lu_g._graphs and len(lu_g._graphs) <= 4
        if t == 0:
            first_graph = lu_g._graphs[key][2]
        if t == 2:
            assert lu_g._graphs[key][2] is first_graph
            again, d_again = run(lu_g, B, adjoint)                             # identical call: identical bits
            assert torch.equal(again, got) and d_again == d_e
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):                                       # a replay on a side stream
                on_side = lu_g.solve(B, adjoint=adjoint)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            assert torch.equal(on_side, ref)
        if t == 5:
            assert (False, m1) not in lu_g._graphs                              # evicted, oldest first
    assert lu_g._graphs[(False, m1)][2] is not first_graph                      # captured again
    ex = exact_lu_solve(f, B.cpu().numpy())
    assert np.abs(got.cpu().numpy() - ex).max() <= 1e-12 * np.abs(ex).max()


def test_second_device(rb):
    """One process, one factorisation: solve through SparseLU on cuda:0, then on cuda:1.  The
    kernels' dynamic shared memory opt-in must be made on each device."""
    import torch
    from rla4mor_b200.factorization import SparseLU
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    A, f, _ = case("fem80")
    n, m = A.shape[0], 65
    V = _rhs("second device", m, n, 0)
    ex = {adj: exact_lu_solve(f, V, adj).astype(np.float64) for adj in (False, True)}
    results = {}
    for dev in ("cuda:0", "cuda:1"):
        lu = SparseLU(f, device=dev)
        B = torch.from_numpy(V).to(dev)
        for adjoint in (False, True):
            for _ in range(2):                                                  # eager + capture, then replay
                out = lu.solve(B, adjoint=adjoint)
                assert out.device == torch.device(dev)
                got = out.cpu().numpy()
                slu = f.solve(np.ascontiguousarray(V.T), trans="T" if adjoint else "N").T
                err_gpu = np.linalg.norm(got - ex[adjoint], axis=1)
                err_slu = np.linalg.norm(slu - ex[adjoint], axis=1)
                assert np.all(err_gpu <= np.maximum(4 * err_slu, 8 * U_ROUND * np.linalg.norm(ex[adjoint], axis=1)))
                results.setdefault(adjoint, []).append(out.cpu())
    for adjoint in (False, True):                                               # same kernels, same bits
        assert all(torch.equal(r, results[adjoint][0]) for r in results[adjoint])
