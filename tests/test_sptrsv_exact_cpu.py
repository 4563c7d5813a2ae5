"""The checks of tests/test_sptrsv_exact_gpu.py can fail: on the CPU, without a GPU.

The NumPy replay of the device schedule (`_replay` of tests/test_sptrsv_plan.py: the kernels'
arithmetic, step by step, in schedule order) passes the componentwise bound; the same replay with
one external term of relative size ~1e-14 dropped, or with one single row left undivided, does
not.  A kernel that made either mistake on the device would fail the GPU tests in the same way.
The exact residual and the extended-precision substitution are checked against rational
arithmetic on a small factor.  The loss of accuracy of the schedule's explicit group inverses
on ill-conditioned group blocks is measured against SuperLU and plain substitution."""
from fractions import Fraction

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.linalg import splu, spsolve_triangular

from rla4mor_b200.factorization import plan_triangular
from test_sptrsv_exact_gpu import (U_ROUND, assert_within_bound, case, componentwise_bound, exact_lu_solve,
                                   exact_residual, factors, group_block_condition, replay_lu_solve, substitute)
from test_sptrsv_plan import _fem, _replay


def _frac(v):
    return Fraction(*np.longdouble(v).as_integer_ratio())               # exact for np.longdouble


@pytest.fixture(scope="module")
def lu():
    return splu(_fem(24))


def test_reference_matches_rational_arithmetic():
    """exact_residual and substitute against Fraction on a 12 x 12 lower factor with entries of
    very different magnitudes."""
    rs = np.random.RandomState(4)
    n, m = 12, 3
    T = sp.tril(sp.random(n, n, 0.5, random_state=rs), -1).tocsr() * 1e3
    T = (T + sp.diags(rs.uniform(0.5, 2.0, n) * 10.0 ** rs.randint(-8, 8, n))).tocsr()
    B = rs.standard_normal((n, m))
    X = substitute(T, B, True)
    Xd = X.astype(np.float64)
    R = exact_residual(T, Xd, B)
    Td = T.toarray()
    for c in range(m):
        xq = [None] * n
        for i in range(n):
            s = Fraction(B[i, c]) - sum(Fraction(Td[i, j]) * xq[j] for j in range(i) if Td[i, j] != 0)
            xq[i] = s / Fraction(Td[i, i])
        for i in range(n):
            rq = Fraction(B[i, c]) - sum(Fraction(Td[i, j]) * Fraction(Xd[j, c]) for j in range(n) if Td[i, j] != 0)
            scale = abs(B[i, c]) + sum(abs(Td[i, j] * Xd[j, c]) for j in range(n))
            assert abs(float(_frac(R[i, c]) - rq)) <= (n + 2) * 2.0 ** -64 * scale      # far below u
            assert abs(float(_frac(X[i, c]) - xq[i])) <= 1e-17 * abs(float(xq[i]))


def test_exact_lu_solve_inverts_the_matrix(lu):
    A = _fem(24)
    B = np.random.RandomState(1).standard_normal((3, A.shape[0]))
    for adjoint in (False, True):
        x = exact_lu_solve(lu, B, adjoint).astype(np.float64)
        M = A.T if adjoint else A
        assert np.abs((M @ x.T).T - B).max() < 1e-13


@pytest.mark.parametrize("which", ["L", "U", "Ut", "Lt"])
def test_replay_of_the_schedule_within_bound(lu, which):
    T, lower, unit = {"L": (lu.L, True, True), "U": (lu.U, False, False),
                      "Ut": (lu.U.T, True, False), "Lt": (lu.L.T, False, True)}[which]
    T = T.tocsr()
    p = plan_triangular(T, lower)
    assert p["ngroups"] > 0 and (p["step_kind"] == 0).any()
    B = np.random.RandomState(2).standard_normal((T.shape[0], 5))
    assert_within_bound(T, lower, _replay(p, B, unit), B, p, what=which)


def _single_row(p, T, rows_ok):
    """Position of a single (ungrouped) row whose row of T satisfies rows_ok(i)."""
    in_group = np.zeros(p["n"], dtype=bool)
    for g0, nr in zip(p["grp_start"][:p["ngroups"]], p["grp_rows"][:p["ngroups"]]):
        in_group[g0:g0 + nr] = True
    for q in np.flatnonzero(~in_group):
        if rows_ok(int(p["order"][q])):
            return int(q)
    raise AssertionError("no such row")


def test_bound_rejects_a_dropped_small_term(lu):
    """One external entry of a single row made ~1e-14 of its row's terms; the replay that leaves
    it out fails the bound, the exact replay passes."""
    T = lu.U.tocsr().astype(np.float64)
    B = np.random.RandomState(3).standard_normal((T.shape[0], 4))
    p = plan_triangular(T, False)
    q = _single_row(p, T, lambda i: 2 <= T.indptr[i + 1] - T.indptr[i] <= 4)
    i = int(p["order"][q])
    x = _replay(p, B, False)
    e = p["rowptr"][q]                                   # an external entry of that row (schedule CSR)
    j = int(p["order"][p["col"][e]])
    k = T.indptr[i] + int(np.flatnonzero(T.indices[T.indptr[i]:T.indptr[i + 1]] == j)[0])
    row_scale = np.abs(B[i]).max() + (abs(T[i]) @ np.abs(x)).max()
    T.data[k] = 1e-14 * row_scale / np.abs(x[j]).max()
    p = plan_triangular(T, False)                         # same schedule, new value
    exact = _replay(p, B, False)
    assert_within_bound(T, False, exact, B, p, what="exact replay")
    dropped = dict(p, val=p["val"].copy())
    dropped["val"][dropped["rowptr"][q]] = 0.0
    x_bad = _replay(dropped, B, False)
    with pytest.raises(AssertionError, match="componentwise bound"):
        assert_within_bound(T, False, x_bad, B, p, what="one term dropped")
    # the error is about 1e-14 of the row: invisible to a normwise 1e-12 check
    ref = substitute(T, B, False).astype(np.float64)
    assert np.linalg.norm(x_bad - ref) / np.linalg.norm(ref) < 1e-12


def test_bound_rejects_an_undivided_single_row(lu):
    T = lu.U.tocsr()
    B = np.random.RandomState(5).standard_normal((T.shape[0], 4))
    p = plan_triangular(T, False)
    q = _single_row(p, T, lambda i: True)
    undivided = dict(p, diag=p["diag"].copy(), diag_eff=p["diag_eff"].copy())
    undivided["diag"][q] = undivided["diag_eff"][q] = 1.0
    x_bad = _replay(undivided, B, False)
    with pytest.raises(AssertionError, match="componentwise bound"):
        assert_within_bound(T, False, x_bad, B, p, what="one row undivided")


def test_bound_is_not_vacuous(lu):
    """The bound is a few gamma_w of the row's terms: on this factor at most ~1e-13 of them."""
    T = lu.L.tocsr()
    B = np.random.RandomState(6).standard_normal((T.shape[0], 2))
    x = substitute(T, B, True).astype(np.float64)
    bnd = componentwise_bound(T, True, x, B)
    scale = np.abs(B) + abs(T) @ np.abs(x)
    assert (bnd / scale).max() < 1e3 * U_ROUND


@pytest.mark.parametrize("name,lossy", [("symmetric_indefinite", True), ("fem80", False)])
def test_explicit_group_inverse_accuracy(name, lossy):
    """A group is resolved as x = Dinv y with the explicit inverse of its triangular block D, whose
    forward error can exceed substitution's by up to || |Dinv| |D| ||.  On the symmetric-mode
    factor of the indefinite matrix of the GPU tests (group blocks with || |Dinv| |D| || ~ 1e5)
    the NumPy replay of the schedule has 17x (forward) and 20x (adjoint) SuperLU's largest
    relative error over these 127 right-hand sides (5.8e-12 against 3.5e-13, 1.0e-11 against
    5.3e-13), while float64 substitution with the same factors stays within 4x of SuperLU (2.6e-13,
    6.9e-13); on the FEM Laplacian (|| |Dinv| |D| || ~ 10) the replay is as accurate as SuperLU."""
    A, f, _ = case(name)
    n, m = A.shape[0], 127
    for adjoint in (False, True):
        V = np.random.RandomState(8 + adjoint).standard_normal((m, n))
        ex = exact_lu_solve(f, V, adjoint).astype(np.float64)
        (T1, l1, _), (T2, l2, _) = factors(f, adjoint)
        p_in, p_out = (f.perm_c, f.perm_r) if adjoint else (f.perm_r, f.perm_c)
        Y = np.empty((n, m))
        Y[p_in] = V.T
        sub = spsolve_triangular(T2, spsolve_triangular(T1, Y, lower=l1), lower=l2)[p_out].T
        slu = f.solve(np.ascontiguousarray(V.T), trans="T" if adjoint else "N").T

        def rel(x):
            return float(np.max(np.linalg.norm(x - ex, axis=1) / np.linalg.norm(ex, axis=1)))

        e_replay, e_slu, e_sub = rel(replay_lu_solve(f, V, adjoint)), rel(slu), rel(sub)
        cond = max(group_block_condition(T, plan_triangular(T, lower)) for T, lower in ((T1, l1), (T2, l2)))
        assert e_sub < 4 * e_slu
        if lossy:
            assert cond > 1e4 and e_replay > 5 * e_slu, (cond, e_replay, e_slu)
        else:
            assert cond < 100 and e_replay < 2 * e_slu, (cond, e_replay, e_slu)
