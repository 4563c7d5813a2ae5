"""CPU-only checks of the GMRES full-order solve (fom_solve.affine_gmres, AffineModel.solve_batch with
method='gmres'): the NumPy restatement of the iteration against spsolve, argument validation that
raises before anything reaches the device, and CG's rejection of non-symmetric terms."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch
from scipy.sparse.linalg import splu, spsolve

from gmres_ref import convection_diffusion_terms, gmres_ref
from rla4mor_b200 import fom_solve
from rla4mor_b200.sketched_reductor import AffineModel
from rla4mor_b200.vectorarray import DeviceVectorSpace, MatrixOperator


@pytest.mark.parametrize("th,restart", [((1.0, 100.0, 50.0, 0.0), 30),      # convection-dominated
                                        ((1.0, 100.0, 50.0, 0.0), 500),     # no restart
                                        ((1.0, 0.0, 0.0, -200.0), 30),      # indefinite
                                        ((1.0, 20.0, -10.0, -80.0), 10)])   # both, short cycles
def test_reference_agrees_with_spsolve(th, restart):
    terms = convection_diffusion_terms(24)
    lu = splu((terms[0] + terms[3]).tocsc())
    A = sum(t * M for t, M in zip(th, terms)).tocsr()
    f = np.random.RandomState(0).standard_normal(A.shape[0])
    x, it, resid, info = gmres_ref(A, f, lu.solve, 1e-12, restart, 2000)
    assert info == 0 and 0 < it < 2000 and resid <= 1e-12
    r = f - A @ x
    assert np.sqrt(r @ lu.solve(r)) <= 1e-12 * np.sqrt(f @ lu.solve(f))
    u = spsolve(A.tocsc(), f)
    assert np.linalg.norm(x - u) <= 1e-9 * np.linalg.norm(u)


def test_reference_conventions():
    terms = convection_diffusion_terms(12)
    lu = splu((terms[0] + terms[3]).tocsc())
    A = (terms[0] + 30 * terms[1] - 60 * terms[3]).tocsr()
    f = np.random.RandomState(1).standard_normal(A.shape[0])
    u = spsolve(A.tocsc(), f)
    # R^-1 A = I: one step; an exact x0: no step; b = 0: 0 in 0 steps
    assert gmres_ref((terms[0] + terms[3]).tocsr(), f, lu.solve, 1e-12, 30, 100)[1] == 1
    assert gmres_ref(A, f, lu.solve, 1e-10, 30, 100, x0=u)[1] <= 1
    x, it, resid, info = gmres_ref(A, 0 * f, lu.solve, 1e-10, 30, 100, x0=np.ones_like(f))
    assert it == 0 and info == 0 and not x.any()
    # out of iterations: the last iterate; not attainable: info 1, not a false 0
    x, it, resid, info = gmres_ref(A, f, lu.solve, 1e-10, 5, 3)
    assert info == 1 and it == 3 and np.all(np.isfinite(x)) and resid > 1e-10
    assert gmres_ref(A, f, lu.solve, 1e-17, 30, 200)[3] == 1
    # a negated preconditioner is not SPD: breakdown
    x, it, resid, info = gmres_ref(A, f, lambda v: -lu.solve(v), 1e-10, 30, 100)
    assert info == 2 and np.isnan(x).all()


class _Fom:
    """What AffineModel.solve_batch reads before it reaches the device (host tensors)."""

    def __init__(self, n=6, Q=3, Pf=2, operators=None):
        self.operators = operators if operators is not None else [None] * Q
        self.rhs = [torch.zeros((1, n), dtype=torch.float64) for _ in range(Pf)]
        self.operator_coefficients = [lambda mu, q=q: mu[q] for q in range(Q)]
        self.rhs_coefficients = [1.0] * Pf
        self.solution_space = DeviceVectorSpace(n)
        self._affine = None

    thetas = AffineModel.thetas
    thetas_batch = AffineModel.thetas_batch
    solve = AffineModel.solve
    solve_batch = AffineModel.solve_batch


def _args(P=4, **kw):
    return dict(theta_lhs=np.ones((P, 3)), theta_rhs=np.ones((P, 2)), preconditioner=None, **kw)


@pytest.mark.parametrize("restart", [0, -3, 2.5, 30.0, "30", True])
def test_restart_is_validated(restart):
    with pytest.raises(ValueError, match="restart"):
        _Fom().solve_batch(**_args(method="gmres", restart=restart))
    with pytest.raises(ValueError, match="restart"):
        fom_solve.affine_gmres(None, None, np.ones((1, 3)), np.ones((1, 1)), None, restart=restart)


def test_method_is_validated():
    with pytest.raises(ValueError, match="method='bicgstab'"):
        _Fom().solve_batch(**_args(method="bicgstab"))
    with pytest.raises(ValueError, match="restart= applies to method='gmres' only"):
        _Fom().solve_batch(**_args(restart=30))
    with pytest.raises(ValueError, match="restart= applies to method='gmres' only"):
        _Fom().solve(theta_lhs=np.ones(3), theta_rhs=np.ones(2), preconditioner=None, method="cg", restart=10)


@pytest.mark.parametrize("th,tf", [(np.ones((4, 2)), np.ones((4, 2))),
                                   (np.ones((4, 3)), np.ones((3, 2))),
                                   (np.ones(3), np.ones((1, 2)))])
def test_theta_shapes_are_validated(th, tf):
    with pytest.raises(ValueError, match=r"expected shapes \(P, 3\) and \(P, 2\)"):
        _Fom().solve_batch(theta_lhs=th, theta_rhs=tf, preconditioner=None, method="gmres")


@pytest.mark.parametrize("x0", [np.zeros((3, 6)), np.zeros(6)])
def test_x0_shape_is_validated(x0):
    with pytest.raises(ValueError, match=r"x0: expected shape \(4, 6\)"):
        _Fom().solve_batch(**_args(x0=x0, method="gmres", restart=5))


def test_other_arguments_are_validated():
    for kw, what in [(dict(tol=-1.0), "tol"), (dict(tol=float("nan")), "tol"), (dict(maxiter=-1), "maxiter"),
                     (dict(maxiter=2.5), "maxiter")]:
        with pytest.raises(ValueError, match=what):
            fom_solve.affine_gmres(None, None, np.ones((1, 3)), np.ones((1, 1)), None, **kw)


def _host_operator(M):
    """A sparse MatrixOperator whose arrays stay on the host (what AffineCsr reads of it)."""
    op = MatrixOperator.__new__(MatrixOperator)
    op.sparse, op._host, op.shape = True, sp.csr_matrix(M), M.shape
    op.rowptr = torch.from_numpy(op._host.indptr.astype(np.int64))
    op.source = op.range = DeviceVectorSpace(M.shape[0])
    return op


def test_cg_still_rejects_non_symmetric_terms():
    terms = convection_diffusion_terms(5)
    ops = [_host_operator(M) for M in terms[:3]]
    A = fom_solve.AffineCsr(ops)                    # GMRES takes them
    assert not A.symmetric and fom_solve.AffineCsr([ops[0]]).symmetric
    fom = _Fom(n=25, Pf=2, operators=ops)
    with pytest.raises(ValueError, match="affine term 1 is not symmetric .*CG needs a symmetric positive definite"):
        fom.solve_batch(**_args(method="cg"))
    with pytest.raises(ValueError, match="affine term 1 is not symmetric"):
        fom_solve.affine_cg(A, None, np.ones((1, 3)), np.ones((1, 1)), None)
    with pytest.raises(ValueError, match="not square"):
        fom_solve.AffineCsr([_host_operator(sp.csr_matrix(np.ones((2, 3))))])


def test_chunking_rule():
    n, m = 10 ** 6, 30
    per_row = (2 * m + 5) * n * 8 + (m + 3) * ((n + 255) // 256) * 8
    assert fom_solve.gmres_rows_per_chunk(n, m, 64, 4 * 64 * per_row) == 64
    assert fom_solve.gmres_rows_per_chunk(n, m, 64, 4 * 10 * per_row) == 10
    assert fom_solve.gmres_rows_per_chunk(n, m, 64, 0) == 1
