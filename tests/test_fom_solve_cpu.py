"""CPU-only checks of the full-order solve (rla4mor_b200.fom_solve, AffineModel.solve_batch): the
union-pattern merge of the affine terms, the symmetry check, and argument validation that raises
before anything reaches the device."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from rla4mor_b200 import fom_solve
from rla4mor_b200.sketched_reductor import AffineModel
from rla4mor_b200.vectorarray import DeviceVectorSpace, IdentityOperator


def _terms(n=60):
    rs = np.random.RandomState(0)
    ex = np.ones(n)
    lap = sp.diags([-ex[:-1], 2 * ex, -ex[:-1]], [-1, 0, 1]).tocsr()
    S = sp.random(n, n, density=0.05, random_state=1, format="csr")
    S = (S + S.T).tocsr()
    rows = np.repeat(np.arange(n), np.diff(S.indptr))
    S.data[(rows + S.indices) % 5 == 0] = 0.0                    # explicit zeros, kept in the pattern
    D = sp.diags(rs.uniform(1, 2, n)).tocsr()
    far = sp.csr_matrix(([3.0, 3.0], ([0, n - 1], [n - 1, 0])), shape=(n, n))
    return [lap, S, D, far]


def test_union_pattern_reproduces_every_term_exactly():
    terms = _terms()
    indptr, indices, values = fom_solve.union_pattern(terms)
    n = terms[0].shape[0]
    assert indptr.dtype == np.int64 and indices.dtype == np.int32 and values.shape == (4, indices.size)
    for i in range(n):                                            # sorted columns, no duplicates
        cols = indices[indptr[i]:indptr[i + 1]]
        assert np.all(np.diff(cols) > 0)
    for q, A in enumerate(terms):
        M = sp.csr_matrix((values[q], indices, indptr), shape=(n, n))
        assert np.array_equal(M.toarray(), A.toarray())           # exact copies, 0 elsewhere
        # every stored entry of the term, explicit zeros included, is a position of the union
        Ac = A.tocoo()
        got = M.toarray()[Ac.row, Ac.col]
        assert np.array_equal(got, Ac.data)
    stored = set()
    for A in terms:
        Ac = A.tocoo()
        stored |= set(zip(Ac.row.tolist(), Ac.col.tolist()))
    assert indices.size == len(stored)


def test_union_pattern_sums_duplicate_entries():
    A = sp.csr_matrix((np.array([1.0, 2.0, 5.0]), np.array([0, 0, 1]), np.array([0, 2, 3])), shape=(2, 2))
    indptr, indices, values = fom_solve.union_pattern([A])
    assert indices.tolist() == [0, 1] and values[0].tolist() == [3.0, 5.0]


def test_non_symmetric_term_is_rejected():
    terms = _terms()
    fom_solve.check_symmetric(terms)
    bad = terms[1].tolil()
    bad[3, 7] = bad[7, 3] + 1.0
    with pytest.raises(ValueError, match="affine term 2 is not symmetric"):
        fom_solve.check_symmetric([terms[0], terms[2], bad.tocsr()])
    # rounding of the two triangles (as D L D assembles them) is accepted
    D = sp.diags(np.random.RandomState(3).uniform(0.01, 1, 60))
    fom_solve.check_symmetric([(D @ terms[0] @ D).tocsr()])


def test_terms_that_are_not_sparse_matrix_operators_are_rejected():
    with pytest.raises(ValueError, match="not a sparse MatrixOperator"):
        fom_solve.AffineCsr([IdentityOperator(DeviceVectorSpace(5))])


class _Fom:
    """What AffineModel.solve_batch reads before it reaches the device (host tensors)."""

    def __init__(self, n=6, Q=3, Pf=2):
        self.operators = [None] * Q
        self.rhs = [torch.zeros((1, n), dtype=torch.float64) for _ in range(Pf)]
        self.operator_coefficients = [lambda mu, q=q: mu[q] for q in range(Q)]
        self.rhs_coefficients = [1.0] * Pf
        self.solution_space = DeviceVectorSpace(n)
        self._affine = None

    thetas = AffineModel.thetas
    thetas_batch = AffineModel.thetas_batch
    solve = AffineModel.solve
    solve_batch = AffineModel.solve_batch


@pytest.mark.parametrize("th,tf", [(np.ones((4, 2)), np.ones((4, 2))),       # Q wrong
                                   (np.ones((4, 3)), np.ones((3, 2))),       # P differs
                                   (np.ones(3), np.ones((1, 2))),            # not 2-D
                                   (np.ones((4, 3)), np.ones((4, 1)))])      # Pf wrong
def test_theta_shapes_are_validated(th, tf):
    with pytest.raises(ValueError, match=r"expected shapes \(P, 3\) and \(P, 2\)"):
        _Fom().solve_batch(theta_lhs=th, theta_rhs=tf, preconditioner=None)


def test_theta_arguments_are_validated():
    fom = _Fom()
    with pytest.raises(ValueError, match="not both"):
        fom.solve_batch(mus=[[1, 2, 3]], theta_lhs=np.ones((1, 3)), preconditioner=None)
    with pytest.raises(ValueError, match="give mus= or both"):
        fom.solve_batch(theta_lhs=np.ones((1, 3)), preconditioner=None)
    with pytest.raises(ValueError, match=r"expected shapes \(P, 3\)"):
        fom.solve(theta_lhs=np.ones(4), theta_rhs=np.ones(2), preconditioner=None)
    with pytest.raises(TypeError):
        fom.solve_batch(theta_lhs=np.ones((1, 3)), theta_rhs=np.ones((1, 2)))     # preconditioner is required


@pytest.mark.parametrize("x0", [np.zeros((3, 6)), np.zeros((4, 5)), np.zeros(6)])
def test_x0_shape_is_validated(x0):
    with pytest.raises(ValueError, match=r"x0: expected shape \(4, 6\)"):
        _Fom().solve_batch(theta_lhs=np.ones((4, 3)), theta_rhs=np.ones((4, 2)), preconditioner=None, x0=x0)
    with pytest.raises(ValueError, match=r"x0: expected shape \(4, 6\)"):
        fom_solve.check_block(torch.from_numpy(x0), 4, 6, "x0", "cpu")


def test_x0_copy_is_new():
    x0 = torch.ones((2, 3), dtype=torch.float32)
    got = fom_solve.check_block(x0, 2, 3, "x0", "cpu")
    assert got.dtype == torch.float64 and got.data_ptr() != x0.data_ptr() and bool((got == 1).all())
