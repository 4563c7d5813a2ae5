"""Full-order solves of the affine model on the device (fom_solve.affine_cg, AffineModel.solve /
solve_batch; csrc/affine_cg.cu): the affine SpMM and its fused dot products against SciPy, the
block preconditioned CG against spsolve and in the dual norm of the preconditioner, its
per-row masking, reproducibility, failure paths, and snapshots feeding SketchedReductor."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch
from scipy.sparse.linalg import splu, spsolve

from test_reductor_gpu import _fem_terms

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rb():
    import rla4mor_b200
    rla4mor_b200.lib()
    return rla4mor_b200


def _sym_random(n, density, seed):
    S = sp.random(n, n, density=density, random_state=seed, format="csr")
    return (S + S.T).tocsr()


def _model(rb, nx, Q=4):
    from rla4mor_b200.factorization import InverseLuOperator
    from rla4mor_b200.sketched_reductor import AffineModel
    terms, n = _fem_terms(nx, Q)
    f = np.random.RandomState(7).standard_normal(n)
    ops_dev = [rb.MatrixOperator(A, source_id="STATE", range_id="STATE") for A in terms]
    R = sum(terms[1:], terms[0]).tocsc()
    prec = InverseLuOperator(rb.MatrixOperator(R, source_id="STATE", range_id="STATE"), symetric=True)
    coef = [(lambda q: (lambda mu: mu[q]))(q) for q in range(Q)]
    fom = AffineModel(ops_dev, [f], operator_coefficients=coef)
    return fom, terms, f, prec, splu(R)


_CACHE = {}


def _cached_model(rb, nx):
    if nx not in _CACHE:
        _CACHE[nx] = _model(rb, nx)
    return _CACHE[nx]


def _thetas(P, lo, hi, Q=4, seed=0):
    return np.random.RandomState(seed).uniform(lo, hi, (P, Q))


@pytest.mark.parametrize("Q", [1, 4])
@pytest.mark.parametrize("P", [1, 7, 64, 65])
def test_affine_spmm_matches_scipy(rb, P, Q):
    from rla4mor_b200 import fom_solve
    nx = 40
    terms, n = _fem_terms(nx, 4)
    # different patterns: the FEM term, a diagonal, a random symmetric pattern with explicit zeros
    D = sp.diags(np.random.RandomState(1).uniform(1, 2, n)).tocsr()
    S = _sym_random(n, 5e-4, 2)
    rows = np.repeat(np.arange(n), np.diff(S.indptr))
    S.data[(rows + S.indices) % 7 == 0] = 0.0                  # explicit zeros, symmetric
    mats = [terms[0], D, S, terms[3]][:Q]
    A = fom_solve.AffineCsr([rb.MatrixOperator(M) for M in mats])
    rs = np.random.RandomState(P)
    th = rs.uniform(-1, 2, (P, Q))
    X = rs.standard_normal((P, n))
    Y, d = fom_solve.affine_spmm(A, th, torch.from_numpy(X).cuda(), dots=True)
    Y, d = Y.cpu().numpy(), d.cpu().numpy()
    ref = np.stack([sum(th[p, q] * (mats[q] @ X[p]) for q in range(Q)) for p in range(P)])
    assert np.linalg.norm(Y - ref) <= 1e-14 * np.linalg.norm(ref)
    dref = np.einsum("pi,pi->p", X, ref)
    assert np.all(np.abs(d - dref) <= 1e-13 * np.einsum("pi,pi->p", np.abs(X), np.abs(ref)))
    # Y alone, without the dot epilogue: the same bits
    assert np.array_equal(fom_solve.affine_spmm(A, th, torch.from_numpy(X).cuda()).cpu().numpy(), Y)


@pytest.mark.parametrize("lo,hi", [(0.1, 1.0), (0.01, 10.0)])
@pytest.mark.parametrize("P", [1, 5, 64])
@pytest.mark.parametrize("nx", [32, 100])
def test_solve_batch_accuracy(rb, nx, P, lo, hi):
    from rla4mor_b200 import fom_solve
    fom, terms, f, prec, lu = _cached_model(rb, nx)
    th = _thetas(P, lo, hi, seed=nx + P)
    tf = np.ones((P, 1))
    for tol in (1e-10, 1e-12):
        X, iters, resid, info = fom_solve.affine_cg(fom.operators, fom.rhs, th, tf, prec, tol=tol, maxiter=3000)
        X, info, resid = X.cpu().numpy(), info.cpu().numpy(), resid.cpu().numpy()
        assert np.all(info == 0) and np.all(resid <= tol)
        fnorm = np.sqrt(f @ lu.solve(f))
        for p in range(P):
            A = sum(th[p, q] * terms[q] for q in range(4)).tocsc()
            r = f - A @ X[p]
            # the true residual in the dual norm of R, recomputed on the host
            assert np.sqrt(r @ lu.solve(r)) <= 2 * tol * fnorm
            if tol == 1e-12:
                u = spsolve(A, f)
                assert np.linalg.norm(X[p] - u) <= 1e-9 * np.linalg.norm(u)


def test_reproducible_and_single_mu_agrees(rb):
    fom, terms, f, prec, lu = _cached_model(rb, 32)
    th = _thetas(5, 0.1, 1.0, seed=3)
    U1 = fom.solve_batch(theta_lhs=th, theta_rhs=np.ones((5, 1)), preconditioner=prec).to_numpy()
    U2 = fom.solve_batch(theta_lhs=th, theta_rhs=np.ones((5, 1)), preconditioner=prec).to_numpy()
    assert np.array_equal(U1, U2)
    for p in (0, 3):
        u = fom.solve(mu=th[p], preconditioner=prec)
        assert len(u) == 1 and u.space == fom.solution_space
        assert np.linalg.norm(u.to_numpy()[0] - U1[p]) <= 1e-12 * np.linalg.norm(U1[p])
    # mus= goes through the model's coefficients: the same rows
    U3 = fom.solve_batch(mus=list(th), preconditioner=prec).to_numpy()
    assert np.array_equal(U3, U1)


def test_masking_rows_independent_of_block(rb):
    """A row's iterates depend on its own data only: the same row in two blocks whose other rows
    converge at different iterations."""
    from rla4mor_b200 import fom_solve
    fom, terms, f, prec, lu = _cached_model(rb, 32)
    th = _thetas(6, 0.01, 10.0, seed=11)
    th[2] = 1.0                                         # R itself: converges in one iteration
    X1, it1, _, _ = fom_solve.affine_cg(fom.operators, fom.rhs, th, np.ones((6, 1)), prec, tol=1e-10, maxiter=3000)
    sub = [4, 2, 0]
    X2, it2, _, _ = fom_solve.affine_cg(fom.operators, fom.rhs, th[sub], np.ones((3, 1)), prec, tol=1e-10, maxiter=3000)
    it1, it2 = it1.cpu().numpy(), it2.cpu().numpy()
    assert it1[2] <= 1 < it1.max()
    assert np.array_equal(it1[sub], it2)
    assert np.allclose(X1[sub].cpu().numpy(), X2.cpu().numpy(), rtol=0, atol=1e-12 * float(X1.abs().max()))


def test_initial_guess_and_zero_rhs(rb):
    from rla4mor_b200 import fom_solve
    fom, terms, f, prec, lu = _cached_model(rb, 32)
    th = _thetas(3, 0.1, 1.0, seed=5)
    tf = np.array([[1.0], [0.0], [2.0]])
    exact = np.stack([spsolve(sum(th[p, q] * terms[q] for q in range(4)).tocsc(), tf[p, 0] * f) for p in range(3)])
    X, iters, resid, info = fom_solve.affine_cg(fom.operators, fom.rhs, th, tf, prec, tol=1e-10, x0=exact)
    iters = iters.cpu().numpy()
    assert np.all(info.cpu().numpy() == 0) and np.all(iters <= 1)
    assert np.linalg.norm(X.cpu().numpy() - exact) <= 1e-10 * np.linalg.norm(exact)
    # zero right-hand side: 0 in 0 iterations, with or without an initial guess
    for x0 in (None, np.ones((3, f.size))):
        X, iters, resid, info = fom_solve.affine_cg(fom.operators, fom.rhs, th, tf, prec, tol=1e-10, x0=x0)
        assert int(iters[1]) == 0 and int(info[1]) == 0 and not X[1].any()
    # the caller's x0 is not modified
    x0 = torch.ones((3, f.size), dtype=torch.float64, device="cuda")
    fom_solve.affine_cg(fom.operators, fom.rhs, th, tf, prec, x0=x0)
    assert bool((x0 == 1).all())


def test_failure_paths(rb):
    from rla4mor_b200 import fom_solve
    fom, terms, f, prec, lu = _cached_model(rb, 32)
    th = _thetas(4, 0.01, 10.0, seed=9)
    tf = np.ones((4, 1))
    X, iters, resid, info = fom_solve.affine_cg(fom.operators, fom.rhs, th, tf, prec, maxiter=2, check=False)
    assert np.all(info.cpu().numpy() == 1) and np.all(iters.cpu().numpy() == 2)
    assert torch.isfinite(X).all() and bool((resid > 1e-10).all())
    with pytest.raises(rb.RlaError, match="4 of 4 rows failed.*not converged"):
        fom.solve_batch(theta_lhs=th, theta_rhs=tf, preconditioner=prec, maxiter=2)
    # an indefinite A(mu) in row 1: negative curvature, a NaN row, the other rows unaffected
    th[1] = [-10.0, 0.1, 0.1, 0.1]
    X, iters, resid, info = fom_solve.affine_cg(fom.operators, fom.rhs, th, tf, prec, maxiter=3000, check=False)
    info = info.cpu().numpy()
    assert info[1] == 2 and torch.isnan(X[1]).all() and np.all(info[[0, 2, 3]] == 0)
    with pytest.raises(rb.RlaError, match="row 1, breakdown"):
        fom.solve_batch(theta_lhs=th, theta_rhs=tf, preconditioner=prec, maxiter=3000)


def test_snapshots_feed_the_reductor(rb):
    """u(mu_1..mu_m) from solve_batch through extend_basis: the Galerkin ROM reproduces them and its
    estimator vanishes there (to the CG tolerance)."""
    fom, terms, f, prec, lu = _cached_model(rb, 32)
    tol = 1e-10
    mus = list(_thetas(6, 0.1, 1.0, seed=21))
    red = rb.SketchedReductor(fom, inverse_product=prec)
    U = fom.solve_batch(mus=mus, preconditioner=red.inverse_product, tol=tol)
    red.extend_basis(U)
    rom = red.reduce()
    a = rom.solve_batch(mus=mus)
    urec = (a @ red.rb).cpu().numpy()
    Un = U.to_numpy()
    assert np.linalg.norm(urec - Un, axis=1).max() <= 1e3 * tol * np.linalg.norm(Un, axis=1).min()
    est = rom.estimate_error_batch(a, mus=mus).cpu().numpy()
    fnorm = np.sqrt(f @ lu.solve(f))
    assert np.all(est <= 1e3 * tol * fnorm)
