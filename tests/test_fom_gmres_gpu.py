"""Restarted GMRES for the affine full-order model on the device (fom_solve.affine_gmres,
AffineModel.solve_batch(method='gmres'); csrc/affine_gmres.cu): accuracy on convection-diffusion
and indefinite models against spsolve and in the dual norm of the preconditioner, iteration counts
against the NumPy restatement (tests/gmres_ref.py), GMRES against CG on SPD rows, per-row
independence, chunking, initial guesses, failure paths, and snapshots feeding a minres reductor."""
import numpy as np
import pytest
import torch
from scipy.sparse.linalg import splu, spsolve

from gmres_ref import convection_diffusion_terms, gmres_ref
from test_fom_solve_gpu import _cached_model, _thetas

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rb():
    import rla4mor_b200
    rla4mor_b200.lib()
    return rla4mor_b200


_CD = {}


def _cd_model(rb, nx):
    """Convection-diffusion-reaction, terms [L, Dx, Dy, M], R = L + M (the preconditioner)."""
    if nx not in _CD:
        from rla4mor_b200.factorization import InverseLuOperator
        from rla4mor_b200.sketched_reductor import AffineModel
        terms = convection_diffusion_terms(nx)
        f = np.random.RandomState(7).standard_normal(nx * nx)
        ops_dev = [rb.MatrixOperator(A, source_id="STATE", range_id="STATE") for A in terms]
        R = (terms[0] + terms[3]).tocsc()
        prec = InverseLuOperator(rb.MatrixOperator(R, source_id="STATE", range_id="STATE"), symetric=True)
        coef = [(lambda q: (lambda mu: mu[q]))(q) for q in range(4)]
        _CD[nx] = (AffineModel(ops_dev, [f], operator_coefficients=coef), terms, f, prec, splu(R))
    return _CD[nx]


def _cd_thetas(P, kind, seed):
    """kind 'conv': theta = (1, a, b, 0), |a|, |b| <= 100; 'indef': |a|, |b| <= 2 and a reaction
    -c, c in [57, 71]: A(mu) has two negative eigenvalues, and c stays in the gap between the
    Laplacian's eigenvalues 2 pi^2 * (5/2, 4) ~ 49.3, 78.9 (convection shifts them by at most
    (a^2 + b^2) / 4 <= 2), so that tol = 1e-12 is attainable on every row."""
    rs = np.random.RandomState(seed)
    th = np.ones((P, 4))
    th[:, 1:3] = rs.uniform(-100, 100, (P, 2))
    th[:, 3] = 0.0
    if kind == "indef":
        th[:, 1:3] /= 50
        th[:, 3] = -rs.uniform(57, 71, P)
    return th


def _A(terms, th):
    return sum(th[q] * terms[q] for q in range(len(terms))).tocsr()


@pytest.mark.parametrize("kind", ["conv", "indef"])
@pytest.mark.parametrize("P", [1, 5, 64])
@pytest.mark.parametrize("nx", [32, 100])
def test_accuracy(rb, nx, P, kind):
    from rla4mor_b200 import fom_solve
    fom, terms, f, prec, lu = _cd_model(rb, nx)
    th = _cd_thetas(P, kind, seed=nx + P)
    fnorm = np.sqrt(f @ lu.solve(f))
    check = range(P) if P <= 5 else range(0, P, 9)
    for tol in (1e-10, 1e-12):
        X, iters, resid, info = fom_solve.affine_gmres(fom.operators, fom.rhs, th, np.ones((P, 1)), prec, tol=tol,
                                                       maxiter=3000)
        X, info, resid = X.cpu().numpy(), info.cpu().numpy(), resid.cpu().numpy()
        assert np.all(info == 0) and np.all(resid <= tol)
        for p in check:
            A = _A(terms, th[p])
            r = f - A @ X[p]
            assert np.sqrt(r @ lu.solve(r)) <= 2 * tol * fnorm
            if tol == 1e-12:
                u = spsolve(A.tocsc(), f)
                assert np.linalg.norm(X[p] - u) <= 1e-9 * np.linalg.norm(u)


@pytest.mark.parametrize("restart", [30, 3000])
@pytest.mark.parametrize("kind", ["conv", "indef"])
def test_iterations_match_reference(rb, kind, restart):
    from rla4mor_b200 import fom_solve
    fom, terms, f, prec, lu = _cd_model(rb, 32)
    th = _cd_thetas(4, kind, seed=3)
    X, iters, resid, info = fom_solve.affine_gmres(fom.operators, fom.rhs, th, np.ones((4, 1)), prec, tol=1e-10,
                                                   restart=restart, maxiter=3000)
    iters = iters.cpu().numpy()
    for p in range(4):
        x, it, res, inf = gmres_ref(_A(terms, th[p]), f, lu.solve, 1e-10, restart, 3000)
        assert inf == 0 and abs(int(iters[p]) - it) <= 1, (p, int(iters[p]), it)
        assert np.linalg.norm(X[p].cpu().numpy() - x) <= 1e-8 * np.linalg.norm(x)


def test_spd_rows_gmres_not_more_steps_than_cg(rb):
    from rla4mor_b200 import fom_solve
    fom, terms, f, prec, lu = _cached_model(rb, 32)
    th = _thetas(6, 0.01, 10.0, seed=4)
    tol = 1e-10
    Xc, itc, _, _ = fom_solve.affine_cg(fom.operators, fom.rhs, th, np.ones((6, 1)), prec, tol=tol, maxiter=3000)
    Xg, itg, _, infog = fom_solve.affine_gmres(fom.operators, fom.rhs, th, np.ones((6, 1)), prec, tol=tol,
                                               restart=3000, maxiter=3000)
    itc, itg = itc.cpu().numpy(), itg.cpu().numpy()
    assert np.all(infog.cpu().numpy() == 0) and np.all(itg <= itc), (itg, itc)
    for p in range(6):
        u = spsolve(_A(terms, th[p]).tocsc(), f)
        for X in (Xc, Xg):
            assert np.linalg.norm(X[p].cpu().numpy() - u) <= 1e3 * tol * np.linalg.norm(u)


def test_cg_breakdown_row_converges(rb):
    """The thermal-block row theta = (-10, 0.1, 0.1, 0.1) on which CG breaks down (A(mu) indefinite)."""
    fom, terms, f, prec, lu = _cached_model(rb, 32)
    th = _thetas(4, 0.01, 10.0, seed=9)
    th[1] = [-10.0, 0.1, 0.1, 0.1]
    U = fom.solve_batch(theta_lhs=th, theta_rhs=np.ones((4, 1)), preconditioner=prec, tol=1e-12, maxiter=3000,
                        method="gmres").to_numpy()
    for p in range(4):
        u = spsolve(_A(terms, th[p]).tocsc(), f)
        assert np.linalg.norm(U[p] - u) <= 1e-9 * np.linalg.norm(u)


def test_deterministic_independent_and_chunked(rb, monkeypatch):
    from rla4mor_b200 import fom_solve
    fom, terms, f, prec, lu = _cd_model(rb, 32)
    th = _cd_thetas(6, "conv", seed=11)
    th[2] = [1.0, 0.0, 0.0, 1.0]                        # R itself: one step
    th[4] = _cd_thetas(1, "indef", seed=12)[0]          # an indefinite row among convective ones
    tf = np.ones((6, 1))
    run = lambda t, g: fom_solve.affine_gmres(fom.operators, fom.rhs, t, g, prec, tol=1e-10, restart=20, maxiter=3000)
    X1, it1, r1, _ = run(th, tf)
    X2, it2, r2, _ = run(th, tf)
    assert torch.equal(X1, X2) and torch.equal(it1, it2) and torch.equal(r1, r2)
    it1 = it1.cpu().numpy()
    assert it1[2] <= 1 < it1.max()
    scale = 1e-12 * float(X1.abs().max())
    sub = [4, 2, 0]
    X3, it3, _, _ = run(th[sub], tf[sub])
    assert np.array_equal(it1[sub], it3.cpu().numpy())
    assert np.allclose(X1[sub].cpu().numpy(), X3.cpu().numpy(), rtol=0, atol=scale)
    monkeypatch.setattr(fom_solve, "KRYLOV_MEMORY_FRACTION", 1e-12)      # one row per chunk
    assert fom_solve.gmres_rows_per_chunk(f.size, 20, 6, torch.cuda.mem_get_info()[0]) == 1
    X4, it4, _, _ = run(th, tf)
    assert np.array_equal(it1, it4.cpu().numpy())
    assert np.allclose(X1.cpu().numpy(), X4.cpu().numpy(), rtol=0, atol=scale)


def test_initial_guess_and_zero_rhs(rb):
    from rla4mor_b200 import fom_solve
    fom, terms, f, prec, lu = _cd_model(rb, 32)
    th = _cd_thetas(3, "indef", seed=5)
    tf = np.array([[1.0], [0.0], [2.0]])
    exact = np.stack([spsolve(_A(terms, th[p]).tocsc(), tf[p, 0] * f) for p in range(3)])
    X, iters, resid, info = fom_solve.affine_gmres(fom.operators, fom.rhs, th, tf, prec, tol=1e-10, x0=exact)
    assert np.all(info.cpu().numpy() == 0) and np.all(iters.cpu().numpy() <= 1)
    assert np.linalg.norm(X.cpu().numpy() - exact) <= 1e-10 * np.linalg.norm(exact)
    for x0 in (None, np.ones((3, f.size))):
        X, iters, resid, info = fom_solve.affine_gmres(fom.operators, fom.rhs, th, tf, prec, tol=1e-10, x0=x0)
        assert int(iters[1]) == 0 and int(info[1]) == 0 and not X[1].any()
        assert np.all(info.cpu().numpy() == 0)
    x0 = torch.ones((3, f.size), dtype=torch.float64, device="cuda")
    fom_solve.affine_gmres(fom.operators, fom.rhs, th, tf, prec, x0=x0)
    assert bool((x0 == 1).all())


def test_failure_paths(rb):
    from rla4mor_b200 import fom_solve
    fom, terms, f, prec, lu = _cd_model(rb, 32)
    th = _cd_thetas(4, "conv", seed=9)
    tf = np.ones((4, 1))
    X, iters, resid, info = fom_solve.affine_gmres(fom.operators, fom.rhs, th, tf, prec, maxiter=3, check=False)
    assert np.all(info.cpu().numpy() == 1) and np.all(iters.cpu().numpy() == 3)
    assert torch.isfinite(X).all() and bool((resid > 1e-10).all())
    with pytest.raises(rb.RlaError, match="4 of 4 rows failed.*not converged"):
        fom.solve_batch(theta_lhs=th, theta_rhs=tf, preconditioner=prec, maxiter=3, method="gmres")
    # not attainable: out of iterations, never a false convergence
    X, iters, resid, info = fom_solve.affine_gmres(fom.operators, fom.rhs, th[:2], tf[:2], prec, tol=1e-17,
                                                   maxiter=300, check=False)
    assert np.all(info.cpu().numpy() == 1) and torch.isfinite(X).all() and bool((resid > 1e-17).all())

    class Negated:
        source = prec.source

        def apply(self, V):
            out = prec.apply(V)
            return type(out)(out.space, -out.data)

    X, iters, resid, info = fom_solve.affine_gmres(fom.operators, fom.rhs, th, tf, Negated(), check=False)
    assert np.all(info.cpu().numpy() == 2) and torch.isnan(X).all() and torch.isnan(resid).all()
    with pytest.raises(rb.RlaError, match="row 0, breakdown"):
        fom.solve_batch(theta_lhs=th, theta_rhs=tf, preconditioner=Negated(), method="gmres")


def test_snapshots_feed_the_minres_reductor(rb):
    """GMRES snapshots of a non-symmetric model through extend_basis: the minres ROM reproduces them
    and its estimator vanishes there (to the GMRES tolerance)."""
    fom, terms, f, prec, lu = _cd_model(rb, 32)
    tol = 1e-10
    mus = list(np.concatenate([_cd_thetas(3, "conv", seed=21), _cd_thetas(3, "indef", seed=22)]))
    red = rb.SketchedReductor(fom, inverse_product=prec, projection="minres")
    U = fom.solve_batch(mus=mus, preconditioner=red.inverse_product, tol=tol, method="gmres", restart=40)
    red.extend_basis(U)
    rom = red.reduce()
    a = rom.solve_batch(mus=mus)
    urec = (a @ red.rb).cpu().numpy()
    Un = U.to_numpy()
    assert np.linalg.norm(urec - Un, axis=1).max() <= 1e3 * tol * np.linalg.norm(Un, axis=1).min()
    est = rom.estimate_error_batch(a, mus=mus).cpu().numpy()
    fnorm = np.sqrt(f @ lu.solve(f))
    assert np.all(est <= 1e3 * tol * fnorm)
