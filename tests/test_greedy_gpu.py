"""The weak greedy on the device (rla4mor_b200.greedy.rb_greedy): parity with the NumPy reference
(tests/greedy_ref.py) for Galerkin + CG on the thermal-block model and minres + GMRES on the
convection-diffusion model, reproduced snapshots, the stopping rules, partial and failed
extensions, determinism and sweep chunking, the interface, and the warm start."""
import numpy as np
import pytest
import torch

from greedy_ref import greedy_ref
from test_fom_gmres_gpu import _cd_model, _cd_thetas
from test_fom_solve_gpu import _cached_model, _thetas

pytestmark = pytest.mark.gpu

NX, P = 32, 300


@pytest.fixture(scope="module")
def rb():
    import rla4mor_b200
    rla4mor_b200.lib()
    return rla4mor_b200


def _gauss(rb, fom, k=200):
    return rb.GaussianEmbedding(source=fom.solution_space, options={"range_dim": k}, _seed=11)


def _check_parity(res, ref, slack):
    """The same rows, or a tie in the reference's estimates; the same max_errs to 1e-8 relative.
    `slack` is the absolute difference the snapshot tolerance allows (the device's snapshots are
    Krylov solutions, the reference's direct ones)."""
    assert len(res["max_errs"]) == len(ref["max_errs"]) and res["stop"] == ref["stop"]
    assert res["basis_sizes"] == ref["basis_sizes"]
    for i, sel in enumerate(res["selected"]):
        est, own = ref["history"][i]["est"], ref["history"][i]["own"]
        for d, o in zip(sel, own):
            if d != o:
                assert abs(est[d] - est[o]) <= 1e-10 * est[o] + slack, (i, d, o, est[d], est[o])
    for i, (d, o) in enumerate(zip(res["max_errs"], ref["max_errs"])):
        assert abs(d - o) <= 1e-8 * o + slack, (i, d, o)


@pytest.mark.parametrize("batch", [1, 4])
@pytest.mark.parametrize("embedding", ["identity", "gaussian"])
def test_galerkin_cg_matches_reference(rb, embedding, batch):
    fom, terms, f, prec, lu = _cached_model(rb, NX)
    th, tf = _thetas(P, 0.1, 1.0, seed=batch), np.ones((P, 1))
    emb = _gauss(rb, fom) if embedding == "gaussian" else None
    red = rb.SketchedReductor(fom, embedding_primal=emb, inverse_product=prec)
    tol = 1e-12
    res = rb.rb_greedy(fom, red, theta_lhs=th, theta_rhs=tf, batch=batch, max_basis_size=20, tol=tol, maxiter=3000)
    assert res["stop"] == "max_basis_size" and res["basis_sizes"][-1] == 20
    theta = None if emb is None else emb.get_matrix_device().cpu().numpy()
    R = sum(terms[1:], terms[0])
    ref = greedy_ref(terms, [f], th, tf, R=R, theta=theta, batch=batch, max_basis_size=20, follow=res["selected"])
    _check_parity(res, ref, 1e2 * tol * ref["max_errs"][0])


def test_minres_gmres_matches_reference_and_is_monotone(rb, monkeypatch):
    from rla4mor_b200 import fom_solve, greedy
    fom, terms, f, prec, lu = _cd_model(rb, NX)
    th, tf = _cd_thetas(P, "conv", seed=5), np.ones((P, 1))
    red = rb.SketchedReductor(fom, inverse_product=prec, projection="minres")
    tol = 1e-12
    res = rb.rb_greedy(fom, red, theta_lhs=th, theta_rhs=tf, batch=4, max_basis_size=20, method="gmres", restart=60,
                       tol=tol, maxiter=3000)
    R = terms[0] + terms[3]
    ref = greedy_ref(terms, [f], th, tf, R=R, projection="minres", batch=4, max_basis_size=20, follow=res["selected"])
    _check_parity(res, ref, 1e2 * tol * ref["max_errs"][0])
    # the sketched residual is minimised over nested spaces (identity online embedding)
    e = res["max_errs"]
    assert all(b <= a * (1 + 1e-10) for a, b in zip(e, e[1:])), e
    # the least-squares sweep does not depend on the chunking
    rom = red.reduce()
    dth, dtf = torch.from_numpy(th).cuda(), torch.from_numpy(tf).cuda()
    r, kp = red.srb.shape[0], red.embedding_online.range.dim
    est1, a1 = greedy._sweep(rom, dth, dtf, r, kp)
    monkeypatch.setattr(fom_solve, "KRYLOV_MEMORY_FRACTION", 1e-12)          # one row per chunk
    est2, a2 = greedy._sweep(rom, dth, dtf, r, kp)
    assert a1 is not None and a2 is None and torch.equal(est1, est2)


@pytest.mark.parametrize("projection", ["galerkin", "minres"])
def test_snapshots_are_reproduced_after_each_extension(rb, projection):
    """A snapshot in the span is reproduced by the Galerkin and least-squares ROMs, so right after
    its extension the estimate at every selected mu is at the level of the snapshot tolerance.  The
    estimator measures ||Theta R^-1 r||, which is within a mesh-dependent factor of the solver's
    ||r||_{R^-1}: the test allows 1e3 tol ||f(mu)||_{R^-1}, as the snapshot tests of solve_batch do."""
    if projection == "galerkin":
        fom, terms, f, prec, lu = _cached_model(rb, NX)
        th, method = _thetas(P, 0.1, 1.0, seed=7), "cg"
    else:
        fom, terms, f, prec, lu = _cd_model(rb, NX)
        th, method = _cd_thetas(P, "conv", seed=7), "gmres"
    tf = np.ones((P, 1))
    fnorm = np.sqrt(f @ lu.solve(f))
    tol = 1e-10
    red = rb.SketchedReductor(fom, embedding_primal=_gauss(rb, fom), inverse_product=prec, projection=projection)
    for _ in range(4):
        res = rb.rb_greedy(fom, red, theta_lhs=th, theta_rhs=tf, batch=2, max_extensions=1, method=method, tol=tol,
                           maxiter=3000)
        assert res["extensions"] == 1 and res["stop"] == "max_extensions"
        sel = res["selected"][0]
        est = res["rom"].estimate_error_batch(theta_lhs=th[sel], theta_rhs=tf[sel]).cpu().numpy()
        assert np.all(est <= 1e3 * tol * fnorm), (est, fnorm)
        assert res["max_errs"][1] <= res["max_errs"][0] * (1 + 1e-10) or projection == "galerkin"


def test_stopping_rules(rb, monkeypatch):
    from rla4mor_b200 import greedy, reductor_ops
    fom, terms, f, prec, lu = _cached_model(rb, NX)
    th, tf = _thetas(P, 0.1, 1.0, seed=3), np.ones((P, 1))

    def run(**kw):
        red = rb.SketchedReductor(fom, inverse_product=prec)
        res = rb.rb_greedy(fom, red, theta_lhs=th, theta_rhs=tf, batch=2, **kw)
        assert len(res["max_errs"]) == res["extensions"] + 1 == len(res["basis_sizes"]) == len(res["timings"])
        assert len(res["selected"]) == len(res["fom_iterations"]) == res["extensions"]
        assert res["basis_sizes"][-1] == red.srb.shape[0] and res["rom"] is not None and res["time"] > 0
        for t in res["timings"][:-1]:
            assert set(t) == {"reduce", "sweep", "solve", "extend", "total"}
        assert set(res["timings"][-1]) == {"reduce", "sweep", "total"}
        return res

    base = run(max_extensions=3)
    assert base["stop"] == "max_extensions" and base["extensions"] == 3 and base["basis_sizes"] == [0, 2, 4, 6]
    e = base["max_errs"]
    atol = e[2]
    res = run(atol=atol)
    assert res["stop"] == "atol" and res["extensions"] == next(i for i, x in enumerate(e) if x <= atol)
    assert res["max_errs"] == e[:res["extensions"] + 1]
    rtol = e[2] / e[0] * (1 + 1e-12)
    res = run(rtol=rtol)
    assert res["stop"] == "rtol" and res["extensions"] == next(i for i, x in enumerate(e) if x <= rtol * e[0])
    res = run(max_basis_size=5)
    assert res["stop"] == "max_basis_size" and res["basis_sizes"] == [0, 2, 4, 5]
    assert run(max_extensions=0)["stop"] == "max_extensions"
    # the default max_basis_size is the batched envelope
    assert greedy.batched_envelope(rb.SketchedReductor(fom, inverse_product=prec)) == reductor_ops.rom_solve_batch_max_r()
    assert reductor_ops.rom_solve_batch_max_r() == 169
    red = rb.SketchedReductor(fom, embedding_primal=_gauss(rb, fom, k=100), inverse_product=prec, projection="minres")
    assert greedy.batched_envelope(red) == min(reductor_ops.rom_lstsq_batch_max_r(), 100) == 100
    red = rb.SketchedReductor(fom, inverse_product=prec, projection="minres")
    assert greedy.batched_envelope(red) == reductor_ops.rom_lstsq_batch_max_r() == 137
    monkeypatch.setattr(reductor_ops, "rom_solve_batch_max_r", lambda: 3)
    res = run()
    assert res["stop"] == "max_basis_size" and res["basis_sizes"] == [0, 2, 3]


def test_partial_and_failed_extensions(rb):
    fom, terms, f, prec, lu = _cached_model(rb, NX)
    th = _thetas(10, 0.1, 1.0, seed=4)
    th[1] = th[0]                     # the empty ROM's estimates are all equal: rows 0 and 1 are selected
    red = rb.SketchedReductor(fom, inverse_product=prec)
    res = rb.rb_greedy(fom, red, theta_lhs=th, theta_rhs=np.ones((10, 1)), batch=2, max_extensions=2)
    assert res["selected"][0] == [0, 1] and res["basis_sizes"] == [0, 1, 3]
    assert res["stop"] == "max_extensions" and res["extensions"] == 2
    # one mu, A(mu) = R: its snapshot is in the span after the first extension
    red = rb.SketchedReductor(fom, inverse_product=prec)
    res = rb.rb_greedy(fom, red, theta_lhs=np.ones((3, 4)), theta_rhs=np.ones((3, 1)))
    assert res["stop"] == "extension_failed" and res["extensions"] == 1 and res["basis_sizes"] == [0, 1]
    assert len(res["max_errs"]) == 2 and len(res["selected"]) == 2 and red.srb.shape[0] == 1


def test_deterministic_and_chunked(rb, monkeypatch):
    from rla4mor_b200 import fom_solve, greedy
    fom, terms, f, prec, lu = _cached_model(rb, NX)
    th, tf = _thetas(P, 0.1, 1.0, seed=6), np.ones((P, 1))
    runs = []
    for _ in range(2):
        red = rb.SketchedReductor(fom, embedding_primal=_gauss(rb, fom), inverse_product=prec)
        res = rb.rb_greedy(fom, red, theta_lhs=th, theta_rhs=tf, batch=4, max_extensions=3)
        runs.append((res, red))
    (r1, red1), (r2, red2) = runs
    assert r1["selected"] == r2["selected"] and r1["max_errs"] == r2["max_errs"]
    assert all(torch.equal(x, y) for x, y in zip(r1["rom"].lhs, r2["rom"].lhs))
    assert all(torch.equal(x, y) for x, y in zip(red1.s_lhs, red2.s_lhs)) and torch.equal(red1.rb, red2.rb)
    rom = red1.reduce()
    dth, dtf = torch.from_numpy(th).cuda(), torch.from_numpy(tf).cuda()
    r, kp = red1.srb.shape[0], red1.embedding_online.range.dim
    est1, _ = greedy._sweep(rom, dth, dtf, r, kp)
    monkeypatch.setattr(fom_solve, "KRYLOV_MEMORY_FRACTION", 1e-12)          # one row per chunk
    est2, a2 = greedy._sweep(rom, dth, dtf, r, kp)
    assert a2 is None and torch.equal(est1, est2)
    # the whole greedy with one-row sweeps: the same run
    red = rb.SketchedReductor(fom, embedding_primal=_gauss(rb, fom), inverse_product=prec)
    r3 = rb.rb_greedy(fom, red, theta_lhs=th, theta_rhs=tf, batch=4, max_extensions=3)
    assert r3["selected"] == r1["selected"] and r3["max_errs"] == r1["max_errs"]


def test_interface(rb):
    fom, terms, f, prec, lu = _cached_model(rb, NX)
    th = _thetas(50, 0.1, 1.0, seed=8)
    mus = list(th)
    red = rb.SketchedReductor(fom, inverse_product=prec)
    r1 = rb.rb_greedy(fom, red, mus, batch=2, max_extensions=2)
    red = rb.SketchedReductor(fom, inverse_product=prec)
    r2 = rb.rb_greedy(fom, red, theta_lhs=th, theta_rhs=np.ones((50, 1)), batch=2, max_extensions=2)
    assert r1["selected"] == r2["selected"] and r1["max_errs"] == r2["max_errs"]
    assert r2["max_err_mus"] == [s[0] for s in r2["selected"]] + [r2["max_err_mus"][-1]]
    assert all(m is mus[i] for m, i in zip(r1["max_err_mus"], r2["max_err_mus"]))
    red = rb.SketchedReductor(fom, inverse_product=prec)
    bad = [dict(theta_lhs=th[:, :3], theta_rhs=np.ones((50, 1))),
           dict(theta_lhs=th, theta_rhs=np.ones((49, 1))),
           dict(theta_lhs=th, theta_rhs=np.ones((50, 2))),
           dict(theta_lhs=th),
           dict(theta_lhs=th[:0], theta_rhs=np.ones((0, 1))),
           dict(theta_lhs=th, theta_rhs=np.ones((50, 1)), batch=0),
           dict(theta_lhs=th, theta_rhs=np.ones((50, 1)), batch=1.5),
           dict(theta_lhs=th, theta_rhs=np.ones((50, 1)), method="bicg")]
    for kw in bad:
        with pytest.raises(ValueError):
            rb.rb_greedy(fom, red, **kw)
    with pytest.raises(ValueError):
        rb.rb_greedy(fom, red, mus, theta_lhs=th, theta_rhs=np.ones((50, 1)))
    with pytest.raises(ValueError, match="preconditioner"):
        rb.rb_greedy(fom, rb.SketchedReductor(fom), mus)
    assert red.srb.shape[0] == 0 and red.rb.shape[0] == 0


def test_warm_start(rb, monkeypatch):
    """Warm-started snapshots agree with cold solve_batch solutions to the solve tolerance, and take
    fewer iterations once the ROM has a basis."""
    from rla4mor_b200 import fom_solve, sketched_reductor
    fom, terms, f, prec, lu = _cached_model(rb, NX)
    th, tf = _thetas(P, 0.01, 1.0, seed=9), np.ones((P, 1))
    calls = []
    solve = sketched_reductor.solve_rows

    def spy(*args, **kw):
        out = solve(*args, **kw)
        calls.append((args[2].cpu().numpy(), kw["x0"], out[0].clone(), out[1].cpu().numpy()))
        return out

    monkeypatch.setattr(sketched_reductor, "solve_rows", spy)
    tol = 1e-10
    red = rb.SketchedReductor(fom, inverse_product=prec)
    res = rb.rb_greedy(fom, red, theta_lhs=th, theta_rhs=tf, batch=3, max_extensions=4, tol=tol)
    assert len(calls) == 4 and calls[0][1] is None and all(c[1] is not None for c in calls[1:])
    assert res["fom_iterations"] == [c[3].tolist() for c in calls]
    fnorm = np.sqrt(f @ lu.solve(f))
    warm = cold = 0
    for i, (rows, x0, X, iters) in enumerate(calls):
        assert np.array_equal(rows, th[res["selected"][i]])
        U, cit, _, _ = fom_solve.affine_cg(fom.operators, fom.rhs, rows, np.ones((3, 1)), prec, tol=tol)
        Xh = X.cpu().numpy()
        for p in range(3):
            r = f - sum(rows[p, q] * terms[q] for q in range(4)) @ Xh[p]
            assert np.sqrt(r @ lu.solve(r)) <= 2 * tol * fnorm          # the solver's own test, recomputed
        # both within the tolerance of the solution: kappa(R^-1 A) <= 100 here, and the 2-norm adds
        # a factor of R's conditioning
        assert torch.linalg.norm(X - U, dim=1).max() <= 1e-6 * torch.linalg.norm(U, dim=1).min()
        if i:
            warm, cold = warm + int(iters.sum()), cold + int(cit.sum())
    assert warm < cold, (warm, cold)
