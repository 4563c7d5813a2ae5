"""The weak greedy without a GPU: the NumPy reference (tests/greedy_ref.py) against the residual
dual norm computed directly, and the selection rule of rla4mor_b200.greedy on CPU tensors."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from greedy_ref import greedy_ref, select


def _tiny_model(nx=10):
    """Two SPD terms of a 5-point Laplacian split by halves of the grid, plus the identity."""
    n = nx * nx
    e = np.ones(nx)
    T = sp.diags([-e[:-1], 2 * e, -e[:-1]], [-1, 0, 1])
    L = (sp.kron(sp.eye(nx), T) + sp.kron(T, sp.eye(nx))).tocsr()
    left = sp.diags((np.arange(n) % nx < nx // 2).astype(float) + 0.05)
    terms = [(left @ L @ left).tocsr(), (L - left @ L @ left + sp.eye(n)).tocsr(), sp.eye(n, format="csr")]
    f = np.random.RandomState(0).standard_normal(n)
    return terms, [f, np.linspace(0, 1, n)]


@pytest.mark.parametrize("with_product", [False, True])
def test_reference_estimates_are_residual_dual_norms(with_product):
    """With Theta^T Theta = R (the identity, or R's Cholesky factor), the sketched estimate is
    ||f(mu) - A(mu) U a||_{R^-1} exactly, at every iteration and every training row."""
    terms, rhs = _tiny_model()
    n = terms[0].shape[0]
    rs = np.random.RandomState(1)
    TH = rs.uniform(0.1, 1.0, (40, 3))
    TF = rs.uniform(0.5, 1.5, (40, 2))
    R = (terms[0] + terms[1] + terms[2]).tocsc() if with_product else None
    theta = np.linalg.cholesky(R.toarray()).T if with_product else None
    out = greedy_ref(terms, rhs, TH, TF, R=R, theta=theta, batch=2, max_extensions=4)
    assert out["stop"] == "max_extensions" and len(out["max_errs"]) == out["extensions"] + 1 == 5
    assert out["basis_sizes"] == [0, 2, 4, 6, 8]
    Rd = np.eye(n) if R is None else R.toarray()
    for h in out["history"]:
        for p in range(0, 40, 3):
            f = TF[p, 0] * rhs[0] + TF[p, 1] * rhs[1]
            A = sum(TH[p, q] * terms[q] for q in range(3))
            res = f - A @ (h["a"][p] @ h["rb"])
            dual = np.sqrt(res @ np.linalg.solve(Rd, res))
            fnorm = np.sqrt(f @ np.linalg.solve(Rd, f))
            assert abs(h["est"][p] - dual) <= 1e-12 * fnorm, (p, h["est"][p], dual)
    # the selected snapshots are reproduced: their estimate vanishes once they are in the basis
    last = out["history"][-1]["est"]
    for sel in out["selected"]:
        assert np.all(last[sel] <= 1e-10 * out["max_errs"][0])
    # the sketched Galerkin condition (Theta U)^T Theta R^-1 res = 0 is U^T res = 0 when Theta^T Theta = R
    h = out["history"][-1]
    for p in (0, 7):
        f = TF[p] @ np.stack(rhs)
        res = f - sum(TH[p, q] * terms[q] for q in range(3)) @ (h["a"][p] @ h["rb"])
        assert np.linalg.norm(h["rb"] @ res) <= 1e-10 * np.linalg.norm(f)


def test_reference_follows_another_run_and_stops():
    terms, rhs = _tiny_model()
    rs = np.random.RandomState(2)
    TH, TF = rs.uniform(0.1, 1.0, (30, 3)), np.ones((30, 2))
    own = greedy_ref(terms, rhs, TH, TF, max_extensions=3)
    assert own["selected"] == [h["own"][:1] for h in own["history"][:3]]
    forced = greedy_ref(terms, rhs, TH, TF, max_extensions=3, follow=[[5], [6], [7]])
    assert forced["selected"] == [[5], [6], [7]]
    e = own["max_errs"]
    assert greedy_ref(terms, rhs, TH, TF, atol=e[2] * (1 + 1e-12))["stop"] == "atol"
    assert greedy_ref(terms, rhs, TH, TF, rtol=e[2] / e[0] * (1 + 1e-12))["extensions"] == 2
    small = greedy_ref(terms, rhs, TH, TF, batch=2, max_basis_size=3)
    assert small["stop"] == "max_basis_size" and small["basis_sizes"] == [0, 2, 3]
    # a repeated row in one batch of 2 grows the basis by one; a training set of one mu fails to extend
    rep = greedy_ref(terms, rhs, np.repeat(TH[:1], 4, axis=0), TF[:4], batch=2)
    assert rep["stop"] == "extension_failed" and rep["basis_sizes"] == [0, 1] and rep["extensions"] == 1


def test_select_largest_ties_batch_and_nan():
    from rla4mor_b200 import RlaError
    from rla4mor_b200.greedy import select_largest
    est = torch.tensor([1.0, 3.0, 2.0, 3.0, 0.5, 3.0], dtype=torch.float64)
    assert select_largest(est, 1) == ([1], 3.0)
    assert select_largest(est, 4) == ([1, 3, 5, 2], 3.0)
    assert select(est.numpy(), 4) == [1, 3, 5, 2]
    assert select_largest(est, 100) == ([1, 3, 5, 2, 0, 4], 3.0)          # batch beyond the rows: all of them
    big = torch.zeros(5000, dtype=torch.float64)                          # ties over a long sort
    big[[4999, 17, 2500]] = 1.0
    assert select_largest(big, 5)[0] == [17, 2500, 4999, 0, 1]
    est[4] = float("nan")
    est[2] = float("nan")
    with pytest.raises(RlaError, match="2 of 6 error estimates are NaN.*training row 2"):
        select_largest(est, 1)
    with pytest.raises(ValueError):
        select_largest(torch.empty(0, dtype=torch.float64), 1)


def test_sweep_chunk_rule():
    from rla4mor_b200 import fom_solve
    from rla4mor_b200.greedy import sweep_rows_per_chunk
    per_row = 8 * (16 + 1 + 4 + 1 + 8) + 4                               # r = 16, Q = 4, Pf = 1, k' = 1000
    free = 4 * 1000 * per_row
    assert fom_solve.KRYLOV_MEMORY_FRACTION == 0.25
    assert sweep_rows_per_chunk(10 ** 6, 16, 1000, 4, 1, free) == 1000
    assert sweep_rows_per_chunk(300, 16, 1000, 4, 1, free) == 300
    assert sweep_rows_per_chunk(300, 16, 1000, 4, 1, 10) == 1
