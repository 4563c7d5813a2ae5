"""The ROM over a parameter set (csrc/rom_batch.cu; SketchedRom.solve_batch / estimate_error_batch /
output_batch) against the per-mu methods, the oracle and the executed-reference fixture."""
import json
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from golden_util import GOLDEN, rel_fro
from oracle import reductor_oracle as ro

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rb():
    import rla4mor_b200
    rla4mor_b200.lib()
    return rla4mor_b200


def _terms(nx, Q):
    """Q block-wise 5-point terms on an nx x nx grid, shifted so that every A(mu) with positive
    coefficients is well conditioned (condition number below ~20)."""
    n = nx * nx
    ex = np.ones(nx)
    T = sp.diags([-ex[:-1], 2 * ex, -ex[:-1]], [-1, 0, 1])
    L = (sp.kron(sp.eye(nx), T) + sp.kron(T, sp.eye(nx))).tocsr()
    idx = np.arange(n)
    blk = (idx // nx >= nx // 2) * 2 + (idx % nx >= nx // 2)
    return [(sp.diags((blk == q % 4) + 0.1) @ L @ sp.diags((blk == q % 4) + 0.1) + 0.5 * sp.eye(n)).tocsr()
            for q in range(Q)], n


_ROMS = {}


def _reduced(rb, r, Q, Pf, k=300):
    """A Galerkin ROM of dimension r built by SketchedReductor (SRHT sketch, online Gaussian sketch)."""
    key = (r, Q, Pf, k)
    if key not in _ROMS:
        terms, n = _terms(24, Q)
        rs = np.random.RandomState(r * 100 + Q * 10 + Pf)
        space = rb.DeviceVectorSpace(n, id="STATE")
        ops_dev = [rb.MatrixOperator(A, source_id="STATE", range_id="STATE") for A in terms]
        emb = rb.SrhtEmbedding(source=space, options={"range_dim": k}, _seed=1)
        onl = rb.GaussianEmbedding(source=emb.range, options={"range_dim": k // 2}, _seed=2)
        fom = rb.sketched_reductor.AffineModel(ops_dev, [rs.standard_normal(n) for _ in range(Pf)],
                                               output=rs.standard_normal((2, n)), solution_space=space)
        red = rb.SketchedReductor(fom, embedding_primal=emb, embedding_online=onl)
        red.extend_basis(rs.standard_normal((r, n)))
        _ROMS[key] = red.reduce()
    return _ROMS[key]


def _thetas(P, Q, Pf, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    th = 0.1 + 0.9 * torch.rand(P, Q, dtype=torch.float64, device="cuda", generator=g)
    tf = torch.randn(P, Pf, dtype=torch.float64, device="cuda", generator=g)
    return th, tf


def _rows(P):
    return sorted(set(range(0, P, max(1, P // 40))) | {P - 1})


def _est_bound(rom, th, tf, a):
    """1e-14 (sum_q |th_q| ||S_q|| ||a|| + sum_j |tf_j| ||g_j||) per row: the rounding scale of the estimate."""
    sn = torch.stack([torch.linalg.matrix_norm(S, ord=2) for S in rom.est_lhs_rows])
    gn = torch.stack([torch.linalg.norm(g) for g in rom.est_rhs]) if rom.est_rhs else torch.zeros(0, device=th.device,
                                                                                                 dtype=torch.float64)
    return 1e-14 * ((th.abs() @ sn) * torch.linalg.norm(a, dim=1) + tf.abs() @ gn)


@pytest.mark.parametrize("Pf", [0, 1, 3])
@pytest.mark.parametrize("Q", [1, 4])
@pytest.mark.parametrize("r", [1, 7, 37, 64, 128])
def test_solve_and_estimate_batch_match_per_mu(rb, r, Q, Pf):
    rom = _reduced(rb, r, Q, Pf)
    for P in (1, 5, 1000, 1031):                           # 1031: no multiple of any tile
        th, tf = _thetas(P, Q, Pf, seed=P + r)
        a = rom.solve_batch(th, tf)
        est = rom.estimate_error_batch(a, th, tf)
        assert a.shape == (P, r) and est.shape == (P,)
        bound = _est_bound(rom, th, tf, a)
        for p in _rows(P):
            if Pf:
                ref = rom.solve(th[p], tf[p])
                assert float(torch.linalg.norm(a[p] - ref) / torch.linalg.norm(ref)) <= 1e-12, (P, p)
            else:
                assert float(torch.linalg.norm(a[p])) == 0.0               # A(mu) a = 0
            e1 = rom.estimate_error(a[p], th[p].tolist(), tf[p].tolist())
            e2 = ro.residual_norm([S.cpu().numpy() for S in rom.est_lhs], th[p].tolist(),
                                  [g.cpu().numpy() for g in rom.est_rhs], tf[p].tolist(), a[p].cpu().numpy())
            for ref in (e1, e2):
                d = abs(float(est[p]) - ref)
                assert d <= 1e-12 * ref or d <= float(bound[p]), (P, p, d, ref)
        assert torch.equal(rom.output_batch(a, th, tf), a @ rom.output_functional)


def test_mus_and_default_a(rb):
    rom = _reduced(rb, 7, 4, 1)
    mus = [[0.2 + 0.1 * p, 0.5, 1.0, 0.3 + 0.01 * p] for p in range(9)]
    rom.fom.operator_coefficients = [lambda mu, i=i: mu[i] for i in range(4)]
    rom.fom.rhs_coefficients = [lambda mu: 2.0 - mu[0]]
    th = torch.tensor(mus, dtype=torch.float64, device="cuda")
    tf = (2.0 - th[:, :1]).contiguous()
    assert torch.equal(rom.solve_batch(mus=mus), rom.solve_batch(th, tf))
    assert torch.equal(rom.estimate_error_batch(mus=mus), rom.estimate_error_batch(None, th, tf))
    assert torch.equal(rom.output_batch(mus=mus), rom.output_batch(None, th, tf))


def _dense_rom(rb, lhs, rhs, kp=40, seed=0):
    """A SketchedRom straight from reduced matrices (random estimator data)."""
    from rla4mor_b200.sketched_reductor import SketchedRom
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = lhs[0].shape[0]
    est = ([torch.randn(r, kp, dtype=torch.float64, device="cuda", generator=g) for _ in lhs],
           [torch.randn(kp, dtype=torch.float64, device="cuda", generator=g) for _ in rhs])
    dev = lambda x: torch.as_tensor(x, dtype=torch.float64, device="cuda")
    return SketchedRom(None, [dev(M) for M in lhs], [dev(v) for v in rhs],
                       torch.zeros((r, 1), dtype=torch.float64, device="cuda"), est, least_squares=False)


def test_row_swaps(rb):
    rs = np.random.RandomState(3)
    r = 7
    A0 = rs.standard_normal((r, r))
    A0[0, 0] = 0.0                                          # zero leading entry
    A1 = rs.standard_normal((r, r))
    A1[:, 0] = 0.0
    A1[r - 1, 0] = 50.0                                     # the first pivot is in the last row
    A2 = np.triu(rs.standard_normal((r, r)), 1)[::-1].copy()   # anti-triangular: a swap at every step
    A2[np.arange(r), r - 1 - np.arange(r)] = 1.0 + np.arange(r)
    rom = _dense_rom(rb, [A0, A1, A2], [rs.standard_normal(r)])
    th = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [1.0, 1.0, 0.0], [0.0, 0.0, 1.0], [0.0, 1.0, 0.5]])
    tf = np.ones((5, 1))
    a = rom.solve_batch(th, tf).cpu().numpy()
    for p in range(5):
        A = sum(t * M for t, M in zip(th[p], (A0, A1, A2)))
        ref = np.linalg.solve(A, rom.rhs[0].cpu().numpy())
        assert np.linalg.norm(a[p] - ref) <= 1e-12 * np.linalg.norm(ref), p


def test_singular_mu_among_many(rb):
    from rla4mor_b200 import reductor_ops as ops
    rs = np.random.RandomState(5)
    r = 9
    M = rs.standard_normal((r, r)) + 5 * np.eye(r)
    S = rs.standard_normal((r, r))
    S[:, 3] = 0.0                                           # A = S is exactly singular: U(4, 4) = 0
    rom = _dense_rom(rb, [M, S], [rs.standard_normal(r)])
    P, bad = 300, 123
    th = np.column_stack([np.ones(P), 0.01 * rs.standard_normal(P)])
    th[bad] = (0.0, 1.0)
    tf = np.ones((P, 1))
    a, info = ops.rom_solve_batch(torch.stack(rom.lhs), torch.stack(rom.rhs), torch.tensor(th), torch.tensor(tf),
                                  check=False)
    info = info.cpu().numpy()
    assert info[bad] == 4 and np.count_nonzero(info) == 1
    with pytest.raises(rb.RlaError, match=r"1 of 300 .*row 123"):
        rom.solve_batch(th, tf)
    a2 = rom.solve_batch(th, tf, check=False)
    assert torch.isnan(a2[bad]).all() and not torch.isnan(a2[:bad]).any() and not torch.isnan(a2[bad + 1:]).any()
    good = np.delete(np.arange(P), bad)
    th_good = torch.tensor(th[good], device="cuda")
    assert torch.equal(a2[good], rom.solve_batch(th_good, torch.ones((P - 1, 1), dtype=torch.float64)))
    est = rom.estimate_error_batch(a2, th, tf)
    assert torch.isnan(est[bad]) and not torch.isnan(est[good]).any()


@pytest.mark.parametrize("kp", [1, 33, 1001])
def test_residual_kernel_ragged_and_strided(rb, kp):
    from rla4mor_b200 import reductor_ops as ops
    g = torch.Generator(device="cuda").manual_seed(kp)
    Q, r, Pf, P = 3, 13, 2, 517
    W = torch.randn(Q * r + Pf, kp, dtype=torch.float64, device="cuda", generator=g)
    big = torch.randn(P, 2 * r + 3, dtype=torch.float64, device="cuda", generator=g)
    a = big[:, 3:3 + r]                                     # strided rows, odd offset
    th, tf = _thetas(P, Q, Pf, seed=kp)
    est = ops.residual_norm_batch(W, Q, r, th, tf, a)
    X = torch.cat([(th[:, :, None] * a[:, None, :]).reshape(P, Q * r), -tf], dim=1)
    ref = torch.linalg.norm(X @ W, dim=1)
    assert float(torch.max(torch.abs(est - ref) / ref)) <= 1e-12
    assert torch.equal(est, ops.residual_norm_batch(W, Q, r, th, tf, a))           # run to run
    Wodd = torch.zeros(W.shape[0], kp + 1, dtype=torch.float64, device="cuda")[:, 1:]   # 8-byte aligned rows
    Wodd.copy_(W)
    assert float(torch.max(torch.abs(ops.residual_norm_batch(Wodd, Q, r, th, tf, a) - ref) / ref)) <= 1e-12


def test_residual_memory_at_scale(rb):
    from rla4mor_b200 import reductor_ops as ops
    P, kp, Q, r, Pf = 100000, 2000, 4, 64, 1
    g = torch.Generator(device="cuda").manual_seed(0)
    W = torch.randn(Q * r + Pf, kp, dtype=torch.float64, device="cuda", generator=g)
    a = torch.randn(P, r, dtype=torch.float64, device="cuda", generator=g)
    th, tf = _thetas(P, Q, Pf, seed=1)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    est = ops.residual_norm_batch(W, Q, r, th, tf, a)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base < P * kp * 8 // 8
    assert torch.equal(est, ops.residual_norm_batch(W, Q, r, th, tf, a))
    rows = torch.arange(0, P, 997, device="cuda")
    X = torch.cat([(th[rows, :, None] * a[rows, None, :]).reshape(-1, Q * r), -tf[rows]], dim=1)
    ref = torch.linalg.norm(X @ W, dim=1)
    assert float(torch.max(torch.abs(est[rows] - ref) / ref)) <= 1e-12


# ----------------------------------------------------------- executed-reference fixture
def _load_reductor():
    z = np.load(os.path.join(GOLDEN, "reductor_reference.npz"))
    meta = json.loads(str(z["__meta__"]))
    n = meta["n"]
    A = [sp.csr_matrix((z[f"A{q}__data"], z[f"A{q}__indices"], z[f"A{q}__indptr"]), shape=(n, n)) for q in range(3)]
    R = sp.csr_matrix((z["R__data"], z["R__indices"], z["R__indptr"]), shape=(n, n))
    return z, meta, A, R


@pytest.mark.parametrize("cfg", ["gauss_galerkin", "gauss_minres", "srht_galerkin", "srht_minres"])
def test_batch_reproduces_executed_reference(rb, cfg):
    from rla4mor_b200.factorization import InverseLuOperator
    from rla4mor_b200.sketched_reductor import AffineModel, EmptyRom
    z, meta, A, R = _load_reductor()
    kind, projection = cfg.split("_")
    ops_dev = [rb.MatrixOperator(x, source_id="S", range_id="S") for x in A]
    space = ops_dev[0].source
    fom = AffineModel(ops_dev, list(z["f"]), operator_coefficients=[1.0, lambda mu: mu[0], lambda mu: mu[1]],
                      rhs_coefficients=[1.0, lambda mu: mu[0]], output=z["out"], solution_space=space)
    Rop = rb.MatrixOperator(R.tocsc(), source_id="S", range_id="S")
    cls = rb.GaussianEmbedding if kind == "gauss" else rb.SrhtEmbedding
    emb = cls(source=space, options={"range_dim": meta["k"]}, _seed=meta["seed_primal"], range_id="SK")
    onl = rb.GaussianEmbedding(source=emb.range, options={"range_dim": meta["k_online"]}, _seed=meta["seed_online"])
    red = rb.SketchedReductor(fom, embedding_primal=emb, embedding_online=onl, product=Rop,
                              inverse_product=InverseLuOperator(Rop), projection=projection, orthonormalize=False)
    mus = meta["test"]
    if projection == "galerkin":
        rom0 = red.reduce()
        assert isinstance(rom0, EmptyRom)
        est0 = rom0.estimate_error_batch(mus=mus)
        assert rom0.solve_batch(mus=mus).shape == (len(mus), 0)
        for j, mu in enumerate(mus):
            ref = float(z[f"{cfg}__empty_est{j}"].ravel()[0])
            assert abs(float(est0[j]) - ref) < 1e-10 * ref
            assert abs(float(est0[j]) - rom0.estimate_error(mu=mu)) <= 1e-14 * ref
        assert torch.equal(rom0.output_batch(mus=mus), torch.stack([rom0.output(mu=mu) for mu in mus]))
    off = 0
    for nb in meta["blocks"]:
        red.extend_basis(z["U"][off:off + nb])
        red.orthonormalize_basis(offset=red.srb.shape[0] - nb)
        off += nb
    rom = red.reduce(seed=meta["reduce_seed"] if projection == "galerkin" else tuple(meta["minres_seeds"]))
    a = rom.solve_batch(mus=mus)
    est = rom.estimate_error_batch(a, mus=mus)
    out = rom.output_batch(a, mus=mus)
    for j, mu in enumerate(mus):
        assert rel_fro(a[j].cpu().numpy(), z[f"{cfg}__sol{j}"][0]) < 1e-9
        ref = float(z[f"{cfg}__est{j}"].ravel()[0])
        assert abs(float(est[j]) - ref) < 1e-8 * max(1.0, float(est[j]))
        assert rel_fro(out[j].cpu().numpy(), z[f"{cfg}__output{j}"].ravel()) < 1e-9
        if projection == "minres":                          # the per-mu loop: the same solve call
            assert torch.equal(a[j], rom.solve(mu=mu))


def test_pymor_adapter_multi_row_estimate(rb):
    stub = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_pymor_stub")
    if stub not in sys.path:
        sys.path.insert(0, stub)
    from pymor.vectorarrays.numpy import NumpyVectorSpace
    from rla4mor_b200.pymor_adapter import ResidualErrorEstimator
    rom = _reduced(rb, 37, 4, 3)
    rom.fom.operator_coefficients = [1.0, lambda mu: mu[0], lambda mu: mu[1], 0.5]
    rom.fom.rhs_coefficients = [1.0, lambda mu: -mu[0], 2.0]
    mu = [0.7, 1.3]
    U = NumpyVectorSpace(37).from_numpy(np.random.RandomState(0).standard_normal((11, 37)))
    got = ResidualErrorEstimator(rom).estimate_error(U, mu)
    assert got.shape == (11,)
    for i, row in enumerate(U.to_numpy()):
        ref = rom.estimate_error(a=torch.as_tensor(row, device="cuda"), mu=mu)
        assert abs(got[i] - ref) <= 1e-12 * ref
