"""The batched least-squares (minres) ROM solve (csrc/rom_batch.cu: rom_lstsq_batch_kernel;
reductor_ops.rom_lstsq_batch; SketchedRom.solve / solve_batch of a least-squares ROM) against a host
SVD solver, with and without the offline compression of the stack, for bit-equality with the
single-mu solve, rank deficiency, and the executed-reference fixture."""
import ctypes
import json
import os

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from golden_util import GOLDEN, rel_fro

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rb():
    import rla4mor_b200
    rla4mor_b200.lib()
    return rla4mor_b200


def _dev(x):
    return torch.as_tensor(np.asarray(x), dtype=torch.float64, device="cuda")


def _ls_rom(lhs, rhs, kp_est=30, seed=0):
    """A least-squares SketchedRom from host matrices M_q (k', r) and vectors g_j (k',), with random
    estimator data (the reduced solve does not read it)."""
    from rla4mor_b200.sketched_reductor import SketchedRom
    rs = np.random.RandomState(seed + 1)
    r = lhs[0].shape[1]
    est = ([_dev(rs.standard_normal((r, kp_est))) for _ in lhs], [_dev(rs.standard_normal(kp_est)) for _ in rhs])
    return SketchedRom(None, [_dev(M) for M in lhs], [_dev(g) for g in rhs], _dev(np.ones((r, 2))), est,
                       least_squares=True)


def _well_conditioned(r, Q, Pf, kp, seed):
    """M_q = U + 0.1 G_q / sqrt(k'): with coefficients in [0.1, 1] every M(mu) has condition below ~3."""
    rs = np.random.RandomState(seed)
    U = np.linalg.qr(rs.standard_normal((kp, r)))[0]
    lhs = [U + 0.1 * rs.standard_normal((kp, r)) / np.sqrt(kp) for _ in range(Q)]
    return lhs, [rs.standard_normal(kp) for _ in range(Pf)]


def _thetas(P, Q, Pf, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    th = 0.1 + 0.9 * torch.rand(P, Q, dtype=torch.float64, device="cuda", generator=g)
    tf = torch.randn(P, Pf, dtype=torch.float64, device="cuda", generator=g)
    return th, tf


def _rows(P):
    return sorted(set(range(0, P, max(1, P // 40))) | {P - 1})


def _host_lstsq(lhs, rhs, th, tf):
    """numpy.linalg.lstsq (SVD) of the assembled system, and its condition number."""
    M = sum(t * A for t, A in zip(th, lhs))
    b = sum((t * g for t, g in zip(tf, rhs)), np.zeros(M.shape[0]))
    x, _, _, s = np.linalg.lstsq(M, b, rcond=None)
    return x, s[0] / s[-1]


def _launches(rb):
    return rb.lib().rla_launch_count()


@pytest.mark.parametrize("Pf", [0, 1, 3])
@pytest.mark.parametrize("Q", [1, 4])
@pytest.mark.parametrize("r", [1, 7, 37, 64, 128])
def test_solve_batch_matches_host_lstsq(rb, r, Q, Pf):
    N = Q * r + Pf
    for kp in (max(r, N - 1), 2 * N + 3):              # N >= k': the stack as is; N < k': compressed
        lhs, rhs = _well_conditioned(r, Q, Pf, kp, seed=r * 100 + Q * 10 + Pf + kp)
        rom = _ls_rom(lhs, rhs)
        for P in (1, 5, 1000, 1031):
            th, tf = _thetas(P, Q, Pf, seed=P + r)
            n0 = _launches(rb)
            a = rom.solve_batch(th, tf)
            assert _launches(rb) - n0 == 1                # one kernel launch for the whole set
            assert a.shape == (P, r) and rom._ls_stack.shape == (N, min(N, kp))
            a_h, th_h, tf_h = a.cpu().numpy(), th.cpu().numpy(), tf.cpu().numpy()
            for p in _rows(P):
                ref, cond = _host_lstsq(lhs, rhs, th_h[p], tf_h[p])
                assert cond <= 1e3
                if Pf:
                    assert np.linalg.norm(a_h[p] - ref) <= 1e-12 * np.linalg.norm(ref), (kp, P, p)
                else:
                    assert np.linalg.norm(a_h[p]) == 0.0                      # b(mu) = 0
        assert torch.equal(rom.estimate_error_batch(a, th, tf), rom.estimate_error_batch(None, th, tf))


def test_ill_conditioned_family(rb):
    """kappa(M(mu)) ~ 1e8 with consistent right-hand sides: the error stays below 1e-14 kappa."""
    rs = np.random.RandomState(7)
    r, kp = 24, 200
    U = np.linalg.qr(rs.standard_normal((kp, r)))[0]
    V1, V2 = (np.linalg.qr(rs.standard_normal((r, r)))[0] for _ in range(2))
    B0 = V1 @ np.diag(np.logspace(0, -8, r)) @ V2.T
    B1 = 1e-10 * rs.standard_normal((r, r))
    lhs, rhs = [U @ B0, U @ B1], [U @ rs.standard_normal(r), U @ rs.standard_normal(r)]
    rom = _ls_rom(lhs, rhs)
    th, tf = _thetas(257, 2, 2, seed=3)
    a = rom.solve_batch(th, tf).cpu().numpy()
    th_h, tf_h = th.cpu().numpy(), tf.cpu().numpy()
    worst = 0.0
    for p in _rows(257):
        ref, cond = _host_lstsq(lhs, rhs, th_h[p], tf_h[p])
        assert 1e7 <= cond <= 1e9
        err = np.linalg.norm(a[p] - ref) / np.linalg.norm(ref)
        assert err <= 1e-14 * cond, (p, err, cond)
        worst = max(worst, err)
    assert worst > 0.0                                     # the family really is ill-conditioned


@pytest.mark.parametrize("r,Q,Pf,kp", [(5, 3, 2, 40), (37, 4, 1, 400), (128, 2, 1, 512)])
def test_compression_is_transparent(rb, r, Q, Pf, kp):
    from rla4mor_b200 import reductor_ops as ops
    lhs, rhs = _well_conditioned(r, Q, Pf, kp, seed=r)
    rom = _ls_rom(lhs, rhs)
    raw = torch.cat([_dev(M).T for M in lhs] + [_dev(g).reshape(1, -1) for g in rhs], dim=0).contiguous()
    comp = rom._lstsq_stack()
    assert raw.shape == (Q * r + Pf, kp) and comp.shape == (Q * r + Pf, Q * r + Pf)
    th, tf = _thetas(1031, Q, Pf, seed=kp)
    a_raw = ops.rom_lstsq_batch(raw, Q, r, th, tf)[0]
    a_comp = ops.rom_lstsq_batch(comp, Q, r, th, tf)[0]
    rel = torch.linalg.norm(a_raw - a_comp, dim=1) / torch.linalg.norm(a_raw, dim=1)
    assert float(rel.max()) <= 1e-12


def test_bit_equality_and_determinism(rb):
    from rla4mor_b200 import reductor_ops as ops
    r, Q, Pf, kp = 29, 3, 2, 300
    lhs, rhs = _well_conditioned(r, Q, Pf, kp, seed=11)
    rom = _ls_rom(lhs, rhs)
    P = 777
    th, tf = _thetas(P, Q, Pf, seed=5)
    a = rom.solve_batch(th, tf)
    for p in _rows(P):
        assert torch.equal(rom.solve(th[p], tf[p]), a[p])                    # P = 1 against the batch
        assert torch.equal(rom.solve(th[p].tolist(), tf[p].tolist()), a[p])
    assert torch.equal(rom.solve_batch(th, tf), a)                           # run to run
    g = torch.Generator(device="cuda").manual_seed(0)
    th_big = torch.randn(P, Q + 4, dtype=torch.float64, device="cuda", generator=g)
    tf_big = torch.randn(P, Pf + 3, dtype=torch.float64, device="cuda", generator=g)
    th_big[:, 1:1 + Q], tf_big[:, 3:3 + Pf] = th, tf
    th_s, tf_s = th_big[:, 1:1 + Q], tf_big[:, 3:3 + Pf]                     # strided rows, odd offsets
    assert th_s.stride(0) == Q + 4 and tf_s.stride(0) == Pf + 3
    assert torch.equal(rom.solve_batch(th_s, tf_s), a)
    # strided a through the C entry point (row stride r + 5, offset 2)
    W = rom._lstsq_stack()
    out = torch.full((P, r + 5), -7.0, dtype=torch.float64, device="cuda")
    info = torch.full((P,), -1, dtype=torch.int32, device="cuda")
    lib = rb.lib()
    rb._lib.check(lib.rla_rom_lstsq_batch_f64(W.data_ptr(), W.stride(0), Q, r, Pf, W.shape[1], th_s.data_ptr(),
                                              th_s.stride(0), tf_s.data_ptr(), tf_s.stride(0), P,
                                              ctypes.c_void_p(out.data_ptr() + 16), r + 5, info.data_ptr(),
                                              rb._lib.stream_ptr()), "rla_rom_lstsq_batch_f64")
    assert torch.equal(out[:, 2:2 + r], a) and bool((out[:, :2] == -7.0).all()) and bool((out[:, 2 + r:] == -7.0).all())
    assert not bool(info.any())
    a_ops, info_ops = ops.rom_lstsq_batch(W, Q, r, th_s, tf_s)
    assert torch.equal(a_ops, a) and not bool(info_ops.any())


def test_rank_deficiency(rb):
    from rla4mor_b200 import reductor_ops as ops
    rs = np.random.RandomState(5)
    r, kp = 9, 60
    M = np.linalg.qr(rs.standard_normal((kp, r)))[0] + 0.05 * rs.standard_normal((kp, r))
    S = rs.standard_normal((kp, r))
    S[:, 3] = 0.0                                           # M(mu) = S: column 4 (1-based) is zero
    rom = _ls_rom([M, S], [rs.standard_normal(kp)])
    P, bad, zero = 300, 123, 200
    th = np.column_stack([np.ones(P), 0.01 * rs.standard_normal(P)])
    th[bad] = (0.0, 1.0)
    th[zero] = (0.0, 0.0)                                   # M(mu) = 0
    tf = np.ones((P, 1))
    a, info = ops.rom_lstsq_batch(rom._lstsq_stack(), 2, r, torch.tensor(th), torch.tensor(tf), check=False)
    info = info.cpu().numpy()
    assert info[bad] == 4 and info[zero] == 1 and np.count_nonzero(info) == 2
    with pytest.raises(rb.RlaError, match=r"2 of 300 .*rank-deficient.*row 123"):
        rom.solve_batch(th, tf)
    with pytest.raises(rb.RlaError, match=r"rank-deficient"):
        rom.solve(th[zero], tf[zero])
    a2 = rom.solve_batch(th, tf, check=False)
    good = np.delete(np.arange(P), [bad, zero])
    assert torch.isnan(a2[bad]).all() and torch.isnan(a2[zero]).all() and not torch.isnan(a2[good]).any()
    assert torch.equal(a2[good], rom.solve_batch(th[good], tf[good]))      # the others do not notice
    est = rom.estimate_error_batch(a2, th, tf)
    assert torch.isnan(est[bad]) and torch.isnan(est[zero]) and not torch.isnan(est[good]).any()


def test_memory_at_scale(rb):
    """P = 1e5, k' = 2000: the compressed stack and the result, nothing proportional to P k'."""
    r, Q, Pf, kp, P = 64, 4, 1, 2000, 100000
    lhs, rhs = _well_conditioned(r, Q, Pf, kp, seed=1)
    rom = _ls_rom(lhs, rhs)
    th, tf = _thetas(P, Q, Pf, seed=2)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    a = rom.solve_batch(th, tf)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base < P * kp * 8 // 8
    a_h, th_h, tf_h = a.cpu().numpy(), th.cpu().numpy(), tf.cpu().numpy()
    for p in range(0, P, 9973):
        ref, _ = _host_lstsq(lhs, rhs, th_h[p], tf_h[p])
        assert np.linalg.norm(a_h[p] - ref) <= 1e-12 * np.linalg.norm(ref)


def test_outside_envelope_loops_per_mu(rb):
    """r above rom_lstsq_batch_max_r(): the per-mu torch solve runs, and agrees with the host."""
    from rla4mor_b200 import reductor_ops as ops
    r = ops.rom_lstsq_batch_max_r() + 1
    lhs, rhs = _well_conditioned(r, 1, 1, r + 20, seed=4)
    rom = _ls_rom(lhs, rhs)
    th, tf = _thetas(3, 1, 1, seed=1)
    n0 = _launches(rb)
    a = rom.solve_batch(th, tf)
    assert _launches(rb) == n0 and rom._ls_stack is None
    for p in range(3):
        assert torch.equal(a[p], rom.solve(th[p], tf[p]))
        ref, _ = _host_lstsq(lhs, rhs, th[p].cpu().numpy(), tf[p].cpu().numpy())
        assert np.linalg.norm(a[p].cpu().numpy() - ref) <= 1e-12 * np.linalg.norm(ref)


# ----------------------------------------------------------- executed-reference fixture
@pytest.mark.parametrize("cfg", ["gauss_minres", "srht_minres"])
def test_minres_fixture_on_the_kernel(rb, cfg, monkeypatch):
    from rla4mor_b200.factorization import InverseLuOperator
    from rla4mor_b200.sketched_reductor import AffineModel
    z = np.load(os.path.join(GOLDEN, "reductor_reference.npz"))
    meta = json.loads(str(z["__meta__"]))
    n = meta["n"]
    A = [sp.csr_matrix((z[f"A{q}__data"], z[f"A{q}__indices"], z[f"A{q}__indptr"]), shape=(n, n)) for q in range(3)]
    R = sp.csr_matrix((z["R__data"], z["R__indices"], z["R__indptr"]), shape=(n, n))
    ops_dev = [rb.MatrixOperator(x, source_id="S", range_id="S") for x in A]
    space = ops_dev[0].source
    fom = AffineModel(ops_dev, list(z["f"]), operator_coefficients=[1.0, lambda mu: mu[0], lambda mu: mu[1]],
                      rhs_coefficients=[1.0, lambda mu: mu[0]], output=z["out"], solution_space=space)
    Rop = rb.MatrixOperator(R.tocsc(), source_id="S", range_id="S")
    cls = rb.GaussianEmbedding if cfg.startswith("gauss") else rb.SrhtEmbedding
    emb = cls(source=space, options={"range_dim": meta["k"]}, _seed=meta["seed_primal"], range_id="SK")
    onl = rb.GaussianEmbedding(source=emb.range, options={"range_dim": meta["k_online"]}, _seed=meta["seed_online"])
    red = rb.SketchedReductor(fom, embedding_primal=emb, embedding_online=onl, product=Rop,
                              inverse_product=InverseLuOperator(Rop), projection="minres", orthonormalize=False)
    off = 0
    for nb in meta["blocks"]:
        red.extend_basis(z["U"][off:off + nb])
        red.orthonormalize_basis(offset=red.srb.shape[0] - nb)
        off += nb
    rom = red.reduce(seed=tuple(meta["minres_seeds"]))

    def no_lstsq(*args, **kwargs):
        raise AssertionError("the per-mu torch.linalg.lstsq ran")
    monkeypatch.setattr(torch.linalg, "lstsq", no_lstsq)
    mus = meta["test"]
    n0 = _launches(rb)
    a = rom.solve_batch(mus=mus)
    assert _launches(rb) - n0 == 1
    for j, mu in enumerate(mus):
        assert rel_fro(a[j].cpu().numpy(), z[f"{cfg}__sol{j}"][0]) < 1e-9
        assert torch.equal(rom.solve(mu=mu), a[j])
