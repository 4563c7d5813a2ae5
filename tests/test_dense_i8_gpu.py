"""The int8 path of float64 sketches (csrc/gemm_i8.cu, kinds 0 and 2): bit-for-bit equal to the NumPy
replay of its slicing and flush order, inside the normwise bound of its header on adversarial blocks,
and within 1e-14 of the FP64 tensor-pipe path at a sketch-sized n."""
from fractions import Fraction

import numpy as np
import pytest
import torch

import ozaki_ref as oz
from golden_util import rel_fro

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dense():
    import rla4mor_b200
    rla4mor_b200.lib()
    from rla4mor_b200 import dense
    return dense


def theta(dense, seed, kind, k, n, row0=0, col0=0):
    return dense.theta_materialize(seed, kind, 1.0, k, n, row0=row0, col0=col0).cpu().numpy()


@pytest.mark.parametrize("m,k,n,row0,col0,kind,accumulate", [
    (200, 100, 40003, 5, 48, 0, False),        # three exponent blocks, the last ragged; cluster pairs
    (400, 70, 20000, 9, 32, 0, False),         # clusters of four along m
    (70, 33, 1000, 0, 0, 2, True),             # one tile along m (no pair), one short block
    (257, 65, 16384 + 31, 3, 16, 0, True),
])
def test_bitwise_equal_to_the_numpy_replay(dense, m, k, n, row0, col0, kind, accumulate):
    rs = np.random.RandomState(m + n)
    u = rs.standard_normal((m, n)) * 2.0 ** rs.randint(-20, 20, (m, 1))
    u[1, : n // 2] = 0.0                                     # an all-zero block
    th = theta(dense, 11, kind, k, n, row0, col0)
    y0 = rs.standard_normal((m, k))
    out = torch.from_numpy(y0.copy()).cuda() if accumulate else None
    got = dense.embed_apply_rng(11, kind, 0.5, k, torch.from_numpy(u).cuda(), row0=row0, col0=col0,
                                out=out, accumulate=accumulate).cpu().numpy()
    want = oz.replay(u, th, 0.5, y0 if accumulate else None)
    assert np.array_equal(got, want)


def exact_dot(a, b):
    return sum(Fraction(float(x)) * Fraction(float(y)) for x, y in zip(a, b) if x != 0 and y != 0)


def test_normwise_bound_on_adversarial_blocks(dense):
    n, k = 2048, 6
    rs = np.random.RandomState(5)
    rows = [
        rs.standard_normal(n) * 2.0 ** rs.randint(-600, 601, n),                 # 2^-600 .. 2^600 in one row
        np.where(np.arange(n) == 777, 3.0e200, rs.standard_normal(n) * 1e-3),    # one spike
        np.zeros(n),                                                              # all-zero block
        rs.standard_normal(n) * 2.0 ** -1060,                                    # subnormals
        np.concatenate([rs.standard_normal(n // 2), rs.standard_normal(n // 2) * 1e-300]),
    ]
    u = np.stack(rows)
    th = theta(dense, 4, 0, k, n)
    got = dense.embed_apply_rng(4, 0, 1.0, k, torch.from_numpy(u).cuda()).cpu().numpy()
    Lb, nb = min(oz.L, n), 1
    for c in range(u.shape[0]):
        for i in range(k):
            mx = np.max(np.abs(u[c]))
            un, tn = (mx * np.linalg.norm(u[c] / mx) if mx > 0 else 0.0), np.linalg.norm(th[i])
            bound = (2.0 ** -53 * np.sqrt(Lb) * un * (tn / 4 + 15 * np.sqrt(n)) + (nb + 10) * 2.0 ** -52 * un * tn
                     + 2.0 ** -1073 * nb)
            err = abs(Fraction(float(got[c, i])) - exact_dot(u[c], th[i]))
            assert err <= Fraction(bound), (c, i, float(err), bound)


def test_nan_block_takes_the_fp64_path(dense):
    n, k = 3000, 8
    rs = np.random.RandomState(6)
    u = rs.standard_normal((4, n))
    u[2, 1234] = np.nan
    th = theta(dense, 9, 0, k, n)
    got = dense.embed_apply_rng(9, 0, 1.0, k, torch.from_numpy(u).cuda()).cpu().numpy()
    assert np.isnan(got[2]).all()
    ok = [0, 1, 3]
    assert rel_fro(got[ok], u[ok] @ th.T) < 1e-14


def test_agrees_with_the_dmma_path_at_sketch_size(dense):
    m, k, n = 512, 64, 2 ** 20
    g = torch.Generator(device="cuda").manual_seed(3)
    u = torch.randn((m, n), dtype=torch.float64, device="cuda", generator=g)
    th = dense.theta_materialize(0, 0, 1.0, k, n)
    y8 = dense.embed_apply_rng(0, 0, 1.0, k, u)
    yd = dense.gauss_apply_explicit(th, u)                   # FP64 tensor pipe, the same Theta
    assert rel_fro(y8.cpu().numpy(), yd.cpu().numpy()) < 1e-14
    again = dense.embed_apply_rng(0, 0, 1.0, k, u)
    assert torch.equal(y8, again)                            # deterministic
