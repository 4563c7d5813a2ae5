"""The device MT19937 Gaussian draw (csrc/mt19937.cu) is bit-identical to NumPy's
RandomState(seed).normal: whole matrices, batches of block seeds, sub-ranges, the host fix-up path,
and the embeddings that draw their Theta with it."""
import numpy as np
import pytest
import torch

import rla4mor_b200 as rb
from rla4mor_b200 import dense, mt19937
from oracle import embeddings_oracle as eo

pytestmark = pytest.mark.gpu


def _numpy(seeds, rows, n, scale):
    return np.vstack([np.random.RandomState(s).normal(size=(b, n), loc=0, scale=scale) for s, b in zip(seeds, rows)])


def _equal(dev, host):
    return dev.shape == host.shape and torch.equal(dev, torch.from_numpy(np.ascontiguousarray(host)).to(dev.device))


@pytest.mark.parametrize("k,n,seed", [(1, 1, 0), (3, 1001, 5), (7, 2 ** 20 + 3, 2 ** 32 - 2), (100, 10 ** 6, 17)])
def test_matrix_equals_numpy(k, n, seed):
    scale = 1 / np.sqrt(k)
    assert _equal(mt19937.gaussian_matrix([seed], [k], n, scale), _numpy([seed], [k], n, scale))


def test_block_batch_and_host_download():
    b = rb.BlockGaussianEmbedding(source=rb.DeviceVectorSpace(3001), options={"range_dim": 70, "max_block_size": 32},
                                  _seed=9)
    ref = _numpy(b.block_seeds, b.block_sizes, 3001, 1 / np.sqrt(70))
    assert _equal(mt19937.gaussian_matrix(list(b.block_seeds), b.block_sizes, 3001, 1 / np.sqrt(70)), ref)
    # drawn in pieces of a few rows and downloaded piece by piece
    host = mt19937.gaussian_matrix_host(list(b.block_seeds), b.block_sizes, 3001, 1 / np.sqrt(70), chunk_bytes=5 * 8 * 3001)
    assert np.array_equal(host, ref)


def test_sub_ranges():
    seeds, counts = [3, 4, 5], [50001, 7, 200000]
    refs = [np.random.RandomState(s).normal(size=c, loc=0, scale=0.5) for s, c in zip(seeds, counts)]
    plan = mt19937.NormalPlan(seeds, counts)
    for first, count in (([1, 0, 12345], [50000, 7, 3]), ([49999, 6, 199999], [2, 1, 1]), ([777, 3, 0], [0, 2, 200000])):
        offset = np.concatenate([[5], 5 + np.cumsum(count)[:-1]])
        out = torch.full((5 + sum(count),), float("nan"), dtype=torch.float64, device="cuda")
        plan.execute(out, first, count, offset, 0.5)
        ref = np.concatenate([r[f:f + c] for r, f, c in zip(refs, first, count)])
        assert torch.isnan(out[:5]).all() and _equal(out[5:], ref), (first, count)


def test_host_fixup_path():
    """w = 0.5 finishes every pair with the C library's log on the host: the same numbers.  w = 0
    trusts the extended log everywhere; how many pairs it gets wrong is reported, not asserted."""
    n, scale = 400_000, 1 / np.sqrt(3)
    ref = np.random.RandomState(21).normal(size=n, loc=0, scale=scale)
    plan = mt19937.NormalPlan([21], [n])
    out = torch.empty(n, dtype=torch.float64, device="cuda")
    flagged = {}
    for w in (mt19937.W_DEFAULT, 0.5, 0.0):
        out.fill_(float("nan"))
        flagged[w] = plan.execute(out, 0, n, 0, scale, w=w)
        if w:
            assert _equal(out, ref), w
    wrong = int((out.cpu().numpy() != ref).sum())
    assert flagged[0.5] == (n + 1) // 2 and flagged[0.0] == 0
    print(f"flagged pairs: {flagged[mt19937.W_DEFAULT]} of {(n + 1) // 2} at w = 2^-5; "
          f"{wrong} of {n} outputs differ from NumPy with w = 0")


@pytest.fixture
def no_numpy_normal(monkeypatch):
    class Guard(np.random.RandomState):
        def normal(self, *a, **k):
            raise AssertionError("Theta was drawn by NumPy on the host")
    monkeypatch.setattr(np.random, "RandomState", Guard)


def test_embeddings_draw_on_device(no_numpy_normal):
    n, k = 5003, 40
    g = rb.GaussianEmbedding(source=rb.DeviceVectorSpace(n), options={"range_dim": k}, _seed=6)
    b = rb.BlockGaussianEmbedding(source=rb.DeviceVectorSpace(n), options={"range_dim": k, "max_block_size": 16},
                                  _seed=7)
    x = np.random.RandomState(1).standard_normal((9, n))
    g.apply(x), b.apply(x), b.get_block_device(1), b.get_random_matrix()


def test_embeddings_equal_the_numpy_draws():
    n, k = 5003, 40
    theta = eo.gaussian_random_matrix(k, n, 6)
    g = rb.GaussianEmbedding(source=rb.DeviceVectorSpace(n), options={"range_dim": k}, _seed=6)
    assert np.array_equal(g._random_matrix, theta)
    assert _equal(g.get_matrix_device(), theta)
    assert np.array_equal(g.get_random_matrix(), theta)
    x = np.random.RandomState(1).standard_normal((9, n))
    xd = torch.from_numpy(x).cuda()
    assert _equal(g.apply(xd), dense.gauss_apply_explicit(torch.from_numpy(theta).cuda(), xd).cpu().numpy())

    b = rb.BlockGaussianEmbedding(source=rb.DeviceVectorSpace(n), options={"range_dim": k, "max_block_size": 16},
                                  _seed=7)
    full = eo.block_gaussian_random_matrix(k, n, 7, 16)
    for i, (lo, hi) in enumerate(((0, 16), (16, 32), (32, 40))):
        assert _equal(b.get_block_device(i), full[lo:hi])
        assert np.array_equal(b._get_random_block(i), full[lo:hi])
    y = b.apply(xd)
    ref = torch.cat([dense.gauss_apply_explicit(torch.from_numpy(full[lo:hi]).cuda(), xd)
                     for lo, hi in ((0, 16), (16, 32), (32, 40))], dim=1)
    assert torch.equal(y, ref)
    assert _equal(b._compute_random_matrix_device(), full)
    assert np.array_equal(b.get_random_matrix(), full)
