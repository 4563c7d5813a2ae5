"""The adjoint of the on-the-fly Gaussian embeddings with Theta generated in the kernel
(csrc/adjoint_rng.cu, `dense.embed_adjoint_rng`, `GaussianEmbedding.apply_adjoint`,
`BlockGaussianEmbedding.apply_adjoint`): bit-identity with the product over the materialised Theta,
parity of the embedding classes with V @ get_matrix(), memory at scale, one launch for all blocks,
adjointness against the forward sketch, and the pyMOR adapter."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import embeddings_oracle as eo
from golden_util import rel_fro

pytestmark = pytest.mark.gpu
MODES = ("mt19937", "philox", "philox_rademacher", "philox_tf32")


@pytest.fixture(scope="module")
def rb():
    import rla4mor_b200
    rla4mor_b200.lib()
    return rla4mor_b200


def _even_ld(v):
    """v stored with an even leading dimension (16-byte rows): gemm_nn takes its DMMA path."""
    m, k = v.shape
    buf = torch.zeros((m, k + (k & 1)), dtype=v.dtype, device=v.device)
    buf[:, :k] = v
    return buf[:, :k]


def _reference(seeds, starts, kind, scale, v, n):
    """gemm_nn(V, Theta materialised) on its tensor-pipe path: Theta and the result are stored with
    an even number of columns (the extra column is sliced off; no element depends on another column)."""
    from rla4mor_b200 import dense
    from rla4mor_b200.reductor_ops import gemm_nn
    npad = n + (n & 1)
    theta = torch.cat([dense.theta_materialize(s, kind, scale, starts[b + 1] - starts[b], npad)
                       for b, s in enumerate(seeds)], dim=0)
    return gemm_nn(_even_ld(v), theta)[:, :n]


@pytest.mark.parametrize("kind", [0, 1, 2])
def test_kernel_bit_identical_to_materialised_product(rb, kind):
    from rla4mor_b200 import dense
    g = torch.Generator(device="cuda").manual_seed(kind)
    for m in (1, 7, 64, 129, 300):
        for k in (1, 3, 17, 2000):
            for n in (1, 5, 4097, 100003):
                v = torch.randn(m, k, dtype=torch.float64, device="cuda", generator=g)
                scale = 1.0 / np.sqrt(k)
                ref = _reference([11 + k], [0, k], kind, scale, v, n)
                got = dense.embed_adjoint_rng([11 + k], [0, k], kind, scale, _even_ld(v), n)
                assert torch.equal(got, ref), (kind, m, k, n)
                if n == 4097:
                    # odd leading dimension (8-byte copies of V) and a strided, unaligned view
                    assert torch.equal(dense.embed_adjoint_rng([11 + k], [0, k], kind, scale, v.contiguous(), n), ref)
                    wide = torch.zeros((m, k + 3), dtype=torch.float64, device="cuda")
                    wide[:, 1:1 + k] = v
                    assert torch.equal(dense.embed_adjoint_rng([11 + k], [0, k], kind, scale, wide[:, 1:1 + k], n), ref)


@pytest.mark.parametrize("kind", [0, 1, 2])
def test_kernel_block_tables(rb, kind):
    """Several blocks with sizes that are not multiples of 4 (and an empty one) in one call."""
    from rla4mor_b200 import dense
    g = torch.Generator(device="cuda").manual_seed(10 + kind)
    for sizes in ([1, 2], [5, 0, 7, 5], [3] * 5 + [2], [200] * 9 + [199, 1], [37, 963, 1000]):
        k = sum(sizes)
        starts = list(np.concatenate([[0], np.cumsum(sizes)]))
        seeds = [2 ** 63 + 977 * i + kind for i in range(len(sizes))]
        for m, n in ((7, 4097), (129, 1000), (2, 3)):
            v = torch.randn(m, k, dtype=torch.float64, device="cuda", generator=g)
            ref = _reference(seeds, starts, kind, 0.25, v, n)
            assert torch.equal(dense.embed_adjoint_rng(seeds, starts, kind, 0.25, _even_ld(v), n), ref), (sizes, m, n)
            assert torch.equal(dense.embed_adjoint_rng(seeds, starts, kind, 0.25, v, n), ref), (sizes, m, n)
    # run to run
    v = torch.randn(300, 2000, dtype=torch.float64, device="cuda", generator=g)
    a = dense.embed_adjoint_rng([5, 6], [0, 1000, 2000], kind, 0.5, v, 50000)
    assert torch.equal(a, dense.embed_adjoint_rng([5, 6], [0, 1000, 2000], kind, 0.5, v, 50000))


def test_kernel_rejects_bad_arguments(rb):
    from rla4mor_b200 import dense
    from rla4mor_b200._lib import lib, stream_ptr
    v = torch.ones((2, 4), dtype=torch.float64, device="cuda")
    out = torch.empty((2, 8), dtype=torch.float64, device="cuda")
    table = torch.tensor([1, 0, 4], dtype=torch.int64, device="cuda")
    call = lambda kind, nb, n, vp, ldo: lib().rla_embed_adjoint_rng_f64(kind, 1.0, table.data_ptr(), table[1:].data_ptr(), nb,
                                                                       n, vp, 2, 4, out.data_ptr(), ldo, stream_ptr())
    assert call(0, 1, 8, v.data_ptr(), 8) == 0
    assert call(3, 1, 8, v.data_ptr(), 8) == -1              # kind
    assert call(0, 0, 8, v.data_ptr(), 8) == -1              # no block
    assert call(0, 1, 8, v.data_ptr(), 7) == -1              # ldo < n
    assert call(0, 1, 8, None, 8) == -1                      # null pointer
    with pytest.raises(AssertionError):
        dense.embed_adjoint_rng([1], [0, 3], 0, 1.0, v, 8)  # table and V disagree on k
    with pytest.raises(AssertionError):
        dense.embed_adjoint_rng([1, 2], [0, 3, 2], 0, 1.0, v[:, :2], 8)


def _embeddings(rb, n, k, seed, mode, Q=None):
    opts = {"range_dim": k, "rng": mode}
    kw = dict(sqrt_product=Q) if Q is not None else dict(source=rb.DeviceVectorSpace(n))
    return (rb.GaussianEmbedding(options=opts, _seed=seed, **kw),
            rb.BlockGaussianEmbedding(options=dict(opts, max_block_size=7), _seed=seed, **kw))


@pytest.mark.parametrize("mode", MODES)
def test_embeddings_match_explicit_matrix(rb, mode):
    n, k, seed = 3001, 30, 4
    v = np.random.RandomState(0).standard_normal((5, k))
    gauss, block = _embeddings(rb, n, k, seed, mode)
    for emb in (gauss, block):
        theta = emb.get_random_matrix()
        if mode == "mt19937":                                         # NumPy's draw, as the reference makes it
            ref_theta = eo.gaussian_random_matrix(k, n, seed) if emb is gauss else \
                eo.block_gaussian_random_matrix(k, n, seed, 7)
            assert np.array_equal(theta, ref_theta)
        got = emb.apply_adjoint(v)
        assert isinstance(got, np.ndarray) and rel_fro(got, v @ theta) < 1e-13, type(emb).__name__
        V = emb.range.from_numpy(v)
        W = emb.apply_adjoint(V)
        assert W in emb.source and rel_fro(W.to_numpy(), v @ theta) < 1e-13
        assert rel_fro(emb.H.apply(V).to_numpy(), v @ theta) < 1e-13
        vt = torch.from_numpy(v).cuda()
        assert rel_fro(emb.apply_adjoint(vt).cpu().numpy(), v @ theta) < 1e-13
        assert rel_fro(emb.apply_adjoint(vt.float()).cpu().numpy(), v.astype(np.float32) @ theta) < 1e-13
        vc = v + 1j * np.random.RandomState(1).standard_normal(v.shape)
        assert rel_fro(emb.apply_adjoint(vc), vc @ theta) < 1e-13                      # complex block
        with pytest.raises(AssertionError):
            emb.apply_adjoint(rb.DeviceVectorSpace(k, id="OTHER").from_numpy(v))       # not in emb.range
        if mode != "mt19937":
            assert emb._matrix_dev is None
    # with the device matrix already built, GaussianEmbedding keeps the product with it
    gauss.get_matrix_device()
    assert rel_fro(gauss.apply_adjoint(v), v @ gauss.get_random_matrix()) < 1e-13


@pytest.mark.parametrize("mode", MODES)
def test_embeddings_with_sqrt_product(rb, mode):
    n, k, seed = 700, 30, 6
    Qm = np.random.RandomState(2).standard_normal((n, n))
    Q = rb.MatrixOperator(Qm, source_id="S", range_id="S")
    v = np.random.RandomState(3).standard_normal((4, k))
    for emb, ref_emb in zip(_embeddings(rb, n, k, seed, mode, Q), _embeddings(rb, n, k, seed, mode, Q)):
        mat = ref_emb.get_matrix()
        assert rel_fro(emb.apply_adjoint(emb.range.from_numpy(v)).to_numpy(), v @ mat) < 1e-13
        with pytest.raises(TypeError):
            emb.apply_adjoint(v + 1j * v)


def test_no_theta_at_scale(rb):
    """k x n = 2000 x 2^22: Theta would take 67 GB; the adjoint holds nothing but its result."""
    from rla4mor_b200 import dense
    from rla4mor_b200.reductor_ops import gemm_nn
    n, k, m = 2 ** 22, 2000, 8
    emb = rb.GaussianEmbedding(source=rb.DeviceVectorSpace(n), options={"range_dim": k, "rng": "philox"}, _seed=21)
    v = torch.randn(m, k, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = emb.apply_adjoint(v)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base < 2 * m * n * 8
    assert emb._matrix_dev is None and emb._matrix is None
    for c in (0, 2 ** 21 + 12, n - 4096):
        slab = dense.theta_materialize(21, dense.KIND_NORMAL, 1.0 / np.sqrt(k), k, 4096, col0=c)
        assert torch.equal(out[:, c:c + 4096], gemm_nn(v, slab)), c


def test_one_launch_for_all_blocks(rb):
    n, k = 50000, 95
    emb = rb.BlockGaussianEmbedding(source=rb.DeviceVectorSpace(n), options={"range_dim": k, "max_block_size": 10,
                                                                             "rng": "philox"}, _seed=3)
    assert emb.n_blocks == 10
    v = torch.randn(16, k, dtype=torch.float64, device="cuda")
    emb.apply_adjoint(v)
    before = rb.lib().rla_launch_count()
    w = emb.apply_adjoint(v)
    assert rb.lib().rla_launch_count() - before == 1
    assert rel_fro(w.cpu().numpy(), v.cpu().numpy() @ emb.get_random_matrix()) < 1e-13


def test_adjointness_against_forward_sketch(rb):
    """<Theta u, v> = <u, Theta^T v>; `apply` runs on the int8 tensor cores, the adjoint on DMMA."""
    n, k = 2 ** 20, 64
    for emb in (rb.GaussianEmbedding(source=rb.DeviceVectorSpace(n), options={"range_dim": k, "rng": "philox"}, _seed=8),
                rb.BlockGaussianEmbedding(source=rb.DeviceVectorSpace(n),
                                          options={"range_dim": k, "max_block_size": 20, "rng": "philox"}, _seed=8)):
        g = torch.Generator(device="cuda").manual_seed(1)
        u = torch.randn(4, n, dtype=torch.float64, device="cuda", generator=g)
        v = torch.randn(3, k, dtype=torch.float64, device="cuda", generator=g)
        lhs = emb.apply(u) @ v.T
        rhs = u @ emb.apply_adjoint(v).T
        assert float(torch.linalg.norm(lhs - rhs) / torch.linalg.norm(lhs)) < 1e-12


@pytest.mark.parametrize("mode", ["philox", "mt19937"])
def test_pymor_adapter_block_adjoint(mode):
    stub = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_pymor_stub")
    if stub not in sys.path:
        sys.path.insert(0, stub)
    import rla4mor_b200.pymor_adapter as rla
    from pymor.vectorarrays.numpy import NumpyVectorSpace
    n, k = 2000, 25
    emb = rla.BlockGaussianEmbedding(source=NumpyVectorSpace(n, id="S"),
                                     options={"range_dim": k, "max_block_size": 8, "rng": mode}, _seed=12, range_id="SK")
    v = np.random.RandomState(4).standard_normal((3, k))
    ref = emb._dev.apply_adjoint(v)
    W = emb.apply_adjoint(emb.range.from_numpy(v))
    assert W in emb.source and np.array_equal(W.to_numpy(), ref)
    assert np.array_equal(emb.H.apply(emb.range.from_numpy(v)).to_numpy(), ref)
    assert rel_fro(ref, v @ emb.get_random_matrix()) < 1e-13
