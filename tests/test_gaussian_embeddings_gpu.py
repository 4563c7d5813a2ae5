"""GaussianEmbedding and BlockGaussianEmbedding share one model of Theta, a table of row blocks: a
Gaussian embedding is a table of one block.  Complex blocks through `apply`, the one-block
equivalence of the two classes, and the block adjoint over a device matrix built beforehand."""
import numpy as np
import pytest
import torch

from golden_util import rel_fro

pytestmark = pytest.mark.gpu
MODES = ("mt19937", "philox", "philox_rademacher", "philox_tf32")


@pytest.fixture(scope="module")
def rb():
    import rla4mor_b200
    rla4mor_b200.lib()
    return rla4mor_b200


def _both(rb, mode, n=3001, k=30, seed=4, **kw):
    opts = {"range_dim": k, "rng": mode}
    if "sqrt_product" not in kw:
        kw["source"] = rb.DeviceVectorSpace(n)
    return (rb.GaussianEmbedding(options=opts, _seed=seed, **kw),
            rb.BlockGaussianEmbedding(options=dict(opts, max_block_size=7), _seed=seed, **kw))


@pytest.mark.parametrize("mode", ["mt19937", "philox", "philox_tf32"])
def test_complex_apply(rb, mode):
    """Theta is real: a complex block is sketched as its real and imaginary parts."""
    n = 1001
    rs = np.random.RandomState(0)
    uc = rs.standard_normal((5, n)) + 1j * rs.standard_normal((5, n))
    for emb in _both(rb, mode, n):
        ref = uc @ emb.get_random_matrix().T
        y = emb.apply(uc)
        assert isinstance(y, np.ndarray) and y.dtype == np.complex128, type(emb).__name__
        assert rel_fro(y, ref) < 1e-12, type(emb).__name__
        yt = emb.apply(torch.from_numpy(uc).cuda())
        assert yt.is_cuda and yt.is_complex() and rel_fro(yt.cpu().numpy(), ref) < 1e-12
    Qm = rs.standard_normal((n, n)) + 1j * rs.standard_normal((n, n))
    Q = rb.MatrixOperator(Qm, source_id="S", range_id="S")
    for emb in _both(rb, mode, n, sqrt_product=Q):
        with pytest.raises(TypeError):
            emb.apply(Q.source.from_numpy(uc))


@pytest.mark.parametrize("mode", MODES)
def test_one_block_is_a_gaussian_embedding(rb, mode):
    """A block embedding whose blocks hold all k rows and the Gaussian embedding of its one block seed
    are the same operator, bit for bit."""
    n, k = 3001, 30

    def pair():
        block = rb.BlockGaussianEmbedding(source=rb.DeviceVectorSpace(n),
                                          options={"range_dim": k, "rng": mode, "max_block_size": 64}, _seed=4)
        gauss = rb.GaussianEmbedding(source=rb.DeviceVectorSpace(n), options={"range_dim": k, "rng": mode},
                                     _seed=int(block.block_seeds[0]))
        assert block.n_blocks == 1
        return gauss, block

    g = torch.Generator(device="cuda").manual_seed(1)
    u = torch.randn(9, n, dtype=torch.float64, device="cuda", generator=g)
    v = torch.randn(4, k, dtype=torch.float64, device="cuda", generator=g)
    gauss, block = pair()
    assert torch.equal(gauss.apply(u), block.apply(u))
    assert torch.equal(gauss.apply_adjoint(v), block.apply_adjoint(v))       # before any device matrix
    assert torch.equal(gauss.get_matrix_device(), block.get_matrix_device())
    gauss, block = pair()
    assert np.array_equal(gauss.get_random_matrix(), block.get_random_matrix())


@pytest.mark.parametrize("mode", MODES)
def test_block_adjoint_over_a_built_device_matrix(rb, mode):
    """After get_matrix_device() the block adjoint is the product with that matrix."""
    n, k = 3001, 30
    _, block = _both(rb, mode, n, k)
    v = np.random.RandomState(2).standard_normal((5, k))
    block.get_matrix_device()
    assert rel_fro(block.apply_adjoint(v), v @ block.get_random_matrix()) < 1e-13
