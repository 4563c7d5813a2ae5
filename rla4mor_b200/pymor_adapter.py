"""pyMOR front end of the B200 sketching engine (SURVEY.md section 8f rank 4).

Importing this module needs pyMOR (it is NOT imported by `rla4mor_b200/__init__.py`; the engine
itself has no pyMOR dependency).  It provides, as pyMOR `Operator`s with the reference's names,
constructor signatures and rule registration:

    RandomEmbedding, SrhtEmbedding, GaussianEmbedding, BlockGaussianEmbedding,
    IdentityEmbedding, EmbeddingVectorized        rla/embeddings.py:22-467
    InverseLuOperator                               utilities/factorization.py:88-138
    LsOperator                                      utilities/other_operators.py:12-39
    SketchedReductor, ResidualErrorEstimator        mor/sketched_reductor.py:22-219
    register_rules()                                rla/__init__.py:15-21

so `project(emb @ inv @ op, None, U)`, `contract(expand(emb @ ...))`, `emb.with_(_seed=s)` and the
`hasattr(emb, 'n_blocks')` probes of preconditioners/preconditioned_reductor.py:185,215 keep
working, with every `apply` running in librla_b200.so.  pyMOR's NumpyVectorArrays are host arrays:
the adapter uploads a block once per call and downloads the (small) sketch; `SketchedReductor`
below keeps the basis, the sketches and the affine images on the device for its whole life and
only hands the small reduced matrices back to pyMOR.

    import rla4mor_b200.pymor_adapter as rla          # instead of `import rla.embeddings`
    S = rla.SrhtEmbedding(source=fom.solution_space, options={'range_dim': 1000}, _seed=0)
    red = rla.SketchedReductor(fom, embedding_primal=S, inverse_product=rla.InverseLuOperator(R))
"""
from importlib.util import find_spec

if find_spec("pymor") is None:                                     # pragma: no cover
    raise ImportError("rla4mor_b200.pymor_adapter needs pyMOR (the engine itself, `import rla4mor_b200`, does not)")

import numpy as np
import scipy.sparse as sps
from pymor.algorithms.rules import match_class
from pymor.algorithms.simplify import ContractRules, ExpandRules
from pymor.core.base import BasicObject, ImmutableObject
from pymor.models.basic import StationaryModel
from pymor.operators.constructions import IdentityOperator, LincombOperator, VectorArrayOperator
from pymor.operators.interface import Operator
from pymor.operators.numpy import NumpyMatrixOperator
from pymor.tools.frozendict import FrozenDict
from pymor.vectorarrays.numpy import NumpyVectorSpace

from . import embeddings as _dev
from . import factorization as _fact
from . import sketched_reductor as _sr
from .vectorarray import DeviceVectorArray, DeviceVectorSpace, MatrixOperator


# ------------------------------------------------------------------ space / operator bridges
def _dspace(space):
    return DeviceVectorSpace(space.dim, id=space.id)


def _device_operator(op):
    """A pyMOR operator as a device operator: matrix operators are uploaded (CSR or dense), our own
    adapters hand over the device object they wrap, anything else is applied by pyMOR on the host."""
    if op is None or isinstance(op, IdentityOperator):
        return None
    if isinstance(op, (InverseLuOperator,)):
        return op._dev
    if isinstance(op, NumpyMatrixOperator):
        return MatrixOperator(op.matrix, source_id=op.source.id, range_id=op.range.id)
    return _HostOperator(op)


class _HostOperator:
    """Fallback: a pyMOR operator the engine knows nothing about, applied through host arrays."""
    linear = True

    def __init__(self, op):
        self.op = op
        self.source, self.range = _dspace(op.source), _dspace(op.range)

    def apply(self, U, mu=None):
        return self.range.from_numpy(self.op.apply(self.op.source.from_numpy(U.to_numpy()), mu=mu).to_numpy())

    def apply_adjoint(self, V, mu=None):
        return self.source.from_numpy(self.op.apply_adjoint(self.op.range.from_numpy(V.to_numpy()), mu=mu).to_numpy())


# ------------------------------------------------------------------------------ embeddings
class RandomEmbedding(Operator):
    """rla/embeddings.py:22-122 as a pyMOR Operator around a device embedding (`self._dev`)."""
    linear = True
    _dev_class = None

    def _setup(self, source, sqrt_product, options, range_id, _seed):
        assert not (source is None) or not (sqrt_product is None)
        if options is None:
            options = dict()
        self.options = FrozenDict(options)
        if sqrt_product is None:
            self.sqrt_product = IdentityOperator(source)
        self.source = self.sqrt_product.source
        q = _device_operator(sqrt_product)
        kw = dict(options=dict(options), range_id=range_id, _seed=_seed)
        self._dev = self._dev_class(sqrt_product=q, **kw) if q is not None else \
            self._dev_class(source=_dspace(self.source), **kw)
        self._seed = self._dev._seed
        self.range = NumpyVectorSpace(self._dev.range.dim, id=range_id)

    # -- the operator interface
    def apply(self, U, mu=None):
        assert U in self.source
        return self.range.from_numpy(self._dev.apply(U.to_numpy()))

    def apply_adjoint(self, V, mu=None):
        assert V in self.range
        return self.source.from_numpy(self._dev.apply_adjoint(V.to_numpy()))

    # -- rla/embeddings.py:69-122
    def compute_dim(self):
        return self._dev.compute_dim()

    def get_matrix(self):
        return self._dev.get_matrix()

    def get_random_matrix(self):
        return self._dev.get_random_matrix()

    def get_matrix_device(self):
        return self._dev.get_matrix_device()

    def set_seed(self, seed=None):
        self._dev.set_seed(seed)
        self._seed = self._dev._seed

    def update(self):
        self._dev.update()

    def as_range_array(self):
        return self.range.from_numpy(self.get_matrix().T)

    def as_source_array(self):
        return self.source.from_numpy(self.get_matrix())

    def _compute_matrix(self):
        return self._dev._compute_matrix()

    def _compute_random_matrix(self):
        return self._dev._compute_random_matrix()


class SrhtEmbedding(RandomEmbedding):
    _dev_class = _dev.SrhtEmbedding

    def __init__(self, source=None, sqrt_product=None, options=None, range_id=None, _seed=None):
        self.__auto_init(locals())
        self._setup(source, sqrt_product, options, range_id, _seed)

    def _get_random_rows(self, indices):
        return self._dev._get_random_rows(indices)


class GaussianEmbedding(RandomEmbedding):
    _dev_class = _dev.GaussianEmbedding

    def __init__(self, source=None, sqrt_product=None, options=None, range_id=None, _seed=None):
        self.__auto_init(locals())
        self._setup(source, sqrt_product, options, range_id, _seed)


class IdentityEmbedding(RandomEmbedding):
    _dev_class = _dev.IdentityEmbedding

    def __init__(self, source=None, sqrt_product=None, options=None, range_id=None, _seed=None):
        self.__auto_init(locals())
        self._setup(source, sqrt_product, options, range_id, _seed)


class BlockGaussianEmbedding(RandomEmbedding):
    _dev_class = _dev.BlockGaussianEmbedding

    def __init__(self, source=None, sqrt_product=None, options=None, range_id=None, _seed=None):
        assert options is not None and "max_block_size" in options.keys()
        self.__auto_init(locals())
        self._setup(source, sqrt_product, options, range_id, _seed)
        self.block_sizes, self.n_blocks, self.block_seeds = self._dev.block_sizes, self._dev.n_blocks, self._dev.block_seeds

    def get_block(self, ind):
        return self._dev.get_block(ind)

    def _get_random_block(self, ind):
        return self._dev._get_random_block(ind)


class EmbeddingVectorized(RandomEmbedding):
    """rla/embeddings.py:318-369: sketch of vec(U) by an inner embedding."""

    def __init__(self, source, n_vectors, embedding, options=None, range_id=None, _seed=None):
        if options is None:
            options = dict()
        self.__auto_init(locals())
        self._dev = _dev.EmbeddingVectorized(_dspace(source), n_vectors, embedding._dev, options=options,
                                             range_id=range_id, _seed=_seed)
        self._seed = self._dev._seed
        self.options = FrozenDict(self._dev.options)
        self.range = embedding.range

    def apply(self, U, mu=None):
        assert U in self.source
        assert len(U) == self.n_vectors
        return self.range.from_numpy(self._dev.apply(U.to_numpy()))

    def apply_adjoint(self, U, mu=None):
        pass


# ------------------------------------------------------------------- operators around the sketch
class InverseLuOperator(Operator):
    """utilities/factorization.py:88-138: SuperLU on the host (as in the reference), every
    application as sparse triangular solves on the device."""
    linear = True

    def __init__(self, operator, factorization=None, symetric=False, splu_kwargs=None):
        self.__auto_init(locals())
        self.source, self.range = operator.range, operator.source
        self._dev = _fact.InverseLuOperator(MatrixOperator(operator.matrix, source_id=operator.source.id,
                                                           range_id=operator.range.id),
                                            factorization=factorization, symetric=symetric, splu_kwargs=splu_kwargs)
        self.factorization = self._dev.factorization

    def apply(self, U, mu=None):
        assert U in self.source
        return self.source.from_numpy(self._dev.apply(self._dev.source.from_numpy(U.to_numpy())).to_numpy())

    def apply_adjoint(self, U, mu=None):
        assert U in self.source
        return self.source.from_numpy(self._dev.apply_adjoint(self._dev.source.from_numpy(U.to_numpy())).to_numpy())

    def apply_inverse(self, U, mu=None, **kwargs):
        return self.operator.apply(U)

    def apply_inverse_adjoint(self, U, mu=None, **kwargs):
        return self.operator.apply_adjoint(U)


class LsOperator(Operator):
    """utilities/other_operators.py:12-39: `apply_inverse` means least squares."""

    def __init__(self, operator):
        self.__auto_init(locals())
        self.source, self.range, self.linear = operator.source, operator.range, operator.linear

    def apply(self, U, mu=None, **kwargs):
        return self.operator.apply(U, mu, **kwargs)

    def apply_adjoint(self, U, mu=None, **kwargs):
        return self.operator.apply_adjoint(U, mu, **kwargs)

    def apply_inverse(self, U, mu=None, **kwargs):
        kwargs.pop("least_squares", None)
        return self.operator.apply_inverse(U, mu=mu, least_squares=True, **kwargs)

    def apply_inverse_adjoint(self, U, mu=None, **kwargs):
        kwargs.pop("least_squares", None)
        return self.operator.apply_inverse_adjoint(U, mu=mu, least_squares=True, **kwargs)

    def assemble(self, mu=None):
        return self.operator.assemble(mu)


_registered = False


def register_rules():
    """What rla/__init__.py:15-21 does for the reference's classes: `expand` / `contract` must treat
    an embedding (and the LU / least-squares wrappers) as a leaf instead of rebuilding it from
    its children."""
    global _registered
    if _registered:
        return

    @match_class(RandomEmbedding, InverseLuOperator, LsOperator)
    def action_Nothing(self, op):
        return op

    ContractRules.insert_rule(0, action_Nothing)
    ExpandRules.insert_rule(0, action_Nothing)
    _registered = True


register_rules()


# ------------------------------------------------------------------------------- reductor
def _terms(op):
    if isinstance(op, LincombOperator):
        return list(op.operators), list(op.coefficients)
    return [op], [1.0]


def to_affine_model(fom):
    """pyMOR StationaryModel with LincombOperators of matrix operators / vector operators ->
    the engine's device-resident AffineModel (affine terms uploaded once)."""
    ops, cop = _terms(fom.operator)
    rhs, crhs = _terms(fom.rhs)
    dev_ops = []
    for o in ops:
        assert isinstance(o, NumpyMatrixOperator), "affine terms must be NumpyMatrixOperators"
        dev_ops.append(MatrixOperator(o.matrix if sps.issparse(o.matrix) else np.asarray(o.matrix),
                                      source_id=o.source.id, range_id=o.range.id))
    f = [o.as_range_array().to_numpy()[0] for o in rhs]
    out = None
    if fom.output_functional is not None:
        from pymor.algorithms.to_matrix import to_matrix
        out = to_matrix(fom.output_functional, format="dense")
    return _sr.AffineModel(dev_ops, f, operator_coefficients=cop, rhs_coefficients=crhs, output=out,
                           solution_space=_dspace(fom.solution_space))


class ResidualErrorEstimator(ImmutableObject):
    """mor/sketched_reductor.py:210-219 on the device ROM: the norms of all rows of U are one
    batched estimate (SketchedRom.estimate_error_batch) with theta(mu) repeated."""

    def __init__(self, rom_dev, name=None):
        self.__auto_init(locals())

    def estimate_error(self, U, mu, m=None):
        import torch
        a = U.to_numpy()
        th, tf = self.rom_dev.fom.thetas(mu)
        rows = len(a)
        est = self.rom_dev.estimate_error_batch(
            a=torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda"),
            theta_lhs=np.tile(np.asarray(th, dtype=np.float64), (rows, 1)).reshape(rows, len(th)),
            theta_rhs=np.tile(np.asarray(tf, dtype=np.float64), (rows, 1)).reshape(rows, len(tf)))
        return est.cpu().numpy()


class SketchedReductor(BasicObject):
    """mor/sketched_reductor.py:22-208 with the reference's constructor; `fom` is a pyMOR
    StationaryModel.  The full-space work (sketches, SpMM, LU solves, basis update) runs and
    stays on the device; `reduce()` returns a pyMOR StationaryModel built from the small
    reduced matrices, with the FOM's own parameter functionals as coefficients."""

    def __init__(self, fom, embedding_primal=None, embedding_online=None, product=None, inverse_product=None,
                 save_rb=True, orthonormalize=True, projection='galerkin', log_level=20):
        assert projection in ('galerkin', 'minres')
        self.__auto_init(locals())
        self.logger.setLevel(log_level)
        self._affine = to_affine_model(fom)
        self._dev = _sr.SketchedReductor(
            self._affine,
            embedding_primal=None if embedding_primal is None else embedding_primal._dev,
            embedding_online=None if embedding_online is None else embedding_online._dev,
            product=_device_operator(product), inverse_product=_device_operator(inverse_product),
            save_rb=save_rb, orthonormalize=orthonormalize, projection=projection, log_level=log_level)
        self.rom = None

    # the reference's attributes, as pyMOR arrays (downloaded on access)
    @property
    def srb(self):
        return NumpyVectorSpace(self._dev.srb.shape[1], id=self._dev.embedding_primal.range.id).from_numpy(self._dev.srb.cpu().numpy())

    @property
    def rb(self):
        return self.fom.solution_space.from_numpy(self._dev.rb.cpu().numpy())

    def extend_basis(self, U, **kwargs):
        self._dev.extend_basis(U.to_numpy(), **kwargs)

    def orthonormalize_basis(self, offset=0, T=None, return_T=False, **kwargs):
        T = self._dev.orthonormalize_basis(offset=offset, T=T, return_T=True, **kwargs)
        return T.cpu().numpy() if return_T else None

    def reduce(self, embedding=None, seed=None, rom_log_level=30):
        if embedding is not None:
            embedding = tuple(e._dev for e in embedding) if isinstance(embedding, (tuple, list)) else embedding._dev
        rom_dev = self._dev.reduce(embedding=embedding, seed=seed)
        cop, crhs = self._affine.operator_coefficients, self._affine.rhs_coefficients
        estimator = ResidualErrorEstimator(rom_dev)
        n_out = self._dev.output_functional.shape[1]
        out = NumpyMatrixOperator(self._dev.output_functional.T.cpu().numpy().reshape(n_out, -1)) if n_out else None
        if isinstance(rom_dev, _sr.EmptyRom):
            r = 0
            lhs = LincombOperator([NumpyMatrixOperator(np.zeros((0, 0))) for _ in cop], cop)
            rhs = LincombOperator([NumpyMatrixOperator(np.zeros((0, 1))) for _ in crhs], crhs)
        else:
            lhs = LincombOperator([NumpyMatrixOperator(M.cpu().numpy()) for M in rom_dev.lhs], cop)
            rhs = LincombOperator([NumpyMatrixOperator(v.cpu().numpy().reshape(-1, 1)) for v in rom_dev.rhs], crhs)
            if rom_dev.least_squares:
                lhs = LsOperator(lhs)
        rom = StationaryModel(lhs, rhs, out, error_estimator=estimator)
        rom.logger.setLevel(rom_log_level)
        return rom
