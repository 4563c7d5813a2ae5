"""B200 drop-in for the reference's `rla/embeddings.py` operator API.

Same class names, constructor signatures, `options` keys, dimension formulas and
method semantics as rla/embeddings.py:22-467 -- `RandomEmbedding`, `SrhtEmbedding`,
`GaussianEmbedding`, `IdentityEmbedding`, `EmbeddingVectorized`,
`BlockGaussianEmbedding` with `apply`, `apply_adjoint`, `get_matrix`,
`get_random_matrix`, `as_source_array`, `as_range_array`, `set_seed`, `update`,
`compute_dim`, `with_`, and for the block variant `get_block`, `_get_random_block`,
`block_sizes`, `n_blocks`, `block_seeds`.  Errors are `AssertionError`s in the same
places (embeddings.py:131,154,168,176,240,353-354,379).

All arithmetic runs in librla_b200.so (sm_100a CUDA); there is no CPU fallback.
Blocks of vectors are `(len, dim)` row arrays: `DeviceVectorArray`s (the stand-in
for pyMOR VectorArrays, see vectorarray.py), or plain NumPy arrays / CUDA tensors,
in which case the result comes back as the same kind.

One option is new: `options['rng']`
  * 'mt19937' (default): Theta is NumPy's legacy RandomState(seed).normal draw, exactly
    as the reference makes it (embeddings.py:269,458), and is applied by the explicit-Theta
    tensor-core GEMM -- same seed, same Theta, same sketch as the reference to 1e-12.
    With a CUDA device the draw itself runs on the GPU (csrc/mt19937.cu: MT19937 jump-ahead,
    bit-identical to NumPy's stream) and host copies such as `_random_matrix` are downloads
    of it; without one NumPy draws it.  Block seeds (:403) stay host draws;
  * 'philox' / 'philox_rademacher': Theta is generated on the fly inside the GEMM
    from a counter-based RNG and never materialised (the only way k x n = 2000 x 2**22
    fits anywhere), by `apply` and by `apply_adjoint` alike (csrc/adjoint_rng.cu generates it
    inside the adjoint's product); `get_random_matrix()` exports exactly what the kernels used;
  * 'philox_tf32': the normals of 'philox' rounded to TF32 (10 explicit mantissa bits).
    With this mode (and with 'philox_rademacher') Theta is exact in TF32, and FLOAT32
    blocks are sketched on the generation-5 tensor cores (tcgen05 kind::tf32 with a
    two-part split of the block and FP64 accumulation of 64-term partial sums,
    csrc/gemm32.cu: 1e-5 relative, ~4x the FP64 path); FP64 blocks use the same Theta.
SRHT signs and row indices are always the reference's NumPy draws (bit-exact).

The two Gaussian classes share one model of Theta, a table of row blocks: block b is rows
0 .. size_b - 1 of the stream of seed_b.  A `BlockGaussianEmbedding` lists its blocks; a
`GaussianEmbedding` is the table of one block (its seed, k rows), so every way of producing Theta,
`apply` and `apply_adjoint` are written once for both.  Theta is real, so a complex block is
sketched (and taken through the adjoint) as its real and imaginary parts; that needs an identity
`sqrt_product`, otherwise `TypeError`, as for the SRHT.  `apply_adjoint` multiplies by
`get_matrix_device()` when a Theta or matrix is already on the device (a `GaussianEmbedding` in
'mt19937' always holds its draw there); otherwise the Philox modes run one kernel over all blocks
with Theta generated inside it, and 'mt19937' draws one block at a time and accumulates.
"""
import logging

import numpy as np

from . import dense
from .srht import SrhtPlan, draw_signs_and_indices
from ._lib import check, lib, require_cuda, stream_ptr
from .vectorarray import DeviceVectorArray, DeviceVectorSpace, IdentityOperator, as_device_block
from . import mt19937

_logger = logging.getLogger("rla4mor_b200.embeddings")
_warned_once = set()


def _warning_once(msg):
    if msg not in _warned_once:
        _warned_once.add(msg)
        _logger.warning(msg)


class FrozenDict(dict):
    """Immutable dict (the reference freezes `options`, embeddings.py:136)."""

    def _blocked(self, *a, **k):
        raise TypeError("FrozenDict is immutable")

    __setitem__ = __delitem__ = clear = pop = popitem = setdefault = update = _blocked

    def __hash__(self):
        return hash(tuple(sorted((k, repr(v)) for k, v in self.items())))


class Concatenation:
    """`emb @ op`: apply right-to-left (what pyMOR's ConcatenationOperator does for the
    expressions at mor/sketched_reductor.py:69,73)."""
    linear = True

    def __init__(self, operators):
        self.operators = tuple(operators)
        self.source = self.operators[-1].source
        self.range = self.operators[0].range

    def apply(self, U, mu=None):
        for op in reversed(self.operators):
            U = op.apply(U, mu=mu)
        return U

    def __matmul__(self, other):
        ops = other.operators if isinstance(other, Concatenation) else (other,)
        return Concatenation(self.operators + tuple(ops))


def _cuda_available():
    try:
        import torch
    except ImportError:
        return False
    return torch.cuda.is_available()


def _wrap_result(kind, space, t):
    if kind == "va":
        return DeviceVectorArray(space, t)
    if kind == "np":
        return t.cpu().numpy()
    return t


def _is_host_tensor(U):
    """A CPU torch tensor: a block that lives in (ideally pinned) host memory and is streamed
    to the GPU in pieces instead of being copied whole."""
    try:
        import torch
    except ImportError:
        return False
    return isinstance(U, torch.Tensor) and not U.is_cuda and U.dim() == 2


def _unwrap(U):
    """-> (CUDA tensor (len, dim), kind)"""
    if isinstance(U, DeviceVectorArray):
        return U.data, "va"
    if isinstance(U, np.ndarray):
        return as_device_block(U), "np"
    return as_device_block(U), "torch"


class RandomEmbedding:
    """Base class -- rla/embeddings.py:22-122.

    Attributes: sqrt_product (operator Q with Q^H Q = R), options (FrozenDict),
    _random_matrix (l2 -> l2 matrix), _matrix (U -> l2 matrix), _seed.
    """
    linear = True
    _init_args = ("source", "sqrt_product", "options", "range_id", "_seed")

    # -- abstract (embeddings.py:44-66)
    def compute_dim(self):
        raise NotImplementedError

    def _compute_matrix(self):
        raise NotImplementedError

    def _compute_random_matrix(self):
        raise NotImplementedError

    # -- embeddings.py:69-100
    def get_matrix(self):
        if self._matrix is None:
            if getattr(self, "_matrix_dev", None) is not None:
                self._matrix = self._matrix_dev.cpu().numpy()        # host view of the device-built matrix
            else:
                self._matrix = self._compute_matrix()
        return self._matrix

    def get_random_matrix(self):
        # the reference caches into `_matrix` here (embeddings.py:98-99); kept as is
        if self._matrix is None:
            self._matrix = self._compute_random_matrix()
        return self._matrix

    def set_seed(self, seed=None):                       # embeddings.py:102-106
        if seed is None:
            seed = np.random.randint(0, high=2 ** 32 - 1)
        self._seed = seed
        self.update()
        if not isinstance(self, SrhtEmbedding):          # SrhtEmbedding.update() is a no-op (:145-146): cache survives
            self._matrix_dev = None

    def update(self):                                    # embeddings.py:108-113
        if not (self._random_matrix is None):
            self._random_matrix = self._compute_random_matrix()
        if not (self._matrix is None):
            self._matrix = self._compute_matrix()

    def as_range_array(self):                            # embeddings.py:115-117
        return DeviceVectorArray(self.range, self.get_matrix_device().T.contiguous())

    def as_source_array(self):                           # embeddings.py:120-122
        return DeviceVectorArray(self.source, self.get_matrix_device())

    # -- device-resident forms of the explicit matrices (consumed by
    #    preconditioners/preconditioned_reductor.py:107-119,185-194 and preconditioned_rom.py:66):
    #    nothing goes through host NumPy; get_matrix() is the host view of the same tensor
    def get_matrix_device(self):
        """The U -> l2 matrix (k, n) as a CUDA tensor, built on the device: explicit SRHT rows
        from the closed form, Theta from the kernel's generator (or the uploaded MT19937 draw),
        Q^H applied by the device operator."""
        if getattr(self, "_matrix_dev", None) is None:
            if self._matrix is not None:                 # same cache as get_matrix (incl. the get_random_matrix quirk)
                import scipy.sparse as sp
                m = self._matrix.toarray() if sp.issparse(self._matrix) else self._matrix
                self._matrix_dev = as_device_block(np.ascontiguousarray(m))
            else:
                self._matrix_dev = self._compute_matrix_device()
        return self._matrix_dev

    def _compute_matrix_device(self):
        return self._adjoint_sqrt_product_device(self._compute_random_matrix_device())

    def _compute_random_matrix_device(self):
        import scipy.sparse as sp
        m = self._compute_random_matrix()
        return as_device_block(np.ascontiguousarray(m.toarray() if sp.issparse(m) else m))

    def _adjoint_sqrt_product_device(self, rmat):
        """Q^H applied to the rows of a (k, n_Q) CUDA matrix (embeddings.py:185,261): conj(Q^H conj(rows))."""
        Q = self.sqrt_product
        if isinstance(Q, IdentityOperator):
            return rmat
        return Q.apply_adjoint(DeviceVectorArray(Q.range, rmat.conj() if rmat.is_complex() else rmat)).data

    # -- pyMOR machinery the call sites rely on
    def with_(self, **kwargs):
        """New embedding with some constructor arguments replaced (fresh caches), as
        `embedding_online.with_(_seed=seed)` at mor/sketched_reductor.py:128."""
        args = {name: getattr(self, "_arg_" + name) for name in self._init_args}
        unknown = set(kwargs) - set(args)
        assert not unknown, f"with_: unknown arguments {unknown}"
        args.update(kwargs)
        return type(self)(**args)

    def __matmul__(self, other):
        ops = other.operators if isinstance(other, Concatenation) else (other,)
        return Concatenation((self,) + tuple(ops))

    @property
    def H(self):
        emb = self

        class _Adjoint:
            linear = True
            source, range = emb.range, emb.source

            def apply(self, V, mu=None):
                return emb.apply_adjoint(V, mu=mu)

            def apply_adjoint(self, U, mu=None):
                return emb.apply(U, mu=mu)
        return _Adjoint()

    # -- helpers
    def _store_args(self, loc):
        for name in self._init_args:
            setattr(self, "_arg_" + name, loc[name])

    def _init(self, args, seeded=True):
        """The constructor body of the embeddings (embeddings.py:132-141 and the like): the argument
        record `with_` uses, with default options and, if `seeded`, a random seed filled in; frozen
        options; Q, the identity by default; the spaces; empty caches."""
        args = dict(args)
        if args["options"] is None:
            args["options"] = dict()
        if seeded and args["_seed"] is None:
            args["_seed"] = np.random.randint(0, high=2 ** 32 - 1)
        self._store_args(args)
        self._seed = args["_seed"]
        self.options = FrozenDict(args["options"])
        sqrt_product = args["sqrt_product"]
        self.sqrt_product = IdentityOperator(args["source"]) if sqrt_product is None else sqrt_product
        self.source = self.sqrt_product.source
        self.range_id = args["range_id"]
        self.range = DeviceVectorSpace(self.compute_dim(), id=self.range_id)
        self._matrix = None
        self._matrix_dev = None
        self._random_matrix = None

    def _apply_sqrt_product(self, U):
        """Q U as a CUDA block, plus the kind of the caller's container."""
        if isinstance(U, DeviceVectorArray):
            assert U in self.source                      # embeddings.py:168
            return self.sqrt_product.apply(U).data, "va"
        t, kind = _unwrap(U)
        assert t.shape[1] == self.source.dim
        if isinstance(self.sqrt_product, IdentityOperator):
            return t, kind
        return self.sqrt_product.apply(DeviceVectorArray(self.source, t)).data, kind

    def _adjoint_sqrt_product(self, rmat):
        """Q^H applied to the rows of a (k, n) host matrix: embeddings.py:185,261."""
        Q = self.sqrt_product
        if isinstance(Q, IdentityOperator):
            return rmat
        return Q.apply_adjoint(Q.range.from_numpy(rmat.conj())).to_numpy().conj()


def _gaussian_dim(opt):
    """embeddings.py:234-247 (also :337-350, :409-422)."""
    range_dim = opt.get('range_dim')
    eps = opt.get('epsilon')
    delta = opt.get('delta')
    d = opt.get('oblivious_dim')
    assert range_dim or all([eps, delta, d])
    if range_dim is None:
        a = 1
        if opt.get('dtype') == complex:
            a = 2
        range_dim = 7.87 * (1 / eps ** 2) * (a * 6.9 * d + np.log(1 / delta))
        range_dim = int(np.ceil(range_dim))
    return range_dim


class SrhtEmbedding(RandomEmbedding):
    """rla/embeddings.py:126-209."""

    def __init__(self, source=None, sqrt_product=None, options=None, range_id=None, _seed=None):
        assert not (source is None) or not (sqrt_product is None)          # :131
        self._init(locals())
        self._plans = {}
        self._order_dev = None

    def update(self):                                                      # :145-146
        pass

    def compute_dim(self):                                                 # :148-164
        opt = self.options
        range_dim = opt.get('range_dim')
        eps = opt.get('epsilon')
        delta = opt.get('delta')
        d = opt.get('oblivious_dim')
        assert range_dim or all([eps, delta, d])
        n = self.source.dim
        if range_dim is None:
            a = 1
            if opt.get('dtype') == complex:
                a = 2
            range_dim = 2 / (eps ** 2 - eps ** 3 / 3)
            range_dim = range_dim * (np.sqrt(a * d) + np.sqrt(8 * np.log(6 * a * n / delta))) ** 2
            range_dim = range_dim * np.log(3 * a * d / delta)
            range_dim = int(np.ceil(range_dim))
        return range_dim

    def _plan(self, dtype, device):
        """Signs / indices drawn as srht.py:162-163 for (self._seed, n, k); cached per seed."""
        n = self.sqrt_product.range.dim
        key = (self._seed, n, self.range.dim, dtype, device.index)
        plan = self._plans.get(key)
        if plan is None:
            signs, sampling = draw_signs_and_indices(n, self.range.dim, self._seed)
            plan = SrhtPlan(n, self.range.dim, signs, sampling, dtype, device)
            self._plans = {key: plan}
            self._order_dev = None
        return plan

    def apply(self, U, mu=None):                                           # :167-172
        torch = require_cuda()
        if _is_host_tensor(U) and isinstance(self.sqrt_product, IdentityOperator):
            # block in host memory: vectors are independent, stream them in groups; the
            # sketch comes back as a pinned host tensor
            from .streaming import apply_streamed
            assert U.shape[1] == self.source.dim
            return apply_streamed(self.apply, U, self.range.dim, return_host=True)
        qu, kind = self._apply_sqrt_product(U)
        if qu.is_complex():
            m = qu.shape[0]
            plan = self._plan(torch.float64 if qu.dtype == torch.complex128 else torch.float32, qu.device)
            y2 = plan.apply(torch.cat([qu.real, qu.imag], dim=0).contiguous())
            squ = torch.complex(y2[:m], y2[m:])
        else:
            squ = self._plan(qu.dtype, qu.device).apply(qu)
        return _wrap_result(kind, self.range, squ)

    def apply_adjoint(self, U, mu=None):                                   # :175-178
        """V @ get_matrix(), evaluated implicitly (scatter -> FWHT -> signs) instead of
        materialising the k x n matrix; same sqrt(n/k) scale as `_get_random_rows`."""
        torch = require_cuda()
        if isinstance(U, DeviceVectorArray):
            assert U in self.range                                         # :176
        v, kind = _unwrap(U)
        assert v.shape[1] == self.range.dim
        n = self.sqrt_product.range.dim
        k = self.range.dim
        plan = self._plan(torch.float64, v.device)
        if self._order_dev is None:
            self._order_dev = torch.from_numpy(np.argsort(plan.idx_host, kind="stable").astype(np.int32)).to(v.device)
        if v.is_complex():
            # the matrix is real: adjoint of the real and imaginary parts separately (the reference
            # multiplies by get_matrix().T, which is complex-safe)
            re = self.apply_adjoint(v.real.contiguous())
            im = self.apply_adjoint(v.imag.contiguous())
            if isinstance(self.sqrt_product, IdentityOperator):
                return _wrap_result(kind, self.source, torch.complex(re, im))
            raise TypeError("SrhtEmbedding.apply_adjoint: complex blocks need an identity sqrt_product")
        v = v.to(torch.float64).contiguous()
        m = v.shape[0]
        out = torch.empty((m, n), dtype=torch.float64, device=v.device)
        with torch.cuda.device(v.device):
            ws = dense._workspace(lib().rla_srht_adjoint_workspace_bytes(m, n), v.device)
            check(lib().rla_srht_adjoint_f64(plan.signs_dev.data_ptr(), n, plan.idx_dev.data_ptr(),
                                             self._order_dev.data_ptr(), k, v.data_ptr(), m, v.stride(0),
                                             self._rows_value(), out.data_ptr(), out.stride(0),
                                             ws.data_ptr(), ws.numel(), stream_ptr()), "rla_srht_adjoint_f64")
        Q = self.sqrt_product
        if not isinstance(Q, IdentityOperator):
            out = Q.apply_adjoint(DeviceVectorArray(Q.range, out)).data
        return _wrap_result(kind, self.source, out)

    def _compute_matrix(self):                                             # :182-186
        return self._adjoint_sqrt_product(self.get_random_matrix())

    def _compute_random_matrix(self):                                      # :189-192
        _warning_once("Computing explicit SRHT matrix")
        return self._get_random_rows(np.arange(self.range.dim))

    def _compute_random_matrix_device(self):
        _warning_once("Computing explicit SRHT matrix")
        return self._get_random_rows_device(np.arange(self.range.dim))

    def _rows_value(self):
        """|entry| of the explicit matrix exactly as the reference forms it:
        fl(fl(sqrt(n/k)) * fl(1 / fl(2**(d/2))))  (embeddings.py:207-208 with srht.py:36)."""
        n = self.sqrt_product.range.dim
        k = self.range.dim
        d = int(np.ceil(np.log2(n)))
        return float(np.sqrt(n / k) * (np.float64(1.0) / np.float64(2 ** (d / 2))))

    def _get_random_rows(self, indices):                                   # :195-209
        return self._get_random_rows_device(indices).cpu().numpy()

    def _get_random_rows_device(self, indices):
        """Rows `indices` of sqrt(n/k) H[s, :n] diag(r) as a CUDA tensor (closed form, bit-identical
        to the reference's one-hot -> fht_oop -> scale route)."""
        torch = require_cuda()
        n = self.sqrt_product.range.dim
        idx = np.asarray(indices, dtype=np.int64).reshape(-1)
        if idx.size and (idx.min() < -self.range.dim or idx.max() >= self.range.dim):
            raise IndexError(f"row index out of range for an embedding of dimension {self.range.dim}")   # sampling[ind], :206
        idx = np.where(idx < 0, idx + self.range.dim, idx)
        plan = self._plan(torch.float64, torch.device("cuda", torch.cuda.current_device()))
        rows = torch.as_tensor(idx, device=plan.device)
        out = torch.empty((len(rows), n), dtype=torch.float64, device=plan.device)
        if len(rows) == 0:
            return out
        with torch.cuda.device(plan.device):
            check(lib().rla_srht_rows_f64(plan.signs_dev.data_ptr(), n, plan.idx_dev.data_ptr(), rows.data_ptr(),
                                          len(rows), self._rows_value(), out.data_ptr(), out.stride(0),
                                          stream_ptr()), "rla_srht_rows_f64")
        return out


class _GaussianBase(RandomEmbedding):
    """What GaussianEmbedding and BlockGaussianEmbedding share: Theta as a table of row blocks.  Block b
    is rows 0 .. size_b - 1 of the stream of seed_b (`_block_seeds`, `_block_sizes`), scaled by
    1/sqrt(k): NumPy's RandomState(seed_b).normal draw in 'mt19937', the kernels' generator
    g(seed_b, row, col) in the Philox modes.  A GaussianEmbedding is the table of one block."""
    # GaussianEmbedding keeps its 'mt19937' draw on the device in `_theta_dev`; the block embedding
    # draws Theta again on every use, as the reference does (:430,452-461)
    _keeps_theta = False
    _theta_dev = None

    def compute_dim(self):                                                 # :234-247, :409-422
        return _gaussian_dim(self.options)

    @property
    def _rng_mode(self):
        mode = self.options.get("rng", "mt19937")
        assert mode in ("mt19937", "philox", "philox_rademacher", "philox_tf32"), f"unknown options['rng'] = {mode!r}"
        return mode

    def _kind(self):
        return {"philox_rademacher": dense.KIND_RADEMACHER, "philox_tf32": dense.KIND_NORMAL_TF32}.get(
            self._rng_mode, dense.KIND_NORMAL)

    def _tf32_ok(self):
        """Theta exact in TF32: float32 blocks can stay float32 (tcgen05 path, csrc/gemm32.cu)."""
        return self._rng_mode in ("philox_rademacher", "philox_tf32")

    @property
    def _scale(self):
        return 1.0 / np.sqrt(self.range.dim)

    def _table(self, blocks=None):
        """(seeds, sizes) of the listed blocks, all by default."""
        seeds, sizes = self._block_seeds, self._block_sizes
        if blocks is None:
            return seeds, sizes
        return [seeds[i] for i in blocks], [sizes[i] for i in blocks]

    # -- Theta
    def _theta_device(self, blocks=None, plan=None):
        """The stacked rows of the listed blocks (all by default) as a CUDA tensor.  'mt19937': NumPy's
        draw made on the device (csrc/mt19937.cu); given `plan`, a NormalPlan over the streams of the
        whole table, the one listed block is drawn from it.  Philox modes: what the kernels generate."""
        torch = require_cuda()
        seeds, sizes = self._table(blocks)
        n = self.sqrt_product.range.dim
        if self._rng_mode != "mt19937":
            parts = [dense.theta_materialize(s, self._kind(), self._scale, b, n) for s, b in zip(seeds, sizes)]
            return parts[0] if len(parts) == 1 else torch.cat(parts, dim=0)
        if self._keeps_theta:
            if self._theta_dev is None:
                self._theta_dev = mt19937.gaussian_matrix(seeds, sizes, n, self._scale)
            return self._theta_dev
        if plan is None:
            return mt19937.gaussian_matrix(seeds, sizes, n, self._scale)
        (i,), (b,) = blocks, sizes
        theta = torch.empty((b, n), dtype=torch.float64, device=plan.device)
        count = np.zeros(len(plan.counts), np.int64)
        count[i] = b * n
        if theta.numel():
            plan.execute(theta.view(-1), 0, count, 0, self._scale)
        return theta

    def _theta_host(self, blocks=None):
        """The same rows as a NumPy array.  'mt19937' is drawn by NumPy itself only where there is no
        CUDA device (an embedding built on the host); otherwise the device draw is downloaded, in
        bounded chunks unless it is kept anyway."""
        seeds, sizes = self._table(blocks)
        n = self.sqrt_product.range.dim
        if self._rng_mode == "mt19937" and not _cuda_available():
            return np.vstack([np.random.RandomState(s).normal(size=(b, n), loc=0, scale=self._scale)
                              for s, b in zip(seeds, sizes)])
        if self._rng_mode == "mt19937" and not self._keeps_theta:
            return mt19937.gaussian_matrix_host(seeds, sizes, n, self._scale)
        return self._theta_device(blocks).cpu().numpy()

    def _compute_random_matrix(self):                                      # :265-270, :444-450
        return self._theta_host()

    def _compute_random_matrix_device(self):
        return self._theta_device()

    def _compute_matrix(self):                                             # :258-262, :437-441
        gauss = self._random_matrix if self._random_matrix is not None else self._compute_random_matrix()
        return self._adjoint_sqrt_product(gauss)

    def update(self):
        self._theta_dev = None
        super().update()

    # -- the operator
    def apply(self, U, mu=None):                                           # :250-254, :425-434
        torch = require_cuda()
        qu, kind = self._apply_sqrt_product(U)
        if qu.is_complex():                                                # Theta is real: sketch both parts in one pass
            if not isinstance(self.sqrt_product, IdentityOperator):
                raise TypeError(f"{type(self).__name__}.apply: complex blocks need an identity sqrt_product")
            m = qu.shape[0]
            y2 = self.sketch_blocks(torch.cat([qu.real, qu.imag], dim=0).to(torch.float64).contiguous())
            return _wrap_result(kind, self.range, torch.complex(y2[:m], y2[m:]))
        if qu.dtype != torch.float64 and not (qu.dtype == torch.float32 and self._tf32_ok()):
            qu = qu.to(torch.float64)
        return _wrap_result(kind, self.range, self.sketch_blocks(qu))

    def sketch_blocks(self, V, blocks=None):
        """Sketch of the real CUDA block V (m, n), already Q U, by the listed row blocks of Theta (all by
        default), their columns side by side: `apply`'s result, or its columns of those blocks.  V is
        float64, or float32 where `_tf32_ok()`."""
        torch = require_cuda()
        seeds, sizes = self._block_seeds, self._block_sizes
        blocks = range(len(sizes)) if blocks is None else blocks
        plan = None
        if self._rng_mode == "mt19937" and not self._keeps_theta and len(blocks):
            # one plan (jump-ahead + acceptance count) for the streams of all blocks
            plan = mt19937.NormalPlan(seeds, [b * self.sqrt_product.range.dim for b in sizes], V.device)

        def sketch(i):                                                     # :430-432
            if self._rng_mode == "mt19937":
                return dense.gauss_apply_explicit(self._theta_device([i], plan).to(V.device), V)
            return dense.embed_apply_rng(seeds[i], self._kind(), self._scale, sizes[i], V)

        if len(blocks) == 1:
            return sketch(blocks[0])
        out = torch.empty((V.shape[0], sum(sizes[i] for i in blocks)), dtype=torch.float64, device=V.device)
        off = 0
        for i in blocks:
            out[:, off:off + sizes[i]].copy_(sketch(i))
            off += sizes[i]
        return out

    def apply_adjoint(self, U, mu=None):
        """V @ get_matrix()  (pyMOR's adjoint of the explicit matrix).  With a Theta or matrix already on
        the device: the product with get_matrix_device().  Otherwise V Theta, then Q^H: in the Philox
        modes one launch over all blocks with Theta generated in the kernel (csrc/adjoint_rng.cu); in
        'mt19937' one plan for all blocks, each block drawn in turn and V[:, block] Theta_b accumulated,
        so one block of Theta is held at a time."""
        from .reductor_ops import gemm_nn
        if self._theta_dev is not None or self._matrix_dev is not None:
            return self._gaussian_adjoint(U, lambda v: gemm_nn(v, self.get_matrix_device()), includes_sqrt_product=True)
        seeds, sizes = self._block_seeds, self._block_sizes
        n = self.sqrt_product.range.dim
        if self._rng_mode != "mt19937":
            starts = np.concatenate([[0], np.cumsum(sizes)])
            return self._gaussian_adjoint(
                U, lambda v: dense.embed_adjoint_rng(seeds, starts, self._kind(), self._scale, v, n))

        def product(v):
            plan = mt19937.NormalPlan(seeds, [b * n for b in sizes], v.device)
            out, off = None, 0
            for i, b in enumerate(sizes):
                w = gemm_nn(v[:, off:off + b], self._theta_device([i], plan))
                out = w if out is None else out.add_(w)
                off += b
            return out
        return self._gaussian_adjoint(U, product)

    def _gaussian_adjoint(self, U, product, includes_sqrt_product=False):
        """V @ get_matrix() from `product(v)`, a real CUDA block times the (k, n) matrix: Theta, then
        Q^H applied here, or the explicit matrix that already holds it (`includes_sqrt_product`).  Theta
        is real, so a complex block goes through as its real and imaginary parts; that needs an identity
        sqrt_product, as SrhtEmbedding.apply_adjoint does."""
        torch = require_cuda()
        if isinstance(U, DeviceVectorArray):
            assert U in self.range
        v, kind = _unwrap(U)
        assert v.shape[1] == self.range.dim
        Q = self.sqrt_product
        if v.is_complex():
            if not isinstance(Q, IdentityOperator):
                raise TypeError(f"{type(self).__name__}.apply_adjoint: complex blocks need an identity sqrt_product")
            m = v.shape[0]
            w2 = product(torch.cat([v.real, v.imag], dim=0).to(torch.float64))
            return _wrap_result(kind, self.source, torch.complex(w2[:m], w2[m:]))
        w = product(v.to(torch.float64))
        if not includes_sqrt_product and not isinstance(Q, IdentityOperator):
            w = Q.apply_adjoint(DeviceVectorArray(Q.range, w)).data
        return _wrap_result(kind, self.source, w)


class GaussianEmbedding(_GaussianBase):
    """rla/embeddings.py:214-270: the table of one block, its seed and k rows."""
    _keeps_theta = True

    def __init__(self, source=None, sqrt_product=None, options=None, range_id=None, _seed=None):
        assert not (source is None) or not (sqrt_product is None)          # :219
        self._init(locals())
        # the reference draws Theta eagerly (:230); on-the-fly modes never hold it
        if self._rng_mode == "mt19937":
            self._random_matrix = self._compute_random_matrix()

    @property
    def _block_seeds(self):
        return [self._seed]

    @property
    def _block_sizes(self):
        return [self.range.dim]

    def apply(self, U, mu=None):                                           # :250-254
        if _is_host_tensor(U) and isinstance(self.sqrt_product, IdentityOperator):
            # block in host memory: streamed by column slabs (on-the-fly Theta: accumulate per
            # slab at full GEMM height) or by groups of vectors (explicit Theta)
            torch = require_cuda()
            from .streaming import apply_streamed, apply_streamed_rng
            assert U.shape[1] == self.source.dim
            k = self.range.dim
            if self._rng_mode == "mt19937" or not (U.dtype == torch.float64 or (U.dtype == torch.float32 and self._tf32_ok())):
                return apply_streamed(self.apply, U, k, return_host=True)
            return apply_streamed_rng(self._seed, self._kind(), self._scale, k, U, return_host=True)
        return super().apply(U, mu)


class IdentityEmbedding(RandomEmbedding):
    """rla/embeddings.py:274-315."""

    def __init__(self, source=None, sqrt_product=None, options=None, range_id=None, _seed=None):
        assert not (source is None) or not (sqrt_product is None)          # :279
        self._init(locals(), seeded=False)
        self._random_matrix = self._compute_random_matrix()

    def compute_dim(self):                                                 # :291-292
        return self.source.dim

    def apply(self, U, mu=None):                                           # :294-295
        qu, kind = self._apply_sqrt_product(U)
        return _wrap_result(kind, self.range, qu)

    def apply_adjoint(self, U, mu=None):                                   # :297-299
        v, kind = _unwrap(U)
        Q = self.sqrt_product
        out = v if isinstance(Q, IdentityOperator) else Q.apply_adjoint(DeviceVectorArray(Q.range, v)).data
        return _wrap_result(kind, self.source, out)

    def update(self):                                                      # :301-302
        pass

    def _compute_matrix(self):                                             # :305-311
        if hasattr(self.sqrt_product, 'get_matrix'):
            return self.sqrt_product.get_matrix()
        vec = np.eye(self.source.dim)
        return self.apply(vec).T

    def _compute_random_matrix(self):                                      # :314-315
        from scipy.sparse import eye
        return eye(self.source.dim)


class EmbeddingVectorized(RandomEmbedding):
    """Sketch a whole block by vectorising it, then applying an inner embedding --
    rla/embeddings.py:318-369."""
    _init_args = ("source", "n_vectors", "embedding", "options", "range_id", "_seed")

    def __init__(self, source, n_vectors, embedding, options=None, range_id=None, _seed=None):
        if options is None:
            options = dict()
        if _seed is None:
            _seed = np.random.randint(0, high=2 ** 32 - 1)
        self._store_args(locals())
        self._seed = _seed
        self.source = source
        self.n_vectors = n_vectors
        self.embedding = embedding
        options = dict(options)
        options['range_dim'] = embedding.range.dim                          # :330
        self.options = FrozenDict(options)
        self.range = embedding.range
        self.range_id = range_id
        self._matrix = None
        self._matrix_dev = None
        self._random_matrix = None

    def compute_dim(self):                                                 # :337-350
        return _gaussian_dim(self.options)

    def apply(self, U, mu=None):                                           # :352-358
        if isinstance(U, DeviceVectorArray):
            assert U in self.source                                        # :353
        t, kind = _unwrap(U)
        assert t.shape[0] == self.n_vectors                                # :354
        x = t.T.contiguous().reshape(1, -1)                                # U.to_numpy().T.flatten()
        if kind == "va":
            return self.embedding.apply(self.embedding.source.from_numpy(x))
        return _wrap_result(kind, self.range, self.embedding.apply(x))

    def apply_adjoint(self, U, mu=None):                                   # :360-361
        pass

    def _compute_matrix(self):                                             # :364-365
        return self.embedding._compute_matrix()

    def _compute_random_matrix(self):                                      # :368-369
        return self.embedding._compute_random_matrix()


class BlockGaussianEmbedding(_GaussianBase):
    """rla/embeddings.py:373-467: Theta in row blocks of at most `max_block_size`
    rows, one seed per block."""

    def __init__(self, source=None, sqrt_product=None, options=None, range_id=None, _seed=None):
        assert not (source is None) or not (sqrt_product is None)          # :378
        assert options is not None and "max_block_size" in options.keys()  # :379
        self._init(locals())
        # block sizes (:393-400)
        max_block_size = options.get("max_block_size")
        m = self.range.dim // max_block_size
        r = self.range.dim % max_block_size
        block_sizes = [max_block_size for i in range(m)]
        if r > 0:
            block_sizes.append(r)
        self.block_sizes = block_sizes
        self.n_blocks = len(block_sizes)
        # block seeds (:402-407)
        block_seeds = np.random.RandomState(self._seed).randint(0, 2 ** 32 - 1, size=len(block_sizes))
        while len(np.unique(block_seeds)) < len(block_seeds):
            self._seed += 1
            block_seeds = np.random.RandomState(self._seed).randint(0, 2 ** 32 - 1, size=len(block_sizes))
        self.block_seeds = block_seeds

    @property
    def _block_seeds(self):
        return [int(s) for s in self.block_seeds]

    @property
    def _block_sizes(self):
        return self.block_sizes

    def _get_random_block(self, ind):                                      # :452-461
        return self._theta_host([ind])

    def get_block(self, ind):                                              # :463-467
        return self._adjoint_sqrt_product(self._get_random_block(ind))

    def get_block_device(self, ind):
        """Block `ind` of the U -> l2 matrix as a CUDA tensor (preconditioned_reductor.py:185-194)."""
        return self._adjoint_sqrt_product_device(self._theta_device([ind]))
