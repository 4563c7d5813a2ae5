"""B200 drop-in for the reference's `SketchedReductor` (mor/sketched_reductor.py:22-219) for
affinely decomposed stationary problems.

The reference drives every step through pyMOR's project / expand / contract rule engine; here
the same sequence of operations is a host-side class over device blocks, method by method:

    extend_basis(U)            :49-86    rb.append(U); output functional L U; Theta U;
                                         Theta R^-1 A_q U per affine term; Theta R^-1 f_p once;
                                         column concatenation; orthonormalize_basis(offset)
    orthonormalize_basis()     :90-118   Gram-Schmidt of the SKETCHED basis, T = pinv(R),
                                         rb <- T^T rb, S_q <- S_q T, output <- output T
    reduce(embedding, seed)    :121-141  empty basis -> _reduce_empty (:189-208)
                                         'galerkin'   -> _reduce_galerkin (:154-168)
                                         'minres'     -> _reduce_minres (:170-187, LsOperator)
    rom.solve / estimate_error / output   StationaryModel + ResidualErrorEstimator (:210-219)

Layout: a block of vectors is (len, dim).  A sketched term is kept as the (r, k) row block
V3 = Theta(R^-1 A_q U) -- the transpose of the k x r matrix of utilities/__init__.py:32-36 --
and exported in the reference's orientation by `sketched_operator_matrices()`.
Everything stays on the device; `fom` is an `AffineModel` (the stand-in for a pyMOR
StationaryModel with LincombOperators; `rla4mor_b200.pymor_adapter` builds one from a real one).
"""
import logging

import numpy as np
import torch

from . import reductor_ops as ops
from .embeddings import IdentityEmbedding
from .vectorarray import DeviceVectorArray, DeviceVectorSpace, MatrixOperator, as_device_block


def _coef(c, mu):
    """Affine coefficient: a number, or a callable / pyMOR-style functional of mu."""
    if hasattr(c, "evaluate"):
        return float(c.evaluate(mu))
    if callable(c):
        return float(c(mu))
    return float(c)


def _theta_rows(fom, theta_lhs, theta_rhs, mus, Q, Pf, dev):
    """theta_lhs (P, Q) and theta_rhs (P, Pf) as given (the fast path), or fom.thetas of every
    entry of `mus` stacked on the host and uploaded once; ValueError on a missing argument or a
    shape mismatch."""
    if mus is not None:
        if theta_lhs is not None or theta_rhs is not None:
            raise ValueError("give either mus= or theta_lhs= / theta_rhs=, not both")
        theta_lhs, theta_rhs = fom.thetas_batch(mus)
    elif theta_lhs is None or theta_rhs is None:
        raise ValueError("give mus= or both theta_lhs= and theta_rhs=")
    th = torch.as_tensor(theta_lhs, dtype=torch.float64, device=dev)
    tf = torch.as_tensor(theta_rhs, dtype=torch.float64, device=dev)
    if th.dim() != 2 or th.shape[1] != Q or tf.dim() != 2 or tf.shape != (th.shape[0], Pf):
        raise ValueError(f"theta_lhs / theta_rhs: expected shapes (P, {Q}) and (P, {Pf}), "
                         f"got {tuple(th.shape)} and {tuple(tf.shape)}")
    return th, tf


class AffineModel:
    """Stationary affine full-order model  sum_q thA_q(mu) A_q u = sum_p thf_p(mu) f_p,
    output L u.  operators: objects with `.apply(DeviceVectorArray)` (e.g. MatrixOperator);
    rhs: (n,) vectors; output: (n_out, n) matrix or None; coefficients default to 1."""

    def __init__(self, operators, rhs, operator_coefficients=None, rhs_coefficients=None, output=None,
                 solution_space=None):
        self.operators = list(operators)
        self.rhs = [as_device_block(f).reshape(1, -1).to(torch.float64) for f in rhs]
        self.operator_coefficients = list(operator_coefficients) if operator_coefficients is not None else [1.0] * len(self.operators)
        self.rhs_coefficients = list(rhs_coefficients) if rhs_coefficients is not None else [1.0] * len(self.rhs)
        assert len(self.operator_coefficients) == len(self.operators) and len(self.rhs_coefficients) == len(self.rhs)
        self.output = None if output is None else as_device_block(output).to(torch.float64)
        if solution_space is None:
            solution_space = getattr(self.operators[0], "source", None) or DeviceVectorSpace(self.rhs[0].shape[1])
        self.solution_space = solution_space
        self._affine = None                      # the terms as one device CSR pattern, built by the first solve

    def thetas(self, mu):
        return ([_coef(c, mu) for c in self.operator_coefficients], [_coef(c, mu) for c in self.rhs_coefficients])

    def thetas_batch(self, mus):
        """The affine coefficients of every mu, evaluated on the host: float64 arrays (P, Q), (P, Pf)."""
        Q, Pf = len(self.operator_coefficients), len(self.rhs_coefficients)
        th, tf = np.empty((len(mus), Q)), np.empty((len(mus), Pf))
        for p, mu in enumerate(mus):
            th[p], tf[p] = self.thetas(mu)
        return th, tf

    def solve(self, mu=None, theta_lhs=None, theta_rhs=None, *, preconditioner, tol=1e-10, maxiter=500, x0=None,
              check=True):
        """The full-order solution u(mu) (pyMOR's StationaryModel.solve) as a DeviceVectorArray of
        length 1 in solution_space: solve_batch of one mu (`mu=`, or theta_lhs (Q,) and theta_rhs
        (Pf,)); x0 is an optional initial guess of length 1."""
        one = lambda t: None if t is None else torch.as_tensor(t, dtype=torch.float64)[None]
        return self.solve_batch(None if mu is None else [mu], one(theta_lhs), one(theta_rhs),
                                preconditioner=preconditioner, tol=tol, maxiter=maxiter, x0=x0, check=check)

    def solve_batch(self, mus=None, theta_lhs=None, theta_rhs=None, *, preconditioner, tol=1e-10, maxiter=500,
                    x0=None, check=True):
        """Full-order solutions u(mu_p) of every mu, a DeviceVectorArray of length P in
        solution_space, by block preconditioned CG on the device (fom_solve.affine_cg: one affine
        SpMM, one application of `preconditioner` to the whole block and a few vector kernels per
        iteration).  The parameters are `mus=` or theta_lhs (P, Q) and theta_rhs (P, Pf), as for
        SketchedRom.solve_batch.  Every term must be a symmetric sparse MatrixOperator and A(mu) SPD;
        `preconditioner` is an SPD operator such as the reductor's `inverse_product`.  Row p stops when
        ||r_p||_{R^-1} <= tol ||b_p||_{R^-1}.  A row that does not converge within `maxiter`
        iterations or breaks down raises RlaError; with check=False it is returned as is (its last
        iterate, or NaN after a breakdown)."""
        from . import fom_solve
        dev = self.rhs[0].device if self.rhs else torch.device("cuda", torch.cuda.current_device())
        th, tf = _theta_rows(self, theta_lhs, theta_rhs, mus, len(self.operators), len(self.rhs), dev)
        n = self.solution_space.dim
        if x0 is not None:
            x0 = fom_solve.check_block(x0, th.shape[0], n, "x0", dev)
        if self._affine is None:
            self._affine = fom_solve.AffineCsr(self.operators)               # once per model
        X = fom_solve.affine_cg(self._affine, self.rhs, th, tf, preconditioner, tol=tol, maxiter=maxiter, x0=x0,
                                check=check)[0]
        return DeviceVectorArray(self.solution_space, X)


class SketchedReductor:
    def __init__(self, fom, *legacy, embedding_primal=None, embedding_online=None, product=None, inverse_product=None,
                 save_rb=True, orthonormalize=True, projection='galerkin', log_level=20):
        assert projection in ('galerkin', 'minres')                       # :25
        if isinstance(fom, (list, tuple)):
            # round-1 calling convention: SketchedReductor(operators, rhs, embedding_primal, ...)
            assert len(legacy) in (1, 2)
            fom = AffineModel(fom, legacy[0])
            if len(legacy) == 2:
                embedding_primal = legacy[1]
        else:
            assert not legacy
        self.fom = fom
        self.logger = logging.getLogger("rla4mor_b200.SketchedReductor")
        self.logger.setLevel(log_level)
        self.mu_basis = []
        self.product = product
        self.inverse_product = inverse_product
        self.space = fom.solution_space
        self.embedding_primal = embedding_primal if embedding_primal is not None else IdentityEmbedding(self.space)   # :35-36
        self.embedding_online = embedding_online if embedding_online is not None else \
            IdentityEmbedding(self.embedding_primal.range)                # :37-38
        self.save_rb, self.orthonormalize, self.projection = save_rb, orthonormalize, projection
        self.batch_bytes = 16 << 30                  # largest block handed to inverse_product in one application
        k = self.embedding_primal.range.dim
        dev = torch.device("cuda", torch.cuda.current_device())
        self.srb = torch.empty((0, k), dtype=torch.float64, device=dev)              # Theta U, (r, k)   :40
        self.rb = torch.empty((0, self.space.dim), dtype=torch.float64, device=dev)  #                   :41
        self.s_lhs = [torch.empty((0, k), dtype=torch.float64, device=dev) for _ in fom.operators]   # residual.operator
        self.s_rhs = None                                                             # residual.rhs: list of (k,)
        n_out = 0 if fom.output is None else fom.output.shape[0]
        self.output_functional = torch.empty((0, n_out), dtype=torch.float64, device=dev)   # (r, n_out) = (L U^T)^T
        self.rom = None

    # -- helpers
    @property
    def operators(self):
        return self.fom.operators

    def _rinv(self, V):
        if self.inverse_product is None:
            return V
        return self.inverse_product.apply(DeviceVectorArray(self.space, V)).data

    def _sketch(self, V):
        return self.embedding_primal.apply(V)

    def extend_basis(self, U, **kwargs):                                  # :49-86
        U = as_device_block(U).to(torch.float64)
        if self.save_rb:
            self.rb = torch.cat([self.rb, U], dim=0)                      # :51-52
        if self.fom.output is not None:                                   # :56-59  project(output, None, U), axis=1 concat
            self.output_functional = torch.cat([self.output_functional, ops.gram(U, self.fom.output)], dim=0)
        su = self._sketch(U)                                              # :63-64
        offset = self.srb.shape[0]
        self.srb = torch.cat([self.srb, su], dim=0)                       # :65
        Uva = DeviceVectorArray(self.space, U)
        images = [A.apply(Uva).data for A in self.fom.operators]          # :69-70 (one term per q after expand)
        first = self.s_rhs is None
        blocks = images + (list(self.fom.rhs) if first else [])           # :72-75: the right-hand sides join the first call
        # R^-1 of ALL affine terms in ONE application (the reference applies it term by term, :69,:73):
        # the columns are independent, so the result is the same bit for bit, but one sparse
        # triangular solve over Q m right-hand sides walks the factor once instead of Q times
        # (n = 10^6, Q = 4, m = 64: 37 ms instead of 4 x 13 ms; its short root levels are latency-bound)
        rows = [b.shape[0] for b in blocks]
        # (the concatenated block, the solver's transposed copy and the result live at the same time:
        # keep the block under a quarter of the free memory)
        limit = min(self.batch_bytes, torch.cuda.mem_get_info()[0] // 4)
        if self.inverse_product is not None and len(blocks) > 1 and sum(rows) * self.space.dim * 8 <= limit:
            solved = list(torch.split(self._rinv(torch.cat(blocks, dim=0)), rows, dim=0))
        else:
            solved = [self._rinv(b) for b in blocks]
        for q in range(len(images)):
            V3 = self._sketch(solved[q])
            self.s_lhs[q] = torch.cat([self.s_lhs[q], V3], dim=0)         # :77-79, concatenate axis=1 of k x m
        if first:
            self.s_rhs = [self._sketch(v).reshape(-1) for v in solved[len(images):]]
        if self.orthonormalize:
            self.orthonormalize_basis(offset=offset, **kwargs)            # :85-86

    def orthonormalize_basis(self, offset=0, T=None, return_T=False, **kwargs):   # :90-118
        if T is None:
            Q, R = ops.gram_schmidt(self.srb, offset=offset, **kwargs)    # :94
            T = ops.pinv_R(R)                                             # :95  (r x r')
        else:
            T = torch.as_tensor(T, dtype=torch.float64, device=self.srb.device)
            Q = ops.lincomb(T.T, self.srb)                                # :97
        if self.save_rb:
            self.rb = ops.lincomb(T.T, self.rb)                           # :99-100  rb.lincomb(T.T)
        self.srb = Q                                                      # :102
        # S_q (k x r) <- S_q T   <=>   V3 (r x k) <- T^T V3              # :104-108
        self.s_lhs = [ops.lincomb(T.T, V3) for V3 in self.s_lhs]
        if self.output_functional.shape[1]:
            self.output_functional = ops.lincomb(T.T, self.output_functional)      # :111
        return T if return_T else None

    def sketched_operator_matrices(self):
        """The k x r matrices the reference holds (utilities/__init__.py:32-36)."""
        return [V3.T.contiguous() for V3 in self.s_lhs]

    def reduce(self, embedding=None, seed=None, rom_log_level=30):        # :121-141
        if self.srb.shape[0] == 0:
            rom = self._reduce_empty()                                    # :123-124
        elif self.projection == 'galerkin':
            if embedding is None:
                embedding = self.embedding_online.with_(_seed=seed)       # :127-128
            rom = self._reduce_galerkin(embedding)
        else:
            if not hasattr(seed, '__len__'):
                seed = (seed, seed)                                       # :132-133
            if embedding is None or tuple(embedding) == (None, None):
                embedding = (self.embedding_online.with_(_seed=seed[0]),
                             self.embedding_online.with_(_seed=seed[1]))  # :134-136
            rom = self._reduce_minres(embedding)
        return rom

    def _sketch_residual(self, embedding=None):                           # :143-152
        if embedding is None:
            embedding = self.embedding_online
        lhs = [embedding.apply(V3) for V3 in self.s_lhs]                  # (r, k')  = (Gamma S_q)^T
        rhs = [embedding.apply(b.reshape(1, -1)).reshape(-1) for b in self.s_rhs]
        return lhs, rhs

    def _reduce_galerkin(self, embedding):                                # :154-168
        est = self._sketch_residual(embedding)
        lhs = [ops.gram(self.srb, V3) for V3 in self.s_lhs]               # :161  (Theta U)^H S_q  (r x r)
        rhs = [ops.gram(self.srb, b.reshape(1, -1)).reshape(-1) for b in self.s_rhs]   # :162
        return SketchedRom(self.fom, lhs, rhs, self.output_functional, est, least_squares=False)

    def _reduce_minres(self, embedding):                                  # :170-187
        lhs, rhs = self._sketch_residual(embedding[0])                    # :173-175  LsOperator(op.operator), op.rhs
        est = self._sketch_residual(embedding[1])                         # :178
        # StationaryModel wants the k' x r matrices: transpose the row blocks once
        return SketchedRom(self.fom, [M.T.contiguous() for M in lhs], rhs, self.output_functional, est,
                           least_squares=True)

    def _reduce_empty(self):                                              # :189-208
        """No basis yet: the ROM solution is empty and the estimator is the dual norm of the
        right-hand side, || f(mu) ||_{R^-1} (ResidualReductor with riesz_representatives, :195-198)."""
        F = torch.cat(self.fom.rhs, dim=0)                                # (P, n)
        G = ops.gram(F, self._rinv(F))                                    # f_p^T R^-1 f_q
        return EmptyRom(self.fom, G, self.output_functional.shape[1])


class SketchedRom:
    """StationaryModel(lhs, rhs, output_functional, error_estimator=ResidualErrorEstimator(...))
    of mor/sketched_reductor.py:165-166,181-182,210-219.  `solve(mu=...)` evaluates the FOM's
    affine coefficients; the round-1 form `solve(theta_lhs, theta_rhs)` takes them directly."""

    def __init__(self, fom, lhs, rhs, output, est, least_squares):
        self.fom, self.lhs, self.rhs, self.output_functional = fom, lhs, rhs, output
        self.est_lhs_rows, self.est_rhs = est                   # (r, k') row blocks, (k',) vectors
        self.est_lhs = [M.T.contiguous() for M in self.est_lhs_rows]       # k' x r, the reference's orientation
        self.least_squares = least_squares
        self._lhs_stack = self._rhs_stack = self._est_stack = None         # built by the first batch call
        self._ls_stack = None                                              # built by the first least-squares solve

    def _thetas(self, theta_lhs, theta_rhs, mu):
        if theta_lhs is None:
            theta_lhs, theta_rhs = self.fom.thetas(mu)
        return theta_lhs, theta_rhs

    def _lstsq_on_device(self):
        """Whether the least-squares solves take the batched QR kernel: r within its shared-memory
        limit and at least r rows (k' >= r; the stack has N = Q r + Pf >= r rows otherwise)."""
        return self._dim <= ops.rom_lstsq_batch_max_r() and self.lhs[0].shape[0] >= self._dim

    def _lstsq_stack(self):
        """The (N, k_eff) stack [M_0^T; ...; M_{Q-1}^T; g_0^T; ...] that reductor_ops.rom_lstsq_batch
        reads, built once.  When N = Q r + Pf is below k', the k' x N matrix Wc = [M_0 ... g_0 ...] is
        replaced by its triangular factor R (Wc = Q R, the stack becomes R^T, k_eff = N): ||Wc x|| =
        ||R x|| for every x, so every mu has the same minimiser, and the per-mu work no longer grows
        with k'."""
        if self._ls_stack is None:
            Wc = torch.cat(list(self.lhs) + [v.reshape(-1, 1) for v in self.rhs], dim=1)
            if Wc.shape[1] < Wc.shape[0]:
                Wc = torch.linalg.qr(Wc, mode="r").R
            self._ls_stack = Wc.T.contiguous()
        return self._ls_stack

    def solve(self, theta_lhs=None, theta_rhs=None, mu=None):
        """The reduced solution of one mu.  A least-squares ROM within the batched kernel's envelope
        solves it as solve_batch does (P = 1, the same bits); a rank-deficient A(mu) raises RlaError."""
        theta_lhs, theta_rhs = self._thetas(theta_lhs, theta_rhs, mu)
        if self.least_squares and self._lstsq_on_device():
            dev = self.output_functional.device
            th = torch.as_tensor(theta_lhs, dtype=torch.float64, device=dev).reshape(1, -1)
            tf = torch.as_tensor(theta_rhs, dtype=torch.float64, device=dev).reshape(1, -1)
            return ops.rom_lstsq_batch(self._lstsq_stack(), len(self.lhs), self._dim, th, tf)[0][0]
        A = sum(t * M for t, M in zip(theta_lhs, self.lhs))
        b = sum(t * v for t, v in zip(theta_rhs, self.rhs))
        if self.least_squares:                                   # LsOperator: apply_inverse(least_squares=True)
            return torch.linalg.lstsq(A, b.reshape(-1, 1)).solution.reshape(-1)
        return torch.linalg.solve(A, b)

    def estimate_error(self, a=None, theta_lhs=None, theta_rhs=None, mu=None):
        theta_lhs, theta_rhs = self._thetas(theta_lhs, theta_rhs, mu)
        if a is None:
            a = self.solve(theta_lhs, theta_rhs)
        return float(ops.residual_norm(self.est_lhs, theta_lhs, self.est_rhs, theta_rhs, a).cpu())

    def output(self, a=None, theta_lhs=None, theta_rhs=None, mu=None):
        if a is None:
            a = self.solve(theta_lhs, theta_rhs, mu)
        return self.output_functional.T @ a

    # -- the same three over a parameter set: row p of every argument and result belongs to mu_p
    @property
    def _dim(self):
        return self.est_lhs_rows[0].shape[0]                    # (r, k') for both projections

    def _thetas_batch(self, theta_lhs, theta_rhs, mus):
        return _theta_rows(self.fom, theta_lhs, theta_rhs, mus, len(self.est_lhs_rows), len(self.est_rhs),
                           self.output_functional.device)

    def _batch_a(self, a, th, tf):
        if a is None:
            return self.solve_batch(th, tf)
        a = torch.as_tensor(a, dtype=torch.float64, device=self.output_functional.device)
        if a.dim() != 2 or a.shape != (th.shape[0], self._dim):
            raise ValueError(f"a: expected shape ({th.shape[0]}, {self._dim}), got {tuple(a.shape)}")
        return a

    def solve_batch(self, theta_lhs=None, theta_rhs=None, mus=None, check=True):
        """Reduced solutions of every mu, (P, r): one launch of the batched LU solve
        (reductor_ops.rom_solve_batch) for a Galerkin ROM, of the batched Householder QR solve
        (reductor_ops.rom_lstsq_batch) for a least-squares (minres) ROM.  A singular or rank-deficient
        A(mu) raises RlaError naming how many and the first; with check=False its row is NaN instead.
        Outside the kernels' envelopes (Galerkin: r above rom_solve_batch_max_r(); least squares: r
        above rom_lstsq_batch_max_r() or k' < r) the per-mu `solve` runs in a loop, which is not
        accelerated."""
        th, tf = self._thetas_batch(theta_lhs, theta_rhs, mus)
        P, r = th.shape[0], self._dim
        if P == 0:
            return torch.empty((0, r), dtype=torch.float64, device=th.device)
        if self.least_squares and self._lstsq_on_device():
            return ops.rom_lstsq_batch(self._lstsq_stack(), len(self.lhs), r, th, tf, check=check)[0]
        if self.least_squares or r > ops.rom_solve_batch_max_r():
            return torch.stack([self.solve(th[p], tf[p]) for p in range(P)])
        if self._lhs_stack is None:
            self._lhs_stack = torch.stack(self.lhs).contiguous()
            self._rhs_stack = torch.stack(self.rhs).contiguous() if self.rhs else torch.empty((0, r), dtype=torch.float64,
                                                                                             device=th.device)
        return ops.rom_solve_batch(self._lhs_stack, self._rhs_stack, th, tf, check=check)[0]

    def estimate_error_batch(self, a=None, theta_lhs=None, theta_rhs=None, mus=None):
        """Sketched residual norms of every mu, (P,): one launch of the batched estimator
        (reductor_ops.residual_norm_batch) for Galerkin and least-squares ROMs alike; `a` (P, r)
        defaults to solve_batch.  A NaN row of `a` gives NaN."""
        th, tf = self._thetas_batch(theta_lhs, theta_rhs, mus)
        a = self._batch_a(a, th, tf)
        if th.shape[0] == 0:
            return torch.empty((0,), dtype=torch.float64, device=th.device)
        if self._est_stack is None:
            # [S_0^T; ...; S_{Q-1}^T; g_0^T; ...] (N, k'), rows padded to an even length for 16-byte copies
            kp = self.est_lhs_rows[0].shape[1] if self.est_lhs_rows else self.est_rhs[0].numel()
            rows = list(self.est_lhs_rows) + [g.reshape(1, -1) for g in self.est_rhs]
            N = sum(x.shape[0] for x in rows)
            W = torch.zeros((N, kp + (kp & 1)), dtype=torch.float64, device=th.device)
            W[:, :kp].copy_(torch.cat(rows, dim=0))
            self._est_stack = W[:, :kp]
        return ops.residual_norm_batch(self._est_stack, len(self.est_lhs_rows), self._dim, th, tf, a)

    def output_batch(self, a=None, theta_lhs=None, theta_rhs=None, mus=None):
        """Outputs of every mu, (P, n_out) = a @ output_functional; `a` defaults to solve_batch."""
        th, tf = self._thetas_batch(theta_lhs, theta_rhs, mus)
        return self._batch_a(a, th, tf) @ self.output_functional


class EmptyRom:
    """ROM of the empty basis (mor/sketched_reductor.py:189-208)."""

    def __init__(self, fom, gram_rhs, n_out):
        self.fom, self.G, self.n_out = fom, gram_rhs, n_out

    def solve(self, theta_lhs=None, theta_rhs=None, mu=None):
        return torch.empty((0,), dtype=torch.float64, device=self.G.device)

    def estimate_error(self, a=None, theta_lhs=None, theta_rhs=None, mu=None):
        if theta_rhs is None:
            _, theta_rhs = self.fom.thetas(mu)
        t = torch.as_tensor(np.asarray(theta_rhs, dtype=np.float64), device=self.G.device)
        return float(torch.sqrt(torch.clamp(t @ self.G @ t, min=0.0)).cpu())

    def output(self, a=None, theta_lhs=None, theta_rhs=None, mu=None):
        return torch.zeros((self.n_out,), dtype=torch.float64, device=self.G.device)

    def _theta_rhs_batch(self, theta_rhs, mus):
        if mus is not None:
            theta_rhs = self.fom.thetas_batch(mus)[1]
        elif theta_rhs is None:
            raise ValueError("give mus= or theta_rhs=")
        tf = torch.as_tensor(theta_rhs, dtype=torch.float64, device=self.G.device)
        if tf.dim() != 2 or tf.shape[1] != self.G.shape[0]:
            raise ValueError(f"theta_rhs: expected shape (P, {self.G.shape[0]}), got {tuple(tf.shape)}")
        return tf

    def solve_batch(self, theta_lhs=None, theta_rhs=None, mus=None, check=True):
        tf = self._theta_rhs_batch(theta_rhs, mus)
        return torch.empty((tf.shape[0], 0), dtype=torch.float64, device=self.G.device)

    def estimate_error_batch(self, a=None, theta_lhs=None, theta_rhs=None, mus=None):
        """sqrt(max(tf_p^T G tf_p, 0)) for every row p."""
        tf = self._theta_rhs_batch(theta_rhs, mus)
        return torch.sqrt(torch.clamp(((tf @ self.G) * tf).sum(dim=1), min=0.0))

    def output_batch(self, a=None, theta_lhs=None, theta_rhs=None, mus=None):
        tf = self._theta_rhs_batch(theta_rhs, mus)
        return torch.zeros((tf.shape[0], self.n_out), dtype=torch.float64, device=self.G.device)
