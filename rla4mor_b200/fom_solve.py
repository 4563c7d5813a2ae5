"""Full-order solves of the affine model over a block of parameter values: pyMOR's
`StationaryModel.solve` (-> `apply_inverse` of A(mu)) for P values mu_p at once.

    A(mu_p) u_p = b_p,   A(mu_p) = sum_q th[p, q] A_q,   b_p = sum_j tf[p, j] f_j

by block preconditioned CG (csrc/affine_cg.cu), one row of every (P, n) block per mu_p.  Every
A_q must be symmetric, and A(mu) positive definite.  The preconditioner is an SPD operator R
applied to the whole block, typically the reductor's `inverse_product` (the sparse LU of the inner
product, factored once).  With R = A(mu_bar) = sum_q A_q and SPD terms,
kappa(R^-1 A(mu)) <= max_q th_q(mu) / min_q th_q(mu), whatever the mesh.  The stopping test uses
the CG quantity <r, R^-1 r> = ||r||^2 in the dual norm of R, the norm the sketched error estimator
approximates: row p stops when ||r_p||_{R^-1} <= tol ||b_p||_{R^-1}.
"""
import numpy as np
import scipy.sparse as sp
import torch

from . import _lib, dense
from . import reductor_ops as ops
from ._lib import RlaError, lib, stream_ptr
from .vectorarray import DeviceVectorArray, MatrixOperator, as_device_block

# |A - A^T| <= SYMMETRY_RTOL max|A| entrywise: assembly such as D L D rounds the two triangles apart
SYMMETRY_RTOL = 1e-12
MAX_TERMS = 32                                 # coefficients of a row held in registers (csrc/affine_cg.cu)
_LIVE = 2                                      # istate mode of a row that is iterating
_INFO = {1: "not converged within maxiter", 2: "breakdown: A(mu) or the preconditioner is not SPD"}


def check_symmetric(matrices):
    """ValueError naming the first term that is not symmetric (CG needs A(mu) SPD)."""
    for q, A in enumerate(matrices):
        A = sp.csr_matrix(A)
        if A.shape[0] != A.shape[1]:
            raise ValueError(f"affine term {q} is not square: shape {A.shape}")
        scale = abs(A).max() if A.nnz else 0.0
        asym = abs(A - A.T).max() if A.nnz else 0.0
        if asym > SYMMETRY_RTOL * scale:
            raise ValueError(f"affine term {q} is not symmetric (max |A - A^T| = {asym:.3g}, max |A| = {scale:.3g}): "
                             "CG needs a symmetric positive definite A(mu)")


def union_pattern(matrices):
    """The Q sparse n x n terms on ONE CSR pattern, the union of theirs: (indptr int64 (n + 1),
    indices int32 (nnz), values float64 (Q, nnz)).  Columns are sorted within a row, every stored
    entry of a term (explicit zeros included) is copied exactly, and a term without an entry at a
    position gets 0 there."""
    csrs = []
    for A in matrices:
        A = sp.csr_matrix(A, dtype=np.float64, copy=True)
        A.sum_duplicates()                                   # canonical: sorted columns, one entry each
        csrs.append(A)
    if not csrs:
        raise ValueError("no affine terms")
    shape = csrs[0].shape
    if any(A.shape != shape for A in csrs):
        raise ValueError(f"affine terms of different shapes: {[A.shape for A in csrs]}")
    # the union pattern: sum of the terms' patterns with every stored entry set to 1 (never cancels)
    ones = [sp.csr_matrix((np.ones(A.nnz), A.indices, A.indptr), shape=shape) for A in csrs]
    U = ones[0]
    for B in ones[1:]:
        U = U + B
    U = sp.csr_matrix(U)
    U.sort_indices()
    n_cols = np.int64(shape[1])
    row_of = lambda A: np.repeat(np.arange(shape[0], dtype=np.int64), np.diff(A.indptr))
    keys = row_of(U) * n_cols + U.indices.astype(np.int64)           # ascending
    values = np.zeros((len(csrs), U.nnz), dtype=np.float64)
    for q, A in enumerate(csrs):
        pos = np.searchsorted(keys, row_of(A) * n_cols + A.indices.astype(np.int64))
        values[q, pos] = A.data
    return U.indptr.astype(np.int64), U.indices.astype(np.int32), values


class AffineCsr:
    """sum_q th_q A_q of sparse `MatrixOperator`s as one device CSR pattern (the union of the terms'
    patterns) with Q value arrays: the operator the affine SpMM of csrc/affine_cg.cu applies with
    one coefficient vector per row of the block.  Built once per model."""

    def __init__(self, operators):
        operators = list(operators)
        if not operators:
            raise ValueError("AffineCsr: no affine terms")
        for q, A in enumerate(operators):
            if not (isinstance(A, MatrixOperator) and A.sparse):
                raise ValueError(f"AffineCsr: affine term {q} ({type(A).__name__}) is not a sparse MatrixOperator")
        if len(operators) > MAX_TERMS:
            raise ValueError(f"AffineCsr: {len(operators)} affine terms, at most {MAX_TERMS} supported")
        mats = [A._host for A in operators]
        check_symmetric(mats)
        indptr, indices, values = union_pattern(mats)
        self.source = operators[0].source
        self.n, self.Q, self.nnz = int(mats[0].shape[0]), len(mats), int(indices.size)
        dev = operators[0].rowptr.device
        self.device = dev
        self.rowptr = torch.from_numpy(indptr).to(dev)
        self.col = torch.from_numpy(indices).to(dev)
        self.val = torch.from_numpy(values).to(dev)


def check_block(x, P, n, name, device):
    """A copy of the (P, n) block x (tensor, array or DeviceVectorArray) as a new contiguous float64
    tensor on `device`; ValueError on a shape mismatch, raised before anything is copied."""
    x = torch.as_tensor(x.data if isinstance(x, DeviceVectorArray) else x)
    if x.dim() != 2 or tuple(x.shape) != (P, n):
        raise ValueError(f"{name}: expected shape ({P}, {n}), got {tuple(x.shape)}")
    return torch.empty((P, n), dtype=torch.float64, device=device).copy_(x)


def affine_spmm(A, th, X, dots=False):
    """Y[p] = sum_q th[p, q] A_q X[p] for every row p of X (P, n), one kernel pass.  With `dots`,
    also <X_p, Y_p> per row (partial sums per 256-entry tile, added in tile order): (Y, d)."""
    X = torch.as_tensor(X.data if isinstance(X, DeviceVectorArray) else X)
    if X.dim() != 2 or X.shape[1] != A.n:
        raise ValueError(f"affine_spmm: X: expected shape (P, {A.n}), got {tuple(X.shape)}")
    P = int(X.shape[0])
    th, ldth = ops._param_rows(th, P, A.Q, "affine_spmm: th", A.device)
    X = X.to(device=A.device, dtype=torch.float64).contiguous()
    Y = torch.empty_like(X)
    d = torch.empty((P,), dtype=torch.float64, device=A.device)
    if P == 0:
        return (Y, d) if dots else Y
    with torch.cuda.device(A.device):
        ws = dense._workspace(lib().rla_affine_cg_workspace_bytes(A.n, P), A.device) if dots else None
        _spmm(A, th, ldth, X, Y, None, ws)
        if dots:
            _lib.check(lib().rla_row_dot_sum_f64(ws.data_ptr(), ws.numel(), A.n, P, d.data_ptr(), stream_ptr()),
                  "rla_row_dot_sum_f64")
    return (Y, d) if dots else Y


def _spmm(A, th, ldth, X, Y, mode, ws):
    _lib.check(lib().rla_affine_spmm_f64(A.rowptr.data_ptr(), A.col.data_ptr(), A.val.data_ptr(), A.nnz, A.Q, A.n,
                                    th.data_ptr(), ldth, X.data_ptr(), A.n, X.shape[0], Y.data_ptr(), A.n,
                                    None if mode is None else mode.data_ptr(),
                                    None if ws is None else ws.data_ptr(), 0 if ws is None else ws.numel(),
                                    stream_ptr()), "rla_affine_spmm_f64")


def _dots(a, b, n, mode, ws):
    _lib.check(lib().rla_row_dot_partials_f64(a.data_ptr(), n, b.data_ptr(), n, n, a.shape[0],
                                         None if mode is None else mode.data_ptr(), ws.data_ptr(), ws.numel(),
                                         stream_ptr()), "rla_row_dot_partials_f64")


def affine_cg(operators, rhs, th, tf, preconditioner, tol=1e-10, maxiter=500, x0=None, check=True):
    """Block preconditioned CG for  (sum_q th[p, q] A_q) x_p = sum_j tf[p, j] f_j,  p = 0 .. P-1.

    operators: the Q symmetric sparse `MatrixOperator`s (or their `AffineCsr`); rhs: the Pf
    right-hand sides f_j ((n,) vectors or one (Pf, n) block); th (P, Q), tf (P, Pf); preconditioner:
    an SPD operator with `.apply(DeviceVectorArray)` (e.g. the reductor's `InverseLuOperator`),
    applied to the whole block once per iteration; x0: optional (P, n) initial guess.

    Each row stops on its own when ||r_p||_{R^-1} <= tol ||b_p||_{R^-1}; its updates are masked
    from then on, so its iterates depend on its own data only.  A row with b_p = 0 is 0 after 0
    iterations.  Returns (X (P, n), iters (P,) int32, resid (P,), info (P,) int32) on the device,
    resid = ||r_p||_{R^-1} / ||b_p||_{R^-1} at the last iterate; info[p]: 0 converged, 1 not
    converged within `maxiter` (the row keeps its last iterate), 2 breakdown (<p, A p> <= 0 or
    <r, R^-1 r> < 0: A(mu) or the preconditioner is not SPD; the row is NaN).  With `check`, a
    nonzero info raises RlaError naming how many rows failed, the first one and why."""
    A = operators if isinstance(operators, AffineCsr) else AffineCsr(operators)
    n, Q, dev = A.n, A.Q, A.device
    th = torch.as_tensor(th)
    P = int(th.shape[0]) if th.dim() == 2 else -1
    if isinstance(rhs, torch.Tensor):
        F = rhs.to(device=dev, dtype=torch.float64).reshape(-1, n)
    else:
        F = torch.cat([as_device_block(f).to(torch.float64).reshape(-1, n) for f in rhs] +
                      [torch.empty((0, n), dtype=torch.float64, device=dev)], dim=0)
    Pf = int(F.shape[0])
    th, ldth = ops._param_rows(th, P, Q, "affine_cg: th", dev)
    tf, _ = ops._param_rows(tf, P, Pf, "affine_cg: tf", dev)
    if not tol >= 0.0:
        raise ValueError(f"affine_cg: tol={tol} must be >= 0")
    if int(maxiter) != maxiter or maxiter < 0:
        raise ValueError(f"affine_cg: maxiter={maxiter} must be a non-negative integer")
    maxiter = int(maxiter)
    if x0 is not None:
        x0 = check_block(x0, P, n, "affine_cg: x0", dev)
    iters = torch.zeros((P,), dtype=torch.int32, device=dev)
    info = torch.zeros((P,), dtype=torch.int32, device=dev)
    if P == 0:
        return (torch.empty((0, n), dtype=torch.float64, device=dev), iters,
                torch.empty((0,), dtype=torch.float64, device=dev), info)
    space = getattr(preconditioner, "source", A.source)

    def precond(V):
        Z = preconditioner.apply(DeviceVectorArray(space, V)).data
        if tuple(Z.shape) != tuple(V.shape):
            raise ValueError(f"affine_cg: the preconditioner returned shape {tuple(Z.shape)} for {tuple(V.shape)}")
        return Z.to(torch.float64).contiguous()

    with torch.cuda.device(dev):
        L, s = lib(), stream_ptr
        wsb = L.rla_affine_cg_workspace_bytes(n, P)
        ws = dense._workspace(wsb, dev)
        state = torch.zeros((5, P), dtype=torch.float64, device=dev)     # rho, rho_b, alpha, beta, resid
        istate = torch.zeros((3, P), dtype=torch.int32, device=dev)     # iterations, info, mode
        mode = istate[2]
        B = ops.gemm_nn(tf.contiguous(), F) if Pf else torch.zeros((P, n), dtype=torch.float64, device=dev)
        if x0 is None:
            X = torch.zeros((P, n), dtype=torch.float64, device=dev)
            R = B                                                         # r_0 = b: <b, R^-1 b> = rho_0
            Z = precond(R)
            _dots(R, Z, n, None, ws)
            ws_b = ws
        else:
            X = x0
            Qv = torch.empty_like(X)
            _spmm(A, th, ldth, X, Qv, None, None)
            R = B.clone()
            state[2].fill_(1.0)
            mode.fill_(_LIVE)
            _lib.check(L.rla_affine_cg_update_r_f64(R.data_ptr(), n, Qv.data_ptr(), n, n, P, state.data_ptr(),
                                                istate.data_ptr(), s()), "rla_affine_cg_update_r_f64")
            ZZ = precond(torch.cat([R, B], dim=0))                         # R^-1 of r_0 and of b in one solve
            Z = ZZ[:P]
            ws_b = dense._workspace(wsb, dev)
            _dots(R, Z, n, None, ws)
            _dots(B, ZZ[P:], n, None, ws_b)
        _lib.check(L.rla_affine_cg_start_f64(ws.data_ptr(), ws_b.data_ptr(), ws.numel(), n, P, float(tol), maxiter,
                                         state.data_ptr(), istate.data_ptr(), s()), "rla_affine_cg_start_f64")
        Pv = Z.clone()
        Qv = torch.empty_like(X)
        while bool((mode == _LIVE).any()):                               # the one device-to-host read per iteration
            _spmm(A, th, ldth, Pv, Qv, mode, ws)
            _lib.check(L.rla_affine_cg_alpha_f64(ws.data_ptr(), ws.numel(), n, P, state.data_ptr(), istate.data_ptr(), s()),
                   "rla_affine_cg_alpha_f64")
            _lib.check(L.rla_affine_cg_update_r_f64(R.data_ptr(), n, Qv.data_ptr(), n, n, P, state.data_ptr(),
                                                istate.data_ptr(), s()), "rla_affine_cg_update_r_f64")
            Z = precond(R)
            _dots(R, Z, n, mode, ws)
            _lib.check(L.rla_affine_cg_beta_f64(ws.data_ptr(), ws.numel(), n, P, float(tol), maxiter, state.data_ptr(),
                                            istate.data_ptr(), s()), "rla_affine_cg_beta_f64")
            _lib.check(L.rla_affine_cg_update_xp_f64(X.data_ptr(), n, Pv.data_ptr(), n, Z.data_ptr(), n, n, P,
                                                 state.data_ptr(), istate.data_ptr(), s()),
                   "rla_affine_cg_update_xp_f64")
        iters.copy_(istate[0])
        info.copy_(istate[1])
        X[info == 2] = float("nan")
        X[state[1] == 0] = 0.0                                            # b_p = 0: x_p = 0
        resid = state[4].clone()
    if check:
        bad = info != 0
        first = torch.argmax(bad.to(torch.int32))
        n_bad, first, why, res = torch.stack([bad.sum().to(torch.float64), first.to(torch.float64),
                                              info[first].to(torch.float64), resid[first]]).tolist()
        if n_bad:
            raise RlaError(f"affine_cg: {int(n_bad)} of {P} rows failed (first: row {int(first)}, {_INFO[int(why)]}"
                           + (f", relative residual {res:.3g} after {maxiter} iterations)" if why == 1 else ")"))
    return X, iters, resid, info

