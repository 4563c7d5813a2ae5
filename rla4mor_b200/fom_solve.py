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
    one coefficient vector per row of the block.  Built once per model.  `symmetric` records whether
    every term is symmetric (to SYMMETRY_RTOL): affine_cg needs it, affine_gmres does not."""

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
        for q, M in enumerate(mats):
            if M.shape[0] != M.shape[1]:
                raise ValueError(f"affine term {q} is not square: shape {M.shape}")
        # GMRES takes any terms, CG symmetric ones only: the first asymmetry is kept for affine_cg's error
        try:
            check_symmetric(mats)
            self.asymmetry = None
        except ValueError as e:
            self.asymmetry = str(e)
        self.symmetric = self.asymmetry is None
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
    if not A.symmetric:
        raise ValueError(A.asymmetry)
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



# ---------------------------------------------------------------------------- GMRES
# The Krylov storage of affine_gmres, 2 m + 5 blocks (P, n), stays within this share of the free
# device memory (the rule of SketchedReductor.extend_basis); a larger P runs in chunks of rows.
KRYLOV_MEMORY_FRACTION = 0.25
# istate rows of csrc/affine_gmres.cu
_G_ITERS, _G_INFO, _G_MODE, _G_NCOL, _G_CYCLES, _G_ACT, _G_ARN, _G_REORTH, _G_RESTART, _G_END = range(10)
_G_MODE_RESTART = 2
_INFO_GMRES = {1: "not converged within maxiter",
               2: "breakdown: the preconditioner is not SPD or A(mu) is singular"}


def _check_restart(restart, who):
    if isinstance(restart, bool) or not isinstance(restart, (int, np.integer)) or restart < 1:
        raise ValueError(f"{who}: restart={restart!r} must be an integer >= 1")
    return int(restart)


def gmres_rows_per_chunk(n, m, P, free_bytes):
    """Rows of the block solved at once: the 2 m + 5 blocks of length n per row (V, W, x, b, U, y,
    z) and the reductions' workspace within KRYLOV_MEMORY_FRACTION of `free_bytes`; at least 1."""
    per_row = (2 * m + 5) * n * 8 + (m + 3) * ((n + 255) // 256) * 8
    return max(1, min(P, int(KRYLOV_MEMORY_FRACTION * free_bytes) // per_row))


def affine_gmres(operators, rhs, th, tf, preconditioner, tol=1e-10, restart=30, maxiter=500, x0=None, check=True):
    """Restarted GMRES(m) for  (sum_q th[p, q] A_q) x_p = sum_j tf[p, j] f_j,  p = 0 .. P-1, where
    A(mu) may be non-symmetric or indefinite (csrc/affine_gmres.cu).

    The arguments are those of affine_cg, plus `restart` = m, the Arnoldi steps of a cycle.  The
    iteration is GMRES on R^-1 A(mu) (left preconditioning by the SPD `preconditioner`) with the
    basis orthogonal in the R inner product, so that row p minimises ||b_p - A x_p||_{R^-1} over its
    Krylov space; a second Gram-Schmidt pass is taken when the first one loses more than half of
    the vector's R-norm (DGKS).  A cycle ends after m steps or when the Givens estimate of the
    residual reaches tol; the row converges only when the residual recomputed at the next cycle
    start satisfies ||r_p||_{R^-1} <= tol ||b_p||_{R^-1}.

    Returns (X (P, n), iters (P,) int32 -- Arnoldi steps, resid (P,) -- the true relative residual
    at the last cycle start, info (P,) int32) on the device: info 0 converged, 1 not converged
    within `maxiter` steps (the row keeps its last iterate), 2 breakdown (<r, R^-1 r> < 0 or
    <z, R z> < 0: the preconditioner is not SPD; a singular A(mu); a non-finite value; the row is
    NaN).  A row with b_p = 0 is 0 after 0 steps.  Rows are independent; the Krylov storage,
    2 m + 5 blocks of (rows, n), is kept within KRYLOV_MEMORY_FRACTION of the free device memory
    by solving the rows in chunks.  With `check`, a nonzero info raises RlaError."""
    X, iters, resid, info, _ = _affine_gmres(operators, rhs, th, tf, preconditioner, tol, restart, maxiter, x0)
    if check:
        _raise_failed("affine_gmres", _INFO_GMRES, info, resid, maxiter)
    return X, iters, resid, info


def _raise_failed(who, reasons, info, resid, maxiter):
    P = info.numel()
    bad = info != 0
    first = torch.argmax(bad.to(torch.int32))
    n_bad, first, why, res = torch.stack([bad.sum().to(torch.float64), first.to(torch.float64),
                                          info[first].to(torch.float64), resid[first]]).tolist()
    if n_bad:
        raise RlaError(f"{who}: {int(n_bad)} of {P} rows failed (first: row {int(first)}, {reasons[int(why)]}"
                       + (f", relative residual {res:.3g} after {maxiter} iterations)" if why == 1 else ")"))


def _affine_gmres(operators, rhs, th, tf, preconditioner, tol, restart, maxiter, x0):
    """affine_gmres without the check: (X, iters, resid, info, cycles)."""
    m = _check_restart(restart, "affine_gmres")
    if not tol >= 0.0:
        raise ValueError(f"affine_gmres: tol={tol} must be >= 0")
    if isinstance(maxiter, bool) or int(maxiter) != maxiter or maxiter < 0:
        raise ValueError(f"affine_gmres: maxiter={maxiter} must be a non-negative integer")
    maxiter = int(maxiter)
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
    th, ldth = ops._param_rows(th, P, Q, "affine_gmres: th", dev)
    tf, _ = ops._param_rows(tf, P, Pf, "affine_gmres: tf", dev)
    if x0 is not None:
        x0 = check_block(x0, P, n, "affine_gmres: x0", dev)
    m = max(1, min(m, maxiter))             # a cycle never outlasts maxiter: the same iterates, less storage
    iters = torch.zeros((P,), dtype=torch.int32, device=dev)
    info = torch.zeros((P,), dtype=torch.int32, device=dev)
    cycles = torch.zeros((P,), dtype=torch.int32, device=dev)
    resid = torch.zeros((P,), dtype=torch.float64, device=dev)
    X = torch.empty((P, n), dtype=torch.float64, device=dev)
    if P == 0:
        return X, iters, resid, info, cycles
    space = getattr(preconditioner, "source", A.source)

    def precond(V):
        Z = preconditioner.apply(DeviceVectorArray(space, V)).data
        if tuple(Z.shape) != tuple(V.shape):
            raise ValueError(f"affine_gmres: the preconditioner returned shape {tuple(Z.shape)} for {tuple(V.shape)}")
        return Z.to(torch.float64).contiguous()

    tf = tf.contiguous()
    with torch.cuda.device(dev):
        chunk = gmres_rows_per_chunk(n, m, P, torch.cuda.mem_get_info(dev)[0])
        for p0 in range(0, P, chunk):
            p1 = min(P, p0 + chunk)
            B = ops.gemm_nn(tf[p0:p1], F) if Pf else torch.zeros((p1 - p0, n), dtype=torch.float64, device=dev)
            out = _gmres_block(A, th[p0:], ldth, B, None if x0 is None else x0[p0:p1], precond, float(tol), m, maxiter)
            for dst, src in zip((X, iters, resid, info, cycles), out):
                dst[p0:p1] = src
    return X, iters, resid, info, cycles


def _gmres_block(A, th, ldth, B, X, precond, tol, m, maxiter):
    """GMRES(m) on the rows of B (P, n) with coefficients th (row stride ldth); X: the initial
    guess (modified in place) or None.  (X, iters, resid, info, cycles)."""
    L, s = lib(), stream_ptr
    P, n = B.shape
    dev = B.device
    f64 = dict(dtype=torch.float64, device=dev)
    ist = torch.zeros((10, P), dtype=torch.int32, device=dev)
    st = torch.zeros((5, P), **f64)                       # <b, R^-1 b>, resid, 1/h, ||z||_R^2 before / after
    hess = torch.zeros((L.rla_affine_gmres_hess_bytes(m, P) // 8,), **f64)
    V = torch.empty((P, m, n), **f64)
    W = torch.empty((P, m, n), **f64)
    U = torch.empty((P, n), **f64)
    ws = dense._workspace(L.rla_affine_gmres_workspace_bytes(n, m, P), dev)
    ws2 = dense._workspace(L.rla_affine_cg_workspace_bytes(n, P), dev)
    hb = torch.empty((P, m + 2), **f64)
    hb2 = torch.empty((P,), **f64)
    act, arn, reorth, rst = ist[_G_ACT], ist[_G_ARN], ist[_G_REORTH], ist[_G_RESTART]
    ist[_G_MODE].fill_(_G_MODE_RESTART)                  # every row starts with its true residual
    act.fill_(_LIVE)
    rst.fill_(_LIVE)
    if X is None:
        X = torch.zeros((P, n), **f64)
        Y = B.clone()                                     # r_0 = b
        Z = precond(Y)
        Zb = Z
    else:
        Y = torch.empty_like(X)
        _spmm(A, th, ldth, X, Y, act, None)
        _lib.check(L.rla_affine_gmres_residual_f64(Y.data_ptr(), B.data_ptr(), n, P, ist.data_ptr(), s()),
                   "rla_affine_gmres_residual_f64")
        ZZ = precond(torch.cat([Y, B], dim=0))            # R^-1 of r_0 and of b in one solve
        Z, Zb = ZZ[:P], ZZ[P:]
    _dots(B, Zb, n, None, ws2)
    _lib.check(L.rla_row_dot_sum_f64(ws2.data_ptr(), ws2.numel(), n, P, st[0].data_ptr(), s()), "rla_row_dot_sum_f64")

    def gram_schmidt_pass(mask_dots, mask_orth):
        _lib.check(L.rla_affine_gmres_dots_f64(Z.data_ptr(), Y.data_ptr(), W.data_ptr(), n, m, P, ist.data_ptr(),
                                               mask_dots.data_ptr(), ws.data_ptr(), ws.numel(), s()),
                   "rla_affine_gmres_dots_f64")
        _lib.check(L.rla_row_dot_sum_f64(ws.data_ptr(), ws.numel(), n, P * (m + 2), hb.data_ptr(), s()),
                   "rla_row_dot_sum_f64")
        _lib.check(L.rla_affine_gmres_orth_f64(Z.data_ptr(), Y.data_ptr(), V.data_ptr(), W.data_ptr(), hb.data_ptr(),
                                               n, m, P, ist.data_ptr(), mask_orth.data_ptr(), ws2.data_ptr(),
                                               ws2.numel(), s()), "rla_affine_gmres_orth_f64")
        _lib.check(L.rla_row_dot_sum_f64(ws2.data_ptr(), ws2.numel(), n, P, hb2.data_ptr(), s()),
                   "rla_row_dot_sum_f64")

    first = True
    while True:
        if not first:
            _spmm(A, th, ldth, U, Y, act, None)           # A v_j, or A x at a restart
            _lib.check(L.rla_affine_gmres_residual_f64(Y.data_ptr(), B.data_ptr(), n, P, ist.data_ptr(), s()),
                       "rla_affine_gmres_residual_f64")
            Z = precond(Y)
        first = False
        gram_schmidt_pass(act, arn)
        _lib.check(L.rla_affine_gmres_dgks_f64(hb.data_ptr(), hb2.data_ptr(), m, P, st.data_ptr(), ist.data_ptr(),
                                               hess.data_ptr(), s()), "rla_affine_gmres_dgks_f64")
        gram_schmidt_pass(reorth, reorth)
        _lib.check(L.rla_affine_gmres_step_f64(hb.data_ptr(), hb2.data_ptr(), m, P, tol, maxiter, st.data_ptr(),
                                               ist.data_ptr(), hess.data_ptr(), s()), "rla_affine_gmres_step_f64")
        _lib.check(L.rla_affine_gmres_normalize_f64(Z.data_ptr(), Y.data_ptr(), V.data_ptr(), W.data_ptr(),
                                                    U.data_ptr(), n, m, P, st.data_ptr(), ist.data_ptr(), s()),
                   "rla_affine_gmres_normalize_f64")
        _lib.check(L.rla_affine_gmres_update_f64(X.data_ptr(), U.data_ptr(), V.data_ptr(), n, m, P, ist.data_ptr(),
                                                 hess.data_ptr(), s()), "rla_affine_gmres_update_f64")
        if not bool((act == _LIVE).any()):                # the one device-to-host read per step
            break
    info = ist[_G_INFO].clone()
    X[info == 2] = float("nan")
    X[st[0] == 0] = 0.0                                   # b_p = 0: x_p = 0
    return X, ist[_G_ITERS].clone(), st[1].clone(), info, ist[_G_CYCLES].clone()
