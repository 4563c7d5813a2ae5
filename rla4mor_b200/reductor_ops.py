"""Device wrappers for the small operations around the sketch (csrc/reductor.cu):
CSR SpMM, V @ Theta, Gram matrices, Gram-Schmidt of the sketched basis, Jacobi SVD of a
k x m sketch and the sketched residual norm.  CUDA tensors in, CUDA tensors out."""
import ctypes

import numpy as np
import torch

from . import _lib, dense
from ._lib import RlaError, check, lib, stream_ptr


def _rows(x):
    return dense._rows(x)


def spmm_csr(rowptr, col, val, shape, u):
    """out[c, i] = sum_j A[i, j] u[c, j]  (A_q.apply(U), mor/sketched_reductor.py:69-70)."""
    u = _rows(u).to(torch.float64)
    n_rows, n_cols = shape
    assert u.shape[1] == n_cols
    m = u.shape[0]
    out = torch.empty((m, n_rows), dtype=torch.float64, device=u.device)
    if m == 0 or n_rows == 0:
        return out
    with torch.cuda.device(u.device):
        check(lib().rla_spmm_csr_f64(rowptr.data_ptr(), col.data_ptr(), val.data_ptr(), n_rows, n_cols,
                                     u.data_ptr(), m, dense._ld(u), out.data_ptr(), out.stride(0), stream_ptr()),
              "rla_spmm_csr_f64")
    return out


def gemm_nn(v, theta):
    """(m, k) @ (k, n) -> (m, n) with m, k small and n long: adjoints (V @ get_matrix()) and the
    basis updates of mor/sketched_reductor.py:97-108 (csrc/lincomb.cu: theta read once per 128
    rows of the result, result written once)."""
    v, theta = _rows(v).to(torch.float64), _rows(theta).to(torch.float64)
    m, k = v.shape
    assert theta.shape[0] == k
    n = theta.shape[1]
    out = torch.empty((m, n), dtype=torch.float64, device=v.device)
    if m == 0 or n == 0:
        return out
    if k == 0:
        return out.zero_()
    with torch.cuda.device(v.device):
        check(lib().rla_gemm_nn_f64(v.data_ptr(), m, k, dense._ld(v), theta.data_ptr(), n, dense._ld(theta),
                                    out.data_ptr(), out.stride(0), None, 0, stream_ptr()),
              "rla_gemm_nn_f64")
    return out


def lincomb(coefficients, rows):
    """pyMOR `VectorArray.lincomb`: rows of the result = coefficients (r', r) @ rows (r, n)
    (rb.lincomb(T.T), mor/sketched_reductor.py:99-100)."""
    return gemm_nn(coefficients, rows)


def gram(a, b):
    """G[i, j] = <a_i, b_j> for row blocks a (r, k), b (q, k): the reduced Galerkin
    matrices (Theta U)^H (Theta R^-1 A_q U) of mor/sketched_reductor.py:161-162."""
    return dense.gauss_apply_explicit(dense._tma_friendly(_rows(b).to(torch.float64)),
                                      dense._tma_friendly(_rows(a).to(torch.float64)))


def gram_schmidt(A, offset=0, atol=1e-13, rtol=1e-13, reiteration_threshold=9e-1):
    """pyMOR-style gram_schmidt(A, offset=offset, return_R=True) on the rows of A
    (mor/sketched_reductor.py:94).  Returns (Q, R) with dependent rows removed."""
    A = _rows(A).to(torch.float64).clone()
    r, k = A.shape
    R = torch.empty((r, r), dtype=torch.float64, device=A.device)
    flags = torch.empty((max(r, 1),), dtype=torch.int32, device=A.device)
    if r == 0:
        return A, R
    with torch.cuda.device(A.device):
        # many-CTA grid-synchronised kernel when the shape allows it (csrc/factor.cu), else one CTA
        ws = dense._workspace(lib().rla_gram_schmidt_workspace_bytes(r, k), A.device)
        check(lib().rla_gram_schmidt_ws_f64(A.data_ptr(), r, k, A.stride(0), int(offset), R.data_ptr(), flags.data_ptr(),
                                            float(atol), float(rtol), float(reiteration_threshold),
                                            ws.data_ptr(), ws.numel(), stream_ptr()),
              "rla_gram_schmidt_ws_f64")
        soff = lib().rla_gram_schmidt_status_offset(r, k)
    keep = flags[:r] == 0
    have_status = soff >= 0 and soff + 4 <= ws.numel()
    # ONE device-to-host read for both answers (number of removed rows, status word of the kernel)
    removed = (flags[:r] != 0).sum().to(torch.int32).view(1)
    word = ws[soff:soff + 4].view(torch.int32) if have_status else torch.zeros_like(removed)
    n_removed, status = torch.cat([removed, word]).tolist()
    all_kept = n_removed == 0
    if have_status and status != 0:
        # a CTA gave up waiting for another CTA's flag (pre-emption, debugger, shared GPU):
        # Q and R are only partly orthogonalised
        raise RlaError("gram_schmidt: the grid-synchronised kernel timed out waiting on a flag; result discarded")
    if not all_kept:
        A, R = A[keep], R[keep]
    return A, R


def pinv_R(R):
    """T = pinv(R) of the Gram-Schmidt factor (mor/sketched_reductor.py:95).  A square R (no row
    removed) is upper triangular with a positive diagonal: T = R^-1 by back substitution on the
    device; a rectangular R (rows removed) goes through the general pseudo-inverse."""
    if R.shape[0] != R.shape[1]:
        return torch.linalg.pinv(R)
    R = _rows(R).to(torch.float64)
    r = R.shape[0]
    T = torch.empty((r, r), dtype=torch.float64, device=R.device)
    if r == 0:
        return T
    with torch.cuda.device(R.device):
        check(lib().rla_trinv_upper_f64(R.data_ptr(), r, R.stride(0), T.data_ptr(), T.stride(0), stream_ptr()),
              "rla_trinv_upper_f64")
    return T


def _round_robin(m, keep_bye=False):
    """Circle-method schedule over m players (rounded up to even): (me - 1) rounds x (me / 2) pairs.
    The pair containing the dummy player is (-1, -1), or (p, -1) with keep_bye."""
    me = m + (m & 1)
    players = list(range(me))
    rounds = []
    for _ in range(me - 1):
        pairs = []
        for i in range(me // 2):
            p, q = players[i], players[me - 1 - i]
            if p >= m or q >= m:
                p, q = (min(p, q), -1) if keep_bye else (-1, -1)
            pairs.append((p, q))
        rounds.append(pairs)
        players = [players[0]] + [players[-1]] + players[1:-1]
    return np.asarray(rounds, dtype=np.int32).reshape(-1)


_PAIRS = {}


def svd_jacobi(S, want_v=False, max_sweeps=30, tol=None, block=True, cluster=True):
    """One-sided Jacobi SVD of the k x m sketch held as a row block S (m, k).
    Returns (U_rows (m, k) orthonormal rows, s (m,), V (m, m) or None), singular values
    sorted descending: S = (V^T diag(s) U_rows) in the row layout, i.e. the k x m matrix
    S^T = U_rows^T diag(s) V.

    Three kernels, in order of preference: the cluster-resident one (`cluster`; the whole
    block in the distributed shared memory of one thread-block cluster, csrc/jacobi_cluster.cu),
    the grid-synchronised block kernel (`block`; csrc/factor.cu) and the launch-per-round one."""
    A = _rows(S).to(torch.float64).clone()
    m, k = A.shape
    if tol is None:
        # rows p, q count as orthogonal when |<a_p, a_q>| <= tol |a_p| |a_q|; a length-k dot product carries
        # sqrt(k) * eps of rounding noise, below which rotations only chase noise (LAPACK xGESVJ: sqrt(m) * eps)
        tol = max(1.0, np.sqrt(k)) * 1.1102230246251565e-16
    s = torch.empty((m,), dtype=torch.float64, device=A.device)
    V = torch.empty((m, m), dtype=torch.float64, device=A.device) if want_v else None
    aligned = A.data_ptr() % 16 == 0 and A.stride(0) % 2 == 0
    C = lib().rla_svd_jacobi_cluster_size(k, m, 1 if want_v else 0) if (cluster and aligned) else 0
    B = lib().rla_svd_jacobi_block_rows(k, m, 1 if want_v else 0) if (block and aligned and not C) else 0
    if C:
        # one launch of ONE cluster: block pairs in distributed shared memory (csrc/jacobi_cluster.cu)
        scratch = torch.zeros((8,), dtype=torch.int32, device=A.device)
        with torch.cuda.device(A.device):
            check(lib().rla_svd_jacobi_cluster_f64(A.data_ptr(), k, m, A.stride(0), s.data_ptr(),
                                                   V.data_ptr() if want_v else None, scratch.data_ptr(),
                                                   int(max_sweeps), float(tol), stream_ptr()),
                  "rla_svd_jacobi_cluster_f64")
    elif B:
        # one persistent launch: block pairs in shared memory, grid barrier per block round (csrc/factor.cu)
        nblk = -(-m // B)
        key = ("blk", nblk, A.device.index)
        if key not in _PAIRS:
            _PAIRS[key] = torch.from_numpy(_round_robin(nblk, keep_bye=True)).to(A.device)
        scratch = torch.empty((lib().rla_svd_jacobi_block_scratch_ints(m, B, int(max_sweeps)),), dtype=torch.int32,
                              device=A.device)
        with torch.cuda.device(A.device):
            check(lib().rla_svd_jacobi_block_f64(A.data_ptr(), k, m, A.stride(0), s.data_ptr(),
                                                 V.data_ptr() if want_v else None, _PAIRS[key].data_ptr(), B,
                                                 scratch.data_ptr(), int(max_sweeps), float(tol), stream_ptr()),
                  "rla_svd_jacobi_block_f64")
    else:
        key = (m, A.device.index)
        if key not in _PAIRS:
            _PAIRS[key] = torch.from_numpy(_round_robin(m)).to(A.device)
        rot = torch.zeros((1,), dtype=torch.int32, device=A.device)
        done = ctypes.c_int(0)
        with torch.cuda.device(A.device):
            check(lib().rla_svd_jacobi_f64(A.data_ptr(), k, m, A.stride(0), s.data_ptr(),
                                           V.data_ptr() if want_v else None, _PAIRS[key].data_ptr(), rot.data_ptr(),
                                           int(max_sweeps), float(tol), ctypes.byref(done), stream_ptr()),
                  "rla_svd_jacobi_f64")
    order = torch.argsort(s, descending=True)
    if B or C:
        host = scratch[:8].cpu() if C else scratch[:3].cpu()    # one read: {sweeps, converged, timeout}[, phase kilo-cycles]
        svd_jacobi.last_phases = host[3:8].tolist() if C else None
        info = host[:3]
        if int(info[2]) != 0:
            raise RlaError("svd_jacobi: the block kernel timed out waiting on a block flag; result discarded")
        svd_jacobi.last_info = info
    s = s[order]
    A = A[order]
    U_rows = A / torch.clamp(s, min=torch.finfo(torch.float64).tiny).unsqueeze(1)
    return U_rows, s, (V[order] if want_v else None)


def residual_norm(S_terms, theta_lhs, b_terms, theta_rhs, a):
    """|| sum_q th_q S_q a - sum_p tr_p b_p ||_2 (mor/sketched_reductor.py:216-219).
    S_terms: list of (k, r) CUDA tensors; b_terms: list of (k,) tensors."""
    dev = a.device if isinstance(a, torch.Tensor) else torch.device("cuda", torch.cuda.current_device())
    Q = len(S_terms)
    S = torch.stack([t.to(torch.float64).contiguous() for t in S_terms]) if Q else torch.empty((0, 1, 0), dtype=torch.float64, device=dev)
    k = S.shape[1] if Q else (b_terms[0].numel() if b_terms else 1)
    r = S.shape[2] if Q else 0
    P = len(b_terms)
    b = torch.stack([t.to(torch.float64).reshape(-1) for t in b_terms]) if P else torch.empty((0, k), dtype=torch.float64, device=dev)
    th = torch.as_tensor(np.asarray(theta_lhs, dtype=np.float64), device=dev)
    tr = torch.as_tensor(np.asarray(theta_rhs, dtype=np.float64), device=dev)
    av = torch.as_tensor(a, dtype=torch.float64, device=dev).reshape(-1).contiguous()
    out = torch.empty((1,), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        check(lib().rla_residual_norm_f64(S.data_ptr(), Q, k, r, th.data_ptr(), av.data_ptr(), b.data_ptr(), P,
                                          tr.data_ptr(), out.data_ptr(), stream_ptr()), "rla_residual_norm_f64")
    return out


# ------------------------------------------------------------- ROM over a parameter set
def _param_rows(x, P, cols, name, device):
    """(P, cols) float64 CUDA rows with unit inner stride and its row stride; ValueError on a
    shape mismatch (raised before anything is copied or launched)."""
    x = torch.as_tensor(x, dtype=torch.float64)
    if x.dim() != 2 or tuple(x.shape) != (P, cols):
        raise ValueError(f"{name}: expected shape ({P}, {cols}), got {tuple(x.shape)}")
    x = x.to(device)
    if cols and (x.stride(1) != 1 or (P > 1 and x.stride(0) < cols)):
        x = x.contiguous()
    return x, (max(x.stride(0), cols) if P > 1 else cols)


def _require_cuda(dev, what):
    if dev.type != "cuda":
        raise ValueError(f"{what}: the ROM's data must be CUDA tensors")


def _stack(terms, shape, name):
    """A list of equally shaped tensors (or one stacked tensor) as one contiguous float64 tensor."""
    if isinstance(terms, torch.Tensor):
        t = terms
    else:
        terms = list(terms)
        t = torch.stack([torch.as_tensor(x).to(torch.float64) for x in terms]) if terms else torch.empty(shape)
    if tuple(t.shape) != tuple(shape):
        raise ValueError(f"{name}: expected shape {tuple(shape)}, got {tuple(t.shape)}")
    return t


def rom_solve_batch_max_r():
    """Largest reduced dimension r of rom_solve_batch (the r x (r + 1) system in one CTA's shared memory)."""
    return int(lib().rla_rom_solve_batch_max_r())


def rom_solve_batch(lhs, rhs, th, tf, check=True):
    """Reduced Galerkin solves  (sum_q th[p, q] A_q) a_p = sum_j tf[p, j] f_j  for every row p
    (StationaryModel.solve, mor/sketched_reductor.py:165-166, over a parameter set; csrc/rom_batch.cu).
    lhs: Q (r, r) matrices (list or (Q, r, r) tensor); rhs: Pf (r,) vectors (list or (Pf, r) tensor);
    th (P, Q), tf (P, Pf).  Returns (a (P, r), info (P,) int32): info[p] = i > 0 when U(i, i) of the
    LU factorisation with partial pivoting is exactly zero, and a_p is then NaN.  With `check`, any
    such row raises RlaError naming how many failed and the first one (one device-to-host read)."""
    Q = len(lhs)
    if Q == 0:
        raise ValueError("rom_solve_batch: no affine terms")
    r = int(lhs[0].shape[0])
    Pf = len(rhs)
    A = _stack(lhs, (Q, r, r), "rom_solve_batch: lhs")
    b = _stack(rhs, (Pf, r), "rom_solve_batch: rhs")
    th = torch.as_tensor(th)
    P = int(th.shape[0]) if th.dim() == 2 else -1
    if r < 1 or r > rom_solve_batch_max_r():
        raise ValueError(f"rom_solve_batch: r={r} outside 1 .. {rom_solve_batch_max_r()}")
    dev = A.device
    th, ldth = _param_rows(th, P, Q, "rom_solve_batch: th", dev)
    tf, ldtf = _param_rows(tf, P, Pf, "rom_solve_batch: tf", dev)
    a = torch.empty((P, r), dtype=torch.float64, device=dev)
    info = torch.zeros((P,), dtype=torch.int32, device=dev)
    if P == 0:
        return a, info
    _require_cuda(dev, "rom_solve_batch")
    A, b = A.to(torch.float64).contiguous(), b.to(device=dev, dtype=torch.float64).contiguous()
    with torch.cuda.device(dev):
        _lib.check(lib().rla_rom_solve_batch_f64(A.data_ptr(), Q, r, b.data_ptr() if Pf else None, Pf, th.data_ptr(), ldth,
                                             tf.data_ptr() if Pf else None, ldtf, P, a.data_ptr(), r, info.data_ptr(),
                                             stream_ptr()), "rla_rom_solve_batch_f64")
    if check:
        bad = info != 0
        n_bad, first = torch.stack([bad.sum(), torch.argmax(bad.to(torch.int32))]).tolist()
        if n_bad:
            raise RlaError(f"rom_solve_batch: {n_bad} of {P} reduced systems are singular "
                           f"(first: row {first}, U({int(info[first])}, {int(info[first])}) = 0)")
    return a, info


def rom_lstsq_batch_max_r():
    """Largest reduced dimension r of rom_lstsq_batch (R and one row panel in one CTA's shared memory)."""
    return int(lib().rla_rom_lstsq_batch_max_r())


def rom_lstsq_batch(W, Q, r, th, tf, check=True):
    """Reduced least-squares solves  a_p = argmin_a || sum_q th[p, q] M_q a - sum_j tf[p, j] g_j ||_2
    for every row p (the minres ROM's LsOperator solve, mor/sketched_reductor.py:170-187, over a
    parameter set; csrc/rom_batch.cu).  W: (Q r + Pf, k_eff) stack [M_0^T; ...; M_{Q-1}^T; g_0^T; ...]
    of the (k_eff, r) matrices M_q and (k_eff,) vectors g_j (unit inner stride, any row stride), with
    k_eff >= r; th (P, Q), tf (P, Pf).  Returns (a (P, r), info (P,) int32): info[p] = i > 0 when
    R(i, i) of the Householder QR is exactly zero, and a_p is then NaN.  With `check`, any such row
    raises RlaError naming how many failed and the first one (one device-to-host read)."""
    if (not isinstance(W, torch.Tensor) or W.dtype != torch.float64 or W.dim() != 2 or W.shape[0] < Q * r
            or (W.shape[1] > 1 and W.stride(1) != 1)):
        raise ValueError("rom_lstsq_batch: W must be a 2-D float64 tensor of Q r + Pf rows with unit inner stride")
    if Q < 1:
        raise ValueError("rom_lstsq_batch: no affine terms")
    if r < 1 or r > rom_lstsq_batch_max_r():
        raise ValueError(f"rom_lstsq_batch: r={r} outside 1 .. {rom_lstsq_batch_max_r()}")
    Pf, ke = int(W.shape[0]) - Q * r, int(W.shape[1])
    if ke < r:
        raise ValueError(f"rom_lstsq_batch: k_eff={ke} < r={r}: the reduced systems are underdetermined")
    th = torch.as_tensor(th)
    P = int(th.shape[0]) if th.dim() == 2 else -1
    dev = W.device
    th, ldth = _param_rows(th, P, Q, "rom_lstsq_batch: th", dev)
    tf, ldtf = _param_rows(tf, P, Pf, "rom_lstsq_batch: tf", dev)
    a = torch.empty((P, r), dtype=torch.float64, device=dev)
    info = torch.zeros((P,), dtype=torch.int32, device=dev)
    if P == 0:
        return a, info
    _require_cuda(dev, "rom_lstsq_batch")
    ldw = W.stride(0) if W.shape[0] > 1 else ke
    with torch.cuda.device(dev):
        _lib.check(lib().rla_rom_lstsq_batch_f64(W.data_ptr(), ldw, Q, r, Pf, ke, th.data_ptr(), ldth,
                                             tf.data_ptr() if Pf else None, ldtf, P, a.data_ptr(), r,
                                             info.data_ptr(), stream_ptr()), "rla_rom_lstsq_batch_f64")
    if check:
        bad = info != 0
        first = torch.argmax(bad.to(torch.int32))
        n_bad, first, i = torch.stack([bad.sum(), first, info[first].to(torch.int64)]).tolist()
        if n_bad:
            raise RlaError(f"rom_lstsq_batch: {n_bad} of {P} reduced systems are rank-deficient "
                           f"(first: row {first}, R({i}, {i}) = 0)")
    return a, info


def residual_norm_batch_workspace_bytes(P, kp):
    """Scratch of residual_norm_batch: one partial sum per row and 128-column tile of the k' sketch."""
    return int(lib().rla_residual_norm_batch_workspace_bytes(int(P), int(kp)))


def residual_norm_batch(W, Q, r, th, tf, a):
    """est[p] = || sum_q th[p, q] S_q a_p - sum_j tf[p, j] g_j ||_2 for every row p
    (ResidualErrorEstimator.estimate_error, mor/sketched_reductor.py:216-219, over a parameter set;
    csrc/rom_batch.cu).  W: (Q r + Pf, k') stack of the (r, k') row blocks S_q^T and the vectors g_j
    (unit inner stride, any row stride); th (P, Q), tf (P, Pf), a (P, r).  Returns (P,)."""
    if (not isinstance(W, torch.Tensor) or W.dtype != torch.float64 or W.dim() != 2 or W.shape[0] < Q * r
            or W.stride(1) != 1):
        raise ValueError("residual_norm_batch: W must be a 2-D float64 tensor of Q r + Pf rows with unit inner stride")
    Pf = int(W.shape[0]) - Q * r
    kp = int(W.shape[1])
    a = torch.as_tensor(a)
    P = int(a.shape[0]) if a.dim() == 2 else -1
    if kp < 1:
        raise ValueError("residual_norm_batch: empty sketch dimension")
    dev = W.device
    a, lda = _param_rows(a, P, r, "residual_norm_batch: a", dev)
    th, ldth = _param_rows(th, P, Q, "residual_norm_batch: th", dev)
    tf, ldtf = _param_rows(tf, P, Pf, "residual_norm_batch: tf", dev)
    est = torch.empty((P,), dtype=torch.float64, device=dev)
    if P == 0:
        return est
    _require_cuda(dev, "residual_norm_batch")
    ldw = W.stride(0) if W.shape[0] > 1 else kp
    with torch.cuda.device(dev):
        ws = dense._workspace(residual_norm_batch_workspace_bytes(P, kp), dev)
        _lib.check(lib().rla_residual_norm_batch_f64(W.data_ptr(), ldw, Q, r, Pf, kp, th.data_ptr() if Q else None, ldth,
                                                 tf.data_ptr() if Pf else None, ldtf, a.data_ptr() if r else None, lda,
                                                 P, est.data_ptr(), ws.data_ptr(), ws.numel(), stream_ptr()),
               "rla_residual_norm_batch_f64")
    return est
