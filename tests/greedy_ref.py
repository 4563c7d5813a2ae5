"""NumPy / SciPy restatement of the weak greedy of rla4mor_b200.greedy.rb_greedy on host data.

Snapshots by direct spsolve; the sketch Theta taken as a (k, n) matrix (the embedding's
get_matrix_device(), or the identity); Gram-Schmidt of the sketched basis as pyMOR does it
(oracle.reductor_oracle.gram_schmidt, T = pinv(R)); Galerkin or least-squares reduced solves;
sketched residual norms with the identity online embedding; the same selection rule (largest
first, ties to the smallest row) and the same stopping tests."""
import numpy as np
from scipy.sparse.linalg import splu, spsolve

from oracle.reductor_oracle import gram_schmidt


def select(est, batch):
    """Row indices of the `batch` largest estimates, largest first, ties to the smallest row."""
    return [int(i) for i in np.argsort(-est, kind="stable")[:batch]]


def greedy_ref(terms, rhs, TH, TF, *, R=None, theta=None, projection="galerkin", batch=1, atol=None, rtol=None,
               max_extensions=None, max_basis_size=169, follow=None):
    """terms: Q sparse n x n; rhs: Pf (n,) vectors; TH (P, Q), TF (P, Pf); R: the inner product
    (sparse SPD, None = identity); theta: the (k, n) primal sketch (None = identity).  `follow`
    (a list of row lists) extends with those rows instead of the reference's own selection, so
    that the reference tracks another run while it still records what it would select.
    Returns a dict like rb_greedy's (max_errs, selected, basis_sizes, extensions, stop) plus
    `history`: per iteration est (P,), a (P, r), rb (r, n), own selection."""
    Q, n = len(terms), terms[0].shape[0]
    rinv = (lambda V: V) if R is None else (lambda V, lu=splu(R.tocsc()): lu.solve(V.T).T)
    sk = (lambda V: V) if theta is None else (lambda V: V @ theta.T)
    F = np.stack(rhs)
    RF = rinv(F)
    G = F @ RF.T                                                   # f_i^T R^-1 f_j: the empty ROM's estimator
    g = sk(RF)                                                     # (Pf, k)
    k = g.shape[1]
    rb, srb = np.zeros((0, n)), np.zeros((0, k))
    S = [np.zeros((0, k)) for _ in range(Q)]                       # Theta R^-1 A_q U as (r, k) row blocks
    out = dict(max_errs=[], selected=[], basis_sizes=[], extensions=0, history=[])
    while True:
        r = srb.shape[0]
        if r == 0:
            a = np.zeros((len(TH), 0))
            est = np.sqrt(np.maximum(np.einsum("pi,ij,pj->p", TF, G, TF), 0.0))
        else:
            a = np.empty((len(TH), r))
            for p in range(len(TH)):
                if projection == "galerkin":
                    A = sum(TH[p, q] * (srb @ S[q].T) for q in range(Q))
                    a[p] = np.linalg.solve(A, srb @ (TF[p] @ g))
                else:
                    M = sum(TH[p, q] * S[q].T for q in range(Q))
                    a[p] = np.linalg.lstsq(M, TF[p] @ g, rcond=None)[0]
            res = sum(TH[:, q:q + 1] * (a @ S[q]) for q in range(Q)) - TF @ g
            est = np.linalg.norm(res, axis=1)
        it = len(out["max_errs"])
        own = select(est, max(1, min(batch, max_basis_size - r)))
        out["history"].append(dict(est=est, a=a, rb=rb.copy(), own=own))
        out["max_errs"].append(float(est[own[0]]))
        out["basis_sizes"].append(r)
        if atol is not None and est[own[0]] <= atol:
            out["stop"] = "atol"
        elif rtol is not None and est[own[0]] <= rtol * out["max_errs"][0]:
            out["stop"] = "rtol"
        elif max_extensions is not None and out["extensions"] >= max_extensions:
            out["stop"] = "max_extensions"
        elif r >= max_basis_size:
            out["stop"] = "max_basis_size"
        if "stop" in out:
            return out
        sel = own if follow is None else list(follow[it])
        U = np.stack([spsolve(sum(TH[p, q] * terms[q] for q in range(Q)).tocsc(), TF[p] @ F) for p in sel])
        rb = np.concatenate([rb, U])
        srb = np.concatenate([srb, sk(U)])
        S = [np.concatenate([S[q], sk(rinv(np.asarray((terms[q] @ U.T).T)))]) for q in range(Q)]
        srb, Rg = gram_schmidt(srb, offset=r)
        T = np.linalg.pinv(Rg)
        S = [T.T @ Sq for Sq in S]
        rb = T.T @ rb
        out["selected"].append(sel)
        if srb.shape[0] == r:
            out["stop"] = "extension_failed"
            return out
        out["extensions"] += 1
