"""NumPy restatement of the restarted GMRES(m) of fom_solve.affine_gmres (csrc/affine_gmres.cu), one
right-hand side at a time, and the convection-diffusion-reaction test problem.

The iteration is written out step by step as the device performs it: left preconditioning by R^-1,
a primal basis v_i and its dual w_i = R v_i, classical Gram-Schmidt in the R inner product with one
DGKS re-orthogonalisation, Givens rotations, and a true-residual test at every cycle start."""
import numpy as np
import scipy.sparse as sp

EPS = np.finfo(np.float64).eps


def convection_diffusion_terms(nx):
    """[L, Dx, Dy, M] on the unit square with nx^2 interior nodes (h = 1 / (nx + 1)), Dirichlet
    boundary: L the 5-point Laplacian, Dx / Dy central first differences (skew-symmetric), M the
    identity.  A(theta) = theta_0 L + theta_1 Dx + theta_2 Dy + theta_3 M; R = L + M is SPD."""
    h = 1.0 / (nx + 1)
    e = np.ones(nx)
    I = sp.eye(nx, format="csr")
    T = sp.diags([-e[:-1], 2 * e, -e[:-1]], [-1, 0, 1], format="csr") / h ** 2
    D = sp.diags([-e[:-1], e[:-1]], [-1, 1], format="csr") / (2 * h)
    L = (sp.kron(I, T) + sp.kron(T, I)).tocsr()
    Dx = sp.kron(I, D).tocsr()
    Dy = sp.kron(D, I).tocsr()
    M = sp.eye(nx * nx, format="csr")
    return [L, Dx, Dy, M]


def gmres_ref(A, b, rinv, tol, m, maxiter, x0=None):
    """GMRES(m) for A x = b in the R inner product, rinv(y) = R^-1 y.  Returns (x, iters, resid,
    info) with the conventions of affine_gmres."""
    n = b.size
    x = np.zeros(n) if x0 is None else np.array(x0, dtype=np.float64)
    bn2 = float(b @ rinv(b))
    if not (np.isfinite(bn2) and bn2 >= 0):
        return np.full(n, np.nan), 0, np.nan, 2
    if bn2 == 0:
        return np.zeros(n), 0, 0.0, 0
    m = max(1, min(m, maxiter))
    it = 0
    while True:
        r = b - A @ x
        z = rinv(r)
        beta2 = float(r @ z)
        if not (np.isfinite(beta2) and beta2 >= 0):
            return np.full(n, np.nan), it, np.nan, 2
        resid = np.sqrt(beta2 / bn2)
        if beta2 <= tol * tol * bn2:
            return x, it, resid, 0
        if it >= maxiter:
            return x, it, resid, 1
        beta = np.sqrt(beta2)
        V, W = [z / beta], [r / beta]
        H = np.zeros((m + 1, m))
        cs, sn = np.zeros(m), np.zeros(m)
        g = np.zeros(m + 1)
        g[0] = beta
        for j in range(m):
            y = A @ V[j]
            z = rinv(y)
            nz2 = float(z @ y)
            h = np.array([z @ w for w in W])
            for k in range(j + 1):
                z = z - h[k] * V[k]
                y = y - h[k] * W[k]
            nzp2 = float(z @ y)
            if not (np.all(np.isfinite(h)) and np.isfinite(nz2) and nz2 >= 0 and np.isfinite(nzp2)):
                return np.full(n, np.nan), it, np.nan, 2
            if nzp2 < 0.5 * nz2:                                  # DGKS: a second pass
                h2 = np.array([z @ w for w in W])
                for k in range(j + 1):
                    z = z - h2[k] * V[k]
                    y = y - h2[k] * W[k]
                h = h + h2
                nzp2 = float(z @ y)
            if nzp2 < 0 and -nzp2 <= EPS * nz2:
                nzp2 = 0.0
            if not (np.all(np.isfinite(h)) and np.isfinite(nzp2) and nzp2 >= 0):
                return np.full(n, np.nan), it, np.nan, 2
            hn = np.sqrt(nzp2)
            H[:j + 1, j] = h
            for k in range(j):
                a, c = H[k, j], H[k + 1, j]
                H[k, j] = cs[k] * a + sn[k] * c
                H[k + 1, j] = -sn[k] * a + cs[k] * c
            rr = np.hypot(H[j, j], hn)
            if not (np.isfinite(rr) and rr > 0):
                return np.full(n, np.nan), it, np.nan, 2
            cs[j], sn[j] = H[j, j] / rr, hn / rr
            H[j, j] = rr
            g[j + 1] = -sn[j] * g[j]
            g[j] = cs[j] * g[j]
            it += 1
            if j + 1 == m or g[j + 1] ** 2 <= tol * tol * bn2 or hn == 0 or it >= maxiter:
                k = j + 1
                yc = np.zeros(k)
                for i in range(k - 1, -1, -1):
                    yc[i] = (g[i] - H[i, i + 1:k] @ yc[i + 1:k]) / H[i, i]
                for i in range(k):
                    x = x + yc[i] * V[i]
                break
            V.append(z / hn)
            W.append(y / hn)
