"""Extended-precision references shared by the exact-arithmetic tests of the kernels.

Products are split exactly into two doubles (Dekker's TwoProduct) and summed in np.longdouble
(the x87 80-bit format: a 64-bit mantissa and a 15-bit exponent), so a dot product of w terms is
off by at most ~ w 2^-64 sum |x_j y_j|, far below float64's unit roundoff."""
import numpy as np
import pytest

U_ROUND = 2.0 ** -53                                   # unit roundoff of float64
_SPLIT = 134217729.0                                   # 2^27 + 1


def gamma(k):
    """gamma_k = k u / (1 - k u) (Higham, Accuracy and Stability, section 3.1)."""
    k = np.asarray(k, dtype=np.float64)
    return k * U_ROUND / (1.0 - k * U_ROUND)


def require_longdouble():
    if np.finfo(np.longdouble).nmant < 63:
        pytest.skip("np.longdouble is not the 64-bit-mantissa extended format on this platform")


def two_product(a, b):
    """a * b = p + e exactly (Dekker's TwoProduct with Veltkamp's split; float64 arithmetic,
    no fused multiply-add).  Exact while no product or split part under- or overflows."""
    p = a * b
    c = _SPLIT * a
    ah = c - (c - a)
    al = a - ah
    c = _SPLIT * b
    bh = c - (c - b)
    bl = b - bh
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p, e


def exact_dots(X, Y, step=1 << 20):
    """S[r, c] = sum_j X[r, j] Y[c, j] and A[r, c] = sum_j |X[r, j]| |Y[c, j]| for finite float64
    X (rx, n) and Y (cy, n), both as np.longdouble (rx, cy).

    Each row of X is first scaled by a power of two (exact) so that its largest entry is near
    2^500: TwoProduct is then exact for entries of any magnitude, subnormal ones included, as long
    as a row spans less than ~2^1400 and |Y| stays within 2^-400 .. 2^400.  S is exact up to the
    rounding of the long-double sums; A carries the relative error of a float64 product of
    absolute values (at most gamma_n), which the tests cover by taking it times (1 + 2 gamma_n)."""
    require_longdouble()
    X = np.asarray(X, dtype=np.float64)
    Y = np.asarray(Y, dtype=np.float64)
    assert np.isfinite(X).all() and np.isfinite(Y).all(), "exact_dots takes finite operands only"
    ymax = np.abs(Y).max(initial=0.0)
    assert ymax < 2.0 ** 400, "Y too large for an exact split"
    rx, n = X.shape
    S = np.zeros((rx, Y.shape[0]), dtype=np.longdouble)
    A = np.zeros((rx, Y.shape[0]), dtype=np.longdouble)
    for r in range(rx):
        mx = np.abs(X[r]).max(initial=0.0)
        if mx == 0.0:
            continue
        sh = 500 - int(np.frexp(mx)[1])
        xs = np.ldexp(X[r], sh)
        assert np.array_equal(np.ldexp(xs, -sh), X[r]), "row scaling not exact"
        for j0 in range(0, n, step):
            x, y = xs[j0:j0 + step], Y[:, j0:j0 + step]
            p, e = two_product(x[None, :], y)
            tiny = (p != 0) & (np.abs(p) < 2.0 ** -960)
            assert not tiny.any(), "products too small for an exact TwoProduct"
            S[r] += p.astype(np.longdouble).sum(axis=1) + e.astype(np.longdouble).sum(axis=1)
            A[r] += (np.abs(y) @ np.abs(x)).astype(np.longdouble)
        S[r] = np.ldexp(S[r], -sh)                                          # exact: 15-bit exponent
        A[r] = np.ldexp(A[r], -sh)
    return S, A
