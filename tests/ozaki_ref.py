"""NumPy model of the int8 slice products of csrc/gemm_i8.cu (Ozaki scheme I): the same slicing of
both operands, exact integer slice products, and the kernel's FP64 flush order."""
import numpy as np

S = 8                 # slices per operand = accumulator levels
L = 1 << 14           # exponent block = flush period
PAIRS_PER_LEVEL_MAX = S


def block_exponent(u_block):
    """Smallest e with max |u| < 2^e (0 for an all-zero block)."""
    return int(np.frexp(np.max(np.abs(u_block)))[1]) if u_block.size else 0


def fix56(v, e):
    """trunc(|v| 2^(56 - e)) as int64, and the sign of v (|v| < 2^e)."""
    v = np.asarray(v, dtype=np.float64)
    return np.floor(np.ldexp(np.abs(v), 56 - e)).astype(np.int64), np.signbit(v)


def digits(v, e):
    """(S, ...) signed 7-bit digits of v 2^-e, most significant first."""
    M, neg = fix56(v, e)
    d = np.stack([(M >> (7 * (S - 1 - s))) & 127 for s in range(S)])
    return np.where(neg, -d, d)


def reconstruct(d, e):
    """sum_s d_s 2^(e - 7 (s + 1)), exactly (as a Python Fraction-free float sum of exact terms)."""
    from fractions import Fraction
    return [sum(Fraction(int(d[s, j])) * Fraction(2) ** (e - 7 * (s + 1)) for s in range(S)) for j in range(d.shape[1])]


def replay(u, theta, scale=1.0, y0=None):
    """The kernel's result for u (m, n) float64 and theta (k, n) (float64 copies of the FP32 draws),
    for inputs of at most three exponent blocks (every chunking of the split-n sums the block
    partials left to right then)."""
    m, n = u.shape
    nb = (n + L - 1) // L
    assert nb <= 3
    tdig = digits(theta, 3).astype(np.float64)               # (S, k, n)
    s = np.zeros((m, theta.shape[0]))
    for b in range(nb):
        sl = slice(b * L, min(n, (b + 1) * L))
        e = np.array([block_exponent(u[c, sl]) for c in range(m)])
        ud = np.stack([digits(u[c, sl], int(e[c])) for c in range(m)], axis=1).astype(np.float64)   # (S, m, len)
        t = None
        for lev in range(S - 1, -1, -1):
            # exact: |digit products| <= 2^14, at most 8 * 2^14 terms of a block -> < 2^31 in float64
            D = sum(ud[i] @ tdig[lev - i, :, sl].T for i in range(lev + 1))
            t = D if t is None else t * 2.0 ** -7 + D        # = fma(t, 2^-7, D): t 2^-7 is exact
        s = s + np.ldexp(t, (e - 11)[:, None])
    return scale * s if y0 is None else y0 + scale * s
