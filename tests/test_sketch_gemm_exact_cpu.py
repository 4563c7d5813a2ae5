"""The checks of tests/test_sketch_gemm_exact_gpu.py can fail: on the CPU, without a GPU.

A NumPy replay of the FP64 sketch GEMM's arithmetic (split-n chunks accumulated term by term,
partials summed in chunk order, then the scale) passes the componentwise bound and the 4x-NumPy
criterion; replays with one subtle mistake do not:
  * one term of relative size ~1e-14 dropped;
  * one chunk's partial rounded to float32;
  * the tail launch reading Theta rows from 0 instead of kc0;
  * the rows of a tile taken from the peer CTA of its cluster pair;
  * in a graded block, an error of 1e-10 in the smallest row, which the normwise comparison at
    1e-12 that the older GEMM tests use accepts.
The reference (exact_dots) is checked against rational arithmetic, and the mirror of the planner
against the set of 35 instantiations the GPU test expects to reach."""
from fractions import Fraction

import numpy as np
import pytest

from exact_ref import U_ROUND, exact_dots, two_product
from test_sketch_gemm_exact_gpu import (CASES, PRODUCTION, check_sampled, entry_errors, graded, instantiations,
                                        plan_gemm, sample_sets, subnormal_rows)


def replay(U, T, scale, kmain, kper, mutant=None, drop=None):
    """The arithmetic of sketch_gemm_kernel + gemm_reduce_kernel in float64: chunks of 16 kper
    columns of n, each accumulated term by term (product rounded, then added); the partials summed
    in chunk order; times scale.  Sketch columns [kmain, k) are the tail launch.  BM = 64 rows per
    tile."""
    m, n = U.shape
    k = T.shape[0]
    Tt = T.copy()
    if mutant == "tail_theta_from_row_0":
        Tt[kmain:] = T[:k - kmain]
    total = np.zeros((m, k))
    for c0 in range(0, n, 16 * kper):
        part = np.zeros((m, k))
        for j in range(c0, min(n, c0 + 16 * kper)):
            term = U[:, j, None] * Tt[None, :, j]
            if mutant == "drop_term" and j == drop[1]:
                term[drop[0]] = 0.0
            part += term
        if mutant == "float32_chunk" and c0 == 0:
            part = part.astype(np.float32).astype(np.float64)
        total += part
    y = scale * total
    if mutant == "rows_of_the_peer_cta":
        y[64:128] = y[0:64]
    return y


def verdict(got, U, T, scale):
    """(every entry within the bound, largest normalised error within 4x NumPy's)."""
    S, A = exact_dots(U, T)
    err, bound, norm = entry_errors(got, S, A, scale, U.shape[1])
    _, _, norm_np = entry_errors(scale * (U @ T.T), S, A, scale, U.shape[1])
    return bool(np.all(err <= bound)), bool(norm.max() <= 4 * max(norm_np.max(), U_ROUND))


def _theta(k, n, seed):
    return np.random.RandomState(seed).standard_normal((k, n)).astype(np.float32).astype(np.float64)


@pytest.mark.parametrize("m,k,n,kmain,kper,inp", [
    (40, 30, 200, 30, 13, "normal"),
    (130, 178, 700, 128, 4, "graded"),          # tail launch, 11 chunks, cancelling rows
    (70, 20, 15, 20, 1, "normal"),               # n < 16
    (20, 9, 1037, 9, 2, "graded"),               # 33 chunks, n odd
])
def test_replay_passes(m, k, n, kmain, kper, inp):
    rs = np.random.RandomState(m + n)
    T = _theta(k, n, n)
    U = graded(m, n, T, rs) if inp == "graded" else rs.standard_normal((m, n))
    if inp == "graded":
        U = subnormal_rows(U, [2], rs)
    got = replay(U, T, 0.3, kmain, kper)
    assert verdict(got, U, T, 0.3) == (True, True)
    rows, cols = sample_sets(m, k, n, 2, rs)
    check_sampled(got, U, T, 0.3, rows, cols, what="replay")
    check_sampled(got, U, T, 0.3, None, None, what="replay")


def test_replay_with_accumulate_passes():
    m, k, n = 50, 40, 300
    rs = np.random.RandomState(1)
    T, U, y0 = _theta(k, n, 2), rs.standard_normal((m, n)), rs.standard_normal((m, k))
    got = y0 + replay(U, T, 0.5, k, 3)
    check_sampled(got, U, T, 0.5, None, None, y0=y0, what="accumulate")
    with pytest.raises(AssertionError):                                    # prior values ignored
        check_sampled(got - y0, U, T, 0.5, None, None, y0=y0, what="accumulate")


def test_dropping_one_small_term_is_rejected():
    """u[7, 21] theta[i, 21] ~ 1e-14 sum_j |u_7j theta_ij| for the median i; the replay drops it."""
    m, k, n = 130, 40, 64
    rs = np.random.RandomState(2)
    T, U = _theta(k, n, 3), rs.standard_normal((m, n))
    U[7, 21] = 0.0
    a = np.abs(U[7]) @ np.abs(T).T
    U[7, 21] = 1e-14 * np.median(a / np.abs(T[:, 21]))
    assert verdict(replay(U, T, 1.0, k, 1), U, T, 1.0) == (True, True)
    assert verdict(replay(U, T, 1.0, k, 1, "drop_term", (7, 21)), U, T, 1.0) == (False, False)


@pytest.mark.parametrize("mutant", ["float32_chunk", "tail_theta_from_row_0", "rows_of_the_peer_cta"])
def test_mutants_are_rejected(mutant):
    m, k, n = 130, 178, 400
    rs = np.random.RandomState(3)
    T, U = _theta(k, n, 4), rs.standard_normal((m, n))
    got = replay(U, T, 0.7, 128, 5, mutant)
    assert verdict(got, U, T, 0.7) == (False, False)
    with pytest.raises(AssertionError):
        check_sampled(got, U, T, 0.7, *sample_sets(m, k, n, 2, rs), what=mutant)


def test_error_in_the_smallest_row_of_a_graded_block_is_rejected():
    """Rows scaled from 2^-300 to 2^300 (no cancellation, so that NumPy's product is a fair
    normwise yardstick): an error of 1e-10 sum |u||theta| in the smallest row passes the normwise
    comparison at 1e-12, not the componentwise bound."""
    m, k, n = 64, 50, 500
    rs = np.random.RandomState(5)
    T = _theta(k, n, 6)
    U = np.ldexp(rs.standard_normal((m, n)), np.round(np.linspace(-300, 300, m)).astype(int)[:, None])
    got = replay(U, T, 1.0, k, 4)
    assert verdict(got, U, T, 1.0) == (True, True)
    bad = got.copy()
    bad[0] += 1e-10 * (np.abs(U[0]) @ np.abs(T).T)
    ref = U @ T.T
    assert np.linalg.norm(bad - ref) / np.linalg.norm(ref) < 1e-12
    assert verdict(bad, U, T, 1.0) == (False, False)


def _frac_dot(x, y):
    return sum(Fraction(float(a)) * Fraction(float(b)) for a, b in zip(x, y))


def test_exact_dots_agree_with_fractions():
    """Random, cancelling (graded) and subnormal rows and one of 2^901: the long-double sums are
    within 2^-60 sum |u||theta| of the rational result."""
    rs = np.random.RandomState(7)
    n, k = 60, 5
    T = _theta(k, n, 8)
    U = np.concatenate([rs.standard_normal((2, n)), graded(4, n, T[:, :], rs)])
    U = subnormal_rows(np.concatenate([U, rs.standard_normal((2, n))]), [6], rs)
    U[7, 3] = 2.0 ** 901
    S, A = exact_dots(U, T)
    for r in range(U.shape[0]):
        for i in range(k):
            ex = _frac_dot(U[r], T[i])
            ab = sum(abs(Fraction(float(a)) * Fraction(float(b))) for a, b in zip(U[r], T[i]))
            assert abs(Fraction(*S[r, i].as_integer_ratio()) - ex) <= ab * Fraction(2) ** -60, (r, i)
            assert abs(Fraction(*A[r, i].as_integer_ratio()) - ab) <= ab * Fraction(2) ** -40, (r, i)


def test_two_product_is_exact():
    rs = np.random.RandomState(9)
    a = rs.standard_normal(1000) * 2.0 ** rs.randint(-400, 400, 1000)
    b = rs.standard_normal(1000) * 2.0 ** rs.randint(-400, 400, 1000)
    p, e = two_product(a, b)
    for x, y, pp, ee in zip(a, b, p, e):
        assert Fraction(float(pp)) + Fraction(float(ee)) == Fraction(float(x)) * Fraction(float(y))


def test_production_set_is_what_the_planner_selects():
    """Over m = 1..1100 and k = 1..300 (every tail width of both tile shapes and every pairing of
    m-tiles), the mirror of plan_gemm selects exactly PRODUCTION; the cases of the GPU test reach
    all of it."""
    seen = set()
    for m in range(1, 1101):
        for k in range(1, 301):
            for mode in (0, 1):
                seen |= instantiations(m, k, 1000, mode)
    seen |= {(wm, wn, ng, mode, cl) for (wm, wn, ng, m1, cl) in seen if m1 == 1 for mode in (2, 3)}
    assert seen == PRODUCTION and len(PRODUCTION) == 35
    reached = set().union(*(instantiations(m, k, n, mode) for mode, m, k, n, _, _ in CASES.values()))
    assert reached == PRODUCTION


def test_sample_sets_hold_the_tile_edges():
    m, k, n = 512, 202, 1500
    rows, cols = sample_sets(m, k, n, 1, np.random.RandomState(0))
    assert {0, 63, 64, 255, 256, 511} <= rows
    (_, kmain, main), (_, _, tail) = plan_gemm(m, k, n, True)
    assert (kmain, main["bn"], tail["ng"]) == (192, 64, 1)
    assert {0, 63, 64, 191, 192, 199, 200, 201} <= cols
