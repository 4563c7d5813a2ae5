"""Host-side checks of the int8 slicing of csrc/gemm_i8.cu (model in ozaki_ref.py): exact where the
accuracy contract says so, and no int32 overflow for the block length and slice count it uses."""
from fractions import Fraction

import numpy as np

import ozaki_ref as oz


def test_int32_levels_cannot_overflow():
    # a level holds at most S pairs of digit products |d_i d_j| <= 127^2, over one block of L terms
    assert oz.PAIRS_PER_LEVEL_MAX * 127 * 127 * oz.L < 2 ** 31 - 1
    assert oz.S * 64 <= 512                                  # S levels x 64 columns of TMEM


def test_fp32_theta_is_exact_in_eight_slices():
    rs = np.random.RandomState(0)
    th = (rs.standard_normal(4000) * 2.0).astype(np.float32)
    th = np.concatenate([th, np.float32([7.99, -7.99, 2.0 ** -20, -(2.0 ** -29), 0.0, -0.0])]).astype(np.float64)
    th = th[np.abs(th) < 8]
    d = oz.digits(th, 3)
    assert np.abs(d).max() <= 127
    for j, r in enumerate(oz.reconstruct(d, 3)):
        assert r == Fraction(float(th[j]))                   # 24 significant bits >= 2^-30: exact


def test_fp64_block_slices_truncate_below_the_block_maximum():
    rs = np.random.RandomState(1)
    u = rs.standard_normal(300) * 2.0 ** rs.randint(-40, 40, 300)
    u[:3] = [2.0 ** -1070, -5e-324, 0.0]                     # subnormals and a zero
    e = oz.block_exponent(u)
    assert np.max(np.abs(u)) < 2.0 ** e <= 2 * np.max(np.abs(u))
    d = oz.digits(u, e)
    assert np.abs(d).max() <= 127
    rec = oz.reconstruct(d, e)
    for j in range(u.size):
        err = abs(Fraction(float(u[j])) - rec[j])
        assert err < Fraction(2) ** (e - 56)                 # truncation of |u| 2^-e after 56 bits
        assert np.sign(float(rec[j])) in (0.0, np.sign(u[j]))
    top = int(np.argmax(np.abs(u)))
    assert rec[top] == Fraction(float(u[top]))               # the block maximum keeps all 53 bits


def test_subnormal_block_is_exact():
    u = np.array([5e-324, -3 * 5e-324, 2.0 ** -1060, 0.0])
    e = oz.block_exponent(u)
    rec = oz.reconstruct(oz.digits(u, e), e)
    assert all(rec[j] == Fraction(float(u[j])) for j in range(u.size))


def test_replay_model_matches_an_exact_product_within_the_contract():
    rs = np.random.RandomState(2)
    m, k, n = 3, 5, 700
    u = rs.standard_normal((m, n)) * 2.0 ** rs.randint(-30, 30, (m, n))
    th = rs.standard_normal((k, n)).astype(np.float32).astype(np.float64)
    got = oz.replay(u, th)
    for c in range(m):
        for i in range(k):
            exact = sum(Fraction(float(a)) * Fraction(float(b)) for a, b in zip(u[c], th[i]))
            un, tn = np.linalg.norm(u[c]), np.linalg.norm(th[i])
            bound = 2.0 ** -53 * np.sqrt(n) * un * (tn / 4 + 15 * np.sqrt(n)) + 11 * 2.0 ** -52 * un * tn
            assert abs(float(Fraction(float(got[c, i])) - exact)) <= bound
