"""CPU checks of the device MT19937 Gaussian draw (csrc/mt19937.cu, csrc/mt19937.cuh) through its
host hooks: the F2 jump-ahead against NumPy's MT19937, a host replay of the segmented
count / scan / write algorithm against RandomState(seed).normal, and the extended log and its
midpoint flag against 60-digit decimal logarithms."""
import math
from decimal import Decimal, getcontext

import numpy as np
import pytest

from rla4mor_b200._lib import check, lib

W = 2.0 ** -5


def _key(seed):
    return np.ascontiguousarray(np.random.RandomState(seed).get_state(legacy=False)["state"]["key"], dtype=np.uint32)


def _jump(key, steps):
    out = np.empty(624, np.uint32)
    check(lib().rla_mt19937_jump_host(key.ctypes.data, int(steps), out.ctypes.data), "rla_mt19937_jump_host")
    return out


def _raw(key, count):
    g = np.random.MT19937()
    g.state = {"bit_generator": "MT19937", "state": {"key": key, "pos": 624}}
    return g.random_raw(count).astype(np.uint32)


@pytest.mark.parametrize("steps", [0, 1, 623, 624, 625, 10 ** 6 + 3, 3 * 624 * 512 + 8])
def test_jump_equals_random_raw(steps):
    key = _key(11)
    assert np.array_equal(_raw(_jump(key, steps), 40), _raw(key, steps + 40)[steps:])


def _attempts(words):
    n = len(words) // 4
    x1, x2, r2 = np.empty(n), np.empty(n), np.empty(n)
    acc = np.empty(n, np.int8)
    check(lib().rla_mt19937_attempts_host(np.ascontiguousarray(words).ctypes.data, n, x1.ctypes.data, x2.ctypes.data,
                                          r2.ctypes.data, acc.ctypes.data), "rla_mt19937_attempts_host")
    return x1, x2, r2, acc.astype(bool)


def _ext_log(x, w):
    x = np.ascontiguousarray(x, dtype=np.float64)
    hi, lo, fl = np.empty(len(x)), np.empty(len(x)), np.empty(len(x), np.int8)
    check(lib().rla_mt19937_ext_log_host(x.ctypes.data, len(x), float(w), hi.ctypes.data, lo.ctypes.data,
                                         fl.ctypes.data), "rla_mt19937_ext_log_host")
    return hi, lo, fl.astype(bool)


def _libm_log(x):
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty(len(x))
    check(lib().rla_libm_log_host(x.ctypes.data, len(x), out.ctypes.data), "rla_libm_log_host")
    return out


def _replay(seed, total, first, count, scale, seg_words=2 * 624):
    """The device algorithm on the host with tiny segments: start states by doubling jumps, per-segment
    accepted counts, exclusive scan, then the write of outputs [first, first + count)."""
    key = _key(seed)
    need = (total + 1) // 2
    states = [key]
    counts = []
    while sum(counts) < need:
        if len(states) <= len(counts):                      # next level of the doubling
            half = len(states)
            states += [_jump(states[j], seg_words * half) for j in range(half)]
        counts.append(int(_attempts(_raw(states[len(counts)], seg_words))[3].sum()))
    base = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.int64)
    out = np.full(count, np.nan)
    for s, b in enumerate(base):
        x1, x2, r2, acc = _attempts(_raw(states[s], seg_words))
        p = b + np.arange(int(acc.sum()))
        x1, x2, r2 = x1[acc], x2[acc], r2[acc]
        hi, _, flag = _ext_log(r2, W)
        lg = np.where(flag, _libm_log(r2), hi)
        f = np.sqrt(-2.0 * lg / r2)
        for o, x in ((2 * p, x2), (2 * p + 1, x1)):
            sel = (o >= first) & (o < first + count)
            out[o[sel] - first] = 0.0 + scale * (f[sel] * x[sel])
    return out


@pytest.mark.parametrize("seed", [0, 5, 12345, 2 ** 32 - 2])
def test_segmented_replay_equals_numpy(seed):
    scale = 1 / np.sqrt(7)
    for total in (0, 1, 2, 2001, 7 * 1001):
        ref = np.random.RandomState(seed).normal(size=total, loc=0, scale=scale)
        assert np.array_equal(_replay(seed, total, 0, total, scale), ref), total
    ref = np.random.RandomState(seed).normal(size=4001, loc=0, scale=scale)
    for first, count in ((1, 4000), (333, 1001), (4000, 1), (1247, 2)):
        assert np.array_equal(_replay(seed, 4001, first, count, scale), ref[first:first + count]), (first, count)


def _sample():
    rs = np.random.RandomState(2024)
    x = np.concatenate([rs.random_sample(600_000),
                        1 - rs.random_sample(300_000) * 2.0 ** -4,         # r2 -> 1: log1p(r2 - 1)
                        2.0 ** rs.uniform(-104, -1, 90_000),                # tiny r2 and every binade
                        1 - rs.randint(1, 5000, 5_000) * 2.0 ** -53,        # the last doubles below 1
                        2.0 ** -rs.randint(1, 105, 5_000) * (1 + rs.randint(-3, 4, 5_000) * 2.0 ** -52)])
    return x[(x > 0) & (x < 1)]


def test_extended_log_error_and_flags():
    """|hi + lo - log x| <= 2^-8 ulp on 10^6 arguments (60-digit decimal reference), and every argument
    where the C library's log is not the correctly rounded value is flagged."""
    getcontext().prec = 60
    x = _sample()
    assert len(x) >= 10 ** 6
    hi, lo, flag = _ext_log(x, W)
    libm = _libm_log(x)
    worst, misrounded = 0.0, 0
    for v, h, l, f, g in zip(x.tolist(), hi.tolist(), lo.tolist(), flag.tolist(), libm.tolist()):
        exact = Decimal(v).ln()
        err = abs(float((Decimal(h) + Decimal(l) - exact) / Decimal(math.ulp(h))))
        worst = max(worst, err)
        cr = float(exact)
        assert h == cr or f, v                                # hi is the correctly rounded log unless flagged
        if g != cr:
            misrounded += 1
            assert f, v
    assert worst <= 2.0 ** -8, worst
    assert misrounded > 0                                     # the fix-up has something to fix
    assert 0.04 < flag.mean() < 0.08


def test_flag_width_extremes_and_libm_batch():
    x = _sample()[:20000]
    assert _ext_log(x, 0.5)[2].all()
    assert not _ext_log(x, 0.0)[2].any()
    assert np.array_equal(_libm_log(x), np.array([math.log(v) for v in x.tolist()]))
