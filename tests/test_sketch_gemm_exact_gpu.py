"""The FP64 sketch GEMM (csrc/gemm.cu: sketch_gemm_kernel<WM, WN, NG, MODE, CL> and
gemm_reduce_kernel) against an extended-precision reference, in every instantiation the planner
selects for production shapes.

The kernel computes y_ci = scale * sum_j u_cj theta_ij with MODE 0 (Theta explicit,
`gauss_apply_explicit`), 2 (Rademacher Theta generated in the kernel) and 1 / 3 (the FP32 normals of
kinds 0 / 2: float64 blocks that the int8 router of gemm_i8.cu hands back because they hold a
non-finite entry or one >= 2^900).  A normwise comparison with NumPy at 1e-12 cannot see an error in
one tile or in a row of small norm; the checks here are per entry:
  * |yhat - y| <= gamma_L |scale| sum_j |u_cj| |theta_ij| + L 2^-1074 with L = n + ceil(n / 16) + 2:
    whatever the split of n into chunks, every product goes through at most n roundings inside its
    chunk (DMMA accumulation), ceil(n / 16) in the chunk sum of the reduce and one in the scale;
    the second term covers the underflow of each of those L roundings.  With accumulate=True one
    more rounding: (1 + u) times that plus u (|y0| + |scale| sum |u||theta|);
  * the largest normalised error |yhat - y| / (|scale| sum |u||theta|) is at most 4x that of NumPy's
    float64 product of the same operands (or of u = 2^-53 when NumPy's is smaller);
  * every byte of the output buffer outside the (m, k) window is unchanged, the operands sit in
    buffers whose padding columns and trailing rows hold NaN, and two calls give the same bits.
y is exact_dots of tests/exact_ref.py (TwoProduct and long-double sums); generated Theta comes from
`dense.theta_materialize`, bit-identical to the kernel's.  Kernel names are recorded with
torch.profiler: the cases together reach all of PRODUCTION, each exactly what the Python mirror of
the planner below predicts.  tests/test_sketch_gemm_exact_cpu.py shows that the checks reject
subtly wrong replays of the kernel's arithmetic.
"""
import functools
import re
import zlib
from fractions import Fraction

import numpy as np
import pytest

from exact_ref import U_ROUND, exact_dots, gamma

pytestmark = pytest.mark.gpu

# ---------------------------------------------------------------- mirror of the planner of gemm.cu

GK = 16
WAVES = 24                                           # RLA_GEMM_WAVES default
KIND_OF_MODE = {1: 0, 2: 1, 3: 2}                    # MODE of the kernel -> kind of embed_apply_rng


def choose_wm(m, rng):
    if m <= 64:
        return 1
    pad2, pad4 = -(-m // 128) * 128, -(-m // 256) * 256
    if not rng or pad2 < pad4:
        return 2
    pair4, pair2 = (pad4 // 256) % 2 == 0, (pad2 // 128) % 2 == 0
    return 4 if (pair4 or not pair2) else 2


def plan_range(m, kcols, n, rng, ng, pairs, sms=148):
    wm = choose_wm(m, rng)
    wn = 8 // wm
    ng = 4 if wm == 1 else ng
    bm, bn = 64 * wm, 8 * wn * ng
    mtiles, ntiles = -(-m // bm), -(-kcols // bn)
    cl = 2 if (rng and pairs and wm >= 2 and mtiles % 2 == 0) else 1
    nk16 = -(-n // GK)
    tiles = mtiles * ntiles
    cmax = max(1, min(max(1, nk16 // 32), -(-sms * WAVES // tiles)))
    chunks, best = cmax, -1.0
    for c in range(max(1, cmax // 4), cmax + 1):
        kper = -(-nk16 // c)
        waves = -(-(-(-nk16 // kper) * tiles) // sms)
        eff = nk16 * tiles / (waves * sms * kper)
        if eff > best + 2e-3:
            best, chunks = eff, c
    kper = -(-nk16 // chunks)
    return dict(wm=wm, wn=wn, ng=ng, cl=cl, bm=bm, bn=bn, mtiles=mtiles, ntiles=ntiles, kper=kper,
                nchunks=-(-nk16 // kper))


def plan_gemm(m, k, n, rng, sms=148):
    """[(kc0, kc1, plan)]: the full-tile launch and the ragged tail launch of plan_gemm."""
    whole = plan_range(m, k, n, rng, 4, True, sms)
    kmain = k // whole["bn"] * whole["bn"]
    ngt = -(-(k - kmain) // (8 * whole["wn"]))
    if whole["wm"] >= 2 and 0 < kmain < k and ngt < 4:
        return [(0, kmain, plan_range(m, kmain, n, rng, 4, True, sms)),
                (kmain, k, plan_range(m, k - kmain, n, rng, ngt, False, sms))]
    return [(0, k, whole)]


def instantiations(m, k, n, mode):
    """Template arguments (WM, WN, NG, MODE, CL) of the sketch_gemm_kernel launches (dispatch_gemm)."""
    return {(p["wm"], p["wn"], p["ng"], mode, p["cl"] if mode != 0 and p["ng"] == 4 else 1)
            for _, _, p in plan_gemm(m, k, n, mode != 0)}


PRODUCTION = frozenset(
    [(1, 8, 4, 0, 1)] + [(2, 4, g, 0, 1) for g in (1, 2, 3, 4)]
    + [x for mode in (1, 2, 3) for x in
       [(1, 8, 4, mode, 1), (2, 4, 4, mode, 1), (2, 4, 4, mode, 2), (4, 2, 4, mode, 2)]
       + [(wm, 8 // wm, g, mode, 1) for wm in (2, 4) for g in (1, 2, 3)]])

_KERNEL = re.compile(r"sketch_gemm_kernel<\s*(\d+),\s*(\d+),\s*(\d+),\s*(\d+),\s*(\d+)\s*>")


def profiled(fn):
    """fn()'s result and the names of the CUDA kernels it launched."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.key for e in prof.key_averages()}


def gemm_instantiations(names):
    return {tuple(int(x) for x in mt.groups()) for s in names for mt in [_KERNEL.search(s)] if mt}


def ran_i8(names):
    return any("sketch_gemm_i8_kernel" in s for s in names)


# ---------------------------------------------------------------- bound and comparison

def length(n):
    return n + -(-n // GK) + 2


def entry_errors(got, S, A, scale, n, y0=None):
    """Per entry: (|yhat - y|, bound, normalised error) as float64 arrays for the computed got and
    the exact S = sum u theta, A = sum |u||theta| (long double, from exact_dots)."""
    L = length(n)
    ld = np.longdouble
    y = S * ld(scale)
    Aa = A * ld(abs(scale)) * ld(1.0 + 2.0 * gamma(n))
    bound = ld(gamma(L)) * Aa + ld(L) * ld(2.0 ** -1074)
    if y0 is not None:
        y = y + ld(1) * y0
        bound = bound * ld(1.0 + U_ROUND) + ld(U_ROUND) * (np.abs(y0).astype(ld) + Aa)
    err = np.abs(got.astype(ld) - y)
    # normalised by what the roundings scale with: sum |u||theta| (plus |y0| when accumulating);
    # entries whose products underflow are left out
    den = Aa if y0 is None else Aa + np.abs(y0).astype(ld)
    norm = np.where(Aa >= ld(2.0 ** -900), err / np.where(Aa > 0, den, ld(1)), ld(0))
    return err, bound, norm.astype(np.float64)


def check_block(got, U, T, scale, y0=None, what=""):
    """Every entry of got (r, c) = scale U T^T (+ y0) within the bound; returns the largest
    normalised error of got and that of NumPy's float64 product of the same operands."""
    S, A = exact_dots(U, T)
    numpy_got = scale * (U @ T.T) if y0 is None else y0 + scale * (U @ T.T)
    err, bound, norm = entry_errors(got, S, A, scale, U.shape[1], y0)
    bad = ~(err <= bound)
    if bad.any():
        r, c = np.argwhere(bad)[0]
        raise AssertionError(f"{what}: {bad.sum()} entries outside the bound, e.g. ({r}, {c}): "
                             f"got {got[r, c]!r}, exact {float(S[r, c] * np.longdouble(scale))!r}, "
                             f"error {float(err[r, c]):.3e} > bound {float(bound[r, c]):.3e}")
    _, _, norm_np = entry_errors(numpy_got, S, A, scale, U.shape[1], y0)
    return float(norm.max(initial=0.0)), float(norm_np.max(initial=0.0))


def check_sampled(got, U, T, scale, rows, cols, y0=None, what=""):
    """check_block over all columns at `rows` and all rows at `cols` (all of got when both are None);
    asserts the 4x-NumPy criterion and returns the ratio of the largest normalised errors."""
    if rows is None:
        parts = [(slice(None), slice(None))]
    else:
        parts = [(np.asarray(sorted(rows)), slice(None)), (slice(None), np.asarray(sorted(cols)))]
    kmax = npmax = 0.0
    for ri, ci in parts:
        g = got[ri][:, ci]
        a, b = check_block(g, U[ri], T[ci], scale, None if y0 is None else y0[ri][:, ci], what=what)
        kmax, npmax = max(kmax, a), max(npmax, b)
    assert kmax <= 4.0 * max(npmax, U_ROUND), \
        f"{what}: largest normalised error {kmax:.3e}, NumPy's {npmax:.3e}"
    return kmax / max(npmax, U_ROUND)


def sample_sets(m, k, n, mode, rs, extra_rows=()):
    """Rows: first and last of every 64-row warp tile, hence of every m-tile and of each CTA of a
    cluster pair; columns: first and last of every tile of the full-tile range and of every 8-wide
    column group of the tail, and k - 1; a few random ones of each."""
    rows = {0, m - 1, *extra_rows}
    for r0 in range(0, m, 64):
        rows |= {r0, min(m, r0 + 64) - 1}
    cols = {0, k - 1}
    for kc0, kc1, p in plan_gemm(m, k, n, mode != 0):
        step = p["bn"] if kc0 == 0 else 8
        for c0 in range(kc0, kc1, step):
            cols |= {c0, min(kc1, c0 + step) - 1}
    rows |= set(rs.randint(0, m, 3).tolist())
    cols |= set(rs.randint(0, k, 3).tolist())
    return rows, cols


# ---------------------------------------------------------------- operands

def nan_padded(a):
    """A view of a (rows x cols) copy of `a` inside a buffer whose padding columns (an even leading
    dimension > cols) and two trailing rows hold NaN: TMA must never read them."""
    import torch
    r, c = a.shape
    buf = torch.full((r + 2, c + 2 + (c & 1)), float("nan"), dtype=torch.float64, device="cuda")
    buf[:r, :c] = torch.from_numpy(np.ascontiguousarray(a))
    return buf[:r, :c]


def graded(m, n, T, rs):
    """Rows scaled from 2^-300 to 2^300; inside a row, even columns of size 2^200 with alternating
    signs, odd columns of size 2^-200.  When n / 2 > k the even part is projected onto the
    orthogonal complement of the even columns of every Theta row, so that sum_j u_j theta_ij
    cancels to ~ 2^-53 of sum |u_j theta_ij| in every sketch entry."""
    k = T.shape[0]
    base = np.abs(rs.standard_normal((m, n))) * np.where(np.arange(n) % 4 < 2, 1.0, -1.0)
    even = base[:, 0::2]
    if even.shape[1] > k + 8:
        q, _ = np.linalg.qr(T[:, 0::2].T)
        even = even - (even @ q) @ q.T
    u = np.empty((m, n))
    u[:, 0::2] = np.ldexp(even, 200)
    u[:, 1::2] = np.ldexp(base[:, 1::2], -200)
    return np.ldexp(u, np.round(np.linspace(-300, 300, m)).astype(int)[:, None])


def subnormal_rows(u, rows, rs):
    for r in rows:
        u[r] = np.ldexp(rs.standard_normal(u.shape[1]), -1050)          # subnormal products
    return u


# ---------------------------------------------------------------- cases
# mode, m, k, n, input, accumulate.  Together they reach every instantiation of PRODUCTION (each
# case exactly `instantiations(m, k, n, mode)`); n odd, n < 16, n not a multiple of 16 and n of
# 23 (12000) and 9 (5000) chunks are among them.  MODEs 1 and 3 carry one entry of +-2^901.
_RNG_SHAPES = [
    ("wm1", 40, 100, 999, "graded", False),
    ("wm2_ng1", 100, 266, 2000, "normal", True),              # main: WM2 NG4 alone, tail t = 10
    ("wm2pair_ng2", 130, 178, 700, "graded", False),          # main: WM2 NG4 in pairs, tail t = 50
    ("wm2pair_ng3_n15", 130, 198, 15, "normal", True),        # tail t = 70
    ("wm4pair_ng1", 512, 202, 1500, "graded", True),          # main: WM4 NG4 in pairs, tail t = 10
    ("wm4_ng2", 512, 84, 333, "normal", False),               # tail t = 20
    ("wm4_ng3_9chunks", 512, 168, 5000, "graded", False),     # tail t = 40
]
CASES = {
    "explicit_wm1_n1037": (0, 40, 300, 1037, "graded", False),
    "explicit_wm2_ng3": (0, 200, 346, 333, "graded", False),
    "explicit_wm2_ng1_n12": (0, 100, 148, 12, "normal", False),
    "explicit_wm2_ng2_23chunks": (0, 384, 296, 12000, "graded", False),
}
for _mode, _tag in ((1, "normal_fallback"), (2, "rademacher"), (3, "tf32_fallback")):
    for _name, *_rest in _RNG_SHAPES:
        CASES[f"{_tag}_{_name}"] = (_mode, *_rest)
FULL_LIMIT = 4 * 10 ** 7                                    # m k n up to which every entry is checked
SEED = 0x5EED


@pytest.fixture(scope="module")
def dense():
    import rla4mor_b200
    rla4mor_b200.lib()
    from rla4mor_b200 import dense
    return dense


def _window_mask(buf, m, k):
    mask = np.ones(tuple(buf.shape), dtype=bool)
    mask[:m, :k] = False
    return mask


@functools.lru_cache(maxsize=None)
def run_case(name):
    """(U, Theta, y0, result, kernel names) of one case; the call is made twice (same bits) and
    every byte of the output buffer outside the window is checked to be untouched."""
    import torch
    from rla4mor_b200 import dense
    mode, m, k, n, inp, accumulate = CASES[name]
    rs = np.random.RandomState(zlib.crc32(name.encode()))
    scale = 1.0 if mode == 0 else 0.75 / np.sqrt(k)
    if mode == 0:
        T = rs.standard_normal((k, n))
    else:
        T = dense.theta_materialize(SEED, KIND_OF_MODE[mode], 1.0, k, n).cpu().numpy()
    U = graded(m, n, T, rs) if inp == "graded" else rs.standard_normal((m, n))
    if inp == "graded" and m >= 8:
        U = subnormal_rows(U, [2], rs)
    hot = None
    if mode in (1, 3):
        hot = m // 3
        U[hot, (7 * n) // 11] = -2.0 ** 901 if m % 2 else 2.0 ** 901
    y0 = rs.standard_normal((m, k)) if accumulate else None
    dU = nan_padded(U)
    dT = nan_padded(T) if mode == 0 else None
    ybuf = torch.full((m + 1, k + 3), float("nan"), dtype=torch.float64, device="cuda")

    def call():
        if y0 is not None:
            ybuf[:m, :k] = torch.from_numpy(y0)
        before = ybuf.cpu()
        out = ybuf[:m, :k]
        if mode == 0:
            dense.gauss_apply_explicit(dT, dU, out=out)
        else:
            dense.embed_apply_rng(SEED, KIND_OF_MODE[mode], scale, k, dU, out=out, accumulate=accumulate)
        torch.cuda.synchronize()
        after = ybuf.cpu()
        mask = _window_mask(after, m, k)
        assert torch.equal(before.view(torch.int64)[mask], after.view(torch.int64)[mask]), \
            f"{name}: bytes outside the (m, k) window of the output changed"
        return after[:m, :k].numpy().copy()

    got, names = profiled(call)
    again = call()
    assert np.array_equal(got.view(np.int64), again.view(np.int64)), f"{name}: two calls differ"
    return dict(U=U, T=T, y0=y0, got=got, names=names, scale=scale, hot=hot)


@pytest.mark.parametrize("name", list(CASES))
def test_every_entry_within_fp64_bound(dense, name):
    mode, m, k, n, inp, accumulate = CASES[name]
    r = run_case(name)
    names = r["names"]
    seen = gemm_instantiations(names)
    assert seen == instantiations(m, k, n, mode), f"{name}: ran {sorted(seen)}"
    assert not ran_i8(names), f"{name}: the int8 kernel ran"
    if m * k * n <= FULL_LIMIT:
        rows = cols = None
    else:
        rows, cols = sample_sets(m, k, n, mode, np.random.RandomState(m + k + n),
                                 () if r["hot"] is None else (r["hot"],))
    ratio = check_sampled(r["got"], r["U"], r["T"], r["scale"], rows, cols, r["y0"], what=name)
    print(f"{name}: largest normalised error / NumPy's = {ratio:.2f}")


def test_cases_reach_every_production_instantiation(dense):
    seen = set()
    for name in CASES:
        seen |= gemm_instantiations(run_case(name)["names"])
    assert seen == PRODUCTION, f"missing {sorted(PRODUCTION - seen)}, unexpected {sorted(seen - PRODUCTION)}"
    assert len(PRODUCTION) == 35


# ---------------------------------------------------------------- the int8 router's boundary

def _i8_header_bound(u, th, scale):
    """The normwise bound of the header of gemm_i8.cu (|scale| times, plus one rounding)."""
    n = u.shape[1]
    Lb, nb = min(1 << 14, n), -(-n // (1 << 14))
    mx = np.abs(u).max(axis=1)
    un = mx * np.linalg.norm(u / np.where(mx > 0, mx, 1.0)[:, None], axis=1)
    tn = np.linalg.norm(th, axis=1)
    b = (2.0 ** -53 * np.sqrt(Lb) * un[:, None] * (tn[None, :] / 4 + 15 * np.sqrt(n))
         + (nb + 10) * 2.0 ** -52 * un[:, None] * tn[None, :] + 2.0 ** -1073 * nb)
    return abs(scale) * b * (1 + 4 * U_ROUND)


@pytest.mark.parametrize("kind", [0, 2])
def test_router_boundary_at_2_pow_900(dense, kind):
    """max |u| just below 2^900 stays on the int8 path (held to its header bound); 2^900 and
    -2^900 go to the FP64 tensor pipe (held to the componentwise bound).  slice_u_kernel tests
    e > IE_MAX for the smallest e with max |u| < 2^e: the same binade as the header's
    max |u| >= 2^IE_MAX."""
    import torch
    m, k, n = 130, 64, 3000
    rs = np.random.RandomState(40 + kind)
    scale = 0.5
    th = dense.theta_materialize(3, kind, 1.0, k, n).cpu().numpy()
    base = rs.standard_normal((m, n))
    mode = kind + 1
    for big, want_i8 in ((np.nextafter(2.0 ** 900, 0.0), True), (2.0 ** 900, False), (-2.0 ** 900, False)):
        u = base.copy()
        u[5, 77] = big
        got, names = profiled(lambda: dense.embed_apply_rng(3, kind, scale, k, torch.from_numpy(u).cuda()))
        got = got.cpu().numpy()
        S, A = exact_dots(u, th)
        if want_i8:
            assert ran_i8(names) and not gemm_instantiations(names), f"max {big!r}: {sorted(names)}"
            err = np.abs(got.astype(np.longdouble) - S * np.longdouble(scale)).astype(np.float64)
            assert np.all(err <= _i8_header_bound(u, th, scale)), f"max {big!r}: outside the int8 bound"
        else:
            assert not ran_i8(names), f"max {big!r}: the int8 kernel ran"
            assert gemm_instantiations(names) == instantiations(m, k, n, mode), sorted(names)
            err, bound, _ = entry_errors(got, S, A, scale, n)
            assert np.all(err <= bound), f"max {big!r}: outside the FP64 bound"


# ---------------------------------------------------------------- non-finite entries

@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_non_finite_entries(dense, mode):
    """+Inf at u[3, 17] gives row 3 = +-Inf with the signs of scale theta_i,17, -Inf at u[7, 100]
    those of -scale theta_i,100, NaN at u[11, 5] a NaN row; with Theta explicit a NaN at theta[9, 40] gives
    a NaN column 9.  Every other entry stays within the bound."""
    import torch
    m, k, n = 130, 150, 500
    rs = np.random.RandomState(50 + mode)
    scale = 1.0 if mode == 0 else -0.3
    if mode == 0:
        th = rs.standard_normal((k, n))
        th[9, 40] = np.nan
    else:
        th = dense.theta_materialize(8, KIND_OF_MODE[mode], 1.0, k, n).cpu().numpy()
    u = rs.standard_normal((m, n))
    u[3, 17], u[7, 100], u[11, 5] = np.inf, -np.inf, np.nan
    du = nan_padded(u)
    if mode == 0:
        got, names = profiled(lambda: dense.gauss_apply_explicit(nan_padded(th), du))
    else:
        got, names = profiled(lambda: dense.embed_apply_rng(8, KIND_OF_MODE[mode], scale, k, du))
    got = got.cpu().numpy()
    assert not ran_i8(names) and gemm_instantiations(names) == instantiations(m, k, n, mode)
    cols = np.ones(k, dtype=bool)
    if mode == 0:
        assert np.isnan(got[:, 9]).all()
        cols[9] = False
    assert np.array_equal(got[3, cols], np.copysign(np.inf, scale * th[cols, 17]))
    assert np.array_equal(got[7, cols], np.copysign(np.inf, -scale * th[cols, 100]))
    assert np.isnan(got[11]).all()
    ok = np.setdiff1d(np.arange(m), [3, 7, 11])
    check_sampled(got[ok][:, cols], u[ok], th[cols], scale, None, None, what=f"mode {mode}")


# ---------------------------------------------------------------- subnormal operands

@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_subnormal_rows_against_fractions(dense, mode):
    """Rows of subnormal entries (every product subnormal) and a row mixing normal and subnormal
    entries, checked against rational arithmetic: the FP64 tensor pipe keeps subnormal operands
    and products (a flush to zero would leave |y| ~ 2^-1045 where the bound allows ~ 2^-1068)."""
    import torch
    m, k, n = 70, 24, 40
    rs = np.random.RandomState(60 + mode)
    scale = 1.0 if mode == 0 else 0.5
    th = (rs.standard_normal((k, n)) if mode == 0
          else dense.theta_materialize(9, KIND_OF_MODE[mode], 1.0, k, n).cpu().numpy())
    u = rs.standard_normal((m, n))
    u[0] = np.ldexp(rs.standard_normal(n), -1050)
    u[1] = np.ldexp(rs.randint(-3, 4, n).astype(float), -1074)                # multiples of the smallest
    u[2, ::2] = np.ldexp(u[2, ::2], -1040)
    if mode in (1, 3):
        u[5, 9] = 2.0 ** 901
    if mode == 0:
        got, names = profiled(lambda: dense.gauss_apply_explicit(torch.from_numpy(th).cuda(), torch.from_numpy(u).cuda()))
    else:
        got, names = profiled(lambda: dense.embed_apply_rng(9, KIND_OF_MODE[mode], scale, k, torch.from_numpy(u).cuda()))
    got = got.cpu().numpy()
    assert not ran_i8(names) and gemm_instantiations(names)
    L = length(n)
    for c in (0, 1, 2):
        for i in range(k):
            exact = Fraction(scale) * sum(Fraction(float(a)) * Fraction(float(b)) for a, b in zip(u[c], th[i]))
            absum = abs(Fraction(scale)) * sum(abs(Fraction(float(a)) * Fraction(float(b))) for a, b in zip(u[c], th[i]))
            bound = Fraction(float(gamma(L))) * absum + L * Fraction(2) ** -1074
            assert abs(Fraction(float(got[c, i])) - exact) <= bound, (c, i, got[c, i], float(exact))
    assert np.all(got[0] != 0) and np.all(got[2] != 0)
    ok = np.arange(3, m)
    check_sampled(got[ok], u[ok], th, scale, None, None, what=f"mode {mode}")


# ---------------------------------------------------------------- offsets

@pytest.mark.parametrize("mode", [1, 2])
def test_offsets_at_the_abi_limits(dense, mode):
    """row0 + k = 2^32 (the largest the ABI allows) and col0 = 2^32 + 48: the kernel's Theta is
    theta_materialize's at the same offsets."""
    import torch
    m, k, n = 130, 70, 600
    row0, col0 = 2 ** 32 - k, 2 ** 32 + 48
    kind = KIND_OF_MODE[mode]
    rs = np.random.RandomState(70 + mode)
    th = dense.theta_materialize(21, kind, 1.0, k, n, row0=row0, col0=col0).cpu().numpy()
    assert not np.array_equal(th, dense.theta_materialize(21, kind, 1.0, k, n).cpu().numpy())
    u = rs.standard_normal((m, n))
    if mode == 1:
        u[4, 4] = np.inf
    got, names = profiled(lambda: dense.embed_apply_rng(21, kind, 1.0, k, torch.from_numpy(u).cuda(),
                                                        row0=row0, col0=col0))
    got = got.cpu().numpy()
    assert not ran_i8(names) and gemm_instantiations(names) == instantiations(m, k, n, mode)
    ok = np.arange(m) != 4 if mode == 1 else np.ones(m, dtype=bool)
    if mode == 1:
        assert np.array_equal(got[4], np.copysign(np.inf, th[:, 4]))
    check_sampled(got[ok], u[ok], th, 1.0, None, None, what=f"mode {mode} offsets")


# ---------------------------------------------------------------- direct C ABI: the non-TMA fallback

def test_c_abi_unaligned_operands_take_the_fallback_kernel(dense):
    """rla_gauss_apply_explicit_f64 with odd leading dimensions and bases 8 bytes off a 16-byte
    boundary (the Python wrapper always copies to a TMA-friendly buffer): gemm_fallback_kernel,
    within the bound, and only the (m, k) window of a strided output written."""
    import torch
    from rla4mor_b200._lib import check, lib, stream_ptr
    m, k, n = 37, 29, 301
    ldu, ldt, ldy = n + 2, n + 4, k + 3                   # n odd: ldu, ldt odd
    rs = np.random.RandomState(80)
    u, th = rs.standard_normal((m, n)), rs.standard_normal((k, n))

    def unaligned(a, ld):
        buf = torch.full((a.shape[0] * ld + 2,), float("nan"), dtype=torch.float64, device="cuda")
        view = buf[1:1 + a.shape[0] * ld].view(a.shape[0], ld)
        view[:, :a.shape[1]] = torch.from_numpy(a)
        return buf, view
    ubuf, uv = unaligned(u, ldu)
    tbuf, tv = unaligned(th, ldt)
    assert uv.data_ptr() % 16 == 8 and tv.data_ptr() % 16 == 8 and ldu % 2 == 1 and ldt % 2 == 1
    ybuf = torch.full((m + 1, ldy), float("nan"), dtype=torch.float64, device="cuda")
    before = ybuf.cpu()
    ws = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    _, names = profiled(lambda: check(lib().rla_gauss_apply_explicit_f64(
        tv.data_ptr(), k, n, ldt, uv.data_ptr(), m, ldu, ybuf.data_ptr(), ldy, ws.data_ptr(), ws.numel(),
        stream_ptr()), "rla_gauss_apply_explicit_f64"))
    assert any("gemm_fallback_kernel" in s for s in names) and not gemm_instantiations(names), sorted(names)
    after = ybuf.cpu()
    mask = _window_mask(after, m, k)
    assert torch.equal(before.view(torch.int64)[mask], after.view(torch.int64)[mask])
    check_sampled(after[:m, :k].numpy(), u, th, 1.0, None, None, what="fallback kernel")


# ---------------------------------------------------------------- C2 size

def test_c2_size_block_with_one_huge_entry(dense):
    """m = 512, n = 2^22, k = 2000, kind 0 with one entry of 2^901: the whole call runs on the FP64
    tensor pipe (<4,2,4,1,2> over 1984 columns in cluster pairs, <4,2,1,1,1> over the last 16) and
    7 rows x 8 columns, at the tile and column-group edges, are within the bound over the full n."""
    import torch
    m, k, n = 512, 2000, 1 << 22
    free, _ = torch.cuda.mem_get_info()
    if free < 48 * 2 ** 30:
        pytest.skip(f"needs ~40 GB of free device memory, {free / 2 ** 30:.0f} GB free")
    g = torch.Generator(device="cuda").manual_seed(12)
    u = torch.randn((m, n), dtype=torch.float64, device="cuda", generator=g)
    hot = 300
    u[hot, 123457] = 2.0 ** 901
    scale = 1.0 / np.sqrt(k)
    y, names = profiled(lambda: dense.embed_apply_rng(7, 0, scale, k, u))
    assert not ran_i8(names)
    assert gemm_instantiations(names) == {(4, 2, 4, 1, 2), (4, 2, 1, 1, 1)} == instantiations(m, k, n, 1)
    rows = [0, 255, 256, 511, hot, 97, 400]
    cols = [0, 63, 64, 1983, 1984, 1991, 1992, 1999]
    U = u[rows].cpu().numpy()
    del u
    T = np.concatenate([dense.theta_materialize(7, 0, 1.0, 1, n, row0=c).cpu().numpy() for c in cols])
    got = y.cpu().numpy()[np.ix_(rows, cols)]
    kmax, npmax = check_block(got, U, T, scale, what="C2")
    assert kmax <= 4.0 * max(npmax, U_ROUND), (kmax, npmax)
    print(f"C2: largest normalised error / NumPy's = {kmax / max(npmax, U_ROUND):.2f}")
