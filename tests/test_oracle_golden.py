"""The CPU oracle against fixtures produced by the reference itself
(oracle/make_golden.py ran /root/reference/rla/srht.py)."""
import numpy as np
import pytest

import oracle
from oracle import embeddings_oracle as eo
from oracle import reductor_oracle as ro
from oracle import srht_oracle as so
from golden_util import srht_cases, fht_cases, emb_golden, rel_fro


@pytest.mark.parametrize("case", list(srht_cases()), ids=lambda c: c["name"])
def test_srht_matches_reference_bitwise(case):
    y = oracle.srht(case["x"], case["k"], seed=case["seed"])
    assert y.shape == case["y"].shape and y.dtype == case["y"].dtype
    if case["cplx"]:
        assert rel_fro(y, case["y"]) < 1e-15
    else:
        assert np.array_equal(y, case["y"])      # same stage order => bit-identical


@pytest.mark.parametrize("case", list(srht_cases()), ids=lambda c: c["name"])
def test_signs_and_indices_bit_exact(case):
    r = oracle.rademacher_signs(case["n"], case["seed"])
    s = oracle.sampling_indices(case["n"], case["k"], case["seed"])
    assert r.dtype == np.int64 and s.dtype == np.int64
    assert np.array_equal(r, case["signs"].astype(np.int64))
    assert np.array_equal(s, case["sampling"])
    y = so.srht_with(case["x"], case["k"], r, s)
    assert rel_fro(y, case["y"]) < 1e-15 if case["cplx"] else np.array_equal(y, case["y"])


@pytest.mark.parametrize("case", list(fht_cases()), ids=lambda c: c["name"])
def test_fht_matches_reference_bitwise(case):
    a = case["a"]
    out = oracle.fht_oop(a)
    b = a.copy()
    oracle.fht_ip(b)
    if np.iscomplexobj(a):
        # numba divides a complex by 2**(d/2) with a complex division; the oracle
        # scales real and imaginary parts separately: equal to rounding only.
        assert rel_fro(out, case["oop"]) < 1e-15 and rel_fro(b, case["ip"]) < 1e-15
    else:
        assert np.array_equal(out, case["oop"])
        assert np.array_equal(b, case["ip"])
    assert np.array_equal(a, case["a"])          # fht_oop never mutates its input


def test_fht_numpy_fallback_equals_c_path():
    a = np.random.RandomState(0).standard_normal((3, 256))
    b = a.copy()
    so._butterflies_numpy(b)
    c = a.copy()
    lib = so._clib()
    if not lib:
        pytest.skip("C oracle not built")
    lib.oracle_fwht_rows_f64(c.ctypes.data, 3, 256, 2)
    assert np.array_equal(b, c)


def test_fht_rejects_non_power_of_two():
    with pytest.raises(AssertionError):
        oracle.fht_oop(np.zeros((2, 12)))
    with pytest.raises(AssertionError):
        oracle.fht_ip(np.zeros((2, 2, 4)))


def test_closed_form_and_involution():
    x = np.random.RandomState(5).standard_normal((3, 37))
    assert rel_fro(oracle.srht(x, 9, seed=4), oracle.srht_closed_form(x, 9, 4)) < 1e-14
    a = np.random.RandomState(6).standard_normal((2, 512))
    assert rel_fro(oracle.fht_oop(oracle.fht_oop(a)), a) < 1e-14
    n = 32
    H = oracle.fht_oop(np.eye(n)) * np.sqrt(n)
    i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    par = np.vectorize(lambda v: bin(v).count("1") & 1)(i & j)
    assert np.array_equal(H, 1.0 - 2.0 * par)


def test_embedding_transcriptions():
    z = emb_golden()
    for tag in ("rows_pow2", "rows_nonpow2", "rows_5000"):
        n, k, seed = (int(v) for v in z[tag + "__meta"])
        rows = eo.srht_random_rows(n, k, seed, z[tag + "__indices"])
        assert np.array_equal(rows, z[tag + "__rows"])
    for tag in ("gauss_small", "gauss_mid"):
        m, n, k, seed = (int(v) for v in z[tag + "__meta"])
        theta = eo.gaussian_random_matrix(k, n, seed)
        assert np.array_equal(theta, z[tag + "__theta"])
        assert rel_fro(eo.gaussian_apply(z[tag + "__U"], theta), z[tag + "__Y"]) < 1e-15
    for tag in ("block_a", "block_b"):
        m, n, k, seed, mbs = (int(v) for v in z[tag + "__meta"])
        assert eo.block_sizes(k, mbs) == list(z[tag + "__sizes"])
        seeds, seed2 = eo.block_seeds(seed, len(z[tag + "__sizes"]))
        assert seed2 == seed and np.array_equal(seeds, z[tag + "__seeds"])
        assert np.array_equal(eo.block_gaussian_random_matrix(k, n, seed, mbs), z[tag + "__theta"])
        assert rel_fro(eo.block_gaussian_apply(z[tag + "__U"], k, seed, mbs), z[tag + "__Y"]) < 1e-15


def test_srht_rows_consistent_with_apply_for_power_of_two():
    n, k, seed = 128, 20, 3
    x = np.random.RandomState(1).standard_normal((4, n))
    mat = eo.srht_matrix(n, k, seed)
    assert rel_fro(x @ mat.T, oracle.srht(x, k, seed)) < 1e-14
    v = np.random.RandomState(2).standard_normal((3, k))
    assert rel_fro(eo.srht_apply_adjoint(v, n, k, seed), v @ mat) < 1e-15


def test_compute_dim_formulas():
    assert eo.srht_compute_dim({"range_dim": 17}, 1000) == 17
    assert eo.gaussian_compute_dim({"range_dim": 5}) == 5
    k = eo.gaussian_compute_dim({"epsilon": 0.5, "delta": 0.01, "oblivious_dim": 10})
    assert k == int(np.ceil(7.87 * 4 * (6.9 * 10 + np.log(100))))
    k2 = eo.gaussian_compute_dim({"epsilon": 0.5, "delta": 0.01, "oblivious_dim": 10, "dtype": complex})
    assert k2 > k
    ks = eo.srht_compute_dim({"epsilon": 0.5, "delta": 0.01, "oblivious_dim": 10}, 10000)
    expect = 2 / (0.25 - 0.125 / 3) * (np.sqrt(10) + np.sqrt(8 * np.log(6 * 10000 / 0.01))) ** 2 * np.log(3 * 10 / 0.01)
    assert ks == int(np.ceil(expect))
    with pytest.raises(AssertionError):
        eo.gaussian_compute_dim({"epsilon": 0.5})


def test_vectorized_apply_layout():
    U = np.arange(12.0).reshape(3, 4)
    got = eo.vectorized_apply(U, lambda x: x)
    assert np.array_equal(got[0], U.T.flatten())


def test_gram_schmidt_and_reductor_identities():
    rs = np.random.RandomState(3)
    A = rs.standard_normal((6, 40))
    Q, R = ro.gram_schmidt(A)
    assert rel_fro(R.T @ Q, A) < 1e-13
    assert rel_fro(Q @ Q.T, np.eye(6)) < 1e-13
    assert np.allclose(R, np.triu(R))
    # offset: the first rows are assumed orthonormal already
    A2 = np.vstack([Q[:3], rs.standard_normal((2, 40))])
    Q2, R2 = ro.gram_schmidt(A2, offset=3)
    assert rel_fro(Q2 @ Q2.T, np.eye(5)) < 1e-13 and rel_fro(R2.T @ Q2, A2) < 1e-13
    # dependent vector is removed
    A3 = np.vstack([A[:2], A[0] + A[1]])
    Q3, R3 = ro.gram_schmidt(A3)
    assert Q3.shape[0] == 2 and R3.shape == (2, 3)
    S = [rs.standard_normal((40, 6)) for _ in range(2)]
    Qo, Ro, T, S2 = ro.orthonormalize_sketch(A, S)
    assert rel_fro(T.T @ A, Qo) < 1e-12
    assert rel_fro(S2[0], S[0] @ T) == 0.0
    lhs, rhs = ro.galerkin_system(Qo, S2, [rs.standard_normal((40, 1))])
    assert lhs[0].shape == (6, 6) and rhs[0].shape == (6, 1)
    a = rs.standard_normal(6)
    b = [rs.standard_normal((40, 1))]
    val = ro.residual_norm(S2, [0.5, 2.0], b, [1.0], a)
    assert np.isclose(val, np.linalg.norm(0.5 * S2[0] @ a + 2.0 * S2[1] @ a - b[0][:, 0]))


def test_factorization_oracle_identities():
    """oracle/factorization_oracle.py restates utilities/factorization.py:17-52,118-132 (SciPy
    SuperLU, the reference's own dependency); pinned by A x = b, A^H x = b and Q^H Q = A."""
    import scipy.sparse as sp
    from oracle import factorization_oracle as fo
    rs = np.random.RandomState(0)
    n = 300
    A = (sp.random(n, n, 0.02, random_state=rs) + 4.0 * sp.eye(n)).tocsc()
    V = rs.standard_normal((5, n))
    slu = fo.factorize(A)
    assert np.linalg.norm((A @ fo.inverse_lu_apply(slu, V).T).T - V) / np.linalg.norm(V) < 1e-12
    assert np.linalg.norm((A.T @ fo.inverse_lu_apply_adjoint(slu, V).T).T - V) / np.linalg.norm(V) < 1e-12
    S = (A @ A.T + sp.eye(n)).tocsc()
    Q = fo.lu_to_cholesky(S)
    assert abs(Q.conj().T @ Q - S).max() < 1e-10
    assert np.linalg.norm(fo.inverse_lu_apply(fo.factorize(S, symetric=True), V) @ S.T - V) / np.linalg.norm(V) < 1e-10


def test_golden_archive_stores_equal_arrays_once(tmp_path):
    from oracle import golden_archive
    rs = np.random.RandomState(0)
    m = rs.standard_normal((33, 301))
    other = m.copy()
    other[7, 9] = np.nextafter(other[7, 9], np.inf)                 # one ulp apart: stored on its own
    arrays = {"a__matrix": m, "a__random_matrix": m.copy(), "a__as_range_array": np.ascontiguousarray(m.T),
              "a__other": other, "a__int": np.arange(5), "a__float": np.arange(5.0), "__meta__": np.array("{}")}
    path = str(tmp_path / "g.npz")
    golden_archive.save(path, arrays)
    assert sorted(np.load(path).files) == sorted(["a__matrix", "a__other", "a__int", "a__float", "__meta__",
                                                  golden_archive.ALIASES])
    z = golden_archive.load(path)
    assert sorted(z.files) == sorted(arrays) and "a__as_range_array" in z and golden_archive.ALIASES not in z
    for name, a in arrays.items():
        assert z[name].dtype == a.dtype and z[name].shape == a.shape and z[name].tobytes() == a.tobytes(), name
