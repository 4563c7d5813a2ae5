"""The CPU oracle against fixtures produced by EXECUTING the reference's own classes
(oracle/make_golden_pymor.py: rla/embeddings.py and mor/sketched_reductor.py imported unmodified
on top of tests/_pymor_stub).  These pin the oracle for the operator classes and for the
reductor arithmetic; the GPU tests compare the product with the same fixtures."""
import json
import os

import numpy as np
import pytest
import scipy.sparse as sp

import oracle
from oracle import embeddings_oracle as eo
from oracle import reductor_oracle as ro
from golden_util import GOLDEN, emb_reference, rel_fro

TOL = 1e-12


@pytest.fixture(scope="module")
def emb():
    z = emb_reference()
    return z, json.loads(str(z["__meta__"]))


def _cases(meta, cls):
    return [t for t, i in meta.items() if not t.startswith("_") and i.get("cls") == cls]


def test_srht_embedding_class(emb):
    z, meta = emb
    for tag in _cases(meta, "SrhtEmbedding"):
        i = meta[tag]
        n, k, seed = i["n"], i["k"], i["seed"]
        Q = z[tag + "__Q"] if i["qrows"] else None
        nq = Q.shape[0] if Q is not None else n
        assert rel_fro(eo.srht_apply(z[tag + "__U"], k, seed, Q), z[tag + "__apply"]) < TOL
        rows = eo.srht_random_rows(nq, k, seed, z[tag + "__rows_idx"])
        assert np.array_equal(rows, z[tag + "__rows"])                       # +-value: bit exact
        assert np.array_equal(eo.srht_random_rows(nq, k, seed, np.arange(k)), z[tag + "__random_matrix"])
        assert rel_fro(eo.srht_matrix(nq, k, seed, Q), z[tag + "__matrix"]) < TOL
        assert rel_fro(eo.srht_apply_adjoint(z[tag + "__V"], nq, k, seed, Q), z[tag + "__apply_adjoint"]) < TOL
        assert rel_fro(eo.srht_apply(z[tag + "__U"], k, seed + 100, Q), z[tag + "__apply_with_seed"]) < TOL
        assert rel_fro(eo.srht_apply(z[tag + "__U"], k, seed + 200, Q), z[tag + "__apply_set_seed"]) < TOL
        # SrhtEmbedding.update() is a no-op (embeddings.py:145-146): a cached matrix survives set_seed
        assert np.array_equal(z[tag + "__matrix_set_seed"], z[tag + "__matrix"])
        # get_random_matrix caches into _matrix (embeddings.py:98-99): get_matrix afterwards is un-Q'd
        assert np.array_equal(z[tag + "__matrix_after_random"], z[tag + "__random_matrix"])


def test_gaussian_embedding_class(emb):
    z, meta = emb
    for tag in _cases(meta, "GaussianEmbedding"):
        i = meta[tag]
        Q = z[tag + "__Q"] if i["qrows"] else None
        nq = Q.shape[0] if Q is not None else i["n"]
        theta = eo.gaussian_random_matrix(i["k"], nq, i["seed"])
        assert np.array_equal(theta, z[tag + "__random_matrix"])
        assert rel_fro(eo.gaussian_apply(z[tag + "__U"], theta, Q), z[tag + "__apply"]) < TOL
        assert rel_fro(eo.gaussian_matrix(theta, Q), z[tag + "__matrix"]) < TOL
        assert rel_fro(eo.gaussian_matrix(theta, Q), z[tag + "__as_source_array"]) < TOL
        assert rel_fro(eo.gaussian_matrix(theta, Q).T, z[tag + "__as_range_array"]) < TOL
        t2 = eo.gaussian_random_matrix(i["k"], nq, i["seed"] + 200)
        assert rel_fro(eo.gaussian_apply(z[tag + "__U"], t2, Q), z[tag + "__apply_set_seed"]) < TOL
        assert rel_fro(eo.gaussian_matrix(t2, Q), z[tag + "__matrix_set_seed"]) < TOL


def test_block_gaussian_embedding_class(emb):
    z, meta = emb
    for tag in _cases(meta, "BlockGaussianEmbedding"):
        i = meta[tag]
        Q = z[tag + "__Q"] if i["qrows"] else None
        nq = Q.shape[0] if Q is not None else i["n"]
        mbs = i["options"]["max_block_size"]
        assert eo.block_sizes(i["k"], mbs) == i["block_sizes"]
        seeds, seed_after = eo.block_seeds(i["seed"], i["n_blocks"])
        assert np.array_equal(seeds, z[tag + "__block_seeds"]) and seed_after == i["seed_after"]
        for b in range(i["n_blocks"]):
            blk = eo.block_gaussian_block(i["k"], nq, i["block_sizes"][b], seeds[b])
            assert np.array_equal(blk, z[tag + f"__random_block{b}"])
            assert rel_fro(eo.gaussian_matrix(blk, Q), z[tag + f"__block{b}"]) < TOL
        assert rel_fro(eo.block_gaussian_apply(z[tag + "__U"], i["k"], i["seed"], mbs, Q), z[tag + "__apply"]) < TOL
        assert np.array_equal(eo.block_gaussian_random_matrix(i["k"], nq, i["seed"], mbs), z[tag + "__random_matrix"])


def test_identity_and_vectorized(emb):
    z, meta = emb
    assert np.array_equal(z["ident__apply"], z["ident__U"])
    Q = z["ident_Q__Q"]
    assert rel_fro(z["ident_Q__U"] @ Q.T, z["ident_Q__apply"]) < TOL
    assert rel_fro(z["ident_Q__V"] @ Q.conj(), z["ident_Q__apply_adjoint"]) < TOL
    v = meta["vectorized"]
    theta = eo.gaussian_random_matrix(v["k2"], v["k1"] * v["n_vectors"], v["seed"])
    y = eo.vectorized_apply(z["vectorized__U"], lambda x: eo.gaussian_apply(x, theta))
    assert rel_fro(y, z["vectorized__apply"]) < TOL
    assert v["apply_adjoint_is_none"] and v["range_dim_option"] == v["k2"]


def test_dimension_formulas(emb):
    _, meta = emb
    for d in meta["_dims"]:
        opt = dict(d["options"])
        if opt.get("dtype") == "complex":
            opt["dtype"] = complex
        assert eo.srht_compute_dim(opt, 1000) == d["srht"]
        assert eo.gaussian_compute_dim(opt) == d["gauss"]


# ------------------------------------------------------------------------------- reductor
def load_reductor():
    z = np.load(os.path.join(GOLDEN, "reductor_reference.npz"))
    meta = json.loads(str(z["__meta__"]))
    n = meta["n"]
    A = [sp.csr_matrix((z[f"A{q}__data"], z[f"A{q}__indices"], z[f"A{q}__indptr"]), shape=(n, n)) for q in range(3)]
    R = sp.csr_matrix((z["R__data"], z["R__indices"], z["R__indptr"]), shape=(n, n))
    return z, meta, A, R


def thetas(mu):
    return [1.0, mu[0], mu[1]], [1.0, mu[0]]


@pytest.mark.parametrize("cfg", ["gauss_galerkin", "gauss_minres", "srht_galerkin", "srht_minres"])
def test_sketched_reductor_oracle_vs_executed_reference(cfg):
    import scipy.sparse.linalg as spla
    z, meta, A, R = load_reductor()
    kind, projection = cfg.split("_")
    n, k = meta["n"], meta["k"]
    lu = spla.splu(R.tocsc())
    if kind == "gauss":
        theta = eo.gaussian_random_matrix(k, n, meta["seed_primal"])
        theta_apply = lambda V: eo.gaussian_apply(V, theta)
    else:
        theta_apply = lambda V: oracle.srht(V, k, seed=meta["seed_primal"])

    def online_apply(seed, V):
        g = eo.gaussian_random_matrix(meta["k_online"], k, seed)
        return eo.gaussian_apply(V, g)

    red = ro.SketchedReductorOracle(A, list(z["f"]), z["out"], theta_apply, online_apply,
                                    Rinv_apply=lambda V: lu.solve(V.T).T, R=R, projection=projection, orthonormalize=False)
    if projection == "galerkin":
        rom0 = red.reduce()
        for j, mu in enumerate(meta["test"]):
            assert rom0.solve(*thetas(mu)).shape == (0,) and z[f"{cfg}__empty_sol{j}"].size == 0
            assert abs(rom0.estimate_error(None, *thetas(mu)) - float(z[f"{cfg}__empty_est{j}"].ravel()[0])) \
                < 1e-10 * float(z[f"{cfg}__empty_est{j}"].ravel()[0])
    off = 0
    for b, nb in enumerate(meta["blocks"]):
        red.extend_basis(z["U"][off:off + nb])
        assert rel_fro(red.srb, z[f"{cfg}__srb_raw{b}"]) < TOL
        assert rel_fro(np.array(red.S), z[f"{cfg}__lhs_raw{b}"]) < TOL
        T = red.orthonormalize_basis(offset=red.srb.shape[0] - nb)
        assert rel_fro(T, z[f"{cfg}__T{b}"]) < 1e-10
        assert rel_fro(red.srb, z[f"{cfg}__srb{b}"]) < 1e-10
        assert rel_fro(red.rb, z[f"{cfg}__rb{b}"]) < 1e-10
        assert rel_fro(np.array(red.S), z[f"{cfg}__lhs{b}"]) < 1e-10
        assert rel_fro(red.out, z[f"{cfg}__out{b}"]) < 1e-10
        off += nb
    assert rel_fro(np.array(red.b), z[f"{cfg}__rhs"]) < TOL
    if projection == "galerkin":
        rom = red.reduce(seed=meta["reduce_seed"])
        assert rel_fro(np.array(rom.lhs), z[f"{cfg}__red_lhs"]) < 1e-10
        assert rel_fro(np.array(rom.rhs), z[f"{cfg}__red_rhs"][:, :, 0]) < 1e-10
    else:
        rom = red.reduce(seed=tuple(meta["minres_seeds"]))
        assert rel_fro(np.array(rom.lhs), z[f"{cfg}__ls_lhs"]) < 1e-10
        assert rel_fro(np.array(rom.rhs), z[f"{cfg}__ls_rhs"]) < 1e-10
    assert rel_fro(np.array(rom.est[0]), z[f"{cfg}__est_lhs"]) < 1e-10
    assert rel_fro(np.array(rom.est[1]), z[f"{cfg}__est_rhs"]) < 1e-10
    for j, mu in enumerate(meta["test"]):
        a = rom.solve(*thetas(mu))
        assert rel_fro(a, z[f"{cfg}__sol{j}"][0]) < 1e-9
        est = rom.estimate_error(a, *thetas(mu))
        assert abs(est - float(z[f"{cfg}__est{j}"].ravel()[0])) < 1e-8 * max(1.0, est)
        assert rel_fro(rom.output(a), z[f"{cfg}__output{j}"].ravel()) < 1e-9
