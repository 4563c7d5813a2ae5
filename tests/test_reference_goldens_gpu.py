"""The CUDA product against fixtures produced by EXECUTING the reference's own classes
(oracle/make_golden_pymor.py: /root/reference/rla/embeddings.py and mor/sketched_reductor.py
imported unmodified on top of tests/_pymor_stub).  Tolerance: relative Frobenius 1e-12 for
sketches (north_star); bit-exact for seeds, block sizes, MT19937 Theta and explicit SRHT rows."""
import json
import os

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from golden_util import GOLDEN, emb_reference, rel_fro

pytestmark = pytest.mark.gpu
TOL = 1e-12


@pytest.fixture(scope="module")
def rb():
    import rla4mor_b200
    rla4mor_b200.lib()
    return rla4mor_b200


@pytest.fixture(scope="module")
def emb():
    z = emb_reference()
    return z, json.loads(str(z["__meta__"]))


def build(rb, z, tag, info, seed="same"):
    cls = getattr(rb, info["cls"])
    options = dict(info["options"])
    seed = info["seed"] if seed == "same" else seed
    rid = "SK" if info["cls"] != "IdentityEmbedding" else ("QS" if info["qrows"] else "S")
    if info["qrows"]:
        Q = rb.MatrixOperator(z[tag + "__Q"], source_id="S", range_id="QS")
        return cls(sqrt_product=Q, options=options, range_id=rid, _seed=seed)
    return cls(source=rb.DeviceVectorSpace(info["n"], id="S"), options=options, range_id=rid, _seed=seed)


def cases(meta, *classes):
    return [t for t, i in meta.items() if not t.startswith("_") and i.get("cls") in classes]


def test_apply_of_every_embedding_class(rb, emb):
    z, meta = emb
    for tag in cases(meta, "SrhtEmbedding", "GaussianEmbedding", "BlockGaussianEmbedding", "IdentityEmbedding"):
        e = build(rb, z, tag, meta[tag])
        assert e.range.dim == meta[tag]["k"]
        U = e.source.from_numpy(z[tag + "__U"])
        Y = e.apply(U)
        assert Y in e.range
        assert rel_fro(Y.to_numpy(), z[tag + "__apply"]) < TOL, tag
        assert rel_fro(e.apply(z[tag + "__U"]), z[tag + "__apply"]) < TOL          # NumPy in, NumPy out
        if meta[tag]["seed"] is not None:
            w = e.with_(_seed=meta[tag]["seed"] + 100)
            assert rel_fro(w.apply(U).to_numpy(), z[tag + "__apply_with_seed"]) < TOL, tag
            e.get_matrix()
            e.set_seed(meta[tag]["seed"] + 200)
            assert rel_fro(e.apply(U).to_numpy(), z[tag + "__apply_set_seed"]) < TOL, tag
            assert rel_fro(e.get_matrix(), z[tag + "__matrix_set_seed"]) < TOL, tag


def test_explicit_matrices_host_and_device(rb, emb):
    z, meta = emb
    for tag in cases(meta, "SrhtEmbedding", "GaussianEmbedding", "BlockGaussianEmbedding"):
        info = meta[tag]
        rm = build(rb, z, tag, info).get_random_matrix()
        if info["cls"] == "SrhtEmbedding" or True:
            assert np.array_equal(rm, z[tag + "__random_matrix"]), tag              # +-value / MT19937: bit exact
        assert rel_fro(build(rb, z, tag, info).get_matrix(), z[tag + "__matrix"]) < TOL, tag
        e = build(rb, z, tag, info)
        md = e.get_matrix_device()
        assert md.is_cuda and rel_fro(md.cpu().numpy(), z[tag + "__matrix"]) < TOL, tag
        assert e._matrix is None                                                      # built on the device, no host copy
        src = build(rb, z, tag, info).as_source_array()
        assert src in e.source and src.data.is_cuda and rel_fro(src.to_numpy(), z[tag + "__as_source_array"]) < TOL
        rng = build(rb, z, tag, info).as_range_array()
        assert rng in e.range and rel_fro(rng.to_numpy(), z[tag + "__as_range_array"]) < TOL
        # caching quirk of get_random_matrix (embeddings.py:98-99)
        e3 = build(rb, z, tag, info)
        e3.get_random_matrix()
        assert np.array_equal(e3.get_matrix(), z[tag + "__matrix_after_random"]), tag


def test_srht_rows_and_adjoint(rb, emb):
    z, meta = emb
    for tag in cases(meta, "SrhtEmbedding"):
        e = build(rb, z, tag, meta[tag])
        assert np.array_equal(e._get_random_rows(z[tag + "__rows_idx"]), z[tag + "__rows"]), tag
        V = e.range.from_numpy(z[tag + "__V"])
        assert rel_fro(e.apply_adjoint(V).to_numpy(), z[tag + "__apply_adjoint"]) < TOL, tag
        with pytest.raises(IndexError):
            e._get_random_rows([meta[tag]["k"]])


def test_block_structure(rb, emb):
    z, meta = emb
    for tag in cases(meta, "BlockGaussianEmbedding"):
        info = meta[tag]
        e = build(rb, z, tag, info)
        assert list(e.block_sizes) == info["block_sizes"] and e.n_blocks == info["n_blocks"]
        assert np.array_equal(np.asarray(e.block_seeds, dtype=np.int64), z[tag + "__block_seeds"])
        assert e._seed == info["seed_after"]
        for b in range(e.n_blocks):
            assert np.array_equal(e._get_random_block(b), z[tag + f"__random_block{b}"])
            assert rel_fro(e.get_block(b), z[tag + f"__block{b}"]) < TOL
            assert rel_fro(e.get_block_device(b).cpu().numpy(), z[tag + f"__block{b}"]) < TOL


def test_identity_vectorized_dims(rb, emb):
    z, meta = emb
    for tag in ("ident", "ident_Q"):
        e = build(rb, z, tag, meta[tag])
        V = e.range.from_numpy(z[tag + "__V"])
        assert rel_fro(e.apply_adjoint(V).to_numpy(), z[tag + "__apply_adjoint"]) < TOL
        assert rel_fro(np.asarray(e.get_matrix().todense() if sp.issparse(e.get_matrix()) else e.get_matrix()),
                       z[tag + "__matrix"]) < TOL
    v = meta["vectorized"]
    inner = rb.GaussianEmbedding(source=rb.DeviceVectorSpace(v["k1"] * v["n_vectors"], id="VEC"),
                                 options={"range_dim": v["k2"]}, _seed=v["seed"])
    vec = rb.EmbeddingVectorized(rb.DeviceVectorSpace(v["k1"], id="SK"), v["n_vectors"], inner, options={}, _seed=v["seed"])
    y = vec.apply(rb.DeviceVectorSpace(v["k1"], id="SK").from_numpy(z["vectorized__U"]))
    assert rel_fro(y.to_numpy(), z["vectorized__apply"]) < TOL
    assert vec.apply_adjoint(None) is None and vec.options["range_dim"] == v["k2"]
    for d in meta["_dims"]:
        opt = dict(d["options"])
        if opt.get("dtype") == "complex":
            opt["dtype"] = complex
        assert rb.SrhtEmbedding(source=rb.DeviceVectorSpace(1000), options=dict(opt), _seed=1).compute_dim() == d["srht"]
        assert rb.BlockGaussianEmbedding(source=rb.DeviceVectorSpace(3), options=dict(opt, max_block_size=10 ** 9),
                                         _seed=1).compute_dim() == d["gauss"]


# ------------------------------------------------------------------------------- reductor
def load_reductor():
    z = np.load(os.path.join(GOLDEN, "reductor_reference.npz"))
    meta = json.loads(str(z["__meta__"]))
    n = meta["n"]
    A = [sp.csr_matrix((z[f"A{q}__data"], z[f"A{q}__indices"], z[f"A{q}__indptr"]), shape=(n, n)) for q in range(3)]
    R = sp.csr_matrix((z["R__data"], z["R__indices"], z["R__indptr"]), shape=(n, n))
    return z, meta, A, R


@pytest.mark.parametrize("cfg", ["gauss_galerkin", "gauss_minres", "srht_galerkin", "srht_minres"])
def test_sketched_reductor_vs_executed_reference(rb, cfg):
    from rla4mor_b200.factorization import InverseLuOperator
    from rla4mor_b200.sketched_reductor import AffineModel
    z, meta, A, R = load_reductor()
    kind, projection = cfg.split("_")
    n, k = meta["n"], meta["k"]
    ops = [rb.MatrixOperator(a, source_id="S", range_id="S") for a in A]
    space = ops[0].source
    fom = AffineModel(ops, list(z["f"]), operator_coefficients=[1.0, lambda mu: mu[0], lambda mu: mu[1]],
                      rhs_coefficients=[1.0, lambda mu: mu[0]], output=z["out"], solution_space=space)
    Rop = rb.MatrixOperator(R.tocsc(), source_id="S", range_id="S")
    Rinv = InverseLuOperator(Rop)
    cls = rb.GaussianEmbedding if kind == "gauss" else rb.SrhtEmbedding
    emb = cls(source=space, options={"range_dim": k}, _seed=meta["seed_primal"], range_id="SK")
    onl = rb.GaussianEmbedding(source=emb.range, options={"range_dim": meta["k_online"]}, _seed=meta["seed_online"])
    red = rb.SketchedReductor(fom, embedding_primal=emb, embedding_online=onl, product=Rop, inverse_product=Rinv,
                              projection=projection, orthonormalize=False)
    if projection == "galerkin":
        rom0 = red.reduce()                                        # _reduce_empty
        for j, mu in enumerate(meta["test"]):
            assert rom0.solve(mu=mu).numel() == 0
            ref = float(z[f"{cfg}__empty_est{j}"].ravel()[0])
            assert abs(rom0.estimate_error(mu=mu) - ref) < 1e-10 * ref
    off = 0
    T_ = lambda t: t.T.cpu().numpy()
    for b, nb in enumerate(meta["blocks"]):
        red.extend_basis(z["U"][off:off + nb])
        assert rel_fro(red.srb.cpu().numpy(), z[f"{cfg}__srb_raw{b}"]) < TOL
        assert rel_fro(np.array([T_(V) for V in red.s_lhs]), z[f"{cfg}__lhs_raw{b}"]) < TOL
        T = red.orthonormalize_basis(offset=red.srb.shape[0] - nb, return_T=True)
        assert rel_fro(T.cpu().numpy(), z[f"{cfg}__T{b}"]) < 1e-10
        assert rel_fro(red.srb.cpu().numpy(), z[f"{cfg}__srb{b}"]) < 1e-10
        assert rel_fro(red.rb.cpu().numpy(), z[f"{cfg}__rb{b}"]) < 1e-10
        assert rel_fro(np.array([T_(V) for V in red.s_lhs]), z[f"{cfg}__lhs{b}"]) < 1e-10
        assert rel_fro(T_(red.output_functional), z[f"{cfg}__out{b}"]) < 1e-10
        off += nb
    assert rel_fro(np.array([v.cpu().numpy() for v in red.s_rhs]), z[f"{cfg}__rhs"]) < TOL
    if projection == "galerkin":
        rom = red.reduce(seed=meta["reduce_seed"])
        assert rel_fro(np.array([M.cpu().numpy() for M in rom.lhs]), z[f"{cfg}__red_lhs"]) < 1e-10
        assert rel_fro(np.array([v.cpu().numpy() for v in rom.rhs]), z[f"{cfg}__red_rhs"][:, :, 0]) < 1e-10
    else:
        rom = red.reduce(seed=tuple(meta["minres_seeds"]))
        assert rel_fro(np.array([M.cpu().numpy() for M in rom.lhs]), z[f"{cfg}__ls_lhs"]) < 1e-10
        assert rel_fro(np.array([v.cpu().numpy() for v in rom.rhs]), z[f"{cfg}__ls_rhs"]) < 1e-10
    assert rel_fro(np.array([M.cpu().numpy() for M in rom.est_lhs]), z[f"{cfg}__est_lhs"]) < 1e-10
    assert rel_fro(np.array([v.cpu().numpy() for v in rom.est_rhs]), z[f"{cfg}__est_rhs"]) < 1e-10
    for j, mu in enumerate(meta["test"]):
        a = rom.solve(mu=mu)
        assert rel_fro(a.cpu().numpy(), z[f"{cfg}__sol{j}"][0]) < 1e-9
        est = rom.estimate_error(a, mu=mu)
        assert abs(est - float(z[f"{cfg}__est{j}"].ravel()[0])) < 1e-8 * max(1.0, est)
        assert rel_fro(rom.output(a).cpu().numpy(), z[f"{cfg}__output{j}"].ravel()) < 1e-9


def test_lincomb_kernel_shapes(rb):
    """out = C @ X on the tall-skinny kernel (csrc/lincomb.cu) for every tile variant, ragged and
    unaligned shapes, against float64 matmul."""
    from rla4mor_b200 import reductor_ops as ops
    g = torch.Generator(device="cuda").manual_seed(3)
    for m, k, n in [(1, 1, 1), (3, 5, 7), (32, 17, 1000), (33, 64, 4097), (64, 64, 12345), (65, 130, 2 ** 15 + 1),
                    (200, 256, 5000), (256, 256, 2 ** 16)]:
        C = torch.randn(m, k, dtype=torch.float64, device="cuda", generator=g)
        X = torch.randn(k, n, dtype=torch.float64, device="cuda", generator=g)
        ref = C @ X
        assert float(torch.linalg.norm(ops.lincomb(C, X) - ref) / torch.linalg.norm(ref)) < 1e-13, (m, k, n)
    Xs = torch.randn(20, 1003, dtype=torch.float64, device="cuda", generator=g)[:, 1:1002]     # odd offset, odd ld
    C = torch.randn(7, 20, dtype=torch.float64, device="cuda", generator=g)
    assert float(torch.linalg.norm(ops.lincomb(C, Xs) - C @ Xs)) < 1e-11
