"""Generate tests/golden/embeddings_reference.npz and reductor_reference.npz by EXECUTING the
reference's own classes (build container only):

    python -m oracle.make_golden_pymor

`/root/reference/rla/embeddings.py`, `mor/sketched_reductor.py`, `utilities/*` import pyMOR at
module level.  pyMOR is not in the image, so `tests/_pymor_stub` (a restatement of the pyMOR
names SURVEY.md App. B lists) is put on sys.path and the UNMODIFIED reference modules are
imported on top of it.  Everything recorded here is an output of the reference's code; the
pyMOR side of each call (matrix-operator apply, gram_schmidt, project/expand/contract) is the
stub's restatement of pyMOR 2023.1 -- see tests/_pymor_stub/pymor/__init__.py.
"""
import json
import os
import sys

import numpy as np
import scipy.sparse as sp

from oracle import golden_archive

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")
REFERENCE = "/root/reference"


def import_reference():
    for p in (os.path.join(ROOT, "tests", "_pymor_stub"), REFERENCE):
        if p not in sys.path:
            sys.path.insert(0, p)
    import rla.embeddings as E                       # noqa: the reference, unmodified
    import mor.sketched_reductor as SR
    import utilities.factorization as F
    return E, SR, F


def dense_Q(n_range, n_source, seed):
    """A dense `sqrt_product` matrix (any full-rank Q defines an inner product Q^H Q)."""
    rs = np.random.RandomState(seed)
    return rs.standard_normal((n_range, n_source)) / np.sqrt(n_source) + np.eye(n_range, n_source)


EMB_CASES = [
    # tag, class, n, m, options, seed, Q rows (None = identity sqrt_product)
    ("srht_pow2", "SrhtEmbedding", 64, 3, {"range_dim": 10}, 0, None),
    ("srht_nonpow2", "SrhtEmbedding", 100, 5, {"range_dim": 16}, 7, None),
    ("srht_5000", "SrhtEmbedding", 5000, 2, {"range_dim": 12}, 5, None),
    ("srht_Q", "SrhtEmbedding", 40, 4, {"range_dim": 9}, 3, 48),
    ("gauss_small", "GaussianEmbedding", 50, 4, {"range_dim": 12}, 3, None),
    ("gauss_mid", "GaussianEmbedding", 301, 7, {"range_dim": 33}, 21, None),
    ("gauss_Q", "GaussianEmbedding", 40, 4, {"range_dim": 9}, 13, 48),
    ("block_a", "BlockGaussianEmbedding", 40, 3, {"range_dim": 10, "max_block_size": 4}, 5, None),
    ("block_b", "BlockGaussianEmbedding", 64, 2, {"range_dim": 33, "max_block_size": 32}, 77, None),
    ("block_Q", "BlockGaussianEmbedding", 40, 3, {"range_dim": 10, "max_block_size": 3}, 6, 48),
    ("ident", "IdentityEmbedding", 30, 3, {}, None, None),
    ("ident_Q", "IdentityEmbedding", 30, 3, {}, None, 30),   # range dim = source dim (embeddings.py:291-292): square Q
]
DIM_OPTIONS = [
    {"epsilon": 0.5, "delta": 0.01, "oblivious_dim": 10},
    {"epsilon": 0.25, "delta": 1e-3, "oblivious_dim": 20, "dtype": "complex"},
]


def make_embeddings(E):
    from pymor.operators.numpy import NumpyMatrixOperator
    from pymor.vectorarrays.numpy import NumpyVectorSpace
    out, meta = {}, {}
    for tag, cls, n, m, options, seed, qrows in EMB_CASES:
        source = NumpyVectorSpace(n, id="S")
        Q = None
        if qrows is not None:
            Qm = dense_Q(qrows, n, 900 + (seed or 0))
            Q = NumpyMatrixOperator(Qm, source_id="S", range_id="QS")
            out[tag + "__Q"] = Qm

        def build(seed_=seed):
            # IdentityEmbedding's range IS the range of sqrt_product (its apply_adjoint hands range
            # vectors straight to sqrt_product.apply_adjoint, embeddings.py:297-299): same id
            rid = "SK" if cls != "IdentityEmbedding" else ("QS" if Q is not None else "S")
            kw = dict(options=dict(options), range_id=rid, _seed=seed_)
            return getattr(E, cls)(sqrt_product=Q, **kw) if Q is not None else getattr(E, cls)(source=source, **kw)
        emb = build()
        U = np.random.RandomState(5000 + (seed or 0)).standard_normal((m, n))
        out[tag + "__U"] = U
        out[tag + "__apply"] = emb.apply(source.from_numpy(U)).to_numpy()
        k = emb.range.dim
        V = np.random.RandomState(6000 + (seed or 0)).standard_normal((2, k))
        out[tag + "__V"] = V
        if cls in ("SrhtEmbedding", "IdentityEmbedding"):
            out[tag + "__apply_adjoint"] = emb.apply_adjoint(emb.range.from_numpy(V)).to_numpy()
        # explicit matrices: fresh objects, because get_random_matrix caches into `_matrix`
        # (embeddings.py:98-99) and would change what get_matrix returns afterwards
        mat = build().get_matrix()
        out[tag + "__matrix"] = mat.toarray() if sp.issparse(mat) else np.asarray(mat)
        rmat = build().get_random_matrix()
        out[tag + "__random_matrix"] = rmat.toarray() if sp.issparse(rmat) else np.asarray(rmat)
        e2 = build()
        out[tag + "__as_source_array"] = e2.as_source_array().to_numpy()
        if cls != "IdentityEmbedding" or Q is None:
            out[tag + "__as_range_array"] = build().as_range_array().to_numpy()
        # the caching quirk itself: get_matrix() AFTER get_random_matrix() on one object
        e3 = build()
        e3.get_random_matrix()
        q = e3.get_matrix()
        out[tag + "__matrix_after_random"] = q.toarray() if sp.issparse(q) else np.asarray(q)
        info = dict(cls=cls, n=n, m=m, options=options, seed=seed, qrows=qrows, k=int(k))
        if cls == "SrhtEmbedding":
            idx = np.array([0, k - 1, 2, 2])
            out[tag + "__rows_idx"] = idx
            out[tag + "__rows"] = build()._get_random_rows(idx)
        if cls == "BlockGaussianEmbedding":
            info["block_sizes"] = [int(b) for b in emb.block_sizes]
            info["n_blocks"] = int(emb.n_blocks)
            info["seed_after"] = int(emb._seed)
            out[tag + "__block_seeds"] = np.asarray(emb.block_seeds, dtype=np.int64)
            for i in range(emb.n_blocks):
                out[tag + f"__block{i}"] = emb.get_block(i)
                out[tag + f"__random_block{i}"] = emb._get_random_block(i)
        if seed is not None:
            # with_(_seed=...) builds a fresh embedding; set_seed() re-seeds in place
            w = emb.with_(_seed=seed + 100)
            out[tag + "__apply_with_seed"] = w.apply(source.from_numpy(U)).to_numpy()
            e4 = build()
            e4.get_matrix()
            e4.set_seed(seed + 200)
            out[tag + "__apply_set_seed"] = e4.apply(source.from_numpy(U)).to_numpy()
            q = e4.get_matrix()
            out[tag + "__matrix_set_seed"] = q.toarray() if sp.issparse(q) else np.asarray(q)
        meta[tag] = info
    # dimension formulas (embeddings.py:148-164, 234-247)
    dims = []
    for o in DIM_OPTIONS:
        opt = dict(o)
        if opt.get("dtype") == "complex":
            opt["dtype"] = complex
        src = NumpyVectorSpace(1000)
        dims.append(dict(options=o,
                         srht=int(E.SrhtEmbedding(source=src, options=dict(opt), _seed=1).compute_dim()),
                         gauss=int(E.BlockGaussianEmbedding(source=NumpyVectorSpace(3), options=dict(opt, max_block_size=10 ** 9), _seed=1).compute_dim())))
    meta["_dims"] = dims
    # EmbeddingVectorized (embeddings.py:318-369): vec of a (n_vectors, k1) block, then an inner embedding
    k1, nv, k2 = 7, 5, 6
    inner = E.GaussianEmbedding(source=NumpyVectorSpace(k1 * nv, id="VEC"), options={"range_dim": k2}, _seed=31)
    vec = E.EmbeddingVectorized(NumpyVectorSpace(k1, id="SK"), nv, inner, options={}, _seed=31)
    W = np.random.RandomState(77).standard_normal((nv, k1))
    out["vectorized__U"] = W
    out["vectorized__apply"] = vec.apply(NumpyVectorSpace(k1, id="SK").from_numpy(W)).to_numpy()
    meta["vectorized"] = dict(k1=k1, n_vectors=nv, k2=k2, seed=31, apply_adjoint_is_none=vec.apply_adjoint(None) is None,
                              range_dim_option=int(vec.options["range_dim"]))
    out["__meta__"] = np.array(json.dumps(meta))
    golden_archive.save(os.path.join(OUT, "embeddings_reference.npz"), out)   # equal attributes stored once
    return len(out)


# ------------------------------------------------------------------ SketchedReductor
def thermal_like_problem(nx=12, seed=0):
    """A small SPD affine problem: A(mu) = A_0 + mu_0 A_1 + mu_1 A_2, f(mu) = f_0 + mu_0 f_1,
    two output functionals, inner product R = K + I."""
    n = nx * nx
    e = np.ones(nx)
    T1 = sp.diags([-e[:-1], 2 * e, -e[:-1]], [-1, 0, 1])
    K = (sp.kron(sp.eye(nx), T1) + sp.kron(T1, sp.eye(nx))).tocsc()
    A = []
    for s in (1, 2, 3):
        d = np.random.RandomState(seed + s).uniform(0.2, 1.0, n)
        D = sp.diags(d)
        A.append((D @ K @ D + sp.diags(d)).tocsc())
    rs = np.random.RandomState(seed)
    f = [rs.standard_normal(n) for _ in range(2)]
    out = rs.standard_normal((2, n))
    R = (K + sp.eye(n)).tocsc()
    return n, A, f, out, R


def make_reductor(E, SR, F):
    from pymor.models.basic import StationaryModel
    from pymor.operators.constructions import LincombOperator, VectorOperator
    from pymor.operators.numpy import NumpyMatrixOperator
    from pymor.parameters.base import Mu
    from pymor.parameters.functionals import ProjectionParameterFunctional

    n, A, f, outm, R = thermal_like_problem()
    rec = {}
    for q, a in enumerate(A):
        a = a.tocsr()
        rec[f"A{q}__data"], rec[f"A{q}__indices"], rec[f"A{q}__indptr"] = a.data, a.indices, a.indptr
    Rc = R.tocsr()
    rec["R__data"], rec["R__indices"], rec["R__indptr"] = Rc.data, Rc.indices, Rc.indptr
    rec["f"] = np.array(f)
    rec["out"] = outm
    A_ops = [NumpyMatrixOperator(a, source_id="S", range_id="S") for a in A]
    space = A_ops[0].source
    th = [ProjectionParameterFunctional("mu", 2, 0), ProjectionParameterFunctional("mu", 2, 1)]
    op = LincombOperator(A_ops, [1.0, th[0], th[1]])
    rhs = LincombOperator([VectorOperator(space.from_numpy(v)) for v in f], [1.0, th[0]])
    fom = StationaryModel(op, rhs, NumpyMatrixOperator(outm, source_id="S"))
    Rop = NumpyMatrixOperator(R, source_id="S", range_id="S")
    Rinv = F.InverseLuOperator(Rop)                      # utilities/factorization.py:88-138
    train = [[0.5, 1.5], [1.0, 0.3], [2.0, 2.0], [0.1, 0.7], [1.3, 1.1]]
    test = [[0.7, 0.9], [1.8, 0.2]]
    U = np.vstack([fom.solve(Mu(mu=m)).to_numpy() for m in train])
    rec["U"] = U
    meta = dict(n=n, k=40, k_online=20, seed_primal=11, seed_online=12, blocks=[2, 3], train=train, test=test,
                reduce_seed=5, minres_seeds=[5, 6], configs=[])
    for tag, kind in (("gauss", "GaussianEmbedding"), ("srht", "SrhtEmbedding")):
        for projection in ("galerkin", "minres"):
            emb = getattr(E, kind)(source=space, options={"range_dim": meta["k"]}, _seed=meta["seed_primal"], range_id="SK")
            onl = E.GaussianEmbedding(source=emb.range, options={"range_dim": meta["k_online"]}, _seed=meta["seed_online"])
            red = SR.SketchedReductor(fom, embedding_primal=emb, embedding_online=onl, product=Rop,
                                      inverse_product=Rinv, projection=projection, orthonormalize=False)
            pre = f"{tag}_{projection}"
            if projection == "galerkin":
                rom0 = red.reduce()                                             # _reduce_empty, :189-208
                for j, m in enumerate(test):
                    u0 = rom0.solve(Mu(mu=m))
                    rec[f"{pre}__empty_sol{j}"] = u0.to_numpy()
                    rec[f"{pre}__empty_est{j}"] = np.asarray(rom0.estimate_error(Mu(mu=m)))
            off = 0
            for b, nb in enumerate(meta["blocks"]):
                Ub = space.from_numpy(U[off:off + nb].copy())
                red.extend_basis(Ub)                                            # :49-83 (orthonormalize=False)
                rec[f"{pre}__srb_raw{b}"] = red.srb.to_numpy().copy()
                rec[f"{pre}__lhs_raw{b}"] = np.array([o.matrix for o in red.residual.operator.operators])
                T = red.orthonormalize_basis(offset=len(red.srb) - nb, return_T=True)   # :85-86 -> :90-118
                rec[f"{pre}__T{b}"] = T
                rec[f"{pre}__srb{b}"] = red.srb.to_numpy().copy()
                rec[f"{pre}__rb{b}"] = red.rb.to_numpy().copy()
                rec[f"{pre}__lhs{b}"] = np.array([o.matrix for o in red.residual.operator.operators])
                rec[f"{pre}__out{b}"] = np.asarray(red.output_functional.matrix)
                off += nb
            rec[f"{pre}__rhs"] = np.array([o.array.to_numpy()[0] for o in red.residual.rhs.operators])
            if projection == "galerkin":
                rom = red.reduce(seed=meta["reduce_seed"])                      # :121-129, :154-168
                rec[f"{pre}__red_lhs"] = np.array([o.matrix for o in rom.operator.operators])
                rec[f"{pre}__red_rhs"] = np.array([o.matrix for o in rom.rhs.operators])
            else:
                rom = red.reduce(seed=tuple(meta["minres_seeds"]))              # :131-137, :170-187
                rec[f"{pre}__ls_lhs"] = np.array([o.matrix for o in rom.operator.operator.operators])
                rec[f"{pre}__ls_rhs"] = np.array([o.array.to_numpy()[0] for o in rom.rhs.operators])
            est_ops = rom.error_estimator.operator
            rec[f"{pre}__est_lhs"] = np.array([o.matrix for o in est_ops.operator.operators])
            rec[f"{pre}__est_rhs"] = np.array([o.array.to_numpy()[0] for o in est_ops.rhs.operators])
            for j, m in enumerate(test):
                mu = Mu(mu=m)
                u = rom.solve(mu)
                rec[f"{pre}__sol{j}"] = u.to_numpy()
                rec[f"{pre}__est{j}"] = np.asarray(rom.estimate_error(mu))
                rec[f"{pre}__output{j}"] = rom.output(mu)
            meta["configs"].append(pre)
    rec["__meta__"] = np.array(json.dumps(meta))
    np.savez_compressed(os.path.join(OUT, "reductor_reference.npz"), **rec)
    return len(rec)


def main():
    assert os.path.isdir(REFERENCE), "the reference tree is only present in the build container"
    os.makedirs(OUT, exist_ok=True)
    E, SR, F = import_reference()
    print("embeddings_reference.npz:", make_embeddings(E), "arrays")
    print("reductor_reference.npz:", make_reductor(E, SR, F), "arrays")
    for fn in ("embeddings_reference.npz", "reductor_reference.npz"):
        print(fn, os.path.getsize(os.path.join(OUT, fn)))


if __name__ == "__main__":
    main()
