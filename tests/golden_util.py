"""Helpers shared by the golden-vector tests (inputs are regenerated from seeds
exactly as oracle/make_golden.py created them)."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def make_input(shape, seed, cplx=False):
    rs = np.random.RandomState(seed)
    x = rs.standard_normal(shape)
    if cplx:
        x = x + 1j * rs.standard_normal(shape)
    return x


def srht_cases():
    z = np.load(os.path.join(GOLDEN, "srht_reference.npz"))
    names = sorted({k.split("__")[0] for k in z.files})
    for name in names:
        m, n, k, seed, cplx = (int(v) for v in z[name + "__meta"])
        shape = (n,) if m < 0 else (m, n)
        x = z[name + "__x"]
        if x.size == 0:
            x = make_input(shape, 1000 + seed, bool(cplx))
        yield dict(name=name, x=x, y=z[name + "__y"], k=k, seed=seed, n=n,
                   signs=z[name + "__signs"], sampling=z[name + "__sampling"], cplx=bool(cplx))


def fht_cases():
    z = np.load(os.path.join(GOLDEN, "fht_reference.npz"))
    tags = sorted({k.split("__")[0] for k in z.files})
    for tag in tags:
        yield dict(name=tag, a=z[tag + "__a"], oop=z[tag + "__oop"], ip=z[tag + "__ip"])


def emb_golden():
    return np.load(os.path.join(GOLDEN, "embeddings_transcribed.npz"))


def emb_reference():
    """embeddings_reference.npz: equal attributes are stored once (oracle/golden_archive.py)."""
    from oracle import golden_archive
    return golden_archive.load(os.path.join(GOLDEN, "embeddings_reference.npz"))


def rel_fro(a, b):
    a = np.asarray(a)
    b = np.asarray(b)
    den = np.linalg.norm(b.ravel())
    return float(np.linalg.norm((a - b).ravel()) / (den if den > 0 else 1.0))
