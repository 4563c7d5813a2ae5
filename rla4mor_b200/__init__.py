"""rla4mor_b200 -- B200-native sketching engine behind rla4mor's embedding API.

Only the hot path of alexandre-pasco/rla4mor lives here: applying random
embeddings Theta (k x n) to blocks of vectors, behind the reference's
`rla/srht.py` and `rla/embeddings.py` interfaces.  Arithmetic runs in
hand-written sm_100a CUDA kernels (`csrc/`, built into librla_b200.so and bound
through the C ABI in include/rla_b200.h); there is no CPU fallback.
"""
from ._lib import RlaError, lib, LIB_PATH, EXPORTED_SYMBOLS  # noqa: F401
from .srht import srht, fht_oop, fht_ip, SrhtPlan, get_plan, draw_signs_and_indices  # noqa: F401

from .vectorarray import DeviceVectorSpace, DeviceVectorArray, IdentityOperator, MatrixOperator  # noqa: F401
from .embeddings import (RandomEmbedding, SrhtEmbedding, GaussianEmbedding, IdentityEmbedding,  # noqa: F401
                         EmbeddingVectorized, BlockGaussianEmbedding, FrozenDict)
from .sketched_reductor import SketchedReductor  # noqa: F401
from .greedy import rb_greedy  # noqa: F401

__all__ = ["RandomEmbedding", "SrhtEmbedding", "GaussianEmbedding", "IdentityEmbedding", "EmbeddingVectorized",
           "BlockGaussianEmbedding", "SketchedReductor", "rb_greedy", "DeviceVectorSpace", "DeviceVectorArray",
           "IdentityOperator", "MatrixOperator","srht", "fht_oop", "fht_ip", "SrhtPlan", "get_plan", "draw_signs_and_indices",
           "RlaError", "lib"]
