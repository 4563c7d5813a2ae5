"""The int8 sketch of float64 blocks (csrc/gemm_i8.cu) when one CTA of a cluster pair flushes several
exponent blocks: m = 256 is one pair of 128-row tiles, k = 4700 is 74 column tiles, so the pair's
148 CTAs fill a 148-SM B200 with one chunk of all three blocks of n = 40003 (bpc = 3).  The TMEM
hand-over between the pair's flush warps and its MMAs then runs twice per CTA.  A sample of sketch
columns must equal the NumPy replay of the slicing and flush order bit for bit."""
import numpy as np
import pytest
import torch

import ozaki_ref as oz

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("kind", [0, 2])
def test_pair_flushing_three_blocks_is_bitwise_equal_to_the_replay(kind):
    import rla4mor_b200
    rla4mor_b200.lib()
    from rla4mor_b200 import dense
    m, k, n, row0, col0 = 256, 4700, 40003, 7, 96
    rs = np.random.RandomState(17 + kind)
    u = rs.standard_normal((m, n)) * 2.0 ** rs.randint(-30, 30, (m, 1))
    u[3, 16384:32768] = 0.0                                         # an all-zero block in the middle
    u[200, :] *= 2.0 ** rs.randint(-40, 40, n)                       # a wide dynamic range inside blocks
    got = dense.embed_apply_rng(5, kind, 0.75, k, torch.from_numpy(u).cuda(), row0=row0, col0=col0).cpu().numpy()
    # both 32-row halves of the pair's Theta tile, the first and the last tile, and the ragged end
    cols = np.unique(np.concatenate([[0, 31, 32, 63, 64, 4607, 4608, 4640, 4699], rs.randint(0, k, 23)]))
    th = np.stack([dense.theta_materialize(5, kind, 1.0, 1, n, row0=row0 + int(c), col0=col0).cpu().numpy()[0]
                   for c in cols])
    want = oz.replay(u, th, 0.75)
    assert np.array_equal(got[:, cols], want)
