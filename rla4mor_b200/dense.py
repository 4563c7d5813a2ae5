"""Device-level wrappers of the dense-embedding kernels (csrc/gemm.cu, csrc/rng.cuh).

Y(m, k) = U(m, n) Theta(k, n)^T in FP64 on the tensor pipe, with Theta explicit
(`gauss_apply_explicit`, the reference's `(Theta @ (QU)^T)^T`, rla/embeddings.py:250-254)
or generated on the fly from the counter-based RNG (`embed_apply_rng`), the adjoint
V(m, k) Theta(k, n) with the same on-the-fly Theta (`embed_adjoint_rng`, csrc/adjoint_rng.cu),
plus the export of what that generator produces (`theta_materialize`, parity tooling).
All inputs are CUDA tensors; there is no CPU path.
"""
import numpy as np
import torch

from ._lib import check, lib, stream_ptr

KIND_NORMAL = 0
KIND_RADEMACHER = 1
KIND_NORMAL_TF32 = 2      # the normals of kind 0 rounded to TF32: exact operands of tcgen05.mma kind::tf32

def _workspace(nbytes, device):
    """Scratch for one call, taken from torch's caching allocator: it is tied to the current
    stream, so concurrent calls on different streams never share a buffer."""
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def _rows(x):
    """A 2-D CUDA tensor with unit inner stride (copy only if needed)."""
    assert x.is_cuda and x.dim() == 2
    if x.stride(1) != 1 or (x.shape[0] > 1 and x.stride(0) < x.shape[1]):
        x = x.contiguous()
    return x


def _ld(x):
    """Leading dimension handed to the kernels.  A single row has no meaningful stride of its own
    (torch reports anything for a size-1 dimension): use the stride when it can be one (a row of
    a padded buffer, as `_tma_friendly` builds for odd n), else the row length."""
    if x.shape[0] > 1:
        return max(x.stride(0), x.shape[1])
    return x.stride(0) if x.stride(0) >= x.shape[1] else x.shape[1]


def _tma_friendly(x):
    """TMA needs a 16-byte aligned base and an even row stride; copy into a padded
    buffer otherwise (odd n)."""
    if x.data_ptr() % 16 == 0 and _ld(x) % 2 == 0:
        return x
    m, n = x.shape
    buf = torch.zeros((m, n + (n & 1)), dtype=x.dtype, device=x.device)
    buf[:, :n] = x
    return buf[:, :n]


def gauss_apply_explicit(theta, u, out=None):
    """(m, n) x (k, n)^T -> (m, k), float64."""
    theta, u = _tma_friendly(_rows(theta)), _tma_friendly(_rows(u))
    assert theta.dtype == torch.float64 and u.dtype == torch.float64
    k, n = theta.shape
    m = u.shape[0]
    assert u.shape[1] == n
    if out is None:
        out = torch.empty((m, k), dtype=torch.float64, device=u.device)
    if m == 0 or k == 0:
        return out
    with torch.cuda.device(u.device):
        ws = _workspace(lib().rla_gemm_workspace_bytes(m, k, n), u.device)
        check(lib().rla_gauss_apply_explicit_f64(theta.data_ptr(), k, n, _ld(theta), u.data_ptr(), m, _ld(u),
                                                 out.data_ptr(), out.stride(0), ws.data_ptr(), ws.numel(),
                                                 stream_ptr()), "rla_gauss_apply_explicit_f64")
    return out


def _tma_friendly_f32(x):
    """float32 rows for TMA: 16-byte aligned base, row stride a multiple of 4 elements."""
    if x.data_ptr() % 16 == 0 and _ld(x) % 4 == 0:
        return x
    m, n = x.shape
    buf = torch.zeros((m, (n + 3) // 4 * 4), dtype=x.dtype, device=x.device)
    buf[:, :n] = x
    return buf[:, :n]


def embed_apply_rng(seed, kind, scale, k, u, row0=0, col0=0, out=None, accumulate=False):
    """Sketch u (m, n) with rows [row0, row0 + k) and columns [col0, col0 + n) of the
    virtual matrix scale * g(seed, row, col); the matrix is never materialised.

    float64 blocks with the FP32 normals of KIND_NORMAL / KIND_NORMAL_TF32 run on the int8 tensor
    cores (csrc/gemm_i8.cu: Theta and per-2^14-column-block scaled U cut into eight 7-bit slices,
    36 exact int8 slice products, FP64 accumulation).  Its error is bounded NORMWISE, about
    2^-49 sqrt(2^14) ||u|| ||theta|| per entry whatever the dynamic range of u (the exact bound is in
    the header of gemm_i8.cu); the componentwise bound in sum |theta| |u| of an FP64 dot product is
    not kept: an entry far below the largest of its 2^14-column block loses its low bits.  Blocks
    with a non-finite entry or one near the FP64 overflow limit, and KIND_RADEMACHER, run on the
    FP64 tensor pipe (csrc/gemm.cu).  float32 blocks with a Theta that
    is exact in TF32 (KIND_RADEMACHER, KIND_NORMAL_TF32) run on the generation-5 tensor cores
    (csrc/gemm32.cu: tcgen05 kind::tf32, two-part split of the block, FP64 accumulation of the
    64-term partial sums); the sketch comes back as float64 either way."""
    if u.dtype == torch.float32 and kind in (KIND_RADEMACHER, KIND_NORMAL_TF32) and col0 % 32 == 0:
        u = _tma_friendly_f32(_rows(u))
        m, n = u.shape
        if out is None:
            assert not accumulate
            out = torch.empty((m, k), dtype=torch.float64, device=u.device)
        if m == 0 or k == 0:
            return out
        with torch.cuda.device(u.device):
            ws = _workspace(lib().rla_gemm32_workspace_bytes(m, k, n), u.device)
            check(lib().rla_embed_apply_rng_f32(int(seed) & (2 ** 64 - 1), int(kind), float(scale), int(row0), int(k),
                                                int(col0), n, u.data_ptr(), m, _ld(u), out.data_ptr(), out.stride(0),
                                                1 if accumulate else 0, ws.data_ptr(), ws.numel(), stream_ptr()),
                  "rla_embed_apply_rng_f32")
        return out
    if u.dtype == torch.float32:
        u = u.to(torch.float64)
    u = _tma_friendly(_rows(u))
    assert u.dtype == torch.float64
    m, n = u.shape
    if out is None:
        assert not accumulate
        out = torch.empty((m, k), dtype=torch.float64, device=u.device)
    if m == 0 or k == 0:
        return out
    with torch.cuda.device(u.device):
        ws = _workspace(lib().rla_gemm_rng_workspace_bytes(m, k, n), u.device)
        check(lib().rla_embed_apply_rng_f64(int(seed) & (2 ** 64 - 1), int(kind), float(scale), int(row0), int(k),
                                            int(col0), n, u.data_ptr(), m, _ld(u), out.data_ptr(), out.stride(0),
                                            1 if accumulate else 0, ws.data_ptr(), ws.numel(), stream_ptr()),
              "rla_embed_apply_rng_f64")
    return out


def embed_adjoint_rng(seeds, row_starts, kind, scale, v, n):
    """out(m, n) = v(m, k) @ Theta(k, n) with Theta generated in the kernel (csrc/adjoint_rng.cu),
    never materialised.  Theta stacks len(seeds) blocks: rows [row_starts[b], row_starts[b + 1]) are
    rows 0 .. size_b - 1 of the virtual matrix scale * g(seeds[b], row, col) that `theta_materialize`
    exports.  Bit-identical to `gemm_nn(v, Theta)` when that product runs on its tensor-pipe path
    (16-byte aligned operands, even leading dimensions).  A float32 v is widened to float64."""
    seeds = np.asarray([int(s) & (2 ** 64 - 1) for s in seeds], dtype=np.uint64)
    row_starts = np.asarray(row_starts, dtype=np.int64)
    nblocks = len(seeds)
    assert nblocks >= 1 and row_starts.shape == (nblocks + 1,) and row_starts[0] == 0, "bad block table"
    assert np.all(np.diff(row_starts) >= 0) and np.all(np.diff(row_starts) < 2 ** 32), "bad block table"
    if v.dtype == torch.float32:
        v = v.to(torch.float64)
    v = _rows(v)
    assert v.dtype == torch.float64
    m, k = v.shape
    n = int(n)
    assert k == row_starts[-1], f"v has {k} columns, the blocks {row_starts[-1]} rows"
    out = torch.empty((m, n), dtype=torch.float64, device=v.device)
    if m == 0 or n == 0:
        return out
    with torch.cuda.device(v.device):
        table = torch.from_numpy(np.concatenate([seeds.view(np.int64), row_starts])).to(v.device)
        check(lib().rla_embed_adjoint_rng_f64(int(kind), float(scale), table.data_ptr(), table[nblocks:].data_ptr(),
                                              nblocks, n, v.data_ptr(), m, _ld(v), out.data_ptr(), out.stride(0),
                                              stream_ptr()), "rla_embed_adjoint_rng_f64")
    return out


def theta_materialize(seed, kind, scale, rows, cols, row0=0, col0=0, device=None):
    """The (rows, cols) block of the virtual matrix, bit-identical to what
    `embed_apply_rng` multiplies by."""
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    out = torch.empty((rows, cols), dtype=torch.float64, device=device)
    if rows == 0 or cols == 0:
        return out
    with torch.cuda.device(device):
        check(lib().rla_theta_materialize_f64(int(seed) & (2 ** 64 - 1), int(kind), float(scale), int(row0), rows,
                                              int(col0), cols, out.data_ptr(), out.stride(0), stream_ptr()),
              "rla_theta_materialize_f64")
    return out
