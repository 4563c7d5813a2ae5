"""Multi-GPU partitioning of the sketch (one process per GPU, torch.distributed).

Two modes (SURVEY.md section 8e):

* column-sharded (default): the m vectors of the block -- rows of the (m, n) array,
  columns of the n x m matrix -- are split across ranks; the embedding descriptor
  (seed, signs, indices) is replicated.  Units are independent: NO collective.  This is
  the reference's only parallelism (numba prange over rows, rla/srht.py:93-96).

* row-sharded (very tall n): the vector dimension is split into contiguous slabs, one
  per rank; every rank sketches its slab and the (m, k) partial sketches are summed with
  ONE all-reduce (NCCL over NVLink on GPUs).
    - Gaussian / Rademacher: rank g applies Theta[:, slab_g] (column offset into the
      virtual matrix).
    - SRHT: H_{2^d} = H_G (x) H_{2^d/G} for a power-of-two world size G: rank g runs the
      SRHT kernel on its slab with the low index bits s & (slab - 1) and its slice of the
      signs, then flips sample i by (-1)^popcount((s_i >> log2 slab) & g).
  Summation order differs from the single-GPU kernel, so results agree to rounding
  (1e-15 relative), not bit for bit.

The functions that touch data take the local sketch as a callable, so the host logic
(partitioning, sign factors, the collective) is testable on CPU with the gloo backend.
"""
import numpy as np


def column_shard(m, rank, world):
    """Half-open range [lo, hi) of the vectors owned by `rank` (balanced, contiguous)."""
    base, rem = divmod(int(m), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def gaussian_slabs(n, world, align=16):
    """Contiguous slabs of the vector dimension, boundaries multiples of `align`
    (the GEMM kernel needs col0 % 16 == 0)."""
    per = -(-int(n) // int(world))
    per = -(-per // align) * align
    return [(min(g * per, n), min((g + 1) * per, n)) for g in range(world)]


def srht_slabs(n, world):
    """Power-of-two slabs of the padded length 2^d; returns (slab_size, [(lo, hi)] clipped to n)."""
    assert world & (world - 1) == 0, "row-sharded SRHT needs a power-of-two world size"
    d = int(np.ceil(np.log2(n))) if n > 1 else 0
    assert (1 << d) >= world, "more ranks than padded elements"
    slab = (1 << d) // world
    return slab, [(min(g * slab, n), min((g + 1) * slab, n)) for g in range(world)]


def srht_slab_descriptor(signs, sampling, n, rank, world):
    """What rank `rank` needs to sketch its slab with the ordinary SRHT kernel:
    (lo, hi, local signs, local indices, +-1 factor per sample)."""
    slab, ranges = srht_slabs(n, world)
    lo, hi = ranges[rank]
    s = np.asarray(sampling, dtype=np.int64)
    local_idx = s & (slab - 1)
    high = s // slab
    par = np.zeros(len(s), dtype=np.int64)
    v = high & rank
    while np.any(v):
        par ^= v & 1
        v >>= 1
    return lo, hi, np.asarray(signs)[lo:hi], local_idx, 1.0 - 2.0 * par


def all_reduce_sum(t, group=None):
    """Sum a tensor over the ranks (no-op without an initialised process group)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


def row_sharded_sketch(local_sketch, factor=None, group=None):
    """partial = local_sketch() [* factor per sample]; returns the all-reduced (m, k) sketch."""
    part = local_sketch()
    if factor is not None:
        part = part * factor
    return all_reduce_sum(part, group)


# ------------------------------------------------------------------ Theta-row-sharded (k split)
def theta_row_shard(k, rank, world):
    """Half-open range [lo, hi) of the SKETCH rows (rows of Theta) owned by `rank`: the
    BlockGaussianEmbedding decomposition (rla/embeddings.py:393-400) spread over ranks.  Every rank
    holds the whole block U; the sketch comes out split along k."""
    return column_shard(k, rank, world)


def block_shard(n_blocks, rank, world):
    """Blocks of a BlockGaussianEmbedding owned by `rank` (contiguous, balanced)."""
    lo, hi = column_shard(n_blocks, rank, world)
    return list(range(lo, hi))


def theta_row_sharded_sketch(local_sketch, k, rank, world, group=None, gather=True, ranges=None):
    """local_sketch(lo, hi) -> this rank's (m, hi - lo) columns of the sketch (rows lo..hi of Theta
    applied to the replicated block).  `ranges` holds every rank's [lo, hi), `theta_row_shard` by
    default.  No reduction is needed -- the slices are disjoint; with `gather` they are concatenated
    along k on every rank by ONE all-gather, else the local slice and its range are returned."""
    import torch
    import torch.distributed as dist
    if ranges is None:
        ranges = [theta_row_shard(k, g, world) for g in range(world)]
    lo, hi = ranges[rank]
    part = local_sketch(lo, hi)
    if not gather:
        return part, (lo, hi)
    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1):
        return part
    m = part.shape[0]
    width = max(ghi - glo for glo, ghi in ranges)     # slices may differ in width: pad to the widest
    buf = torch.zeros((m, width), dtype=part.dtype, device=part.device)
    buf[:, :hi - lo] = part
    parts = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(parts, buf, group=group)
    return torch.cat([parts[g][:, :ghi - glo] for g, (glo, ghi) in enumerate(ranges)], dim=1)


# --------------------------------------------------------------------- device front ends
def gaussian_theta_row_sharded(x, k, seed, rank, world, kind=0, group=None, gather=True):
    """Theta-row-sharded on-the-fly Gaussian / Rademacher sketch on the GPU: rank g generates and
    applies rows [lo_g, hi_g) of the virtual k x n matrix (`row0` of rla_embed_apply_rng_f64) to the
    replicated block x (m, n).  Equal to the single-GPU sketch column for column (same Philox
    counters), bit for bit."""
    from . import dense

    def local(lo, hi):
        return dense.embed_apply_rng(seed, kind, 1.0 / np.sqrt(k), hi - lo, x, row0=lo)
    return theta_row_sharded_sketch(local, k, rank, world, group, gather)


def block_gaussian_theta_row_sharded(embedding, U, rank, world, group=None, gather=True):
    """BlockGaussianEmbedding.apply (rla/embeddings.py:425-434) with the row blocks of Theta dealt to
    the ranks: each rank regenerates only its own blocks (per-block seeds, :402-407) and the
    hstack of :433 becomes an all-gather.  U: replicated CUDA block (m, n)."""
    import torch
    from .vectorarray import as_device_block
    V = as_device_block(U).to(torch.float64)
    offs = np.concatenate([[0], np.cumsum(embedding.block_sizes)])
    shards = [block_shard(embedding.n_blocks, g, world) for g in range(world)]
    ranges = [(int(offs[b[0]]), int(offs[b[-1] + 1])) if b else (0, 0) for b in shards]
    return theta_row_sharded_sketch(lambda lo, hi: embedding.sketch_blocks(V, shards[rank]), int(offs[-1]), rank,
                                    world, group, gather, ranges)


def srht_row_sharded(x_slab, n, k, seed, rank, world, group=None, reducer=None, check=True):
    """Row-sharded SRHT on the GPU: x_slab is this rank's (m, hi - lo) CUDA slab.

    With `reducer` (a peer.PeerSketchReducer for this (m, k)) the local kernel writes its
    partial into peer-mapped memory and ONE kernel applies the slab signs and sums over
    NVLink (csrc/peer.cu); without it the partial is scaled and all-reduced by NCCL."""
    import torch
    from .srht import SrhtPlan, draw_signs_and_indices
    m = x_slab.shape[0]
    slab, ranges = srht_slabs(n, world)
    lo, hi = ranges[rank]
    key = (int(n), int(k), None if seed is None else int(seed), int(rank), int(world), x_slab.dtype, x_slab.device.index)
    desc = _SLAB_PLANS.get(key) if seed is not None else None
    if desc is None:
        # the host draws cost seconds at n = 2**24: once per (seed, n, k, rank, world)
        signs, sampling = draw_signs_and_indices(n, k, seed)
        _, _, lsigns, lidx, fac = srht_slab_descriptor(signs, sampling, n, rank, world)
        plan = None
        if hi > lo:
            if hi - lo < slab:
                lsigns = np.concatenate([lsigns, np.ones(slab - (hi - lo), dtype=lsigns.dtype)])
            plan = SrhtPlan(slab, k, lsigns, lidx, x_slab.dtype, x_slab.device)
        factor = torch.as_tensor(fac, dtype=x_slab.dtype, device=x_slab.device)
        high = torch.as_tensor((np.asarray(sampling, dtype=np.int64) // slab).astype(np.int32), device=x_slab.device)
        desc = (plan, factor, high)
        if seed is not None:
            _SLAB_PLANS[key] = desc
            while len(_SLAB_PLANS) > 8:
                _SLAB_PLANS.pop(next(iter(_SLAB_PLANS)))
    plan, factor, high = desc
    if hi > lo:
        assert x_slab.shape[1] == hi - lo
        if hi - lo < slab:
            # ragged last slab: pad to the slab length so the local indices stay in range
            xp = torch.zeros((m, slab), dtype=x_slab.dtype, device=x_slab.device)
            xp[:, :hi - lo] = x_slab
            x_slab = xp
    scale = 1.0 / np.sqrt(k)
    if reducer is not None:
        assert x_slab.dtype == torch.float64 and (reducer.m, reducer.k) == (m, k)
        part = reducer.partial()
        if hi > lo:
            plan.apply(x_slab, scale=scale, out=part)
        else:
            part.zero_()
        out = reducer.reduce(high=high)
        if check:
            reducer.check_status()      # synchronises; pass check=False inside timed loops and check once afterwards
        return out
    if hi <= lo:
        return all_reduce_sum(torch.zeros((m, k), dtype=x_slab.dtype, device=x_slab.device), group)
    return row_sharded_sketch(lambda: plan.apply(x_slab, scale=scale), factor, group)


_SLAB_PLANS = {}


def gaussian_row_sharded(x_slab, n, k, seed, rank, world, kind=0, group=None, reducer=None, check=True):
    """Row-sharded on-the-fly Gaussian / Rademacher sketch on the GPU (`reducer`: see srht_row_sharded)."""
    import torch
    from . import dense
    lo, hi = gaussian_slabs(n, world)[rank]
    m = x_slab.shape[0]
    if reducer is not None:
        assert (reducer.m, reducer.k) == (m, k)
        part = reducer.partial()
        if hi > lo:
            assert x_slab.shape[1] == hi - lo
            dense.embed_apply_rng(seed, kind, 1.0 / np.sqrt(k), k, x_slab, col0=lo, out=part)
        else:
            part.zero_()
        out = reducer.reduce()
        if check:
            reducer.check_status()
        return out
    if hi <= lo:
        return all_reduce_sum(torch.zeros((m, k), dtype=torch.float64, device=x_slab.device), group)
    assert x_slab.shape[1] == hi - lo
    return row_sharded_sketch(lambda: dense.embed_apply_rng(seed, kind, 1.0 / np.sqrt(k), k, x_slab, col0=lo),
                              None, group)
