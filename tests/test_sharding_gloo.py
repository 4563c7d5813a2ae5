"""Host logic of the multi-GPU paths on CPU: world_size-2 (and 4) gloo groups.
The local sketches are computed with the oracle here (no GPU in this tier); on the GPU
the same functions run with the CUDA kernels (tests/test_sharding_gpu.py)."""
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle
from oracle import embeddings_oracle as eo
from rla4mor_b200 import sharding


def test_partition_arithmetic():
    assert [sharding.column_shard(10, r, 4) for r in range(4)] == [(0, 3), (3, 6), (6, 8), (8, 10)]
    assert sharding.column_shard(3, 3, 4) == (3, 3)
    sl = sharding.gaussian_slabs(1000, 3)
    assert sl[0][0] == 0 and sl[-1][1] == 1000 and all(lo % 16 == 0 for lo, _ in sl)
    assert all(a[1] == b[0] for a, b in zip(sl, sl[1:]))
    slab, rg = sharding.srht_slabs(5000, 4)
    assert slab == 2048 and rg == [(0, 2048), (2048, 4096), (4096, 5000), (5000, 5000)]


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _worker(rank, world, port, n, k, seed, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        x = np.random.RandomState(0).standard_normal((3, n))
        # --- row-sharded SRHT: H_{2^d} = H_G (x) H_{2^d/G}
        signs = oracle.rademacher_signs(n, seed)
        samp = oracle.sampling_indices(n, k, seed)
        lo, hi, lsigns, lidx, fac = sharding.srht_slab_descriptor(signs, samp, n, rank, world)
        slab = sharding.srht_slabs(n, world)[0]

        def local():
            xs = np.zeros((3, slab)); xs[:, :hi - lo] = x[:, lo:hi] * lsigns
            z = oracle.fht_oop(xs) * np.sqrt(slab)                      # unnormalised slab transform
            return torch.from_numpy(z[:, lidx] / np.sqrt(k))
        y = sharding.row_sharded_sketch(local, torch.from_numpy(fac))
        # --- row-sharded Gaussian: Theta[:, slab]
        theta = eo.gaussian_random_matrix(k, n, seed)
        glo, ghi = sharding.gaussian_slabs(n, world)[rank]
        yg = sharding.row_sharded_sketch(lambda: torch.from_numpy(x[:, glo:ghi] @ theta[:, glo:ghi].T))
        # --- column-sharded: no collective, gather only to compare
        clo, chi = sharding.column_shard(3, rank, world)
        part = torch.zeros(3, k, dtype=torch.float64)
        if chi > clo:
            part[clo:chi] = torch.from_numpy(oracle.srht(x[clo:chi], k, seed=seed))
        yc = sharding.all_reduce_sum(part)
        # --- Theta-row-sharded (k split): disjoint slices of the sketch, one all-gather, no reduction
        yt = sharding.theta_row_sharded_sketch(lambda lo, hi: torch.from_numpy(x @ theta[lo:hi].T), k, rank, world)
        sl, rng = sharding.theta_row_sharded_sketch(lambda lo, hi: torch.from_numpy(x @ theta[lo:hi].T), k, rank, world,
                                                    gather=False)
        assert rng == sharding.theta_row_shard(k, rank, world) and sl.shape == (3, rng[1] - rng[0])
        # blocks of a BlockGaussianEmbedding dealt to the ranks (embeddings.py:393-407): uneven column
        # ranges, an empty one with world 4
        sizes = eo.block_sizes(k, 7)
        seeds, _ = eo.block_seeds(seed, len(sizes))
        offs = np.concatenate([[0], np.cumsum(sizes)])
        shards = [sharding.block_shard(len(sizes), g, world) for g in range(world)]
        ranges = [(int(offs[b[0]]), int(offs[b[-1] + 1])) if b else (0, 0) for b in shards]

        def local_blocks(lo, hi):
            cols = [x @ eo.block_gaussian_block(k, n, sizes[i], seeds[i]).T for i in shards[rank]]
            return torch.from_numpy(np.hstack(cols) if cols else np.zeros((3, 0)))
        yb = sharding.theta_row_sharded_sketch(local_blocks, k, rank, world, ranges=ranges)
        if rank == 0:
            np.savez(out, y=y.numpy(), yg=yg.numpy(), yc=yc.numpy(), yt=yt.numpy(), yb=yb.numpy())
    finally:
        dist.destroy_process_group()


def _run(world, n, k, seed, tmp_path):
    out = str(tmp_path / f"res_{world}_{n}.npz")
    mp.spawn(_worker, args=(world, _free_port(), n, k, seed, out), nprocs=world, join=True)
    z = np.load(out)
    x = np.random.RandomState(0).standard_normal((3, n))
    ref = oracle.srht(x, k, seed=seed)
    assert np.linalg.norm(z["y"] - ref) / np.linalg.norm(ref) < 1e-13
    assert np.linalg.norm(z["yc"] - ref) / np.linalg.norm(ref) == 0.0
    refg = eo.gaussian_apply(x, eo.gaussian_random_matrix(k, n, seed))
    assert np.linalg.norm(z["yg"] - refg) / np.linalg.norm(refg) < 1e-13
    # k split: the same dot products (BLAS may block them differently on the host: rounding only)
    assert np.linalg.norm(z["yt"] - refg) / np.linalg.norm(refg) < 1e-14
    refb = eo.block_gaussian_apply(x, k, seed, 7)
    assert np.linalg.norm(z["yb"] - refb) / np.linalg.norm(refb) < 1e-14


def test_world2_pow2(tmp_path):
    _run(2, 4096, 40, 3, tmp_path)


def test_world2_ragged(tmp_path):
    _run(2, 5000, 33, 7, tmp_path)


def test_world4_ragged_with_empty_slab(tmp_path):
    _run(4, 5000, 20, 1, tmp_path)
