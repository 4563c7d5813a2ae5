"""Timing of the Gaussian embeddings' adjoint out(m, n) = V(m, k) Theta(k, n) with Theta generated in
the kernel (csrc/adjoint_rng.cu) against the two materialising paths it replaces, one JSON line per
shape after a line with the card's name, power limit and the FP64 tensor-pipe peak of the same run.

  new    dense.embed_adjoint_rng: Theta generated in the kernel, never in memory
  first  theta_materialize + gemm_nn: what GaussianEmbedding.apply_adjoint did on its first call
         (Theta written to HBM, then read once per 128 rows of V)
  warm   gemm_nn over an already materialised Theta: the later calls of that path

Shapes: (k, n) = (2000, 2^22), m in {1, 8, 64, 256} with one block, and BlockGaussianEmbedding's
blocks of 200 rows at m = 64.  Every path is warmed up, then timed with CUDA events over --reps calls.
Per path: ms, FP64 TFLOP/s = 2 m k n / t, the share of the same-run DMMA peak, Theta entries
generated per second (the new kernel generates Theta once per 128-row tile of V) and the peak device
memory of one call.  `equal` says whether the new result equals the warm path's bit for bit.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rla4mor_b200 as rb  # noqa: E402
from rla4mor_b200 import dense  # noqa: E402
from rla4mor_b200._lib import check, lib, stream_ptr  # noqa: E402
from rla4mor_b200.reductor_ops import gemm_nn  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--k", type=int, default=2000)
ap.add_argument("--logn", type=int, default=22)
ap.add_argument("--ms", default="1,8,64,256")
ap.add_argument("--block", type=int, default=200)
ap.add_argument("--block-m", type=int, default=64)
ap.add_argument("--reps", type=int, default=5)
a = ap.parse_args()
k, n = a.k, 2 ** a.logn
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip().splitlines()
gpu = (q[0].split(", ") + ["", "", ""])[:3] if q else ["", "", ""]
scratch = torch.empty(1 << 20, dtype=torch.uint8, device=dev)
peak = ctypes.c_double()
check(lib().rla_dmma_peak_tflops(ctypes.byref(peak), ctypes.c_void_p(scratch.data_ptr()), stream_ptr()), "dmma peak")
print(json.dumps({"gpu": gpu[0], "power_limit": gpu[1], "max_sm_clock": gpu[2], "dmma_peak_tflops": peak.value,
                  "k": k, "n": n}), flush=True)


def timed(f, reps):
    """(result of the last call, ms per call, peak bytes allocated during one call)"""
    f()                                                         # warm-up: module load, allocator
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    r = f()
    torch.cuda.synchronize()
    mem = torch.cuda.max_memory_allocated() - base
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        r = f()
    e1.record()
    torch.cuda.synchronize()
    return r, e0.elapsed_time(e1) / reps, mem


def materialize(seeds, sizes, scale):
    """The stacked Theta, each block written in place by rla_theta_materialize_f64."""
    theta = torch.empty((k, n), dtype=torch.float64, device=dev)
    off = 0
    for s, b in zip(seeds, sizes):
        check(lib().rla_theta_materialize_f64(s, dense.KIND_NORMAL, scale, 0, b, 0, n, theta[off].data_ptr(), n,
                                              stream_ptr()), "rla_theta_materialize_f64")
        off += b
    return theta


def row(name, m, seeds, sizes):
    scale = 1.0 / np.sqrt(k)
    starts = np.concatenate([[0], np.cumsum(sizes)])
    v = torch.randn(m, k, dtype=torch.float64, device=dev, generator=torch.Generator(device=dev).manual_seed(m))
    flop = 2.0 * m * k * n
    res = {"shape": name, "m": m, "k": k, "n": n, "blocks": len(sizes)}

    def entry(ms, mem, generated):
        t = ms * 1e-3
        return {"ms": ms, "tflops": flop / t / 1e12, "of_dmma_peak": flop / t / 1e12 / peak.value,
                "theta_entries_per_s": generated / t, "peak_mem_gb": mem / 1e9}

    new, ms, mem = timed(lambda: dense.embed_adjoint_rng(seeds, starts, dense.KIND_NORMAL, scale, v, n), a.reps)
    res["new"] = entry(ms, mem, -(-m // 128) * k * n)
    del new
    _, ms, mem = timed(lambda: gemm_nn(v, materialize(seeds, sizes, scale)), max(1, a.reps // 2))
    res["first"] = entry(ms, mem, k * n)
    theta = materialize(seeds, sizes, scale)
    warm, ms, mem = timed(lambda: gemm_nn(v, theta), a.reps)
    res["warm"] = entry(ms, mem, 0)
    del theta
    res["equal"] = bool(torch.equal(dense.embed_adjoint_rng(seeds, starts, dense.KIND_NORMAL, scale, v, n), warm))
    del warm
    torch.cuda.empty_cache()
    print(json.dumps(res), flush=True)


for m in (int(x) for x in a.ms.split(",")):
    row("gaussian", m, [21], [k])
emb = rb.BlockGaussianEmbedding(source=rb.DeviceVectorSpace(n), options={"range_dim": k, "max_block_size": a.block,
                                                                         "rng": "philox"}, _seed=21)
row(f"block{a.block}", a.block_m, [int(s) for s in emb.block_seeds], emb.block_sizes)
