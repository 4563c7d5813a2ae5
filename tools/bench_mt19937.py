"""Timing of the device MT19937 Gaussian draw (csrc/mt19937.cu) against NumPy's host draw, printed
as one JSON line with the card's name and power limit read in the same run.

  * the device draw of a (k, n) Theta (default 2000 x 2^20: 2.1e9 normals, 16.8 GB) split into
    plan (jump-ahead, acceptance count) and execute (write pass, host fix-up), with the kernel and
    copy times of a torch.profiler pass; the flagged fraction and the time of the C library's log
    over that many arguments on this host;
  * NumPy's legacy normal rate on the same host (a bounded sample of --numpy-sample normals);
  * GaussianEmbedding construction at (k, n) and BlockGaussianEmbedding.apply (max_block_size 200,
    m vectors), each for this code and for the parent's host-draw path (restated below: NumPy draws
    Theta, the block is uploaded, then the same GEMM), alternating new / parent / new.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rla4mor_b200 as rb  # noqa: E402
from rla4mor_b200 import dense, mt19937  # noqa: E402
from rla4mor_b200._lib import lib  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--k", type=int, default=2000)
ap.add_argument("--logn", type=int, default=20)
ap.add_argument("--m", type=int, default=64)
ap.add_argument("--block", type=int, default=200)
ap.add_argument("--numpy-sample", type=int, default=2 * 10 ** 7)
ap.add_argument("--skip-parent", action="store_true")
a = ap.parse_args()
k, n = a.k, 2 ** a.logn
scale = 1 / np.sqrt(k)
dev = torch.device("cuda", 0)
res = {"k": k, "n": n, "normals": k * n, "theta_gb": k * n * 8 / 1e9}

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                   text=True).stdout.strip().splitlines()
res["gpu"], res["power_limit"] = (q[0].split(", ") + [""])[:2] if q else ("", "")


def sync_time(f):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = f()
    torch.cuda.synchronize()
    return r, time.perf_counter() - t0


# ---- device draw, split into plan and execute (warm-up draw first: polynomials, module load)
mt19937.gaussian_matrix([1], [1], 1000, 1.0)
out = torch.empty(k * n, dtype=torch.float64, device=dev)
plan, t_plan = sync_time(lambda: mt19937.NormalPlan([123], [k * n], dev))
nflag, t_exec = sync_time(lambda: plan.execute(out, 0, k * n, 0, scale))
res.update(plan_s=t_plan, execute_s=t_exec, draw_s=t_plan + t_exec, flagged_pairs=nflag,
           flagged_fraction=nflag / ((k * n + 1) // 2), theta_gb_per_s=res["theta_gb"] / (t_plan + t_exec))
x = np.random.RandomState(0).random_sample(nflag) * 0.999 + 1e-4
y = np.empty_like(x)
_, res["host_log_s"] = sync_time(lambda: lib().rla_libm_log_host(x.ctypes.data, len(x), y.ctypes.data))
del x, y

from torch.profiler import ProfilerActivity, profile  # noqa: E402
with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    p2 = mt19937.NormalPlan([123], [k * n], dev)
    p2.execute(out, 0, k * n, 0, scale)
    torch.cuda.synchronize()
dev_ms = {}
for ev in prof.key_averages():
    name = ev.key
    for tag in ("mt_jump_kernel", "mt_count_kernel", "mt_write_kernel", "mt_fixup_kernel", "Memcpy DtoH", "Memcpy HtoD"):
        if tag in name:
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            dev_ms[tag] = dev_ms.get(tag, 0.0) + t / 1e3
res["device_ms"] = dev_ms
del p2, plan

# ---- check a sample of the draw against NumPy (first 10^6 normals)
ref = np.random.RandomState(123).normal(size=10 ** 6, loc=0, scale=scale)
res["sample_bit_identical"] = bool(np.array_equal(out[:10 ** 6].cpu().numpy(), ref))
del out
torch.cuda.empty_cache()

# ---- NumPy on this host
_, t_np = sync_time(lambda: np.random.RandomState(5).normal(size=a.numpy_sample, loc=0, scale=scale))
res["numpy_normals_per_s"] = a.numpy_sample / t_np
res["numpy_draw_s_extrapolated"] = k * n / res["numpy_normals_per_s"]
res["speedup_vs_numpy"] = res["numpy_draw_s_extrapolated"] / res["draw_s"]


# ---- embedding level, this code vs the parent's host draw
def construct_new():
    g = rb.GaussianEmbedding(source=rb.DeviceVectorSpace(n), options={"range_dim": k}, _seed=77)
    return g


def construct_parent():
    # the parent's constructor: the eager NumPy draw of Theta
    return np.random.RandomState(77).normal(size=(k, n), loc=0, scale=scale)


U = torch.randn(a.m, n, dtype=torch.float64, device=dev)
be = rb.BlockGaussianEmbedding(source=rb.DeviceVectorSpace(n), options={"range_dim": k, "max_block_size": a.block},
                               _seed=78)


def apply_parent():
    # the parent's BlockGaussianEmbedding.apply: NumPy draws each block, uploads it, one GEMM per block
    result = torch.empty((a.m, k), dtype=torch.float64, device=dev)
    off = 0
    for i, b in enumerate(be.block_sizes):
        gauss = torch.from_numpy(np.random.RandomState(be.block_seeds[i]).normal(size=(b, n), loc=0, scale=scale)).to(dev)
        result[:, off:off + b].copy_(dense.gauss_apply_explicit(gauss, U))
        off += b
    return result


runs = {"construct_new_s": [], "construct_parent_s": [], "block_apply_new_s": [], "block_apply_parent_s": []}
y_new = y_par = None
for rnd, who in enumerate(("new", "parent", "new")):
    if who == "parent" and a.skip_parent:
        continue
    obj, t = sync_time(construct_new if who == "new" else construct_parent)
    runs[f"construct_{who}_s"].append(t)
    del obj
    torch.cuda.empty_cache()
    y, t = sync_time((lambda: be.apply(U)) if who == "new" else apply_parent)
    runs[f"block_apply_{who}_s"].append(t)
    if who == "new":
        y_new = y
    else:
        y_par = y
res.update(runs)
if y_par is not None:
    res["block_apply_bit_identical"] = bool(torch.equal(y_new, y_par))
print(json.dumps(res), flush=True)
