"""Launch-configuration sweep of rom_lstsq_batch_kernel (csrc/rom_batch.cu): the evidence behind
rl_config, the rule that picks threads per CTA, lanes per column G and panel height c from r.

The library launches the kernel with rl_config only, so this tool compiles a small harness that
includes csrc/rom_batch.cu and launches the kernel with an explicit (threads, G, c), into a
temporary directory (nothing is written to the tree), linked against librla_b200.so.  For every
shape (r, Q, Pf, k_eff) it times all fitting configurations of threads {64, 128, 256, 512} x
G {2, 4, 8} x c {32, 64, 128} at P mu with CUDA events (one warm-up, --reps timed launches) and
prints one JSON line each, after a line with the card's name and power limit.  `diff` is the
largest relative row difference to the first configuration: the configurations reorder sums only.
The stack W is Gaussian and the coefficients are in [0.1, 1.1].
"""
import argparse
import ctypes
import itertools
import json
import os
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rla4mor_b200 import _build  # noqa: E402
from rla4mor_b200._lib import LIB_PATH, lib  # noqa: E402

HARNESS = r"""
#include "%s"
extern "C" int sweep_lstsq(const double *W, int64_t ldw, int Q, int r, int Pf, int64_t ke, const double *th,
                           const double *tf, int64_t P, double *a, int32_t *info, int threads, int G, int c) {
    const int smem = (int)(rla::rl_smem_doubles(r, c, G) * sizeof(double));
    if (smem > rla::RL_SMEM_LIMIT) return -1;
    if (cudaFuncSetAttribute(rla::rom_lstsq_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)) return -1;
    int per_sm = 0, dev = 0, sms = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rla::rom_lstsq_batch_kernel, threads, smem);
    if (per_sm < 1) return -1;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int64_t grid = std::min<int64_t>(P, (int64_t)per_sm * sms);
    rla::rom_lstsq_batch_kernel<<<(unsigned)grid, threads, smem>>>(W, ldw, Q, r, Pf, ke, th, Q, tf, Pf, P, a, r,
                                                                   info, G, c);
    return cudaGetLastError() ? -2 : per_sm;
}
"""

ap = argparse.ArgumentParser()
ap.add_argument("--shapes", default="16,3,2,50;16,8,1,64;64,4,1,257;128,2,1,257", help="r,Q,Pf,k_eff separated by ';'")
ap.add_argument("--P", type=int, default=100000)
ap.add_argument("--reps", type=int, default=3)
args = ap.parse_args()

lib()                                                           # builds librla_b200.so if it is missing
tmp = tempfile.mkdtemp(prefix="rla_sweep_")
src, so = os.path.join(tmp, "sweep.cu"), os.path.join(tmp, "libsweep.so")
with open(src, "w") as f:
    f.write(HARNESS % os.path.join(ROOT, "rla4mor_b200", "csrc", "rom_batch.cu"))
libdir = os.path.dirname(LIB_PATH)
cmd = [_build._nvcc(), "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "--shared", "-Xcompiler",
       "-fPIC", src, "-o", so, "-L" + libdir, "-lrla_b200", "-Xlinker", "-rpath," + libdir]
if os.path.exists("/usr/bin/g++"):
    cmd += ["-ccbin", "/usr/bin/g++"]
subprocess.run(cmd, check=True)
L = ctypes.CDLL(so)
vp, i64, ci = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
L.sweep_lstsq.argtypes = [vp, i64, ci, ci, ci, i64, vp, vp, i64, vp, vp, ci, ci, ci]

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip().splitlines()
gpu = (q[0].split(", ") + ["", "", ""])[:3] if q else ["", "", ""]
print(json.dumps({"gpu": gpu[0], "power_limit": gpu[1], "max_sm_clock": gpu[2], "P": args.P}), flush=True)
P = args.P
for shape in args.shapes.split(";"):
    r, Q, Pf, ke = (int(v) for v in shape.split(","))
    g = torch.Generator(device="cuda").manual_seed(r)
    W = torch.randn(Q * r + Pf, ke, dtype=torch.float64, device="cuda", generator=g)
    th = 0.1 + torch.rand(P, Q, dtype=torch.float64, device="cuda", generator=g)
    tf = torch.randn(P, Pf, dtype=torch.float64, device="cuda", generator=g)
    a = torch.empty(P, r, dtype=torch.float64, device="cuda")
    info = torch.empty(P, dtype=torch.int32, device="cuda")
    ref = None
    for threads, G, c in itertools.product([64, 128, 256, 512], [2, 4, 8], [32, 64, 128]):
        call = lambda: L.sweep_lstsq(W.data_ptr(), ke, Q, r, Pf, ke, th.data_ptr(), tf.data_ptr(), P, a.data_ptr(),
                                     info.data_ptr(), threads, G, c)
        per_sm = call()
        if per_sm == -1:                                        # does not fit
            continue
        assert per_sm > 0, "launch failed"
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.reps):
            call()
        e1.record()
        torch.cuda.synchronize()
        if ref is None:
            ref = a.clone()
        d = float(torch.max(torch.linalg.norm(a - ref, dim=1) / torch.linalg.norm(ref, dim=1)))
        print(json.dumps({"r": r, "Q": Q, "Pf": Pf, "ke": ke, "threads": threads, "G": G, "c": c, "per_sm": per_sm,
                          "ms": e0.elapsed_time(e1) / args.reps, "diff": d, "info_nz": int(info.count_nonzero())}),
              flush=True)
