"""Timing of the ROM over a parameter set (csrc/rom_batch.cu: SketchedRom.solve_batch and
estimate_error_batch) against the per-mu methods and a torch formulation, one JSON line per
(shape, P) after a line with the card's name, power limit and the FP64 tensor-pipe peak of the
same run.

The ROMs are built directly from seeded random reduced data: A_q = I + 0.1 G_q / sqrt(r) and
coefficients in [0.1, 1], so every A(mu) is well conditioned; f_j, the sketched terms and the
output functional are Gaussian.

  batch      solve_batch (one launch) and estimate_error_batch given a (two launches)
  per_mu     rom.solve + rom.estimate_error for each of 1000 mu (one host round trip each),
             EXTRAPOLATED linearly to P
  torch      A(mu) and b(mu) by einsum / matmul, torch.linalg.solve on the stacked (P, r, r)
             systems; the residual as X(mu) @ W and a row norm in chunks of 8192 mu

The batch residual kernel's rate counts 2 P N k' flops (N = Q r + Pf) over its time.  Every path
is warmed up, then timed with CUDA events over --reps calls; peak memory is that of one call.
`max_rel_diff_*` compare the batch results with each yardstick (per_mu: over its 1000 mu).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rla4mor_b200._lib import check, lib, stream_ptr  # noqa: E402
from rla4mor_b200.sketched_reductor import SketchedRom  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--shapes", default="16,4,1,200;64,4,1,1000;128,8,2,2000", help="r,Q,Pf,k' separated by ';'")
ap.add_argument("--Ps", default="1000,10000,100000")
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--loop", type=int, default=1000, help="mu of the per-mu yardstick")
args = ap.parse_args()
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip().splitlines()
gpu = (q[0].split(", ") + ["", "", ""])[:3] if q else ["", "", ""]
scratch = torch.empty(1 << 20, dtype=torch.uint8, device=dev)
peak = ctypes.c_double()
check(lib().rla_dmma_peak_tflops(ctypes.byref(peak), ctypes.c_void_p(scratch.data_ptr()), stream_ptr()), "dmma peak")
print(json.dumps({"gpu": gpu[0], "power_limit": gpu[1], "max_sm_clock": gpu[2], "dmma_peak_tflops": peak.value}),
      flush=True)


def timed(f, reps):
    """(result of the last call, ms per call, peak bytes allocated during one call)"""
    f()
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


def make_rom(r, Q, Pf, kp, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    rnd = lambda *s: torch.randn(*s, dtype=torch.float64, device=dev, generator=g)
    eye = torch.eye(r, dtype=torch.float64, device=dev)
    lhs = [eye + 0.1 * rnd(r, r) / r ** 0.5 for _ in range(Q)]
    rhs = [rnd(r) for _ in range(Pf)]
    est = ([rnd(r, kp) for _ in range(Q)], [rnd(kp) for _ in range(Pf)])
    return SketchedRom(None, lhs, rhs, rnd(r, 2), est, least_squares=False)


def thetas(P, Q, Pf, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    return (0.1 + 0.9 * torch.rand(P, Q, dtype=torch.float64, device=dev, generator=g),
            torch.randn(P, Pf, dtype=torch.float64, device=dev, generator=g))


def torch_solve(rom, th, tf):
    A = torch.einsum("pq,qij->pij", th, torch.stack(rom.lhs))
    b = tf @ torch.stack(rom.rhs)
    return torch.linalg.solve(A, b)


def torch_estimate(rom, th, tf, a, chunk=8192):
    W = torch.cat(list(rom.est_lhs_rows) + [g.reshape(1, -1) for g in rom.est_rhs], dim=0)
    out = torch.empty(th.shape[0], dtype=torch.float64, device=dev)
    for p0 in range(0, th.shape[0], chunk):
        t, f, x = th[p0:p0 + chunk], tf[p0:p0 + chunk], a[p0:p0 + chunk]
        X = torch.cat([(t[:, :, None] * x[:, None, :]).reshape(t.shape[0], -1), -f], dim=1)
        out[p0:p0 + chunk] = torch.linalg.norm(X @ W, dim=1)
    return out


def rel_rows(x, ref):
    d = torch.linalg.norm((x - ref).reshape(x.shape[0], -1), dim=1)
    return float(torch.max(d / torch.linalg.norm(ref.reshape(ref.shape[0], -1), dim=1)))


for shape in args.shapes.split(";"):
    r, Q, Pf, kp = (int(v) for v in shape.split(","))
    rom = make_rom(r, Q, Pf, kp, seed=r)
    N = Q * r + Pf
    # per-mu yardstick, once per shape: the single-mu methods, one host round trip per mu
    thl, tfl = thetas(args.loop, Q, Pf, seed=7)
    thl_h, tfl_h = thl.tolist(), tfl.tolist()
    rom.estimate_error(None, thl_h[0], tfl_h[0])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    loop_a = [rom.solve(thl_h[p], tfl_h[p]) for p in range(args.loop)]
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    loop_est = [rom.estimate_error(loop_a[p], thl_h[p], tfl_h[p]) for p in range(args.loop)]
    t2 = time.perf_counter()
    solve_per_mu_ms, est_per_mu_ms = (t1 - t0) * 1e3 / args.loop, (t2 - t1) * 1e3 / args.loop
    a_l = rom.solve_batch(thl, tfl)
    e_l = rom.estimate_error_batch(a_l, thl, tfl)
    loop_diff_a = rel_rows(a_l, torch.stack(loop_a))
    loop_diff_e = float(torch.max(torch.abs(e_l - torch.tensor(loop_est, dtype=torch.float64, device=dev)) / e_l))
    del loop_a
    for P in (int(v) for v in args.Ps.split(",")):
        th, tf = thetas(P, Q, Pf, seed=P)
        a, ms_solve, mem_solve = timed(lambda: rom.solve_batch(th, tf), args.reps)
        est, ms_est, mem_est = timed(lambda: rom.estimate_error_batch(a, th, tf), args.reps)
        flop = 2.0 * P * N * kp
        a_t, ms_tsolve, mem_tsolve = timed(lambda: torch_solve(rom, th, tf), args.reps)
        est_t, ms_test, mem_test = timed(lambda: torch_estimate(rom, th, tf, a), args.reps)
        res = {
            "r": r, "Q": Q, "Pf": Pf, "kp": kp, "P": P, "N": N,
            "batch": {"solve_ms": ms_solve, "estimate_ms": ms_est, "mu_per_s": P / ((ms_solve + ms_est) * 1e-3),
                      "estimate_tflops": flop / (ms_est * 1e-3) / 1e12,
                      "estimate_of_dmma_peak": flop / (ms_est * 1e-3) / 1e12 / peak.value,
                      "solve_peak_mem_mb": mem_solve / 1e6, "estimate_peak_mem_mb": mem_est / 1e6},
            "per_mu_extrapolated": {"from_mu": args.loop, "solve_ms": solve_per_mu_ms * P,
                                    "estimate_ms": est_per_mu_ms * P,
                                    "mu_per_s": 1e3 / (solve_per_mu_ms + est_per_mu_ms)},
            "torch": {"solve_ms": ms_tsolve, "estimate_ms": ms_test, "mu_per_s": P / ((ms_tsolve + ms_test) * 1e-3),
                      "solve_peak_mem_mb": mem_tsolve / 1e6, "estimate_peak_mem_mb": mem_test / 1e6},
            "max_rel_diff_per_mu": {"a": loop_diff_a, "est": loop_diff_e},
            "max_rel_diff_torch": {"a": rel_rows(a, a_t), "est": float(torch.max(torch.abs(est - est_t) / est_t))},
            "est_run_to_run_equal": bool(torch.equal(est, rom.estimate_error_batch(a, th, tf))),
        }
        del a, est, a_t, est_t
        torch.cuda.empty_cache()
        print(json.dumps(res), flush=True)
