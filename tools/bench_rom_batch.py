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

--mode minres times the batched least-squares solve of a minres ROM (rom_lstsq_batch_kernel).  The
ROMs are M_q = U + 0.1 G_q / sqrt(k') (U with orthonormal columns), coefficients in [0.1, 1], so
every M(mu) is well conditioned; g_j are Gaussian.

  kernel     reductor_ops.rom_lstsq_batch on the ROM's stack (compressed once when N < k')
  compress   building that stack (torch.linalg.qr of the k' x N matrix), once per ROM
  torch      M(mu), b(mu) by einsum / matmul and torch.linalg.lstsq on the stacked (P, k', r)
             systems, in chunks of at most 256 MB of systems; timed once over min(P, --torch-max)
             mu (after a warm-up) and EXTRAPOLATED linearly to P beyond that; its agreement
             is over those mu
  per_mu     the per-mu loop of torch.linalg.lstsq over 1000 mu, EXTRAPOLATED linearly to P

The kernel's rate counts, per mu, 2 N k_eff flops of assembly, 2 k_eff r^2 - 2/3 r^3 of QR and
r^2 of back substitution, with k_eff = min(N, k').
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
from rla4mor_b200 import reductor_ops as ops  # noqa: E402
from rla4mor_b200.sketched_reductor import SketchedRom  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--mode", choices=("galerkin", "minres"), default="galerkin")
ap.add_argument("--shapes", default=None, help="r,Q,Pf,k' separated by ';'")
ap.add_argument("--Ps", default=None)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--loop", type=int, default=1000, help="mu of the per-mu yardstick")
ap.add_argument("--torch-max", type=int, default=10000, help="minres: mu of the chunked torch yardstick")
args = ap.parse_args()
if args.shapes is None:
    args.shapes = "16,4,1,200;64,4,1,1000;128,8,2,2000" if args.mode == "galerkin" else \
        "16,3,2,64;16,8,1,64;64,4,1,1000;128,2,1,512"
if args.Ps is None:
    args.Ps = "1000,10000,100000" if args.mode == "galerkin" else "1000,100000"
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


def make_ls_rom(r, Q, Pf, kp, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    rnd = lambda *s: torch.randn(*s, dtype=torch.float64, device=dev, generator=g)
    U = torch.linalg.qr(rnd(kp, r)).Q
    lhs = [U + 0.1 * rnd(kp, r) / kp ** 0.5 for _ in range(Q)]
    est = ([rnd(r, 8) for _ in range(Q)], [rnd(8) for _ in range(Pf)])
    return SketchedRom(None, lhs, [rnd(kp) for _ in range(Pf)], rnd(r, 2), est, least_squares=True)


def lstsq_per_mu(rom, th, tf):
    """The per-mu least-squares solve as SketchedRom.solve ran it before the batched kernel."""
    A = sum(t * M for t, M in zip(th, rom.lhs))
    b = sum(t * v for t, v in zip(tf, rom.rhs))
    return torch.linalg.lstsq(A, b.reshape(-1, 1)).solution.reshape(-1)


def torch_lstsq(rom, th, tf):
    M, G = torch.stack(rom.lhs), torch.stack(rom.rhs)
    kp, r = M.shape[1], M.shape[2]
    chunk = max(1, (256 << 20) // (8 * kp * (r + 1)))
    out = torch.empty(th.shape[0], r, dtype=torch.float64, device=dev)
    for p0 in range(0, th.shape[0], chunk):
        A = torch.einsum("pq,qkr->pkr", th[p0:p0 + chunk], M)
        b = tf[p0:p0 + chunk] @ G
        out[p0:p0 + chunk] = torch.linalg.lstsq(A, b.unsqueeze(-1)).solution[..., 0]
    return out


def run_minres():
    for shape in args.shapes.split(";"):
        r, Q, Pf, kp = (int(v) for v in shape.split(","))
        rom = make_ls_rom(r, Q, Pf, kp, seed=r)
        N = Q * r + Pf

        def build():
            rom._ls_stack = None
            return rom._lstsq_stack()
        W, ms_compress, _ = timed(build, args.reps)
        ke = W.shape[1]
        thl, tfl = thetas(args.loop, Q, Pf, seed=7)
        lstsq_per_mu(rom, thl[0], tfl[0])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loop_a = torch.stack([lstsq_per_mu(rom, thl[p], tfl[p]) for p in range(args.loop)])
        torch.cuda.synchronize()
        per_mu_ms = (time.perf_counter() - t0) * 1e3 / args.loop
        loop_diff = rel_rows(ops.rom_lstsq_batch(W, Q, r, thl, tfl)[0], loop_a)
        for P in (int(v) for v in args.Ps.split(",")):
            th, tf = thetas(P, Q, Pf, seed=P)
            a, ms, mem = timed(lambda: ops.rom_lstsq_batch(W, Q, r, th, tf, check=False)[0], args.reps)
            Pt = min(P, args.torch_max)
            torch_lstsq(rom, th[:64], tf[:64])
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a_t = torch_lstsq(rom, th[:Pt], tf[:Pt])
            e1.record()
            torch.cuda.synchronize()
            ms_t, mem_t = e0.elapsed_time(e1) * P / Pt, torch.cuda.max_memory_allocated() - base
            flop = P * (2.0 * N * ke + 2.0 * ke * r * r - 2.0 / 3.0 * r ** 3 + r * r)
            res = {
                "mode": "minres", "r": r, "Q": Q, "Pf": Pf, "kp": kp, "k_eff": ke, "compressed": ke < kp, "P": P,
                "kernel": {"ms": ms, "tflops": flop / (ms * 1e-3) / 1e12, "mu_per_s": P / (ms * 1e-3),
                           "peak_mem_mb": mem / 1e6},
                "compress_ms_once": ms_compress,
                "torch_lstsq_chunked": {"ms": ms_t, "timed_mu": Pt, "extrapolated": Pt < P, "peak_mem_mb": mem_t / 1e6},
                "per_mu_extrapolated": {"from_mu": args.loop, "ms": per_mu_ms * P},
                "speedup": {"vs_torch": ms_t / ms, "vs_per_mu": per_mu_ms * P / ms},
                "max_rel_diff_torch": rel_rows(a[:Pt], a_t), "max_rel_diff_per_mu": loop_diff,
                "run_to_run_equal": bool(torch.equal(a, ops.rom_lstsq_batch(W, Q, r, th, tf)[0])),
            }
            del a, a_t
            torch.cuda.empty_cache()
            print(json.dumps(res), flush=True)


def run_galerkin():
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


run_minres() if args.mode == "minres" else run_galerkin()
