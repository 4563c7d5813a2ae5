"""Full-order snapshots on the device: AffineModel.solve_batch / fom_solve.affine_cg (block
preconditioned CG, csrc/affine_cg.cu) on the thermal-block-like FEM problem of tools/bench_c4.py:
n = nx^2, Q = 4 SPD terms, R = A(mu_bar) = sum_q A_q factored once by SuperLU (symmetric mode) and
applied on the device as the preconditioner, theta drawn in [0.1, 1]^Q, one right-hand side.

One JSON line per block size P, after a line with the card's name, power limit and the measured
device-copy bandwidth (the HBM yardstick):
  - total time of the solve (CUDA events, after a warm-up solve of the same shape);
  - iterations (min / max over the rows);
  - one iteration's parts, each timed alone on the full block with every row iterating: affine
    SpMM (with its dot epilogue), preconditioner (InverseLuOperator.apply), vector updates
    (r -= alpha Ap; x += alpha p, p = z + beta p) and reductions (<r, z> partials, the alpha and
    beta kernels);
  - the affine SpMM's algorithmic rate nnz (4 + 8 Q) + 2 P n 8 bytes over its time, beside the
    existing single-term CSR SpMM at the same P (nnz 12 + 2 P n 8 bytes);
  - a host yardstick: SuperLU factorisation plus solve of A(mu) for a few mu, extrapolated to P
    (flagged as such), and the device solution's distance to those host solutions.

    python tools/bench_fom_solve.py [--nx 1000] [--Ps 1,16,64,256] [--out profiles/fom_solve_r01.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
from scipy.sparse.linalg import splu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools")]
import rla4mor_b200 as rb                                            # noqa: E402
from rla4mor_b200 import _lib, fom_solve, reductor_ops               # noqa: E402
from rla4mor_b200._lib import lib, stream_ptr                        # noqa: E402
from rla4mor_b200.factorization import InverseLuOperator             # noqa: E402
from rla4mor_b200.sketched_reductor import AffineModel               # noqa: E402
from bench_c4 import fem_terms                                       # noqa: E402


def timed(f, reps):
    """Least of `reps` CUDA-event timings (ms) of f(), after one untimed call."""
    f()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        f()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return min(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=1000)
    ap.add_argument("--Ps", default="1,16,64,256")
    ap.add_argument("--tol", type=float, default=1e-10)
    ap.add_argument("--host-mus", type=int, default=2, help="mu of the SuperLU yardstick")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "fom_solve_r01.jsonl"))
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    out = open(args.out, "w")

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    gpu = (q[0].split(", ") + ["", "", ""])[:3] if q else ["", "", ""]
    big = torch.empty(1 << 29, dtype=torch.float64, device=dev)     # 4 GiB, far above the 126 MB L2
    dst = torch.empty_like(big)
    copy_ms = timed(lambda: dst.copy_(big), 5)
    hbm = 2 * big.numel() * 8 / copy_ms / 1e6                         # GB/s, read + write
    del big, dst
    emit({"gpu": gpu[0], "power_limit": gpu[1], "max_sm_clock": gpu[2], "hbm_copy_GBs": hbm,
          "torch_device": torch.cuda.get_device_name(dev)})

    terms, _, n = fem_terms(args.nx)
    Q = len(terms)
    R = sum(terms[1:], terms[0]).tocsc()
    space = rb.DeviceVectorSpace(n, id="S")
    ops_dev = [rb.MatrixOperator(A, source_id="S", range_id="S") for A in terms]
    t0 = time.time()
    prec = InverseLuOperator(rb.MatrixOperator(R, source_id="S", range_id="S"), symetric=True)
    splu_R_s = time.time() - t0
    f = np.random.RandomState(0).standard_normal(n)
    fom = AffineModel(ops_dev, [f])
    t0 = time.time()
    A = fom_solve.AffineCsr(ops_dev)
    merge_s = time.time() - t0
    fom._affine = A
    nnz = A.nnz
    common = {"n": n, "Q": Q, "nnz_union": nnz, "tol": args.tol, "theta": "uniform [0.1, 1]^Q",
              "preconditioner": "R = sum_q A_q, SuperLU symmetric mode, device triangular solves (CUDA graph)",
              "host_splu_R_s": splu_R_s, "host_union_merge_s": merge_s, "gpu": gpu[0], "power_limit": gpu[1]}

    # host yardstick: SuperLU factorisation + solve of A(mu) for a few mu
    rs = np.random.RandomState(1)
    th_all = rs.uniform(0.1, 1.0, (max(int(x) for x in args.Ps.split(",")), Q))
    host = []
    for p in range(args.host_mus):
        Amu = sum(th_all[p, q] * terms[q] for q in range(Q)).tocsc()
        t0 = time.time()
        u = splu(Amu).solve(f)
        host.append((time.time() - t0, u))
    host_s = float(np.mean([h[0] for h in host]))

    L = lib()
    for P in [int(x) for x in args.Ps.split(",")]:
        th = torch.from_numpy(th_all[:P].copy()).to(dev)
        tf = torch.ones((P, 1), dtype=torch.float64, device=dev)
        res = {}

        def solve():
            res["out"] = fom_solve.affine_cg(A, fom.rhs, th, tf, prec, tol=args.tol, maxiter=1000)

        total_ms = timed(solve, 2 if P >= 64 else 3)
        X, iters, resid, info = res["out"]
        it = iters.cpu().numpy()
        assert np.all(info.cpu().numpy() == 0)
        err = [float(np.linalg.norm(X[p].cpu().numpy() - host[p][1]) / np.linalg.norm(host[p][1]))
               for p in range(min(P, len(host)))]

        # one iteration's parts on the full block, every row iterating
        g = torch.Generator(device=dev).manual_seed(P)
        V = [torch.randn((P, n), dtype=torch.float64, device=dev, generator=g) for _ in range(4)]
        Xv, Pv, Rv, Zv = V
        Qv = torch.empty_like(Pv)
        ws = torch.empty(L.rla_affine_cg_workspace_bytes(n, P), dtype=torch.uint8, device=dev)
        state = torch.full((5, P), 0.5, dtype=torch.float64, device=dev)
        istate = torch.full((3, P), 2, dtype=torch.int32, device=dev)
        istate[0].zero_()
        istate[1].zero_()
        mode = istate[2]
        s = stream_ptr
        spmm_ms = timed(lambda: fom_solve._spmm(A, th, Q, Pv, Qv, mode, ws), 20)
        prec_ms = timed(lambda: prec.apply(rb.DeviceVectorArray(prec.source, Rv)), 5)
        upd_r_ms = timed(lambda: _lib.check(L.rla_affine_cg_update_r_f64(Rv.data_ptr(), n, Qv.data_ptr(), n, n, P,
                                                                         state.data_ptr(), istate.data_ptr(), s())), 20)
        upd_xp_ms = timed(lambda: _lib.check(L.rla_affine_cg_update_xp_f64(Xv.data_ptr(), n, Pv.data_ptr(), n,
                                                                           Zv.data_ptr(), n, n, P, state.data_ptr(),
                                                                           istate.data_ptr(), s())), 20)
        dots_ms = timed(lambda: fom_solve._dots(Rv, Zv, n, mode, ws), 20)

        def scalars():
            # alpha and beta kernels; beta is given an unbounded maxiter and tol 0 so every row stays live
            _lib.check(L.rla_affine_cg_alpha_f64(ws.data_ptr(), ws.numel(), n, P, state.data_ptr(), istate.data_ptr(), s()))
            _lib.check(L.rla_affine_cg_beta_f64(ws.data_ptr(), ws.numel(), n, P, 0.0, 1 << 40, state.data_ptr(),
                                                istate.data_ptr(), s()))
        ws.view(torch.float64).fill_(1.0)
        scal_ms = timed(scalars, 20)
        assert bool((mode == 2).all())
        single_ms = timed(lambda: reductor_ops.spmm_csr(ops_dev[0].rowptr, ops_dev[0].col, ops_dev[0].val,
                                                        ops_dev[0].shape, Pv), 20)
        nnz1 = ops_dev[0].val.numel()
        del V, Xv, Pv, Rv, Zv, Qv
        torch.cuda.empty_cache()
        other = spmm_ms + upd_r_ms + upd_xp_ms + dots_ms + scal_ms
        iter_ms = other + prec_ms
        emit({**common, "P": P, "total_ms": total_ms, "iters_min": int(it.min()), "iters_max": int(it.max()),
              "ms_per_iteration_total": total_ms / max(int(it.max()), 1),
              "per_iteration_ms": {"affine_spmm_with_dot": spmm_ms, "preconditioner": prec_ms,
                                   "update_r": upd_r_ms, "update_xp": upd_xp_ms,
                                   "dot_rz_partials": dots_ms, "alpha_beta_reductions": scal_ms},
              "outside_preconditioner_frac": other / iter_ms,
              "affine_spmm_algorithmic_GBs": (nnz * (4 + 8 * Q) + 2 * P * n * 8) / spmm_ms / 1e6,
              "affine_spmm_frac_of_hbm_copy": (nnz * (4 + 8 * Q) + 2 * P * n * 8) / spmm_ms / 1e6 / hbm,
              "single_term_spmm_ms": single_ms,
              "single_term_spmm_algorithmic_GBs": (nnz1 * 12 + 2 * P * n * 8) / single_ms / 1e6,
              "host_superlu_factor_solve_s_per_mu": host_s,
              "host_superlu_extrapolated_s": host_s * P, "host_extrapolated": True,
              "host_sample_mus": len(host),
              "speedup_vs_host_extrapolated": host_s * P * 1e3 / total_ms,
              "rel_err_vs_superlu": err})
    out.close()


if __name__ == "__main__":
    main()
