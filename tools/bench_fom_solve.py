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

With --method gmres: restarted GMRES(m) (fom_solve.affine_gmres, csrc/affine_gmres.cu, m = --restart)
on a non-symmetric problem, convection-diffusion-reaction on the unit square (terms [L, Dx, Dy, M]:
5-point Laplacian, central first differences, identity; n = nx^2, R = L + M factored once by
SuperLU), with theta drawn from a seed in two sets: convection only, theta = (1, a, b, 0) with
a, b in [-100, 100], and convection with a negative reaction, theta = (1, a / 50, b / 50, -c) with c in
[57, 71] (A(mu) indefinite, c inside a gap of the Laplacian's spectrum).  Per set and block size P: total time, steps and cycles; one step's
parts at the mid-cycle column j = m / 2, each timed alone on the full block (affine SpMM,
preconditioner, multi-dot with its row sums, orthogonalisation with its row sums, the per-row
scalar kernels, normalisation, and the cycle-end update x += V y divided by m); the Gram-Schmidt
kernels' algorithmic rates against the same-run device copy; and host SuperLU in general
(non-symmetric) mode for one mu of each set, extrapolated to P.

    python tools/bench_fom_solve.py --method gmres [--restart 30] [--Ps 1,16,64] [--out profiles/fom_gmres_r01.jsonl]
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
    ap.add_argument("--Ps", default=None, help="block sizes (default 1,16,64,256 for cg, 1,16,64 for gmres)")
    ap.add_argument("--tol", type=float, default=1e-10)
    ap.add_argument("--host-mus", type=int, default=2, help="mu of the SuperLU yardstick (cg)")
    ap.add_argument("--method", choices=["cg", "gmres"], default="cg")
    ap.add_argument("--restart", type=int, default=30, help="GMRES cycle length m")
    ap.add_argument("--out", default=None, help="default profiles/fom_solve_r01.jsonl (cg), fom_gmres_r01.jsonl (gmres)")
    args = ap.parse_args()
    if args.Ps is None:
        args.Ps = "1,16,64,256" if args.method == "cg" else "1,16,64"
    if args.out is None:
        args.out = os.path.join(ROOT, "profiles", "fom_solve_r01.jsonl" if args.method == "cg" else "fom_gmres_r01.jsonl")
    if args.method == "gmres":
        return gmres_main(args)
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


def card_and_copy(dev, emit):
    """The card's name and power limit, and the device-copy bandwidth (GB/s) of a 4 GiB block."""
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    gpu = (q[0].split(", ") + ["", "", ""])[:3] if q else ["", "", ""]
    big = torch.empty(1 << 29, dtype=torch.float64, device=dev)
    dst = torch.empty_like(big)
    copy_ms = timed(lambda: dst.copy_(big), 5)
    hbm = 2 * big.numel() * 8 / copy_ms / 1e6
    del big, dst
    emit({"gpu": gpu[0], "power_limit": gpu[1], "max_sm_clock": gpu[2], "hbm_copy_GBs": hbm,
          "torch_device": torch.cuda.get_device_name(dev)})
    return gpu, hbm


def cdr_terms(nx):
    """[L, Dx, Dy, M] of convection-diffusion-reaction on the unit square, nx^2 interior nodes."""
    import scipy.sparse as sp
    h = 1.0 / (nx + 1)
    e = np.ones(nx)
    I = sp.eye(nx, format="csr")
    T = sp.diags([-e[:-1], 2 * e, -e[:-1]], [-1, 0, 1], format="csr") / h ** 2
    D = sp.diags([-e[:-1], e[:-1]], [-1, 1], format="csr") / (2 * h)
    return [(sp.kron(I, T) + sp.kron(T, I)).tocsr(), sp.kron(I, D).tocsr(), sp.kron(D, I).tocsr(),
            sp.eye(nx * nx, format="csr")]


def cdr_thetas(P, kind, seed):
    rs = np.random.RandomState(seed)
    th = np.ones((P, 4))
    th[:, 1:3] = rs.uniform(-100, 100, (P, 2))
    th[:, 3] = 0.0
    if kind == "indefinite":                # two negative eigenvalues; c in the gap of L's spectrum (49.3, 78.9)
        th[:, 1:3] /= 50
        th[:, 3] = -rs.uniform(57, 71, P)
    return th


def gmres_main(args):
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    out = open(args.out, "w")

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    gpu, hbm = card_and_copy(dev, emit)
    terms = cdr_terms(args.nx)
    n, Q, m = terms[0].shape[0], len(terms), args.restart
    R = (terms[0] + terms[3]).tocsc()
    ops_dev = [rb.MatrixOperator(A, source_id="S", range_id="S") for A in terms]
    t0 = time.time()
    prec = InverseLuOperator(rb.MatrixOperator(R, source_id="S", range_id="S"), symetric=True)
    splu_R_s = time.time() - t0
    f = np.random.RandomState(0).standard_normal(n)
    fom = AffineModel(ops_dev, [f])
    A = fom_solve.AffineCsr(ops_dev)
    nnz = A.nnz
    Ps = [int(x) for x in args.Ps.split(",")]
    L, s = lib(), stream_ptr
    for kind, seed in (("convection", 1), ("indefinite", 2)):
        th_all = cdr_thetas(max(Ps), kind, seed)
        # host yardstick: SuperLU in general (non-symmetric) mode, factorisation + solve of A(mu_0)
        Amu = sum(th_all[0, q] * terms[q] for q in range(Q)).tocsc()
        t0 = time.time()
        u_host = splu(Amu).solve(f)
        host_s = time.time() - t0
        del Amu
        common = {"problem": "convection-diffusion-reaction, unit square, central differences", "theta_set": kind,
                  "theta_seed": seed, "n": n, "Q": Q, "nnz_union": nnz, "tol": args.tol, "restart": m,
                  "preconditioner": "R = L + M, SuperLU symmetric mode, device triangular solves",
                  "host_splu_R_s": splu_R_s, "gpu": gpu[0], "power_limit": gpu[1]}
        for P in Ps:
            th = torch.from_numpy(th_all[:P].copy()).to(dev)
            tf = torch.ones((P, 1), dtype=torch.float64, device=dev)
            res = {}

            def solve():
                res["out"] = fom_solve._affine_gmres(A, fom.rhs, th, tf, prec, args.tol, m, 3000, None)

            total_ms = timed(solve, 1)
            X, iters, resid, info, cycles = res["out"]
            it, cy = iters.cpu().numpy(), cycles.cpu().numpy()
            assert np.all(info.cpu().numpy() == 0)
            err = float(np.linalg.norm(X[0].cpu().numpy() - u_host) / np.linalg.norm(u_host))
            del X, res["out"]
            torch.cuda.empty_cache()

            # one step's parts on the full block at column j = m / 2 (c = j + 1 basis vectors)
            c = m // 2 + 1
            g = torch.Generator(device=dev).manual_seed(P)
            V = torch.randn((P, m, n), dtype=torch.float64, device=dev, generator=g)
            W = torch.randn((P, m, n), dtype=torch.float64, device=dev, generator=g)
            Z, Y, U, Xv = [torch.randn((P, n), dtype=torch.float64, device=dev, generator=g) for _ in range(4)]
            ws = torch.empty(L.rla_affine_gmres_workspace_bytes(n, m, P), dtype=torch.uint8, device=dev)
            ws2 = torch.empty(L.rla_affine_cg_workspace_bytes(n, P), dtype=torch.uint8, device=dev)
            hb = torch.full((P, m + 2), 1e-3, dtype=torch.float64, device=dev)
            hb2 = torch.ones((P,), dtype=torch.float64, device=dev)
            ist0 = torch.zeros((10, P), dtype=torch.int32, device=dev)
            ist0[2].fill_(1)                                   # in a cycle
            ist0[3].fill_(c)
            ist0[5].fill_(2)
            ist0[6].fill_(2)
            ist = ist0.clone()
            st0 = torch.ones((5, P), dtype=torch.float64, device=dev)
            st = st0.clone()
            hess = torch.full((L.rla_affine_gmres_hess_bytes(m, P) // 8,), 0.5, dtype=torch.float64, device=dev)
            act, arn = ist[5], ist[6]
            spmm_ms = timed(lambda: fom_solve._spmm(A, th, Q, U, Y, act, None), 10)
            prec_ms = timed(lambda: prec.apply(rb.DeviceVectorArray(prec.source, Y)), 5)

            def dots():
                _lib.check(L.rla_affine_gmres_dots_f64(Z.data_ptr(), Y.data_ptr(), W.data_ptr(), n, m, P,
                                                       ist.data_ptr(), act.data_ptr(), ws.data_ptr(), ws.numel(), s()))

            def dots_sum():
                _lib.check(L.rla_row_dot_sum_f64(ws.data_ptr(), ws.numel(), n, P * (m + 2), hb.data_ptr(), s()))

            def orth():
                _lib.check(L.rla_affine_gmres_orth_f64(Z.data_ptr(), Y.data_ptr(), V.data_ptr(), W.data_ptr(),
                                                       hb.data_ptr(), n, m, P, ist.data_ptr(), arn.data_ptr(),
                                                       ws2.data_ptr(), ws2.numel(), s()))

            def orth_sum():
                _lib.check(L.rla_row_dot_sum_f64(ws2.data_ptr(), ws2.numel(), n, P, hb2.data_ptr(), s()))

            def scalars():
                ist.copy_(ist0)
                st.copy_(st0)
                _lib.check(L.rla_affine_gmres_dgks_f64(hb.data_ptr(), hb2.data_ptr(), m, P, st.data_ptr(),
                                                       ist.data_ptr(), hess.data_ptr(), s()))
                _lib.check(L.rla_affine_gmres_step_f64(hb.data_ptr(), hb2.data_ptr(), m, P, 0.0, 1 << 40,
                                                       st.data_ptr(), ist.data_ptr(), hess.data_ptr(), s()))

            def normalize():
                _lib.check(L.rla_affine_gmres_normalize_f64(Z.data_ptr(), Y.data_ptr(), V.data_ptr(), W.data_ptr(),
                                                            U.data_ptr(), n, m, P, st.data_ptr(), ist.data_ptr(), s()))

            ist_end = ist0.clone()
            ist_end[9].fill_(2)
            ist_end[3].fill_(m)

            def update():
                _lib.check(L.rla_affine_gmres_update_f64(Xv.data_ptr(), U.data_ptr(), V.data_ptr(), n, m, P,
                                                         ist_end.data_ptr(), hess.data_ptr(), s()))

            dots_ms, dsum_ms, orth_ms, osum_ms = timed(dots, 10), timed(dots_sum, 10), timed(orth, 10), timed(orth_sum, 10)
            scal_ms = timed(scalars, 10)
            ist.copy_(ist0)
            norm_ms = timed(normalize, 10)
            upd_ms = timed(update, 5)
            del V, W, Z, Y, U, Xv, ws
            torch.cuda.empty_cache()
            dots_B, orth_B, norm_B = (c + 2) * P * n * 8, (2 * c + 4) * P * n * 8, 5 * P * n * 8
            upd_B = (m + 2) * P * n * 8
            gs_ms = dots_ms + dsum_ms + orth_ms + osum_ms + scal_ms + norm_ms + upd_ms / m
            step_ms = spmm_ms + prec_ms + gs_ms
            steps = int(it.max()) + int(cy.max())              # Arnoldi steps + true-residual steps
            emit({**common, "P": P, "total_ms": total_ms, "iters_min": int(it.min()), "iters_max": int(it.max()),
                  "cycles_min": int(cy.min()), "cycles_max": int(cy.max()),
                  "ms_per_step_total": total_ms / max(steps, 1),
                  "per_step_ms_at_mid_cycle": {"column_j": c - 1, "affine_spmm": spmm_ms, "preconditioner": prec_ms,
                                               "multidot": dots_ms, "multidot_row_sums": dsum_ms,
                                               "orthogonalisation": orth_ms, "orth_row_sums": osum_ms,
                                               "scalars": scal_ms, "normalisation": norm_ms,
                                               "cycle_end_update_per_cycle": upd_ms,
                                               "cycle_end_update_per_step": upd_ms / m},
                  "step_ms_model": step_ms,
                  "outside_preconditioner_frac": (step_ms - prec_ms) / step_ms,
                  "gs_algorithmic_GBs": {"multidot": dots_B / dots_ms / 1e6, "orthogonalisation": orth_B / orth_ms / 1e6,
                                         "normalisation": norm_B / norm_ms / 1e6, "cycle_end_update": upd_B / upd_ms / 1e6},
                  "gs_frac_of_hbm_copy": {"multidot": dots_B / dots_ms / 1e6 / hbm,
                                          "orthogonalisation": orth_B / orth_ms / 1e6 / hbm,
                                          "normalisation": norm_B / norm_ms / 1e6 / hbm,
                                          "cycle_end_update": upd_B / upd_ms / 1e6 / hbm},
                  "hbm_copy_GBs": hbm,
                  "host_superlu_general_factor_solve_s_per_mu": host_s, "host_superlu_extrapolated_s": host_s * P,
                  "host_extrapolated": True, "host_sample_mus": 1,
                  "speedup_vs_host_extrapolated": host_s * P * 1e3 / total_ms,
                  "rel_err_vs_superlu_row0": err})
    out.close()


if __name__ == "__main__":
    main()
