"""The weak greedy (rla4mor_b200.rb_greedy) on the thermal-block FEM problem of tools/bench_c4.py:
n = nx^2, Q = 4 SPD terms, R = sum_q A_q factored once by SuperLU and applied on the device (the
snapshot solver's preconditioner and the reductor's inverse product), a Gaussian primal embedding
(Theta generated in the kernel) with k rows, the Galerkin projection, one right-hand side, training
theta drawn in [0.1, 1]^4 from a seed.

After a line with the card's name and power limit, one JSON line per iteration of each run
(P training mu, `batch` snapshots per extension, up to r_max): r, max estimate, the host-clock ms
of reduce / sweep / snapshot solve / extend (each phase ends in a device synchronise or a
device-to-host read), the snapshot iterations, and the unattributed remainder of the iteration
(selection bookkeeping and Python between the phases).  One summary line per run, with the
per-mu yardstick: the final ROM swept by the per-mu `rom.estimate_error` loop over 1000 mu,
extrapolated to P (flagged as such) -- what a greedy that estimates one mu at a time (pyMOR's
rb_greedy through the adapter) spends per sweep.

    python tools/bench_greedy.py [--nx 1000] [--runs 10000:1:64,10000:8:128,100000:8:128,100000:1:64]
                                 [--out profiles/greedy_r01.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools")]
import rla4mor_b200 as rb                                            # noqa: E402
from rla4mor_b200 import fom_solve                                   # noqa: E402
from rla4mor_b200.factorization import InverseLuOperator             # noqa: E402
from rla4mor_b200.sketched_reductor import AffineModel               # noqa: E402
from bench_c4 import fem_terms                                       # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=1000)
    ap.add_argument("--k", type=int, default=1000, help="rows of the Gaussian primal embedding")
    ap.add_argument("--runs", default="10000:1:64,10000:8:128,100000:8:128,100000:1:64", help="P:batch:r_max,...")
    ap.add_argument("--tol", type=float, default=1e-10)
    ap.add_argument("--loop-mus", type=int, default=1000, help="mu of the per-mu estimate_error yardstick")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "greedy_r01.jsonl"))
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    out = open(args.out, "w")

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    gpu = (q[0].split(", ") + ["", "", ""])[:3] if q else ["", "", ""]
    emit({"gpu": gpu[0], "power_limit": gpu[1], "max_sm_clock": gpu[2], "torch_device": torch.cuda.get_device_name(dev)})

    terms, _, n = fem_terms(args.nx)
    Q = len(terms)
    ops_dev = [rb.MatrixOperator(A, source_id="S", range_id="S") for A in terms]
    t0 = time.time()
    prec = InverseLuOperator(rb.MatrixOperator(sum(terms[1:], terms[0]).tocsc(), source_id="S", range_id="S"),
                             symetric=True)
    splu_s = time.time() - t0
    fom = AffineModel(ops_dev, [np.random.RandomState(0).standard_normal(n)])
    fom._affine = fom_solve.AffineCsr(ops_dev)
    runs = [tuple(int(x) for x in r.split(":")) for r in args.runs.split(",")]
    TH = np.random.RandomState(1).uniform(0.1, 1.0, (max(P for P, _, _ in runs), Q))

    def reductor():
        emb = rb.GaussianEmbedding(source=fom.solution_space, options={"range_dim": args.k, "rng": "philox"}, _seed=3)
        return rb.SketchedReductor(fom, embedding_primal=emb, inverse_product=prec)

    # warm-up: module loads, the LU solve's graphs, every kernel of the loop at a small size
    rb.rb_greedy(fom, reductor(), theta_lhs=TH[:1000], theta_rhs=np.ones((1000, 1)), batch=8, max_extensions=2,
                 tol=args.tol)
    torch.cuda.synchronize()

    for P, batch, rmax in runs:
        config = {"n": n, "Q": Q, "k": args.k, "P": P, "batch": batch, "r_max": rmax, "tol": args.tol,
                  "projection": "galerkin", "method": "cg", "gpu": gpu[0], "power_limit": gpu[1]}
        th, tf = TH[:P], np.ones((P, 1))
        res = rb.rb_greedy(fom, reductor(), theta_lhs=th, theta_rhs=tf, batch=batch, max_basis_size=rmax,
                           tol=args.tol)
        phases = ("reduce", "sweep", "solve", "extend")
        sums = dict.fromkeys(phases + ("total", "unattributed"), 0.0)
        for i, t in enumerate(res["timings"]):
            rest = t["total"] - sum(t.get(k, 0.0) for k in phases)
            for k in phases + ("total",):
                sums[k] += t.get(k, 0.0)
            sums["unattributed"] += rest
            it = res["fom_iterations"][i] if i < len(res["fom_iterations"]) else []
            emit({"P": P, "batch": batch, "iteration": i, "r": res["basis_sizes"][i], "max_est": res["max_errs"][i],
                  **{k + "_ms": t.get(k) for k in phases}, "total_ms": t["total"], "unattributed_ms": rest,
                  "unattributed_share": rest / t["total"],
                  "fom_iterations": [min(it), max(it)] if it else None})
        # the per-mu yardstick on the final ROM (r = r_max)
        rom = res["rom"]
        m = min(args.loop_mus, P)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loop = [rom.estimate_error(theta_lhs=th[p], theta_rhs=tf[p]) for p in range(m)]
        loop_s = time.perf_counter() - t0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        est = rom.estimate_error_batch(theta_lhs=th, theta_rhs=tf)
        torch.cuda.synchronize()
        batch_sweep_s = time.perf_counter() - t0
        agree = float(np.max(np.abs(est[:m].cpu().numpy() - np.array(loop)) / np.maximum(np.array(loop), 1e-300)))
        ext = [t for t in res["timings"] if "solve" in t]
        emit({"config": config, "stop": res["stop"], "extensions": res["extensions"], "r_final": res["basis_sizes"][-1],
              "max_errs_first_last": [res["max_errs"][0], res["max_errs"][-1]], "greedy_s": res["time"],
              "host_splu_R_s": splu_s,
              "phase_ms_sum": {k: sums[k] for k in phases}, "total_ms_sum": sums["total"],
              "unattributed_ms_sum": sums["unattributed"], "unattributed_share": sums["unattributed"] / sums["total"],
              "max_unattributed_share_of_an_extension": max(
                  (t["total"] - sum(t[k] for k in phases)) / t["total"] for t in ext) if ext else None,
              "final_rom_batched_sweep_ms": batch_sweep_s * 1e3,
              "per_mu_estimate_loop": {"mus": m, "s": loop_s, "extrapolated_to_P_s": loop_s * P / m,
                                       "extrapolated": True, "max_rel_diff_to_batched": agree}})
    out.close()


if __name__ == "__main__":
    main()
