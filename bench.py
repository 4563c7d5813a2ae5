#!/usr/bin/env python
"""bench.py -- sketch throughput of the B200 sketching engine (contract bench).

    python bench.py --gpus N --steps K --warmup W                 # our arm
    python bench.py --impl reference --gpus N --steps K --warmup W # CPU reference arm
    torchrun ... bench.py --gpus N ...                             # N > 1, one rank per GPU

A step is one pass of the hot path over one block of synthetic vectors.  Workloads
(BASELINE.json `configs`):
    gauss_c2 (default)  Gaussian embedding k=2000 on a float64 2^22 x 512 block, Theta
                        generated on the fly (configs[1]; FP64 tensor-pipe bound)
    gauss_c2_f32        the same shape with a FLOAT32 block on the generation-5 tensor cores
                        (tcgen05 kind::tf32, Theta = normals rounded to TF32, FP64 accumulation of
                        64-term partial sums; 1e-5 tolerance); `secondary`
    srht_c3             SRHT k=4000 on a float64 2^24 x 1024 block, column-sharded
                        (configs[2]; HBM bound); run as the `secondary` result
    srht_c1             SRHT k=1000 on 2^16 x 200 (configs[0], the one case the reference runs in
                        full on the CPU: the oracle's whole srht() is timed beside it, L2 flushed
                        between steps because the 105 MB block fits the 126 MB L2); `secondary`
    sketched_reductor_c4  SketchedReductor.extend_basis on an n = 1e6, Q = 4 FEM-like problem with the
                        LU inverse product (configs[3]; tools/bench_c4.py; the inverse product of all Q
                        terms is ONE sparse triangular solve of Q m right-hand sides, whose HBM
                        roofline the line carries); `secondary`, rank 0
    rangefinder_c5      sketch + thin QR / SVD of a 2^23 x 256 block, k=1024, ROW-sharded with one
                        exchange of the (m, k) partials over NVLink peer memory (configs[4]);
                        second `secondary` result (tools/bench_c5.py)
Multi-GPU: column-sharded, no collective.  gauss_c2 scales weakly (every rank sketches its
own 2^22 x 512 block); srht_c3 is the fixed 2^24 x 1024 block split by columns (strong);
rangefinder_c5 is the fixed block split by rows (strong).
Prints ONE JSON line on rank 0.

    python bench.py --dump-outputs bench_out ...

also writes, on rank 0, the sketch that each workload timed in this file (the primary one and,
beside gauss_c2, srht_c3, srht_c1 and gauss_c2_f32) computed in its last timed step, as
bench_out/<workload>.npy (float64, m x k).  A sketch larger than 16 MB is cut to a fixed,
seeded sample of its rows, so the files stay under 64 MB in all.  The input blocks come from seeded generators, so two
builds run with the same arguments can be compared file by file.  A workload whose block had
to be cut to the free memory is not written (its note in the JSON line says so).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "gauss_c2": dict(kind="gauss", m=512, logn=22, k=2000, config="configs[1]"),
    "srht_c3": dict(kind="srht", m=1024, logn=24, k=4000, config="configs[2]"),
    "srht_c1": dict(kind="srht", m=200, logn=16, k=1000, config="configs[0]"),
    # configs[1] with a float32 block: the optional FP32 path of north_star (tcgen05 kind::tf32)
    "gauss_c2_f32": dict(kind="gauss32", m=512, logn=22, k=2000, config="configs[1] (float32 block, optional FP32 path)"),
}


def workload_config(name, world, m_loc=None, note=None):
    """The `config` object of the JSON line -- built by BOTH arms from the same inputs."""
    wl = WORKLOADS[name]
    n = 2 ** wl["logn"]
    strong = name == "srht_c3"
    if m_loc is None:
        m_loc = wl["m"] // world if strong else wl["m"]
    m_total = m_loc * world
    esz = 4 if wl["kind"] == "gauss32" else 8
    cfg = {"workload": name, "baseline_config": wl["config"], "embedding": wl["kind"], "m_total": m_total,
           "m_per_gpu": m_loc, "n": n, "k": wl["k"], "partition": f"columns x{world} (no collective)",
           "scaling": "strong" if strong else "weak",
           "l2": ("inputs larger than L2 (per-GPU block %.1f GB >> 126 MB)" % (m_loc * n * esz / 1e9)) if m_loc * n * esz > 2e8
           else "L2 flushed between timed steps (256 MB write); per-step CUDA events"}
    if note:
        cfg["note"] = note
    return cfg


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="gauss_c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary SRHT result")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the sketch of the last timed step of every workload as DIR/<workload>.npy")
    return ap.parse_args()


DUMP_BYTES_PER_OUTPUT = 16_000_000       # at most four sketches are dumped: 64 MB in all


def dump_sample(out):
    """`out` (m, k) on the device -> host float64 array: all of it, or the rows of a fixed seeded
    sample (in ascending order) when it is larger than DUMP_BYTES_PER_OUTPUT."""
    import torch
    rows = max(1, DUMP_BYTES_PER_OUTPUT // (out.shape[1] * 8))
    if out.shape[0] > rows:
        idx = np.sort(np.random.RandomState(0).choice(out.shape[0], rows, replace=False))
        out = out[torch.from_numpy(idx).to(out.device)]
    return out.to(torch.float64).cpu().numpy()


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------ CPU reference legs
def cpu_gauss_sample(U_host, k_total, k_block, seed=0):
    """One row block of Theta in the reference's BlockGaussianEmbedding decomposition
    (rla/embeddings.py:393-400,425-434,452-461): RandomState.normal + (Theta @ U^T)^T."""
    from oracle import embeddings_oracle as eo
    t0 = time.perf_counter()
    theta = eo.block_gaussian_block(k_total, U_host.shape[1], k_block, seed)
    y = (theta @ U_host.T).T
    dt = time.perf_counter() - t0
    return dt, float(np.abs(y).sum())


def cpu_srht_sample(x_host, k, seed=0):
    import oracle
    t0 = time.perf_counter()
    y = oracle.srht(x_host, k, seed=seed, nthreads=0)
    return time.perf_counter() - t0, float(np.abs(y).sum())


def host_block(m, n, seed=1234):
    """Synthetic N(0,1) block on the host; a 16-vector base is tiled (values do not matter
    for the CPU timing, generation of 17 GB of normals would dominate the run)."""
    rs = np.random.RandomState(seed)
    base = rs.standard_normal((min(m, 16), n))
    reps = -(-m // base.shape[0])
    return np.ascontiguousarray(np.tile(base, (reps, 1))[:m])


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
    except Exception:
        return os.cpu_count() or 1


def all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1, which would leave the CPU arm's BLAS on one core: lift the
    limit of every thread pool in the process to the host's core count."""
    cores = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=cores)
    except Exception:
        pass
    os.environ["OMP_NUM_THREADS"] = str(cores)
    return cores


def run_reference(args):
    """`--impl reference`: the reference's CPU algorithm for the same workload on the host
    cores of this box (oracle port: /root/reference is a Python tree that does not travel
    to the GPU box, so its restatement under oracle/ -- checked against outputs of the executed
    reference, tests/test_reference_goldens_cpu.py -- is what runs here)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = all_host_threads()
    wl = WORKLOADS[args.workload]
    m, n, k = wl["m"], 2 ** wl["logn"], wl["k"]
    extrapolated = True
    if wl["kind"] in ("gauss", "gauss32"):                # the CPU reference has one Gaussian path (float64 Theta)
        kb = 50
        U = host_block(m, n)
        step = lambda: cpu_gauss_sample(U, k, kb)
        sample = (f"one {kb}-row block of Theta (of {k}) over the full {m} x 2^{wl['logn']} block per step: "
                  f"RandomState.normal + dgemm; whole-sketch time = step time x {k // kb}")
        scale = k / kb
        threads = blas_threads()
    else:
        ms = min(m, 8 if wl["logn"] >= 22 else m)
        U = host_block(ms, n)
        step = lambda: cpu_srht_sample(U, k)
        extrapolated = ms < m
        sample = (f"{ms} of {m} vectors per step (srht() incl. its per-call sign/index draw); rate scaled per vector"
                  if extrapolated else f"the whole {m} x 2^{wl['logn']} block per step (srht() incl. its sign/index draw)")
        scale = m / ms
        import oracle.srht_oracle as so
        threads = so.oracle_threads()
    for _ in range(max(1, min(args.warmup, 1))):
        step()
    t = []
    for _ in range(args.steps):
        dt, _ = step()
        t.append(dt)
        if sum(t) > 240:
            break
    full = float(np.mean(t)) * scale                      # seconds for one whole block
    gbs = m * n * 8 / full / 1e9
    line = {
        "impl": "reference", "metric": "sketch throughput", "value": gbs, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": len(t), "warmup": min(args.warmup, 1), "ms_per_step": float(np.mean(t)) * 1e3,
        "higher_is_better": True, "scaling": "strong" if args.workload == "srht_c3" else "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": workload_config(args.workload, max(1, args.gpus)),
        "cols_per_s": m / full,
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": threads, "kind": "port", "sample": sample,
                         "host_cpus": cores, "extrapolated": extrapolated,
                         "note": "one host processes one block at this rate whatever N is (the GPU arm's weak-scaled "
                                 "value is N blocks)"},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    import rla4mor_b200 as rb
    from rla4mor_b200 import dense
    from rla4mor_b200.streaming import apply_streamed

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the sketching engine has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner on STDOUT at NCCL_DEBUG=VERSION; stdout carries only the JSON line
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=300))
    lib = rb.lib()
    peaks, peak_src = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    def reduce_sum(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            return float(t.item())
        return x

    flush_buf = []
    dumps = {}

    def timed(step, steps, warmup, flush=False):
        """K timed steps.  Default: back to back, start-to-end CUDA events.  flush=True (inputs that
        fit the 126 MB L2): a 256 MB buffer is overwritten before every step and each step is
        timed by its own event pair (the flush is outside the timed region)."""
        if flush and not flush_buf:
            flush_buf.append(torch.empty(256 << 20, dtype=torch.uint8, device=dev))
        for _ in range(warmup):
            if flush and flush_buf:
                flush_buf[0].add_(1)
            step()
        barrier()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        l0 = lib.rla_launch_count()
        if flush:
            pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for e0, e1 in pairs:
                flush_buf[0].add_(1)
                e0.record()
                step()
                e1.record()
            torch.cuda.synchronize()
            timed.last_step_ms = [e0.elapsed_time(e1) for e0, e1 in pairs]
            ms = float(sum(timed.last_step_ms))
        else:
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
            evs[0].record()
            for i in range(steps):
                step()
                evs[i + 1].record()
            torch.cuda.synchronize()
            ms = evs[0].elapsed_time(evs[-1])                    # the K timed steps, start to end
            timed.last_step_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
        launches = lib.rla_launch_count() - l0
        clocks = sampler.stop() if rank == 0 else None
        barrier()
        return reduce_max(ms), int(reduce_sum(launches)), clocks

    def run_workload(name, with_e2e, with_cpu, steps, warmup):
        wl = WORKLOADS[name]
        n, k = 2 ** wl["logn"], wl["k"]
        strong = wl["kind"] == "srht" and name == "srht_c3"
        m_total = wl["m"] if strong else wl["m"] * world
        m_loc = wl["m"] // world if strong else wl["m"]
        note = None
        free, _ = torch.cuda.mem_get_info(dev)
        fit = int((free - (6 << 30)) // (n * 8))
        if m_loc > fit:
            note = f"per-GPU block cut from {m_loc} to {fit} vectors to fit {free / 2**30:.0f} GiB free"
            m_loc = fit
            m_total = m_loc * world
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        dt_in = torch.float32 if wl["kind"] == "gauss32" else torch.float64
        esz = 4 if wl["kind"] == "gauss32" else 8
        U = torch.empty((m_loc, n), dtype=dt_in, device=dev)
        for lo in range(0, m_loc, 32):                      # in-place fill, no 2x temporary
            U[lo:lo + 32].normal_(generator=gen)
        out = torch.empty((m_loc, k), dtype=torch.float64, device=dev)
        if wl["kind"] == "gauss":
            emb = rb.GaussianEmbedding(source=rb.DeviceVectorSpace(n), options={"range_dim": k, "rng": "philox"}, _seed=0)
            step = lambda: dense.embed_apply_rng(0, dense.KIND_NORMAL, 1.0 / np.sqrt(k), k, U, out=out)
            apply_fn = emb.apply
            work = 2.0 * k * n * m_loc                       # flops per rank per step
            scratch = torch.empty(1 << 20, dtype=torch.uint8, device=dev)
            import ctypes
            pk = ctypes.c_double(0.0)
            rb._lib.check(lib.rla_dmma_peak_tflops(ctypes.byref(pk), scratch.data_ptr(), rb._lib.stream_ptr()), "dmma peak")
            a_cb = torch.randn(4096, 4096, dtype=torch.float64, device=dev)
            for _ in range(2):
                a_cb @ a_cb
            torch.cuda.synchronize()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record(); a_cb @ a_cb; c1.record(); torch.cuda.synchronize()
            cublas_tf = 2 * 4096 ** 3 / c0.elapsed_time(c1) / 1e9
            del a_cb
            roof = dict(bound="tensor", unit="TFLOP/s", peak=pk.value,
                        peak_source="in-run FP64 DMMA issue-rate microbenchmark (rla_dmma_peak_tflops); "
                                    "MEASURED_PEAKS.json has no FP64 entry",
                        cublas_dgemm_tflops_same_run=cublas_tf,
                        algorithmic="2*k*n*m flops per launch, Theta generated in-kernel (no bytes)")
        elif wl["kind"] == "gauss32":
            emb = rb.GaussianEmbedding(source=rb.DeviceVectorSpace(n), options={"range_dim": k, "rng": "philox_tf32"}, _seed=0)
            step = lambda: dense.embed_apply_rng(0, dense.KIND_NORMAL_TF32, 1.0 / np.sqrt(k), k, U, out=out)
            apply_fn = emb.apply
            work = 2.0 * k * n * m_loc
            tf32_peak = float(peaks.get("bf16_tflops", 1618.2)) / 2.0
            roof = dict(bound="tensor", unit="TFLOP/s", peak=tf32_peak,
                        peak_source="half of the measured dense bf16 figure (MEASURED_PEAKS.json): kind::tf32 runs at half the bf16 rate",
                        algorithmic="2*k*n*m flops per launch (Theta generated in-kernel, no bytes); the kernel issues TWO "
                                    "tf32 MMAs per product (two-part split of the block), so the tensor pipe is busy at twice "
                                    "`frac`; the bound of this kernel is the Theta generator (1024 Philox blocks per 128 x 128 x 32 "
                                    "stage), not the tensor pipe")
        else:
            emb = rb.SrhtEmbedding(source=rb.DeviceVectorSpace(n), options={"range_dim": k}, _seed=0)
            plan = emb._plan(torch.float64, dev)
            step = lambda: plan.apply(U, out=out)
            apply_fn = emb.apply
            work = float(m_loc * n * 8 + m_loc * k * 8 + n + 4 * k)   # algorithmic bytes per rank per step
            roof = dict(bound="hbm", unit="GB/s", peak=float(peaks["hbm_gbs"]), peak_source=peak_src,
                        algorithmic="m*n*8 (read U once) + m*k*8 (write sketch) + n (signs) + 4k (indices) bytes per launch")
        small = m_loc * n * esz < 2e8                        # fits L2: flush between steps
        ms, launches, clocks = timed(step, steps, warmup, flush=small)
        if args.dump_outputs and rank == 0:
            if note:                                         # another block than the seeded one: not comparable
                sys.stderr.write(f"bench.py: no {name}.npy written ({note})\n")
            else:
                dumps[name] = dump_sample(out)
        t_step = ms / steps / 1e3
        achieved = work / t_step / (1e12 if roof["bound"] == "tensor" else 1e9)
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath)).get(name) or {}
            traffic = tj.get("bytes")
            traffic_src = "not measured in this run: dram__bytes_read+write of the ncu --set full capture " + str(tj.get("source", "under profiles/"))
        best = min(timed.last_step_ms) / 1e3
        roof.update(achieved=achieved, frac=achieved / roof["peak"], traffic=traffic, traffic_source=traffic_src,
                    frac_best_step=work / best / (1e12 if roof["bound"] == "tensor" else 1e9) / roof["peak"],
                    achieved_best_step=work / best / (1e12 if roof["bound"] == "tensor" else 1e9),
                    step_ms=[round(v, 3) for v in timed.last_step_ms],
                    kernel="sketch_gemm_kernel" if wl["kind"] == "gauss" else
                    "sketch_gemm_tf32_kernel" if wl["kind"] == "gauss32" else
                    ("srht_ws_kernel" if m_loc * (n // 4096) >= 16384 else "srht_main_kernel"),
                    note="duration = whole step (main kernel + its small reduce/finalize kernel), CUDA events")
        res = {
            "workload": name, "value": m_total * n * esz / t_step / 1e9, "unit": "GB/s",
            "cols_per_s": m_total / t_step, "ms_per_step": ms / steps, "gpu_launches": launches,
            "roofline": roof, "clocks": clocks,
            "config": workload_config(name, world, m_loc, note),
        }
        if wl["kind"] == "srht" and clocks:
            roof["note_power"] = ("frac is the mean over the back-to-back steps; frac_best_step the fastest step. A pure HBM "
                                  "read stream already holds this board at its 1000 W cap (SM clock ~1.6 GHz, "
                                  "profiles/srht_r02_experiments.txt); the 13 FP64 adds per element then run at that clock")
        # ---- end to end: host (pinned) block -> H2D -> sketch -> D2H of the result, per step
        if with_e2e:
            m_e = min(m_loc, max(1, (20 << 30) // (n * esz)))         # at most ~20 GiB of pinned memory
            try:
                host = torch.empty((m_e, n), dtype=dt_in, pin_memory=True)
                host.copy_(U[:m_e])
                torch.cuda.synchronize()
                e_step = lambda: apply_fn(host)                       # host block in, host sketch out
                e_steps = max(2, min(steps, 5))
                ems, _, _ = timed(e_step, e_steps, 1, flush=small)
                te = ems / e_steps / 1e3
                res["e2e"] = {"value": m_e * world * n * esz / te / 1e9, "unit": "GB/s",
                              "h2d_bytes_per_step": int(m_e * n * esz), "d2h_bytes_per_step": int(m_e * k * 8),
                              "api": f"{type(emb).__name__}.apply(pinned host block) -> pinned host sketch; ~1 GiB pieces "
                                     "copied on a side stream under the sketch of the previous piece (streaming.py)",
                              "m_per_gpu": m_e, "ms_per_step": ems / e_steps, "cols_per_s": m_e * world / te}
                if rank == 0 and with_cpu and name == "srht_c1":
                    # configs[0] is the one case the CPU reference runs in full: time it, no extrapolation
                    import oracle.srht_oracle as so
                    all_host_threads()
                    cpu_srht_sample(host.numpy()[:1, :4096].copy(), 16)
                    dts = [cpu_srht_sample(host.numpy(), k)[0] for _ in range(3)]
                    dt = float(np.median(dts))
                    res["cpu_baseline"] = {"value": m_e * n * 8 / dt / 1e9, "unit": "GB/s", "cores": so.oracle_threads(),
                                           "kind": "port", "host_cpus": os.cpu_count(), "extrapolated": False,
                                           "sample": f"the whole {m_e} x 2^{wl['logn']} block, oracle srht() incl. its sign/index "
                                                     f"draw, median of 3: {dt * 1e3:.0f} ms", "cols_per_s": m_e / dt}
                    del host
                elif rank == 0 and with_cpu:
                    res["_host_block"] = host.numpy()
                else:
                    del host
            except RuntimeError as exc:                               # pinned allocation refused
                res["e2e"] = {"value": None, "unit": "GB/s", "error": str(exc)[:200]}
        del U, out
        torch.cuda.empty_cache()
        return res

    secondary = []
    if not args.no_secondary and args.workload == "gauss_c2":
        # configs[2] first: the 137 GB block needs the whole HBM, and every workload is then timed
        # from an idle GPU (the FP64 GEMM leaves the board at its power cap for seconds)
        secondary.append(run_workload("srht_c3", not args.no_e2e, False, max(3, min(args.steps, 10)), max(3, args.warmup)))
        secondary[-1].pop("_host_block", None)
        secondary[-1]["order"] = "timed before the primary workload"
        time.sleep(1.0)
        # configs[0]: the reference's own CPU-sized case, with e2e and the whole CPU srht() beside it
        secondary.append(run_workload("srht_c1", not args.no_e2e, not args.no_cpu_baseline and args.gpus == 1,
                                      max(5, min(args.steps, 20)), max(3, args.warmup)))
        secondary[-1].pop("_host_block", None)
    primary = run_workload(args.workload, not args.no_e2e, not args.no_cpu_baseline, args.steps, args.warmup)
    host_block_np = primary.pop("_host_block", None)
    if not args.no_secondary and args.workload == "gauss_c2":
        try:
            secondary.append(run_workload("gauss_c2_f32", not args.no_e2e, False, max(3, min(args.steps, 10)), max(3, args.warmup)))
            secondary[-1].pop("_host_block", None)
            if secondary[-1].get("roofline"):
                secondary[-1]["dtype"] = "f32 block, tf32 x 2 tensor-core products, FP64 accumulation of 64-term partial sums"
        except Exception as exc:
            secondary.append({"workload": "gauss_c2_f32", "error": f"{type(exc).__name__}: {exc}"[:300]})

    if not args.no_secondary and args.workload == "gauss_c2":
        # configs[4]: row-sharded range finder (sketch + NVLink peer-memory exchange + thin QR / SVD)
        try:
            from tools.bench_c5 import run_c5
            pk = primary["roofline"].get("peak") if primary["roofline"]["bound"] == "tensor" else None
            secondary.append(run_c5(rank, world, dev, steps=max(3, min(args.steps, 10)), warmup=3,
                                    hbm_peak=float(peaks["hbm_gbs"]), dmma_peak=pk))
        except Exception as exc:                                       # never lose the primary line to a secondary
            secondary.append({"workload": "rangefinder_c5", "error": f"{type(exc).__name__}: {exc}"[:300]})
        # configs[3]: SketchedReductor with the LU inverse product (rank 0; the other ranks wait at the barrier)
        if rank == 0:
            try:
                from tools.bench_c4 import run_c4
                secondary.append(run_c4(hbm_peak=float(peaks["hbm_gbs"]), with_cpu=not args.no_cpu_baseline and args.gpus == 1))
            except Exception as exc:
                secondary.append({"workload": "sketched_reductor_c4", "error": f"{type(exc).__name__}: {exc}"[:300]})
        barrier()

    cpu = None
    if rank == 0 and world >= 1 and not args.no_cpu_baseline and args.gpus == 1:
        wl = WORKLOADS[args.workload]
        m, n, k = wl["m"], 2 ** wl["logn"], wl["k"]
        if wl["kind"] == "gauss":
            Uh = host_block_np if host_block_np is not None else host_block(m, n)
            kb = 50
            cpu_gauss_sample(Uh[:8], k, 2)                           # warm BLAS
            dt, _ = cpu_gauss_sample(Uh, k, kb)
            full = dt * (k / kb) * (m / Uh.shape[0])
            cpu = {"value": m * n * 8 / full / 1e9, "unit": "GB/s", "cores": blas_threads(), "kind": "port",
                   "sample": f"one {kb}-row Theta block (of {k}) over {Uh.shape[0]} x 2^{wl['logn']} vectors: "
                             f"{dt:.1f} s; RandomState.normal (1 thread) + OpenBLAS dgemm; scaled x{k // kb}",
                   "host_cpus": os.cpu_count(), "cols_per_s": m / full}
        else:
            ms_ = min(m, 8 if wl["logn"] >= 22 else m)
            Uh = host_block(ms_, n)
            cpu_srht_sample(Uh[:1, :4096].copy(), 16)
            dt, _ = cpu_srht_sample(Uh, k)
            full = dt * m / ms_
            import oracle.srht_oracle as so
            cpu = {"value": m * n * 8 / full / 1e9, "unit": "GB/s", "cores": so.oracle_threads(), "kind": "port",
                   "sample": f"{ms_} of {m} vectors, srht() incl. its per-call sign/index draw: {dt:.1f} s; scaled per vector",
                   "host_cpus": os.cpu_count(), "cols_per_s": m / full}

    if dumps:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dumps.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    if rank == 0:
        line = {
            "metric": "sketch throughput", "value": primary["value"], "unit": "GB/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": primary["ms_per_step"],
            "higher_is_better": True, "scaling": primary["config"]["scaling"], "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": primary["config"], "cols_per_s": primary["cols_per_s"],
            "clocks": primary["clocks"], "e2e": primary.get("e2e"), "gpu_launches": primary["gpu_launches"],
            "roofline": primary["roofline"], "cpu_baseline": cpu,
            "secondary": secondary,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    assert args.warmup >= 0 and args.steps >= 1
    if args.impl == "reference" and args.dump_outputs:
        raise SystemExit("bench.py: --dump-outputs writes the sketches of our arm; the reference arm has none to write")
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3                                            # timing rule: W >= 3
        run_ours(args)


if __name__ == "__main__":
    main()
