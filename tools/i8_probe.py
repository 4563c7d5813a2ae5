"""Driver of tools/micro/i8_probe.cu: the stage-time attribution of the int8 sketch GEMM at the C2
grid.  Prints the card, its power limit and clocks, the probe variants 1-5, and variant 6: the full
sketch_gemm_i8_kernel of the library at the C2 shape (m = 512, n = 2^22, k = 2000), its device time
taken from torch.profiler (the slicing pre-pass and the chunk reduce excluded).

    python tools/i8_probe.py [--out profiles/gemm_i8_r03_probe.txt]

The probe binary is built into a temporary directory."""
import argparse
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

IS, IBM, IBN, IK = 8, 128, 64, 32


def smi():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks_event_reasons.active"
    return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv"], capture_output=True, text=True).stdout.strip()


def full_kernel(reps):
    import torch
    from torch.profiler import profile, ProfilerActivity
    from rla4mor_b200 import dense
    m, k, n = 512, 2000, 2 ** 22
    u = torch.randn(m, n, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    dense.embed_apply_rng(0, 0, 1.0, k, u)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            dense.embed_apply_rng(0, 0, 1.0, k, u)
        torch.cuda.synchronize()
    times = [e.device_time_total / e.count for e in prof.key_averages() if "sketch_gemm_i8_kernel" in e.key]
    if not times:
        raise SystemExit("sketch_gemm_i8_kernel did not run")
    ms = times[0] / 1e3
    macs = IS * (IS + 1) // 2 * (-(-m // IBM) * IBM) * (-(-k // IBN) * IBN) * (n // IK * IK)
    return f"{'6: full sketch_gemm_i8_kernel (library, mean of %d calls)' % reps:<66} {ms:8.2f} ms  {macs / ms / 1e9:6.0f} T int8 MAC/s"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    with tempfile.TemporaryDirectory() as td:
        exe = os.path.join(td, "i8_probe")
        from rla4mor_b200._build import _nvcc
        ccbin = ["-ccbin", "/usr/bin/g++"] if os.path.exists("/usr/bin/g++") else []
        subprocess.run([_nvcc(), "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                        os.path.join(ROOT, "tools", "micro", "i8_probe.cu"), "-o", exe] + ccbin, check=True)
        lines = [smi(), subprocess.run([exe], capture_output=True, text=True, check=True).stdout.rstrip()]
    lines.append(full_kernel(a.reps))
    lines.append(smi())
    text = "\n".join(lines) + "\n"
    print(text, end="")
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
