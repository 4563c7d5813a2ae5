"""Developer timing of the int8 sketch of float64 blocks (csrc/gemm_i8.cu) with its own roofline:
int8 MACs actually issued (36 slice products of a 128 x 64 x 32 tile per stage, padded tiles
included) against the data-sheet dense int8 rate of a B200, 2250 T MAC/s (not reached), and the
FP64 tensor-pipe path (kind 1 on the same block: Rademacher, still DMMA) beside it.
bench.py reports the gauss_c2 step against the DMMA peak with the DMMA kernel's name; this script is
the roofline of the kernel that actually runs."""
import argparse, os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rla4mor_b200 import dense  # noqa: E402

IS, IL, BM, BN, BK = 8, 1 << 14, 128, 64, 32
PAIRS = IS * (IS + 1) // 2
INT8_PEAK_TMACS = 2250.0

ap = argparse.ArgumentParser()
ap.add_argument("--m", type=int, default=512); ap.add_argument("--logn", type=int, default=22)
ap.add_argument("--k", type=int, default=2000); ap.add_argument("--iters", type=int, default=5)
a = ap.parse_args()
n = 2 ** a.logn
u = torch.randn(a.m, n, dtype=torch.float64, device="cuda")


def best_ms(f):
    f(); torch.cuda.synchronize()
    ts = []
    for _ in range(a.iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); f(); e1.record(); torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    return min(ts)


mt, nt, st = -(-a.m // BM), -(-a.k // BN), -(-n // BK)
macs = PAIRS * mt * BM * nt * BN * st * BK
t8 = best_ms(lambda: dense.embed_apply_rng(0, 0, 1.0, a.k, u))
td = best_ms(lambda: dense.embed_apply_rng(0, 1, 1.0, a.k, u))
fl = 2.0 * a.m * a.k * n
print(f"m={a.m} n=2^{a.logn} k={a.k}: int8 path {t8:.2f} ms = {fl / t8 / 1e9:.1f} FP64-equivalent TFLOP/s, "
      f"{macs / t8 / 1e9:.0f} T int8 MAC/s issued = {macs / t8 / 1e9 / INT8_PEAK_TMACS:.3f} of {INT8_PEAK_TMACS:.0f} "
      f"(data sheet); DMMA path (kind 1) {td:.2f} ms", flush=True)
