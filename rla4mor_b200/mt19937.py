"""NumPy's legacy MT19937 Gaussian draws on the device, bit for bit (csrc/mt19937.cu).

`gaussian_matrix(seeds, rows, n, scale)` is the CUDA tensor equal to
    np.vstack([np.random.RandomState(s).normal(size=(b, n), loc=0, scale=scale) for s, b in zip(seeds, rows)])
-- the reference's Theta (rla/embeddings.py:269) or its stacked row blocks (:458) -- and
`gaussian_matrix_host` is the same array in host memory, drawn on the device and downloaded in
bounded chunks.  `NormalPlan` is the plan / execute split underneath: the jump-ahead and the
acceptance count run once per batch of seeds, then any range of any stream is cheap.
"""
import ctypes
import math

import numpy as np
import torch

from ._lib import RlaError, check, lib, stream_ptr

RLA_ERR_WORKSPACE = -3
# Pairs whose extended log lies within W_DEFAULT ulp of a rounding midpoint take the C library's
# log from the host (about 2 W_DEFAULT of all pairs); the exactness argument needs W > 0.019 + 2^-13.
W_DEFAULT = 2.0 ** -5
_ACCEPT = math.pi / 4


def _key(seed):
    st = np.random.RandomState(seed).get_state(legacy=False)
    s = st["state"]
    if s["pos"] != 624 or st["has_gauss"]:
        raise RlaError("mt19937: a fresh RandomState(seed) is expected at position 624")
    return np.asarray(s["key"], dtype=np.uint32)


def _segments(count, seg_words):
    """Segments for `count` normals: the expected attempts plus eight standard deviations."""
    pairs = (count + 1) // 2
    attempts = pairs / _ACCEPT + 8.0 * math.sqrt(pairs * (1 - _ACCEPT)) / _ACCEPT + 64
    return max(1, int(math.ceil(4 * attempts / seg_words)))


class NormalPlan:
    """Segment start states and accepted-pair prefix counts of one batch of seeds (stream i holds
    at least counts[i] normals), in device memory of `device`."""

    def __init__(self, seeds, counts, device=None):
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.counts = [int(c) for c in counts]
        assert len(self.counts) == len(seeds) >= 1 and min(self.counts) >= 0
        keys = np.ascontiguousarray(np.stack([_key(s) for s in seeds]))
        seg_words = lib().rla_mt19937_segment_words()
        nseg = np.array([_segments(c, seg_words) for c in self.counts], dtype=np.int64)
        self._h = None
        while True:
            h = ctypes.c_void_p()
            check(lib().rla_mt19937_plan_create(ctypes.byref(h), keys.ctypes.data, nseg.ctypes.data, len(nseg)),
                  "rla_mt19937_plan_create")
            self._h = h
            with torch.cuda.device(self.device):
                self._ws = torch.empty(lib().rla_mt19937_plan_workspace_bytes(h), dtype=torch.uint8, device=self.device)
                check(lib().rla_mt19937_plan_build(h, self._ws.data_ptr(), self._ws.numel(), stream_ptr()),
                      "rla_mt19937_plan_build")
            short = np.array([2 * lib().rla_mt19937_plan_pairs(h, i) < c for i, c in enumerate(self.counts)])
            if not short.any():
                break
            self._destroy()                                  # rare: more rejections than planned
            nseg = np.where(short, 2 * nseg, nseg)

    def _destroy(self):
        if self._h is not None:
            lib().rla_mt19937_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self._destroy()
        except Exception:
            pass

    def execute(self, out, first, count, offset, scale, w=W_DEFAULT):
        """Normals [first[i], first[i] + count[i]) of stream i into the flat float64 CUDA tensor
        `out` at offset[i].  Returns the number of pairs finished with the host's log."""
        assert out.is_cuda and out.dtype == torch.float64 and out.is_contiguous()
        ns = len(self.counts)
        first, count, offset = (np.ascontiguousarray(np.broadcast_to(np.asarray(a, dtype=np.int64), (ns,)))
                                for a in (first, count, offset))
        pairs = int(np.sum((count + 2) // 2))
        cap = min(pairs, int(pairs * min(1.0, 2.5 * w)) + 4096)
        nflag = ctypes.c_int64(0)
        while True:
            with torch.cuda.device(self.device):
                ws = torch.empty(lib().rla_mt19937_execute_workspace_bytes(self._h, cap), dtype=torch.uint8,
                                 device=self.device)
                staging = torch.empty(max(cap, 1), dtype=torch.float64, pin_memory=True)
                rc = lib().rla_mt19937_normal_f64(self._h, first.ctypes.data, count.ctypes.data, offset.ctypes.data,
                                                  float(scale), float(w), out.data_ptr(), out.numel(), ws.data_ptr(),
                                                  ws.numel(), cap, staging.data_ptr(), ctypes.byref(nflag), stream_ptr())
            if rc == RLA_ERR_WORKSPACE and nflag.value > cap:
                cap = nflag.value
                continue
            check(rc, "rla_mt19937_normal_f64")
            return nflag.value


def gaussian_matrix(seeds, rows, n, scale, device=None, w=W_DEFAULT, plan=None):
    """(sum(rows), n) CUDA float64 tensor: row block i is RandomState(seeds[i]).normal(size=(rows[i], n),
    loc=0, scale=scale)."""
    rows = [int(b) for b in rows]
    counts = [b * n for b in rows]
    plan = NormalPlan(seeds, counts, device) if plan is None else plan
    out = torch.empty((sum(rows), n), dtype=torch.float64, device=plan.device)
    if out.numel():
        plan.execute(out.view(-1), 0, counts, np.cumsum([0] + counts[:-1]), scale, w)
    return out


def gaussian_matrix_host(seeds, rows, n, scale, device=None, chunk_bytes=1 << 30, w=W_DEFAULT):
    """The same array as NumPy in host memory, drawn on the device in pieces of at most
    `chunk_bytes` (whole rows) and downloaded piece by piece."""
    rows = [int(b) for b in rows]
    out = np.empty((sum(rows), n), dtype=np.float64)
    if out.size == 0:
        return out
    plan = NormalPlan(seeds, [b * n for b in rows], device)
    step = max(1, int(chunk_bytes) // (8 * n))
    buf = torch.empty((min(step, max(rows)), n), dtype=torch.float64, device=plan.device)
    ns = len(rows)
    r_out = 0
    for i, b in enumerate(rows):
        for r0 in range(0, b, step):
            r1 = min(b, r0 + step)
            first = np.zeros(ns, np.int64)
            count = np.zeros(ns, np.int64)
            first[i], count[i] = r0 * n, (r1 - r0) * n
            piece = buf[:r1 - r0]
            plan.execute(buf.view(-1), first, count, 0, scale, w)
            torch.from_numpy(out[r_out + r0:r_out + r1]).copy_(piece)
        r_out += b
    return out
