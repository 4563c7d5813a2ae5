"""Weak greedy construction of the reduced basis over a training set on the device: pyMOR's
`rb_greedy` / `weak_greedy`, with every step batched.

One iteration, in pyMOR's order:
    rom = reductor.reduce()
    sweep: a = rom.solve_batch(theta), est = rom.estimate_error_batch(a, theta)   (csrc/rom_batch.cu)
    record max est and its mu; stop on atol / rtol / max_extensions / max_basis_size
    select the `batch` largest estimates (stable descending sort: ties to the smallest row)
    U = fom solve of the selected rows, warm-started from the ROM solution a @ rb
                                                   (csrc/affine_cg.cu / affine_gmres.cu)
    reductor.extend_basis(U); stop if Gram-Schmidt removed every new vector

The training set's theta is evaluated on the host once and uploaded once; the sweeps read it in
place and the snapshot solves index the selected rows out of it.
"""
import logging
import time

import numpy as np
import torch

from . import fom_solve, sketched_reductor
from . import reductor_ops as ops
from ._lib import RlaError
from .sketched_reductor import _theta_rows
from .vectorarray import DeviceVectorArray

logger = logging.getLogger("rla4mor_b200.greedy")


def select_largest(est, batch):
    """The row indices of the `batch` largest entries of est (P,), largest first, ties to the
    smallest index (a stable descending sort; torch.topk leaves the order of ties unspecified),
    and the largest entry: (list of ints, float).  A NaN entry raises RlaError naming the first
    such row.  One device-to-host read."""
    est = torch.as_tensor(est, dtype=torch.float64)
    if est.dim() != 1 or est.numel() == 0:
        raise ValueError(f"select_largest: expected a non-empty (P,) tensor, got shape {tuple(est.shape)}")
    nan = torch.isnan(est)
    order = torch.sort(est, descending=True, stable=True).indices[:batch]
    head = torch.stack([nan.sum().to(torch.float64), torch.argmax(nan.to(torch.int32)).to(torch.float64),
                        est[order[0]]])
    host = torch.cat([head, order.to(torch.float64)]).tolist()     # indices < 2^53: exact in float64
    n_nan, first, top = host[:3]
    if n_nan:
        raise RlaError(f"rb_greedy: {int(n_nan)} of {est.numel()} error estimates are NaN (first: training row "
                       f"{int(first)}): its reduced system is singular or rank-deficient, or its theta is not finite")
    return [int(i) for i in host[3:]], top


def sweep_rows_per_chunk(P, r, kp, Q, Pf, free_bytes):
    """Training rows swept at once: per row the reduced solution (r doubles), the estimate and its
    workspace (one partial per 128 columns of the k' sketch), the solve's info word and the row's
    theta, within fom_solve.KRYLOV_MEMORY_FRACTION of `free_bytes` (the rule of
    SketchedReductor.extend_basis and affine_gmres); at least 1."""
    per_row = 8 * (r + 1 + Q + Pf + (kp + 127) // 128) + 4
    return max(1, min(P, int(fom_solve.KRYLOV_MEMORY_FRACTION * free_bytes) // per_row))


def batched_envelope(reductor):
    """Largest basis whose ROM is swept by the batched kernels: rom_solve_batch_max_r() for a
    Galerkin ROM; min(rom_lstsq_batch_max_r(), k') for a least-squares (minres) ROM, whose batched
    QR solve needs the online sketch dimension k' >= r."""
    if reductor.projection == 'galerkin':
        return ops.rom_solve_batch_max_r()
    return min(ops.rom_lstsq_batch_max_r(), reductor.embedding_online.range.dim)


def _sweep(rom, th, tf, r, kp):
    """Estimates of every training row, (P,), and the reduced solutions (P, r) when the set was
    swept in one chunk (None otherwise).  Each row's solve and estimate depend on that row only, so
    the chunking does not change a bit."""
    P = th.shape[0]
    chunk = sweep_rows_per_chunk(P, r, kp, th.shape[1], tf.shape[1], torch.cuda.mem_get_info(th.device)[0])
    est = torch.empty((P,), dtype=torch.float64, device=th.device)
    for p0 in range(0, P, chunk):
        rows = slice(p0, p0 + chunk)
        a = rom.solve_batch(th[rows], tf[rows], check=False)      # a singular system: NaN, caught by the selection
        est[rows] = rom.estimate_error_batch(a, th[rows], tf[rows])
    return est, (a if chunk >= P else None)


def rb_greedy(fom, reductor, mus=None, *, theta_lhs=None, theta_rhs=None, atol=None, rtol=None, max_extensions=None,
              max_basis_size=None, batch=1, method='cg', tol=1e-10, maxiter=500, restart=None, preconditioner=None):
    """Weak greedy basis generation (pyMOR's `rb_greedy`) with the sketched error estimator of
    `reductor` (a SketchedReductor of the AffineModel `fom`), extending its basis in place.

    The training set is `mus=` or theta_lhs (P, Q) and theta_rhs (P, Pf), validated as by
    SketchedRom.solve_batch.  Each iteration reduces, sweeps the whole set with the batched ROM
    (in chunks of rows within a quarter of the free device memory), records the largest estimate
    and stops on `atol` (max est <= atol), `rtol` (max est <= rtol * max_errs[0]), `max_extensions`
    or `max_basis_size`.  Otherwise it solves the full-order model at the `batch` largest estimates
    (ties to the smallest row) in one `fom` block solve (`method` 'cg' or 'gmres', `tol`, `maxiter`,
    `restart`; `preconditioner` defaults to reductor.inverse_product), warm-started from the ROM
    solutions when the reductor keeps its basis (save_rb), and extends the basis with them.  If
    Gram-Schmidt removes every new vector, the loop stops ('extension_failed').  So every stop
    leaves max_errs with one entry more than extensions, and the last one is the error of the
    returned ROM.

    max_basis_size defaults to batched_envelope(reductor) (169 for Galerkin, min(137, k') for
    minres), and no extension goes past it: beyond the envelope the ROM solves loop over mu on the
    host.  A larger max_basis_size is allowed, and logged once when the basis passes the envelope.

    Returns a dict: rom, max_errs, max_err_mus (mu objects for mus=, else row indices),
    extensions, time (s), selected (row indices per extension), basis_sizes (per entry of
    max_errs), stop ('atol' | 'rtol' | 'max_extensions' | 'max_basis_size' | 'extension_failed'),
    fom_iterations (per extension, per selected row) and timings (per entry of max_errs, host-clock
    ms of each phase, which ends in a device synchronise or a device-to-host read: reduce, sweep
    (with the selection), and for an iteration that extended, solve and extend; total covers the
    whole iteration, so total minus the phases is the driver's own host time)."""
    t_start = time.perf_counter()
    if isinstance(batch, bool) or not isinstance(batch, (int, np.integer)) or batch < 1:
        raise ValueError(f"rb_greedy: batch={batch!r} must be an integer >= 1")
    if method not in ('cg', 'gmres'):
        raise ValueError(f"rb_greedy: method={method!r}, expected 'cg' or 'gmres'")
    if preconditioner is None:
        preconditioner = reductor.inverse_product
    if preconditioner is None:
        raise ValueError("rb_greedy: no preconditioner: give preconditioner= or a reductor with inverse_product")
    dev = reductor.srb.device
    mus = None if mus is None else list(mus)
    th, tf = _theta_rows(fom, theta_lhs, theta_rhs, mus, len(fom.operators), len(fom.rhs), dev)
    th, tf = th.contiguous(), tf.contiguous()
    P = th.shape[0]
    if P == 0:
        raise ValueError("rb_greedy: empty training set")
    envelope = batched_envelope(reductor)
    if max_basis_size is None:
        max_basis_size = envelope
    kp = reductor.embedding_online.range.dim
    res = dict(max_errs=[], max_err_mus=[], extensions=0, selected=[], basis_sizes=[], fom_iterations=[], timings=[])
    ms = lambda t0, t1: (t1 - t0) * 1e3
    warned = False
    while True:
        t0 = time.perf_counter()
        rom = reductor.reduce()
        torch.cuda.synchronize(dev)                      # the reduction ends in no device-to-host read
        t1 = time.perf_counter()
        r = reductor.srb.shape[0]
        if r > envelope and not warned:
            logger.warning(f"basis size {r} is beyond the batched ROM solve's limit {envelope}: "
                           "the sweeps solve the reduced systems mu by mu")
            warned = True
        t2 = time.perf_counter()
        est, a = _sweep(rom, th, tf, r, kp)
        sel, top = select_largest(est, max(1, min(batch, max_basis_size - r)))   # the one read of the sweep
        t3 = time.perf_counter()
        timing = dict(reduce=ms(t0, t1), sweep=ms(t2, t3))
        res['timings'].append(timing)
        res['basis_sizes'].append(r)
        res['max_errs'].append(top)
        res['max_err_mus'].append(sel[0] if mus is None else mus[sel[0]])
        logger.info(f"maximum estimated error after {res['extensions']} extensions (r = {r}): {top:.6g} "
                    f"(training row {sel[0]})")
        if atol is not None and top <= atol:
            res['stop'] = 'atol'
        elif rtol is not None and top <= rtol * res['max_errs'][0]:
            res['stop'] = 'rtol'
        elif max_extensions is not None and res['extensions'] >= max_extensions:
            res['stop'] = 'max_extensions'
        elif r >= max_basis_size:
            res['stop'] = 'max_basis_size'
        if 'stop' in res:
            timing['total'] = ms(t0, time.perf_counter())
            break
        idx = torch.tensor(sel, dtype=torch.int64, device=dev)
        x0 = None
        if reductor.save_rb and r > 0:
            # the ROM solution is the best guess at hand; the solvers stop relative to ||f||_{R^-1},
            # so a warm start only saves iterations
            a_sel = a[idx] if a is not None else rom.solve_batch(th[idx], tf[idx], check=False)
            x0 = ops.lincomb(a_sel, reductor.rb)
        t4 = time.perf_counter()
        X, iters = sketched_reductor.solve_rows(fom, None, th[idx], tf[idx], preconditioner=preconditioner, tol=tol,
                                                maxiter=maxiter, x0=x0, check=True, method=method, restart=restart)[:2]
        iters = iters.tolist()
        t5 = time.perf_counter()
        reductor.extend_basis(DeviceVectorArray(fom.solution_space, X))
        t6 = time.perf_counter()
        timing.update(solve=ms(t4, t5), extend=ms(t5, t6), total=ms(t0, t6))
        res['selected'].append(sel)
        res['fom_iterations'].append(iters)
        if reductor.srb.shape[0] == r:
            logger.info("extension failed: every new vector is in the span of the basis")
            res['stop'] = 'extension_failed'
            break
        res['extensions'] += 1
    res['rom'] = rom
    res['time'] = time.perf_counter() - t_start
    return res
