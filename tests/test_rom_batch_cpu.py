"""CPU-only checks of the ROM's batch evaluation (SketchedRom.solve_batch / estimate_error_batch /
output_batch): the host stacking of the affine coefficients of `mus=`, shape and argument
validation that raises before anything is launched, and the workspace size of the batched
residual norm."""
import numpy as np
import pytest
import torch

import rla4mor_b200 as rb
from rla4mor_b200 import reductor_ops as ops
from rla4mor_b200.sketched_reductor import AffineModel, EmptyRom, SketchedRom


class _Functional:
    """pyMOR-style parameter functional: evaluate(mu)."""

    def __init__(self, i, scale=1.0):
        self.i, self.scale = i, scale

    def evaluate(self, mu):
        return self.scale * mu["mu"][self.i]


class _Fom:
    """Only what the ROM's batch methods read of an AffineModel."""

    def __init__(self, cop, crhs):
        self.operator_coefficients, self.rhs_coefficients = cop, crhs

    thetas = AffineModel.thetas
    thetas_batch = AffineModel.thetas_batch


def _rom(r=5, Q=3, Pf=2, kp=11, least_squares=False):
    g = torch.Generator().manual_seed(0)
    fom = _Fom([1.0, _Functional(0), lambda mu: 2.0 * mu["mu"][1]][:Q], [_Functional(1, -1.0), 0.5][:Pf])
    lhs = [torch.randn(r, r, generator=g, dtype=torch.float64) for _ in range(Q)]
    rhs = [torch.randn(r, generator=g, dtype=torch.float64) for _ in range(Pf)]
    est = ([torch.randn(r, kp, generator=g, dtype=torch.float64) for _ in range(Q)],
           [torch.randn(kp, generator=g, dtype=torch.float64) for _ in range(Pf)])
    out = torch.randn(r, 2, generator=g, dtype=torch.float64)
    return SketchedRom(fom, lhs, rhs, out, est, least_squares=least_squares)


def test_mus_stacking_with_pymor_style_functionals():
    fom = _Fom([1.0, _Functional(0), lambda mu: 2.0 * mu["mu"][1]], [_Functional(1, -1.0), 0.5])
    mus = [{"mu": [0.1 * p, 1.0 + p]} for p in range(7)]
    th, tf = fom.thetas_batch(mus)
    assert th.dtype == np.float64 and th.shape == (7, 3) and tf.shape == (7, 2)
    for p, mu in enumerate(mus):
        t1, t2 = fom.thetas(mu)
        assert np.array_equal(th[p], t1) and np.array_equal(tf[p], t2)
    th0, tf0 = fom.thetas_batch([])
    assert th0.shape == (0, 3) and tf0.shape == (0, 2)
    # the ROM stacks mus= through the same host evaluation
    rom = _rom()
    th_r, tf_r = rom._thetas_batch(None, None, mus)
    assert torch.equal(th_r, torch.from_numpy(th)) and torch.equal(tf_r, torch.from_numpy(tf))


def test_empty_parameter_set_returns_empty_results():
    rom = _rom()
    th, tf = np.zeros((0, 3)), np.zeros((0, 2))
    assert rom.solve_batch(th, tf).shape == (0, 5)
    assert rom.estimate_error_batch(None, th, tf).shape == (0,)
    assert rom.output_batch(None, th, tf).shape == (0, 2)
    assert rom.solve_batch(mus=[]).shape == (0, 5)
    G = torch.eye(2, dtype=torch.float64)
    empty = EmptyRom(_Fom([1.0], [1.0, 2.0]), G, 3)
    assert empty.solve_batch(theta_rhs=np.zeros((0, 2))).shape == (0, 0)
    assert empty.estimate_error_batch(theta_rhs=np.zeros((0, 2))).shape == (0,)
    assert empty.output_batch(theta_rhs=np.zeros((0, 2))).shape == (0, 3)


def test_empty_rom_batch_equals_per_mu():
    g = torch.Generator().manual_seed(1)
    F = torch.randn(3, 50, generator=g, dtype=torch.float64)
    empty = EmptyRom(_Fom([1.0], [1.0, _Functional(0), _Functional(1)]), F @ F.T, 2)
    mus = [{"mu": [0.3 * p - 1.0, 0.7 + p]} for p in range(6)]
    est = empty.estimate_error_batch(mus=mus)
    for p, mu in enumerate(mus):
        assert abs(float(est[p]) - empty.estimate_error(mu=mu)) <= 1e-14 * float(est[p])
    assert torch.equal(empty.output_batch(mus=mus), torch.zeros((6, 2), dtype=torch.float64))


@pytest.mark.parametrize("th,tf", [
    (np.zeros((4, 2)), np.zeros((4, 2))),       # Q mismatch
    (np.zeros((4, 3)), np.zeros((4, 1))),       # Pf mismatch
    (np.zeros((4, 3)), np.zeros((5, 2))),       # P mismatch
    (np.zeros(3), np.zeros(2)),                 # one mu given as vectors
])
def test_rom_rejects_bad_theta_shapes(th, tf):
    rom = _rom()
    for f in (rom.solve_batch, rom.output_batch):
        with pytest.raises(ValueError):
            f(theta_lhs=th, theta_rhs=tf)
    with pytest.raises(ValueError):
        rom.estimate_error_batch(None, th, tf)


def test_rom_rejects_bad_arguments():
    rom = _rom()
    th, tf = np.zeros((4, 3)), np.zeros((4, 2))
    with pytest.raises(ValueError):
        rom.estimate_error_batch(torch.zeros(4, 6, dtype=torch.float64), th, tf)       # a has the wrong r
    with pytest.raises(ValueError):
        rom.output_batch(torch.zeros(3, 5, dtype=torch.float64), th, tf)              # a has the wrong P
    with pytest.raises(ValueError):
        rom.solve_batch(th, tf, mus=[{"mu": [0.0, 1.0]}])                             # both forms
    with pytest.raises(ValueError):
        rom.solve_batch(th)                                                           # theta_rhs missing
    with pytest.raises(ValueError):
        EmptyRom(_Fom([1.0], [1.0, 2.0]), torch.eye(2, dtype=torch.float64), 0).estimate_error_batch(
            theta_rhs=np.zeros((3, 3)))


def test_ops_validate_before_launch():
    """The wrappers check shapes before any copy or launch (and CPU data is refused, not launched)."""
    lhs, rhs = torch.zeros(2, 4, 4, dtype=torch.float64), torch.zeros(1, 4, dtype=torch.float64)
    with pytest.raises(ValueError):
        ops.rom_solve_batch(lhs, rhs, torch.zeros(3, 3), torch.zeros(3, 1))           # th (P, 3), Q = 2
    with pytest.raises(ValueError):
        ops.rom_solve_batch(lhs, rhs, torch.zeros(3, 2), torch.zeros(2, 1))           # tf rows
    with pytest.raises(ValueError):
        ops.rom_solve_batch(torch.zeros(2, 4, 3), rhs, torch.zeros(3, 2), torch.zeros(3, 1))   # non-square A_q
    big = ops.rom_solve_batch_max_r() + 1
    with pytest.raises(ValueError):
        ops.rom_solve_batch(torch.zeros(1, big, big), torch.zeros(1, big), torch.zeros(2, 1), torch.zeros(2, 1))
    with pytest.raises(ValueError):
        ops.rom_solve_batch(lhs, rhs, torch.zeros(3, 2), torch.zeros(3, 1))           # CPU data: refused
    W = torch.zeros(2 * 4 + 1, 10, dtype=torch.float64)
    with pytest.raises(ValueError):
        ops.residual_norm_batch(W, 2, 4, torch.zeros(3, 2), torch.zeros(3, 1), torch.zeros(3, 5))   # a (P, 5)
    with pytest.raises(ValueError):
        ops.residual_norm_batch(W, 2, 4, torch.zeros(3, 2), torch.zeros(3, 2), torch.zeros(3, 4))   # tf (P, 2)
    with pytest.raises(ValueError):
        ops.residual_norm_batch(W, 3, 4, torch.zeros(3, 3), torch.zeros(3, 1), torch.zeros(3, 4))   # W too short
    with pytest.raises(ValueError):
        ops.residual_norm_batch(W.T, 2, 4, torch.zeros(3, 2), torch.zeros(3, 1), torch.zeros(3, 4))  # W strided
    with pytest.raises(ValueError):
        ops.residual_norm_batch(W, 2, 4, torch.zeros(3, 2), torch.zeros(3, 1), torch.zeros(3, 4))   # CPU data
    assert ops.residual_norm_batch(W, 2, 4, torch.zeros(0, 2), torch.zeros(0, 1), torch.zeros(0, 4)).shape == (0,)


def test_entry_points_validate_arguments_without_gpu():
    lib = rb.lib()
    assert lib.rla_rom_solve_batch_max_r() >= 128
    r = lib.rla_rom_solve_batch_max_r()
    assert r * (r + 1) * 8 <= 227 * 1024 < (r + 1) * (r + 2) * 8                # the largest system one CTA holds
    assert lib.rla_rom_solve_batch_f64(None, 1, r + 1, None, 0, None, 1, None, 0, 4, None, r + 1, None, None) == -1
    assert b"largest supported" in lib.rla_last_error()
    assert lib.rla_rom_solve_batch_f64(None, 2, 4, None, 1, None, 1, None, 1, 4, None, 4, None, None) == -1   # ldth < Q
    assert lib.rla_rom_solve_batch_f64(None, 2, 4, None, 1, None, 2, None, 1, 0, None, 4, None, None) == 0    # P = 0
    assert lib.rla_residual_norm_batch_f64(None, 10, 2, 4, 1, 10, None, 2, None, 1, None, 4, 3, None, None, 0,
                                           None) == -1                                           # null pointers
    assert lib.rla_residual_norm_batch_f64(None, 9, 2, 4, 1, 10, None, 2, None, 1, None, 4, 3, None, None, 0,
                                           None) == -1                                           # ldw < k'
    x = np.zeros(64)
    p = x.ctypes.data
    assert lib.rla_residual_norm_batch_f64(p, 10, 2, 4, 1, 10, p, 2, p, 1, p, 4, 3, p, p, 8, None) == -1  # workspace
    assert b"workspace" in lib.rla_last_error()


@pytest.mark.parametrize("P,kp", [(1, 1), (1, 128), (5, 129), (1000, 1000), (100000, 2000), (7, 33)])
def test_workspace_size_formula(P, kp):
    tiles = -(-kp // 128)
    assert ops.residual_norm_batch_workspace_bytes(P, kp) == 8 * P * tiles
    assert ops.residual_norm_batch_workspace_bytes(P, kp) < P * kp * 8 or kp <= 128
    assert ops.residual_norm_batch_workspace_bytes(0, kp) == 0
