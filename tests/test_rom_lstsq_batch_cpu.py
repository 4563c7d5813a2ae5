"""CPU-only checks of the batched least-squares (minres) ROM solve (reductor_ops.rom_lstsq_batch,
rla_rom_lstsq_batch_f64): argument validation that raises before anything is launched, the C
entry point's return codes, and its size limit."""
import numpy as np
import pytest
import torch

import rla4mor_b200 as rb
from rla4mor_b200 import reductor_ops as ops


def test_max_r_holds_r_128():
    assert ops.rom_lstsq_batch_max_r() >= 128
    assert rb.lib().rla_rom_lstsq_batch_max_r() == ops.rom_lstsq_batch_max_r()


def test_ops_validate_before_launch():
    Q, r, Pf, ke = 2, 4, 1, 10
    W = torch.zeros(Q * r + Pf, ke, dtype=torch.float64)
    th, tf = torch.zeros(3, Q), torch.zeros(3, Pf)
    with pytest.raises(ValueError):
        ops.rom_lstsq_batch(W, Q, r, torch.zeros(3, 3), tf)                          # th (P, 3), Q = 2
    with pytest.raises(ValueError):
        ops.rom_lstsq_batch(W, Q, r, th, torch.zeros(2, Pf))                         # tf rows
    with pytest.raises(ValueError):
        ops.rom_lstsq_batch(W, Q, r, th, torch.zeros(3, 2))                          # tf (P, 2), Pf = 1
    with pytest.raises(ValueError):
        ops.rom_lstsq_batch(W, 3, r, torch.zeros(3, 3), tf)                          # W shorter than Q r
    with pytest.raises(ValueError):
        ops.rom_lstsq_batch(W.T, Q, r, th, tf)                                        # W strided
    with pytest.raises(ValueError):
        ops.rom_lstsq_batch(W.to(torch.float32), Q, r, th, tf)                        # W not float64
    with pytest.raises(ValueError):
        ops.rom_lstsq_batch(W[:, :3], Q, r, th, tf)                                   # k_eff = 3 < r
    with pytest.raises(ValueError):
        ops.rom_lstsq_batch(W[:, :0], Q, r, th, tf)                                   # empty rows
    with pytest.raises(ValueError):
        ops.rom_lstsq_batch(W, 0, r, torch.zeros(3, 0), torch.zeros(3, Q * r + Pf))   # no affine terms
    big = ops.rom_lstsq_batch_max_r() + 1
    with pytest.raises(ValueError, match="outside"):
        ops.rom_lstsq_batch(torch.zeros(big + 1, 2 * big, dtype=torch.float64), 1, big, torch.zeros(2, 1),
                            torch.zeros(2, 1))
    with pytest.raises(ValueError, match="CUDA"):
        ops.rom_lstsq_batch(W, Q, r, th, tf)                                          # CPU data: refused
    a, info = ops.rom_lstsq_batch(W, Q, r, torch.zeros(0, Q), torch.zeros(0, Pf))
    assert a.shape == (0, r) and info.shape == (0,)


def test_entry_point_validates_arguments_without_gpu():
    lib = rb.lib()
    m = lib.rla_rom_lstsq_batch_max_r()
    x = np.zeros(64)
    p = x.ctypes.data
    #                                   W  ldw  Q  r   Pf ke  th ldth tf ldtf P  a  lda info stream
    assert lib.rla_rom_lstsq_batch_f64(None, 10, 2, 4, 1, 10, None, 2, None, 1, 3, None, 4, None, None) == -1
    assert b"null pointer" in lib.rla_last_error()
    assert lib.rla_rom_lstsq_batch_f64(p, 2 * m, 1, m + 1, 0, 2 * m, p, 1, None, 0, 3, p, m + 1, p, None) == -1
    assert b"largest supported" in lib.rla_last_error()
    assert lib.rla_rom_lstsq_batch_f64(p, 10, 2, 4, 1, 3, p, 2, p, 1, 3, p, 4, p, None) == -1      # k_eff < r
    assert b"underdetermined" in lib.rla_last_error()
    assert lib.rla_rom_lstsq_batch_f64(p, 10, 2, 4, 1, 10, p, 1, p, 1, 3, p, 4, p, None) == -1     # ldth < Q
    assert lib.rla_rom_lstsq_batch_f64(p, 9, 2, 4, 1, 10, p, 2, p, 1, 3, p, 4, p, None) == -1      # ldw < k_eff
    assert lib.rla_rom_lstsq_batch_f64(p, 10, 2, 4, 1, 10, p, 2, p, 0, 3, p, 4, p, None) == -1     # ldtf < Pf
    assert lib.rla_rom_lstsq_batch_f64(p, 10, 2, 4, 1, 10, p, 2, p, 1, 3, p, 3, p, None) == -1     # lda < r
    assert lib.rla_rom_lstsq_batch_f64(p, 10, 2, 0, 1, 10, p, 2, p, 1, 3, p, 4, p, None) == -1     # r = 0
    assert lib.rla_rom_lstsq_batch_f64(p, 10, 2, 4, 1, 10, p, 2, p, 1, -1, p, 4, p, None) == -1    # P < 0
    assert lib.rla_rom_lstsq_batch_f64(None, 10, 2, 4, 1, 10, None, 2, None, 1, 0, None, 4, None, None) == 0  # P = 0
