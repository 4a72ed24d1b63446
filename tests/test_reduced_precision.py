"""fno_block_precision "half" / "mixed" (SURVEY section 8 f3) without a GPU.

(1) The oracle's statement of the half-precision contraction (`contract_dense_half`: operands rounded to fp16, fp32 accumulation,
    fp16 result) against what the reference's own `einsum_complexhalf` (neuralop/layers/einsum_utils.py:10-36) returned on CPU -- the
    one stage of the reduced-precision path that can execute there (the half FFTs need cuFFT).
(2) The host logic of `_SpectralConvDenseReduced` -- where the tensors are rounded, what is saved, straight-through gradients --
    with the device primitives emulated (transforms: a trivial adjoint pair; contraction: einsum; rounding: the pointwise kernel's
    host check) against the same pipeline written with `oracle.round_half`."""
import contextlib

import pytest
import torch

from neuraloperator_b200 import _lib, spectral_conv as sc
from oracle import spectral_conv_oracle as O
from conftest import reference_checks, stored_rel_err


def test_round_half_is_fp16_rounding_with_straight_through_gradient():
    t = (torch.randn(50) * 100).requires_grad_(True)
    r = O.round_half(t)
    assert torch.equal(r.detach(), t.detach().half().float())
    r.sum().backward()
    assert torch.equal(t.grad, torch.ones_like(t))
    c = torch.randn(20, dtype=torch.complex64)
    rc = O.round_half(c)
    assert torch.equal(torch.view_as_real(rc), torch.view_as_real(c).half().float())


HALF_CASES = [(2, 3, 4, (5, 3)), (1, 8, 8, (6,)), (2, 4, 3, (3, 2, 4))]


def half_case_inputs(shape):
    B, Ci, Co, kept = shape
    torch.manual_seed(3)
    xm = torch.randn(B, Ci, *kept, dtype=torch.complex64)
    w = torch.randn(Ci, Co, *kept, dtype=torch.complex64) / Ci ** 0.5
    return xm, w


@pytest.mark.parametrize("shape", HALF_CASES)
def test_half_contraction_restatement_against_live_einsum_complexhalf(shape):
    """Against what the reference's einsum_complexhalf returned for these operands (stored by oracle/make_golden_reference_checks.py,
    from the string _contract_dense builds, spectral_convolution.py:21-40, the weight passed as cfloat and cast inside)."""
    store, _ = reference_checks()
    xm, w = half_case_inputs(shape)
    ours = O.contract_dense_half(xm, w)
    # same operand rounding; the reference rounds each of the four real products to fp16 before combining them: <= 2 fp16 ulps apart
    assert stored_rel_err(store, f"half{HALF_CASES.index(shape)}", ours) <= 2.0 ** -9


class _Plan:
    def __init__(self, kept):
        self.kept = tuple(kept)


@pytest.fixture
def emulated(monkeypatch):
    real = _lib.load()

    class Host:
        def sc_pointwise(self, op, a, b, out, n, st):
            return real.sc_hostcheck_pointwise(op, a, b, out, n)

        def sc_last_error(self):
            return real.sc_last_error()

    monkeypatch.setattr(sc._lib, "load", lambda: Host())
    monkeypatch.setattr(sc, "_stream_ptr", lambda dev: None)
    monkeypatch.setattr(torch.cuda, "device", lambda dev: contextlib.nullcontext())
    monkeypatch.setattr(sc, "analyze", lambda plan, x, adjoint=False: x.to(torch.complex64) * (1 + 0.5j))
    monkeypatch.setattr(sc, "synthesize", lambda plan, m, bias=None, adjoint=False:
                        ((m * (1 - 0.5j)).real + (bias.reshape(1, -1, *[1] * (m.ndim - 2)) if bias is not None else 0)).contiguous())
    monkeypatch.setattr(sc, "contract_dense", lambda plan, xm, w: torch.einsum("bi...,io...->bo...", xm, w).contiguous())

    def bwd(plan, xm, gm, w, need_dxm=True, need_dweight=True, need_dbias=True):
        return (torch.einsum("bo...,io...->bi...", gm, w.conj()).contiguous() if need_dxm else None,
                torch.einsum("bi...,bo...->io...", xm.conj(), gm).contiguous() if need_dweight else None,
                gm.real.sum(dim=[0] + list(range(2, gm.ndim))) if need_dbias else None)
    monkeypatch.setattr(sc, "contract_dense_backward", bwd)


@pytest.mark.parametrize("round_input", [False, True])
@pytest.mark.parametrize("kept", [(6,), (4, 3), (2, 3, 2)])
def test_reduced_precision_function_host_logic(emulated, kept, round_input):
    B, Ci, Co = 2, 3, 4
    d = len(kept)
    torch.manual_seed(8)
    x = (torch.randn(B, Ci, *kept) * 3).requires_grad_(True)
    w = (torch.randn(Ci, Co, *kept, dtype=torch.complex64)).requires_grad_(True)
    bias = torch.randn(Co, *[1] * d).requires_grad_(True)
    gy = torch.randn(B, Co, *kept)
    y = sc._SpectralConvDenseReduced.apply(x, w, bias, _Plan(kept), round_input)
    y.backward(gy)

    x2, w2, b2 = (t.detach().clone().requires_grad_(True) for t in (x, w, bias))
    xin = O.round_half(x2) if round_input else x2
    xm = O.round_half(xin.to(torch.complex64) * (1 + 0.5j))
    ym = O.round_half(torch.einsum("bi...,io...->bo...", xm, O.round_half(w2)))
    y2 = (ym * (1 - 0.5j)).real + b2
    # backward of the emulated synthesis / analysis pair as the Function computes it: gm = gy * (1 + 0.5j), dx = Re(dxm * (1 - 0.5j))
    gm = gy.to(torch.complex64) * (1 + 0.5j)
    dxm = torch.einsum("bo...,io...->bi...", gm, O.round_half(w2).detach().conj())
    dx_want = (dxm * (1 - 0.5j)).real
    dw_want = torch.einsum("bi...,bo...->io...", xm.detach().conj(), gm)
    assert torch.allclose(y, y2.detach(), rtol=0, atol=1e-6 * y2.abs().max().item())
    assert torch.allclose(x.grad, dx_want, rtol=0, atol=1e-5 * dx_want.abs().max().item())
    assert torch.allclose(w.grad, dw_want, rtol=0, atol=1e-5 * dw_want.abs().max().item())
    assert torch.allclose(bias.grad.reshape(-1), gm.real.sum(dim=[0] + list(range(2, gm.ndim))), atol=1e-5)
    # the saved modes really are fp16 values, and the input was not modified
    assert torch.equal(torch.view_as_real(xm.detach()), torch.view_as_real(xm.detach()).half().float())


def test_reduced_oracle_is_close_to_full_precision_and_differentiable():
    x, w, bias, gy = O.make_inputs(2, 4, 4, (16, 12), (8, 6), seed=2)
    y_full = O.spectral_conv_forward(x, w, bias, (8, 6))
    for precision in ("mixed", "half"):
        xr = x.clone().requires_grad_(True)
        wt = w.tensor.clone().requires_grad_(True)
        y = O.spectral_conv_forward_reduced(xr, O.Weight("dense", tensor=wt), bias, (8, 6), precision)
        assert (y - y_full).abs().max() < 5e-3 * y_full.abs().max()          # fp16 rounding noise
        assert not torch.equal(y, y_full)
        y.backward(gy)
        assert xr.grad is not None and wt.grad is not None and torch.isfinite(xr.grad).all()
