"""The reference's own test file (`neuralop/layers/tests/test_spectral_convolution.py`: `test_SpectralConv` :7-90, `test_SpectralConv2`
:93-125) against `neuraloperator_b200.SpectralConv` WITHOUT a GPU: the whole parameter grid (4 factorizations x 2 implementations x
separable x 1-4 dims x real / complex; Hermitian flag x dims x even / odd sizes x resolution scaling x modes) runs through the
module's own host logic -- plan lookup, weight slicing, which chain runs, operand strides, mutable n_modes, output grids -- with the
device primitives emulated by the oracle's torch.fft statements of the two transforms and by einsums for the contractions.  Every
result is ALSO compared with what the unmodified reference class returned on the same weights (stored by
oracle/make_golden_reference_checks.py).
The GPU twin of this file is tests/test_gpu_zzz_a_reference_suite.py."""
import contextlib
import math
import re

import pytest
import torch

import neuraloperator_b200 as nb
from neuraloperator_b200 import spectral_conv as sc
from oracle import spectral_conv_oracle as O
from conftest import reference_checks, stored_rel_err
from test_factorized_host_logic import _LIB as _CHAIN_LIB, _pair_reduce, _table_contract


class FakePlan:
    """What `Plan` exposes to the Python side, computed by the oracle's index rules instead of the C library."""

    def __init__(self, device, grid, out_grid, n_modes_stored, max_n_modes, fft_norm="forward", flags=0):
        self.dims = O.kept_mode_plan(list(grid), list(n_modes_stored), list(max_n_modes))
        self.kept = tuple(p.kept for p in self.dims)
        self.ndim, self.grid, self.out_grid = len(grid), tuple(grid), tuple(out_grid)
        self.n_modes_total = math.prod(self.kept)
        self.max_n_modes = tuple(int(m) for m in max_n_modes)
        self.fft_norm, self.handle, self.plan_kept, self.device = fft_norm, self, None, device

    def weight_row_range(self, j):
        return self.dims[j].w_index[0], self.dims[j].w_index[0] + self.dims[j].kept

    def workspace_bytes(self, n):
        return 16

    def cut(self, w, lead=2):
        for j in range(self.ndim):
            lo, hi = self.weight_row_range(j)
            if w.shape[lead + j] != hi - lo:
                w = w.narrow(lead + j, lo, hi - lo)
        return w


class _Lib(type(_CHAIN_LIB)):
    """sc_forward_dense / sc_forward_tucker with REAL transforms (the chain emulations of test_factorized_host_logic stay for CP)."""

    def sc_forward_dense(self, plan, x, weight, bias, y, xm, layout, B, Ci, Co, ws, n, st):
        m = O.analyze_modes(x, plan.dims, plan.fft_norm)
        ym = torch.einsum("bi...,io...->bo...", m, plan.cut(weight))
        out = O.synthesize_modes(ym, plan.dims, plan.out_grid, plan.fft_norm)
        y.copy_(out + (bias.reshape(1, -1, *[1] * plan.ndim) if bias is not None else 0))
        return 0

    def sc_forward_tucker(self, plan, plan_kept, x, core, u_in, u_out, u_modes, bias, y, saved, B, Ci, Co, ranks, ws, n, st):
        m = O.analyze_modes(x, plan.dims, plan.fft_norm)
        ym = O.contract_tucker(m, core, [u_in, u_out, *u_modes])
        out = O.synthesize_modes(ym, plan.dims, plan.out_grid, plan.fft_norm)
        y.copy_(out + (bias.reshape(1, -1, *[1] * plan.ndim) if bias is not None else 0))
        return 0


@pytest.fixture
def emulated(monkeypatch):
    return emulate_device(monkeypatch)


def emulate_device(monkeypatch):
    lib = _Lib()
    monkeypatch.setattr(sc._lib, "load", lambda: lib)
    monkeypatch.setattr(sc._lib, "check", lambda rc, what: None)
    monkeypatch.setattr(sc, "_ptr", lambda t: t)
    monkeypatch.setattr(sc, "_ptr_array", lambda ts: list(ts))
    monkeypatch.setattr(sc, "_rank_array", lambda core: [int(r) for r in core.shape])
    monkeypatch.setattr(sc, "_stream_ptr", lambda dev: None)
    monkeypatch.setattr(sc, "_table_contract", _table_contract)
    monkeypatch.setattr(sc, "_pair_reduce", _pair_reduce)
    monkeypatch.setattr(sc, "_cp_factor_args", lambda us, kept: (list(us), list(kept), len(us)))
    monkeypatch.setattr(sc, "get_plan", lambda dev, grid, out, nm, mx, norm="forward", flags=0: FakePlan(dev, grid, out, nm, mx, norm, flags))
    monkeypatch.setattr(sc, "get_complex_plan", lambda dev, grid, out, nm, mx, norm: sc.ComplexPlan(torch.device("cpu"), grid, out, nm, mx, norm))
    monkeypatch.setattr(sc, "analyze", lambda plan, x, adjoint=False: O.analyze_modes(x, plan.dims, plan.fft_norm))
    monkeypatch.setattr(sc, "synthesize", lambda plan, m, bias=None, adjoint=False:
                        O.synthesize_modes(m, plan.dims, plan.out_grid, plan.fft_norm) + (bias.reshape(1, -1, *[1] * plan.ndim) if bias is not None else 0))
    monkeypatch.setattr(sc, "contract_dense", lambda plan, xm, w: torch.einsum("bi...,io...->bo...", xm, plan.cut(w)).contiguous())
    monkeypatch.setattr(torch.cuda, "device", lambda dev: contextlib.nullcontext())
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))       # the module refuses CPU tensors: pretend
    return lib


def assert_close(a, b, tol):
    assert a.shape == b.shape
    assert (a - b).abs().max().item() / max(b.abs().max().item(), 1e-20) < tol


def case_key(prefix, case, twin):
    return f"{prefix}_{re.sub(r'[^0-9A-Za-z.]+', '_', str(case))}_{twin}"


class StoredTwin:
    """Stands for the unmodified reference class holding the same weight (reconstructed dense): `check` compares an output with what
    that class returned for the same input, stored under the case's key, in the order the suite asks."""

    def __init__(self, key):
        self.key, self.n, self.n_modes = key, 0, None

    def check(self, out, x, tol):
        store, _ = reference_checks("reference_suite")
        assert stored_rel_err(store, f"{self.key}__{self.n}", out) < tol
        self.n += 1


def _stored_twins(prefix, case):
    made = []

    def twin_of(conv, **ctor):
        made.append(StoredTwin(case_key(prefix, case, len(made))))
        return made[-1]
    return twin_of


FACTORIZATIONS = ["Dense", "CP", "Tucker", "TT"]
IMPLEMENTATIONS = ["factorized", "reconstructed"]
GRID_1 = [(f, i, s, d, c) for c in (False, True) for d in (1, 2, 3, 4) for s in (False, True) for i in IMPLEMENTATIONS for f in FACTORIZATIONS]
GRID_2 = [(h, d, n, r, m) for m in ((4, 4, 4), (4, 5, 7)) for r in (None, 0.5, 2) for n in (8, 9) for d in (1, 2, 3) for h in (True, False)]
MODES, FEWER_MODES, SIDE = (10, 8, 6, 6), (6, 6, 4, 4), 12


def suite_factorized_vs_dense(device, factorization, implementation, separable, dim, complex_data, tol, twin_of=None):
    """What the reference's `test_SpectralConv` (:7-90) asserts, for one point of its parameter grid, on `device`:
    a conv in any weight form equals its dense twin holding the reconstructed weight; shrinking `n_modes` at run time keeps the output
    shape; a conv with resolution_scaling_factor 0.5 / 2 halves / doubles every spatial extent.  twin_of(conv, **ctor) may return a
    stand-in for the unmodified reference module with the same weight: then every output is checked against it as well."""
    torch.manual_seed(0)
    modes = MODES[:dim]
    make = lambda *a, **k: nb.SpectralConv(*a, **k).to(device)                                            # noqa: E731
    conv = make(3, 3, modes, bias=False, implementation=implementation, factorization=factorization, complex_data=complex_data,
                separable=separable)
    dense = make(3, 3, modes, bias=False, implementation="reconstructed", factorization=None, complex_data=complex_data)
    x = torch.randn(2, 3, *(SIDE,) * dim, dtype=torch.cfloat if complex_data else torch.float32, device=device)
    assert torch.is_complex(conv.weight) and torch.is_complex(dense.weight)
    with torch.no_grad():
        if not separable:                                   # (the full weights have the same shape only then)
            dense.weight.tensor.copy_(conv.weight.to_tensor())
        out = conv(x)
        if not separable:
            assert_close(out, dense(x), tol)
        twin = twin_of(conv, user_modes=modes) if twin_of is not None else None
        if twin is not None:
            twin.check(out, x, tol)
        conv.n_modes = FEWER_MODES[:dim]                    # incremental training shrinks the modes at run time
        fewer = conv(x)
        assert fewer.shape == out.shape
        if twin is not None:
            twin.n_modes = FEWER_MODES[:dim]
            twin.check(fewer, x, tol)
        for factor, side in ((0.5, SIDE // 2), (2, SIDE * 2)):
            scaler = make(3, 4, modes, resolution_scaling_factor=factor)
            xr = torch.randn(2, 3, *(SIDE,) * dim, device=device)
            res = scaler(xr)
            assert res.shape[1] == 4 and list(res.shape[2:]) == [side] * dim
            twin = twin_of(scaler, user_modes=modes, resolution_scaling_factor=factor) if twin_of is not None else None
            if twin is not None:
                twin.check(res, xr, tol)


def suite_real_output_shapes(device, hermitian, dim, side, scaling, modes, tol, twin_of=None):
    """The reference's `test_SpectralConv2` (:93-125): real float32 output of the right (rounded) size for even / odd grids, with and
    without the Hermitian flag, at every resolution scaling; checked against twin_of(conv) as above when given."""
    torch.manual_seed(0)
    modes = modes[:dim]
    want = [side] * dim if scaling is None else [round(side * scaling)] * dim
    conv = nb.SpectralConv(3, 4, modes, enforce_hermitian_symmetry=hermitian, complex_data=False, resolution_scaling_factor=scaling).to(device)
    x = torch.randn(2, 3, *[side] * dim, dtype=torch.float32, device=device)
    with torch.no_grad():
        res = conv(x)
    assert tuple(res.shape) == (2, 4, *want) and res.dtype == torch.float32 and not torch.is_complex(res)
    if twin_of is not None:
        twin_of(conv).check(res, x, tol)


@pytest.mark.parametrize("factorization,implementation,separable,dim,complex_data", GRID_1)
def test_SpectralConv(emulated, factorization, implementation, separable, dim, complex_data):
    suite_factorized_vs_dense(torch.device("cpu"), factorization, implementation, separable, dim, complex_data, 2e-5,
                              twin_of=_stored_twins("g1", (factorization, implementation, separable, dim, complex_data)))


@pytest.mark.parametrize("enforce_hermitian_symmetry,dim,spatial_size,resolution_scaling_factor,modes", GRID_2)
def test_SpectralConv2(emulated, enforce_hermitian_symmetry, dim, spatial_size, modes, resolution_scaling_factor):
    suite_real_output_shapes(torch.device("cpu"), enforce_hermitian_symmetry, dim, spatial_size, resolution_scaling_factor, modes, 2e-5,
                             twin_of=_stored_twins("g2", (enforce_hermitian_symmetry, dim, spatial_size, resolution_scaling_factor, modes)))
