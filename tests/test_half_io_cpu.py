"""16-bit image storage (float16 / bfloat16 x and dx, SC_FLAG_GRID_F16 / SC_FLAG_GRID_BF16) without a GPU.

(1) The element conversion the device kernels use, run on the host (`sc_hostcheck_convert`), against torch's own casts: every
    16-bit pattern widened, and a sweep of float32 values rounded (ties, subnormals, the overflow threshold, signed zeros, inf, NaN).
(2) The plan-level contract: flag constants, the rejected flag combinations, tables independent of the flag.
(3) The host logic of every autograd Function with 16-bit x and the device primitives emulated (the same emulation as
    tests/test_factorized_host_logic.py): y is float32 and equal to the float32 run on x.float(), dx is that run's dx rounded to
    x's dtype, the parameter gradients are unchanged."""
import contextlib
import ctypes
import math
import os
import re

import numpy as np
import pytest
import torch

from neuraloperator_b200 import _lib, spectral_conv as sc
from neuraloperator_b200.build import build_library
from test_factorized_host_logic import KEPT, _c, _Lib, _pair_reduce, _table_contract

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DTYPES = {torch.float16: _lib.FLAG_GRID_F16, torch.bfloat16: _lib.FLAG_GRID_BF16}


@pytest.fixture(scope="module")
def lib():
    build_library()
    return _lib.load()


def _convert(lib, flag, to_16, arr):
    src = np.ascontiguousarray(arr)
    out = np.empty(src.shape, dtype=np.uint16 if to_16 else np.float32)
    rc = lib.sc_hostcheck_convert(flag, int(to_16), src.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p), src.size)
    _lib.check(rc, "sc_hostcheck_convert")
    return out


def _same_bits_nan_as_nan(ours: torch.Tensor, want: torch.Tensor):
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(ours), nan)
    bits = {torch.float32: torch.int32, torch.float16: torch.int16, torch.bfloat16: torch.int16}[want.dtype]
    assert torch.equal(ours[~nan].view(bits), want[~nan].view(bits))


@pytest.mark.parametrize("dtype", list(DTYPES))
def test_load_every_16_bit_pattern(lib, dtype):
    bits = np.arange(1 << 16, dtype=np.uint16)
    ours = torch.from_numpy(_convert(lib, DTYPES[dtype], False, bits))
    want = torch.from_numpy(bits.view(np.int16)).view(dtype).float()
    _same_bits_nan_as_nan(ours, want)


def _store_sweep(dtype):
    finfo = torch.finfo(dtype)
    g = torch.Generator().manual_seed(7)
    vals = [torch.randn(4096, generator=g, dtype=torch.float64) * 10.0 ** torch.randint(-8, 9, (4096,), generator=g)]
    # exact midpoints between neighbouring 16-bit values (ties to even) and their float32 neighbours
    pats = torch.arange(0, 0x7C00 if dtype == torch.float16 else 0x7F80, 7, dtype=torch.int32)
    lo = pats.to(torch.int16).view(dtype).double()
    hi = (pats + 1).to(torch.int16).view(dtype).double()
    mid = ((lo + hi) / 2).float()
    vals += [mid.double(), torch.nextafter(mid, torch.tensor(0.0)).double(), torch.nextafter(mid, torch.tensor(math.inf)).double()]
    # subnormals of the 16-bit type and of float32 itself
    tiny = finfo.smallest_normal
    vals.append(torch.linspace(-2 * tiny, 2 * tiny, 2001, dtype=torch.float64))
    vals.append(torch.tensor([1e-45, -1e-45, 1e-40, 3e-39, -3e-39], dtype=torch.float64))
    # around the overflow threshold: max + half an ulp rounds to inf (to even), anything below it to max
    top = finfo.max
    below_top = torch.tensor([0x7BFE if dtype == torch.float16 else 0x7F7E], dtype=torch.int16).view(dtype).double().item()
    thr = top + (top - below_top) / 2
    edge = torch.tensor([top, thr, -thr, top * 2, -top], dtype=torch.float64).float()
    vals += [edge.double(), torch.nextafter(edge, torch.tensor(0.0)).double(), torch.nextafter(edge, torch.tensor(math.inf)).double()]
    vals.append(torch.tensor([0.0, -0.0, math.inf, -math.inf, math.nan, -math.nan, 3.4e38, -3.4e38], dtype=torch.float64))
    return torch.cat(vals).float()


@pytest.mark.parametrize("dtype", list(DTYPES))
def test_store_rounds_like_torch_cast(lib, dtype):
    x = _store_sweep(dtype)
    ours = torch.from_numpy(_convert(lib, DTYPES[dtype], True, x.numpy()).view(np.int16)).view(dtype)
    want = x.to(dtype)
    assert torch.isinf(want).any() and (want == 0).any() and torch.isnan(want).any()
    _same_bits_nan_as_nan(ours, want)


def test_convert_rejects_unknown_flag(lib):
    a = np.zeros(4, dtype=np.float32)
    assert lib.sc_hostcheck_convert(_lib.FLAG_RESAMPLE, 1, a.ctypes.data_as(ctypes.c_void_p), a.ctypes.data_as(ctypes.c_void_p), 4) != 0
    assert b"SC_FLAG_GRID_F16" in lib.sc_last_error()


def test_flag_constants_match_header():
    header = open(os.path.join(ROOT, "include", "spectral_conv_b200.h")).read()
    assert int(re.search(r"SC_FLAG_GRID_F16\s*=\s*(\d+)", header).group(1)) == _lib.FLAG_GRID_F16
    assert int(re.search(r"SC_FLAG_GRID_BF16\s*=\s*(\d+)", header).group(1)) == _lib.FLAG_GRID_BF16
    assert int(re.search(r"SC_FLAG_RESAMPLE\s*=\s*(\d+)", header).group(1)) == _lib.FLAG_RESAMPLE
    assert len({_lib.FLAG_RESAMPLE, _lib.FLAG_GRID_F16, _lib.FLAG_GRID_BF16}) == 3
    assert sc._GRID_FLAGS == {torch.float32: 0, torch.float16: _lib.FLAG_GRID_F16, torch.bfloat16: _lib.FLAG_GRID_BF16}


def _problem(grid, modes, flags, out=None):
    prob = _lib.ScProblem()
    prob.ndim = len(grid)
    for j, (n, m) in enumerate(zip(grid, modes)):
        prob.grid[j] = n
        prob.out_grid[j] = (out or grid)[j]
        prob.n_modes[j] = prob.max_n_modes[j] = m
    prob.flags = flags
    return prob


@pytest.mark.parametrize("flags,msg", [
    (_lib.FLAG_GRID_F16 | _lib.FLAG_GRID_BF16, b"exclude each other"),
    (_lib.FLAG_GRID_F16 | _lib.FLAG_RESAMPLE, b"SC_FLAG_RESAMPLE"),
    (_lib.FLAG_GRID_BF16 | _lib.FLAG_RESAMPLE, b"SC_FLAG_RESAMPLE"),
])
def test_plan_create_rejects_invalid_flag_combinations(lib, flags, msg):
    handle = ctypes.c_void_p()
    prob = _problem((16, 12), (8, 7), flags)
    assert lib.sc_plan_create(ctypes.byref(prob), ctypes.byref(handle)) != 0
    assert msg in lib.sc_last_error()
    assert not handle.value


def _tables(lib, prob):
    out = []
    for which in range(8):
        dims = [0] if which < 4 else range(prob.ndim - 1)
        for dim in dims:
            rows, cols = ctypes.c_int64(), ctypes.c_int64()
            _lib.check(lib.sc_problem_table(ctypes.byref(prob), which, dim, None, 0, ctypes.byref(rows), ctypes.byref(cols)), "query")
            buf = np.empty(rows.value * cols.value, dtype=np.float32)
            _lib.check(lib.sc_problem_table(ctypes.byref(prob), which, dim, buf.ctypes.data_as(ctypes.c_void_p), buf.size,
                                            ctypes.byref(rows), ctypes.byref(cols)), "table")
            out.append(buf)
    return out


@pytest.mark.parametrize("grid,modes,out", [((16, 12), (8, 7), None), ((30, 20), (12, 9), (24, 24)), ((64,), (17,), None),
                                            ((8, 6, 10), (4, 4, 6), None)])
def test_tables_do_not_depend_on_the_storage_flag(lib, grid, modes, out):
    base = _tables(lib, _problem(grid, modes, 0, out))
    for flag in DTYPES.values():
        for a, b in zip(base, _tables(lib, _problem(grid, modes, flag, out))):
            assert np.array_equal(a, b)


def test_one_plan_per_storage_dtype(monkeypatch):
    class _FakePlan:
        def __init__(self, device, grid, out_grid, n_modes, max_n_modes, fft_norm, flags=0):
            self.flags = flags

    monkeypatch.setattr(sc, "Plan", _FakePlan)
    monkeypatch.setattr(sc, "_PLAN_CACHE", type(sc._PLAN_CACHE)())
    dev = torch.device("cuda", 0)
    plans = {dt: sc.get_plan(dev, [16, 12], [16, 12], [8, 7], [8, 7], "forward", flags=f) for dt, f in sc._GRID_FLAGS.items()}
    assert len({id(p) for p in plans.values()}) == 3
    assert {dt: p.flags for dt, p in plans.items()} == sc._GRID_FLAGS
    assert sc.get_plan(dev, [16, 12], [16, 12], [8, 7], [8, 7], "forward", flags=_lib.FLAG_GRID_BF16) is plans[torch.bfloat16]


# ---- host logic of the autograd Functions with 16-bit x --------------------------------------------------------------------------
class _Lib16(_Lib):
    """The emulation of tests/test_factorized_host_logic.py plus the dense entry points; dx is written into the caller's buffer with
    copy_, i.e. rounded to nearest even when that buffer is 16-bit, as the library's store does."""

    def sc_forward_dense(self, plan, x, w, b, y, xm, layout, B, Ci, Co, ws, n, st):
        assert x.dtype == plan.grid_dtype
        xm.copy_(x.to(torch.complex64))
        out = torch.einsum("bi...,io...->bo...", xm, w).real
        y.copy_(out + (b.reshape(1, -1, *[1] * (out.ndim - 2)) if b is not None else 0))
        return 0

    def sc_backward_dense(self, plan, gy, w, xm, layout, dx, dw, db, B, Ci, Co, ws, n, st, ev):
        assert gy.dtype == torch.float32 and (dx is None or dx.dtype == plan.grid_dtype)
        gm = gy.to(torch.complex64)
        if dx is not None:
            dx.copy_(torch.einsum("bo...,io...->bi...", gm, w.conj()).real)
        if dw is not None:
            dw.copy_(torch.einsum("bi...,bo...->io...", xm.conj(), gm))
        if db is not None:
            db.copy_(gy.sum(dim=[0] + list(range(2, gy.ndim))))
        return 0

    def sc_forward_tucker(self, plan, plan_kept, x, *rest):
        assert x.dtype == plan.grid_dtype
        return super().sc_forward_tucker(plan, plan_kept, x.float(), *rest)

    def sc_forward_cp(self, plan, x, *rest):
        assert x.dtype == plan.grid_dtype
        return super().sc_forward_cp(plan, x.float(), *rest)

    def sc_forward_tt(self, plan, plan_kept, x, *rest):
        assert x.dtype == plan.grid_dtype
        return super().sc_forward_tt(plan, plan_kept, x.float(), *rest)


class _Plan16:
    def __init__(self, kept, dtype):
        self.kept, self.ndim, self.n_modes_total, self.handle = tuple(kept), len(kept), math.prod(kept), self
        self.grid = self.out_grid = tuple(kept)
        self.grid_dtype = dtype

    def workspace_bytes(self, n):
        return 16


@pytest.fixture
def emulated16(monkeypatch):
    lib16 = _Lib16()
    monkeypatch.setattr(sc._lib, "load", lambda: lib16)
    monkeypatch.setattr(sc, "_ptr_array", lambda ts: list(ts))
    monkeypatch.setattr(sc, "_rank_array", lambda core: [int(r) for r in core.shape])
    monkeypatch.setattr(sc._lib, "check", lambda rc, what: None)
    monkeypatch.setattr(sc, "_ptr", lambda t: t)
    monkeypatch.setattr(sc, "_stream_ptr", lambda dev: None)
    monkeypatch.setattr(sc, "_table_contract", _table_contract)
    monkeypatch.setattr(sc, "_pair_reduce", _pair_reduce)
    monkeypatch.setattr(sc, "_cp_factor_args", lambda us, kept: (list(us), list(kept), len(us)))

    def analyze(plan, x, adjoint=False):
        assert x.dtype == (torch.float32 if adjoint else plan.grid_dtype)
        return x.to(torch.complex64)

    def synthesize(plan, m, bias=None, adjoint=False):
        out = (m.real + (bias.reshape(1, -1, *[1] * (m.ndim - 2)) if bias is not None else 0)).contiguous()
        return out.to(plan.grid_dtype) if adjoint else out

    monkeypatch.setattr(sc, "analyze", analyze)
    monkeypatch.setattr(sc, "synthesize", synthesize)
    monkeypatch.setattr(sc, "contract_dense", lambda plan, xm, w: torch.einsum("bi...,io...->bo...", xm, w).contiguous())
    monkeypatch.setattr(sc, "contract_dense_backward", lambda plan, xm, gm, w, **kw: (
        torch.einsum("bo...,io...->bi...", gm, w.conj()).contiguous(),
        torch.einsum("bi...,bo...->io...", xm.conj(), gm).contiguous(), None))
    monkeypatch.setattr(torch.cuda, "device", lambda dev: contextlib.nullcontext())


def _run(apply, x, params, gy):
    x = x.detach().clone().requires_grad_(True)
    ps = [p.detach().clone().requires_grad_(True) for p in params]
    y = apply(x, *ps)
    y.backward(gy)
    return y.detach(), x.grad, [p.grad for p in ps]


def _check_half_vs_float(apply, x32, params, gy, dtype):
    """apply(plan, x, *params): the 16-bit run against the float32 run on the widened input."""
    x16 = (x32 * 40).to(dtype)           # large enough that some dx entries need real rounding
    y16, dx16, g16 = _run(lambda x, *p: apply(_Plan16(x32.shape[2:], dtype), x, *p), x16, params, gy)
    y32, dx32, g32 = _run(lambda x, *p: apply(_Plan16(x32.shape[2:], torch.float32), x, *p), x16.float(), params, gy)
    assert y16.dtype == torch.float32 and torch.equal(y16, y32)
    assert dx16.dtype == dtype and torch.equal(dx16, dx32.to(dtype))
    assert not torch.equal(dx16.float(), dx32)       # the rounding really happened
    for a, b in zip(g16, g32):
        assert a.dtype == b.dtype and torch.equal(a, b)


def _gy(B, C, kept):
    return torch.randn(B, C, *kept) * 1e3


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("kept", KEPT[:3])
def test_dense_function(emulated16, dtype, kept):
    d, B, Ci, Co = len(kept), 2, 3, 4
    torch.manual_seed(10)
    params = [_c(Ci, Co, *kept), torch.randn(Co, *[1] * d)]
    _check_half_vs_float(lambda plan, x, w, b: sc._SpectralConvDense.apply(x, w, b, plan, None),
                         torch.randn(B, Ci, *kept), params, _gy(B, Co, kept), dtype)


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("kept", KEPT[:3])
def test_tucker_function(emulated16, dtype, kept):
    d, B, Ci, Co = len(kept), 2, 3, 4
    torch.manual_seed(11)
    ranks = [2, 3] + [2 + (j % 2) for j in range(d)]
    params = [torch.randn(Co, *[1] * d), _c(*ranks), _c(Ci, ranks[0]), _c(Co, ranks[1]), *[_c(k, r) for k, r in zip(kept, ranks[2:])]]
    _check_half_vs_float(lambda plan, x, b, core, ui, uo, *um: sc._SpectralConvTucker.apply(x, b, plan, plan, core, ui, uo, *um),
                         torch.randn(B, Ci, *kept), params, _gy(B, Co, kept), dtype)


@pytest.mark.parametrize("in_c", [False, True])
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("kept", KEPT[:3])
def test_cp_functions(emulated16, dtype, kept, in_c):
    d, B, Ci, Co, R = len(kept), 2, 3, 4, 5
    torch.manual_seed(12)
    fn = sc._SpectralConvCPCall if in_c else sc._SpectralConvCP
    params = [torch.randn(Co, *[1] * d), _c(R), _c(Ci, R), _c(Co, R), *[_c(k, R) for k in kept]]
    _check_half_vs_float(lambda plan, x, b, lam, ui, uo, *um: fn.apply(x, b, plan, lam, ui, uo, *um),
                         torch.randn(B, Ci, *kept), params, _gy(B, Co, kept), dtype)


@pytest.mark.parametrize("in_c", [False, True])
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("kept", KEPT[:3])
def test_tt_functions(emulated16, dtype, kept, in_c):
    d, B, Ci, Co = len(kept), 2, 3, 4
    torch.manual_seed(13)
    fn = sc._SpectralConvTTCall if in_c else sc._SpectralConvTT
    r = [1, 3, 4] + [2 + j for j in range(d - 1)] + [1]
    params = [torch.randn(Co, *[1] * d), _c(1, Ci, r[1]), _c(r[1], Co, r[2]), *[_c(r[2 + j], kept[j], r[3 + j]) for j in range(d)]]
    _check_half_vs_float(lambda plan, x, b, *cores: fn.apply(x, b, plan, plan, *cores),
                         torch.randn(B, Ci, *kept), params, _gy(B, Co, kept), dtype)


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("kept", KEPT[:3])
def test_separable_function(emulated16, dtype, kept):
    d, B, C = len(kept), 2, 3
    torch.manual_seed(14)
    params = [_c(C, *kept), torch.randn(C, *[1] * d)]
    _check_half_vs_float(lambda plan, x, w, b: sc._SpectralConvSeparable.apply(x, w, b, plan),
                         torch.randn(B, C, *kept), params, _gy(B, C, kept), dtype)
