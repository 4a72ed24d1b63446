"""`SpectralConv`: B200-native drop-in for `neuralop.layers.spectral_convolution.SpectralConv`.

Same constructor signature (reference spectral_convolution.py:285-305), same `forward(x, output_shape=None)`,
`transform`, mutable `n_modes`, `max_n_modes`, `weight`, `bias` (:383-415) -- so it can be passed as
`conv_module=` to the reference's `FNOBlocks` / `FNO` / `TFNO` (fno_block.py:163,210-240; fno.py:208,315).
Everything between the input tensor and the output tensor runs in hand-written sm_100a kernels behind the
C ABI of `include/spectral_conv_b200.h`; there is no PyTorch / cuFFT / CPU fallback.  PyTorch is used for
device memory, the stream, and the autograd graph node.
"""
import ctypes
import threading
from collections import OrderedDict
from typing import List, Optional, Sequence, Tuple, Union

import torch
from torch.autograd.function import once_differentiable
from torch import nn

from . import _lib
from .factorized import FactorizedWeight

Number = Union[int, float]


# --------------------------------------------------------------------------------------------------
# plans (kept-mode index set + twiddle tables), cached per shape: n_modes and the grid may change between
# calls (incremental training mutates n_modes, resolution invariance changes the grid)
# --------------------------------------------------------------------------------------------------
class Plan:
    def __init__(self, device: torch.device, grid, out_grid, n_modes_stored, max_n_modes, fft_norm: str, flags: int = 0):
        lib = _lib.load()
        prob = _lib.ScProblem()
        d = len(grid)
        if not 1 <= d <= _lib.SC_MAX_DIMS:
            raise NotImplementedError(f"SpectralConv supports 1..{_lib.SC_MAX_DIMS} spatial dims, got {d}")
        if fft_norm not in _lib.NORMS:
            raise ValueError(f"unknown fft_norm {fft_norm!r}")
        prob.ndim = d
        for j in range(d):
            prob.grid[j] = int(grid[j])
            prob.out_grid[j] = int(out_grid[j])
            prob.n_modes[j] = int(n_modes_stored[j])
            prob.max_n_modes[j] = int(max_n_modes[j])
        prob.fft_norm = _lib.NORMS[fft_norm]
        prob.flags = int(flags)
        self._lib = lib
        self.device = device
        self.handle = ctypes.c_void_p()
        with torch.cuda.device(device):
            _lib.check(lib.sc_plan_create(ctypes.byref(prob), ctypes.byref(self.handle)), "sc_plan_create")
        kept = (ctypes.c_int32 * _lib.SC_MAX_DIMS)()
        lib.sc_plan_kept_modes(self.handle, kept)
        self.ndim = d
        self.grid = tuple(int(g) for g in grid)
        self.out_grid = tuple(int(g) for g in out_grid)
        self.kept = tuple(int(kept[j]) for j in range(d))
        self.n_modes_total = 1
        for k in self.kept:
            self.n_modes_total *= k
        self.max_n_modes = tuple(int(m) for m in max_n_modes)
        self.grid_dtype = _GRID_DTYPES[int(flags) & (_lib.FLAG_GRID_F16 | _lib.FLAG_GRID_BF16)]   # x and dx; y / gy are float32
        self._bins = {}
        self._ws_bytes = {}
        self.plan_kept = None        # lazily: the same problem with weight extents == kept modes (factorized chains)

    def mode_bins(self, dim: int) -> Tuple[List[int], List[int]]:
        """(unshifted spectrum bins read, weight rows used) for kept slots of `dim` -- for index-set checks."""
        if dim not in self._bins:
            self._bins[dim] = self._mode_bins(dim)
        b, r = self._bins[dim]
        return list(b), list(r)

    def weight_row_range(self, dim: int) -> Tuple[int, int]:
        """[first, last+1) rows of the weight's mode axis `dim` that the kept block uses (`weight[slices_w]`, :489)."""
        _, rows = self.mode_bins(dim)
        return rows[0], rows[0] + len(rows)

    def _mode_bins(self, dim: int) -> Tuple[List[int], List[int]]:
        k = self.kept[dim]
        bins = (ctypes.c_int32 * k)()
        rows = (ctypes.c_int32 * k)()
        _lib.check(self._lib.sc_plan_mode_bins(self.handle, dim, bins, rows), "sc_plan_mode_bins")
        return list(bins), list(rows)

    def workspace_bytes(self, n_images: int) -> int:
        b = self._ws_bytes.get(n_images)
        if b is None:
            b = self._ws_bytes[n_images] = int(self._lib.sc_workspace_bytes(self.handle, n_images))
        return b

    def set_fast_path(self, enable: bool):
        _lib.check(self._lib.sc_plan_set_fast_path(self.handle, int(bool(enable))), "sc_plan_set_fast_path")

    def set_reserved_sms(self, n_sms: int):
        """Leave `n_sms` SMs free in the persistent transform launches (room for a concurrent NCCL collective)."""
        _lib.check(self._lib.sc_plan_set_reserved_sms(self.handle, int(n_sms)), "sc_plan_set_reserved_sms")

    def uses_fast_path(self) -> int:
        return int(self._lib.sc_plan_uses_fast_path(self.handle))

    def __del__(self):
        try:
            if self.handle:
                self._lib.sc_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


# storage of x / dx -> plan flag; the kernels compute in fp32 either way (a 16-bit value widens to float exactly)
_GRID_FLAGS = {torch.float32: 0, torch.float16: _lib.FLAG_GRID_F16, torch.bfloat16: _lib.FLAG_GRID_BF16}
_GRID_DTYPES = {flag: dtype for dtype, flag in _GRID_FLAGS.items()}

_PLAN_CACHE: "OrderedDict[tuple, Plan]" = OrderedDict()
_PLAN_LOCK = threading.RLock()      # re-entrant: building a ComplexPlan (under the lock) asks get_plan for its contraction plan
_PLAN_CACHE_MAX = 64


def get_plan(device: torch.device, grid, out_grid, n_modes_stored, max_n_modes, fft_norm="forward", flags: int = 0) -> Plan:
    if device.type != "cuda":
        raise RuntimeError("neuraloperator_b200.SpectralConv runs on CUDA (sm_100a) only; there is no CPU path")
    idx = device.index if device.index is not None else torch.cuda.current_device()
    key = (idx, tuple(grid), tuple(out_grid), tuple(n_modes_stored), tuple(max_n_modes), fft_norm, int(flags))
    with _PLAN_LOCK:
        plan = _PLAN_CACHE.get(key)
        if plan is not None:
            _PLAN_CACHE.move_to_end(key)
            return plan
        plan = Plan(torch.device("cuda", idx), grid, out_grid, n_modes_stored, max_n_modes, fft_norm, flags)
        _PLAN_CACHE[key] = plan
        while len(_PLAN_CACHE) > _PLAN_CACHE_MAX:
            _PLAN_CACHE.popitem(last=False)
        return plan


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream_ptr(device) -> ctypes.c_void_p:
    """cudaStream_t of PyTorch's current stream on `device` (the raw getter skips building a torch.cuda.Stream object)."""
    if _raw_stream is not None and device.index is not None:
        return ctypes.c_void_p(_raw_stream(device.index))
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _ptr(t: Optional[torch.Tensor]) -> ctypes.c_void_p:
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _rank_array(core) -> ctypes.Array:
    return (ctypes.c_int32 * core.ndim)(*[int(r) for r in core.shape])


def _ptr_array(tensors) -> ctypes.Array:
    """Host array of device pointers (`const sc_complex* const*` arguments)."""
    return (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


def _workspace(plan: Plan, n_images: int, device) -> torch.Tensor:
    return torch.empty(max(plan.workspace_bytes(n_images), 16), dtype=torch.uint8, device=device)


# --------------------------------------------------------------------------------------------------
# thin functional wrappers over the C ABI (also what the parity tests call)
# --------------------------------------------------------------------------------------------------
def analyze(plan: Plan, images: torch.Tensor, adjoint: bool = False) -> torch.Tensor:
    """images (n0, n1, *grid) in plan.grid_dtype -> kept modes (n0, n1, *kept) complex64 (adjoint: float32 images on out_grid)."""
    lib = _lib.load()
    spatial = plan.out_grid if adjoint else plan.grid
    dtype = torch.float32 if adjoint else plan.grid_dtype
    assert images.dtype == dtype and images.is_contiguous() and tuple(images.shape[2:]) == spatial
    n_images = images.shape[0] * images.shape[1]
    modes = torch.empty((*images.shape[:2], *plan.kept), dtype=torch.complex64, device=images.device)
    ws = _workspace(plan, n_images, images.device)
    with torch.cuda.device(images.device):
        _lib.check(lib.sc_analyze(plan.handle, _ptr(images), n_images, _ptr(modes), int(adjoint), _ptr(ws),
                                  ws.numel(), _stream_ptr(images.device)), "sc_analyze")
    return modes


def synthesize(plan: Plan, modes: torch.Tensor, bias: Optional[torch.Tensor] = None, adjoint: bool = False) -> torch.Tensor:
    """kept modes -> images: float32 on out_grid (+ bias), or with adjoint=True the gradient on grid in plan.grid_dtype."""
    lib = _lib.load()
    assert modes.dtype == torch.complex64 and modes.is_contiguous() and tuple(modes.shape[2:]) == plan.kept
    n_images = modes.shape[0] * modes.shape[1]
    spatial = plan.grid if adjoint else plan.out_grid
    out = torch.empty((*modes.shape[:2], *spatial), dtype=plan.grid_dtype if adjoint else torch.float32, device=modes.device)
    ws = _workspace(plan, n_images, modes.device)
    b = bias.reshape(-1).contiguous() if bias is not None else None
    with torch.cuda.device(modes.device):
        _lib.check(lib.sc_synthesize(plan.handle, _ptr(modes), n_images, modes.shape[1], _ptr(b), _ptr(out),
                                     int(adjoint), _ptr(ws), ws.numel(), _stream_ptr(modes.device)), "sc_synthesize")
    return out


def contract_dense(plan: Plan, xm: torch.Tensor, weight: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    B, Ci = xm.shape[:2]
    Co = weight.shape[1]
    assert weight.dtype == torch.complex64 and weight.is_contiguous() and weight.shape[0] == Ci
    ym = torch.empty((B, Co, *plan.kept), dtype=torch.complex64, device=xm.device)
    with torch.cuda.device(xm.device):
        _lib.check(lib.sc_contract_dense(plan.handle, _ptr(xm), _ptr(weight), _ptr(ym), B, Ci, Co,
                                         _stream_ptr(xm.device)), "sc_contract_dense")
    return ym


def contract_dense_backward(plan: Plan, xm, gm, weight, need_dxm=True, need_dweight=True, need_dbias=True):
    lib = _lib.load()
    B, Co = gm.shape[:2]
    Ci = weight.shape[0]
    dxm = torch.empty((B, Ci, *plan.kept), dtype=torch.complex64, device=gm.device) if need_dxm else None
    dw = torch.empty_like(weight) if need_dweight else None
    db = torch.empty(Co, dtype=torch.float32, device=gm.device) if need_dbias else None
    with torch.cuda.device(gm.device):
        _lib.check(lib.sc_contract_dense_backward(plan.handle, _ptr(xm), _ptr(gm), _ptr(weight), _ptr(dxm), _ptr(dw),
                                                  _ptr(db), B, Ci, Co, _stream_ptr(gm.device)),
                   "sc_contract_dense_backward")
    return dxm, dw, db


class _SpectralConvDense(torch.autograd.Function):
    """y = SpectralConv.forward(x) with a dense weight; saves only the kept input modes (B,Ci,*kept)."""

    @staticmethod
    def forward(ctx, x, weight, bias, plan: Plan, reducer=None):
        lib = _lib.load()
        B, Ci = x.shape[:2]
        Co = weight.shape[1]
        dev = x.device
        y = torch.empty((B, Co, *plan.out_grid), dtype=torch.float32, device=dev)
        xm = torch.empty((B, Ci, *plan.kept), dtype=torch.complex64, device=dev)
        n_max = B * max(Ci, Co)
        ws = _workspace(plan, n_max, dev)
        b = bias.reshape(-1) if bias is not None else None
        layout = ctypes.c_int32(0)
        with torch.cuda.device(dev):
            _lib.check(lib.sc_forward_dense(plan.handle, _ptr(x), _ptr(weight), _ptr(b), _ptr(y), _ptr(xm), ctypes.byref(layout),
                                            B, Ci, Co, _ptr(ws), ws.numel(), _stream_ptr(dev)), "sc_forward_dense")
        ctx.x_dtype = x.dtype            # dx is stored like x (16-bit image storage)
        ctx.saved_layout = int(layout.value)      # xm is opaque: the library says how it ordered the saved modes
        ctx.plan = plan
        ctx.reducer = reducer
        ctx.has_bias = bias is not None
        ctx.bias_shape = bias.shape if bias is not None else None
        ctx.save_for_backward(xm, weight)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        lib = _lib.load()
        xm, weight = ctx.saved_tensors
        plan = ctx.plan
        need_dx, need_dw, need_db = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.has_bias and ctx.needs_input_grad[2]
        gy = gy.contiguous()
        if gy.dtype != torch.float32:
            gy = gy.float()
        B, Ci = xm.shape[:2]
        Co = weight.shape[1]
        dev = gy.device
        dx = torch.empty((B, Ci, *plan.grid), dtype=ctx.x_dtype, device=dev) if need_dx else None
        if need_dw and need_db:
            # dweight and dbias share one allocation so that a data-parallel reducer moves them with ONE collective; a peer-memory
            # reducer hands out its symmetric buffer, so that the kernels write the gradients where the collective reads them
            n_w = weight.numel() * 2
            owner = getattr(ctx.reducer, "grad_buffer", None) if ctx.reducer is not None and ctx.reducer.world_size() > 1 else None
            flat = owner(n_w + Co, dev) if owner is not None else torch.empty(n_w + Co, dtype=torch.float32, device=dev)
            dw = torch.view_as_complex(flat[:n_w].view(*weight.shape, 2))
            db = flat[n_w:]
        else:
            dw = torch.empty_like(weight) if need_dw else None
            db = torch.empty(Co, dtype=torch.float32, device=dev) if need_db else None
        ws = _workspace(plan, B * max(Ci, Co), dev)
        reducer = ctx.reducer
        data_parallel = reducer is not None and reducer.world_size() > 1 and (dw is not None or db is not None)
        # data parallel: the library records `grads_ready` right after the dweight (+dbias) launch; the reducer's collective
        # stream waits on it, so the all-reduce runs underneath the dxm contraction and the dx synthesis kernel
        ev = reducer.grads_ready_event() if data_parallel else ctypes.c_void_p(0)
        with torch.cuda.device(dev):
            _lib.check(lib.sc_backward_dense(plan.handle, _ptr(gy), _ptr(weight), _ptr(xm), ctx.saved_layout, _ptr(dx), _ptr(dw),
                                             _ptr(db), B, Ci, Co, _ptr(ws), ws.numel(), _stream_ptr(dev), ev), "sc_backward_dense")
            if data_parallel:
                reducer.reduce_in_backward([dw, db], after_event=ev)
        if db is not None:
            db = db.reshape(ctx.bias_shape)
        return dx, dw, db, None, None


def spectral_conv_dense(x, weight, bias, plan: Plan, reducer=None):
    return _SpectralConvDense.apply(x, weight, bias, plan, reducer)


# --------------------------------------------------------------------------------------------------
# Tucker-factorized contraction without reconstructing the weight (reference `_contract_tucker`, :76-103)
# --------------------------------------------------------------------------------------------------
def _table_contract(table, s_p, s_q, conj, src, n_outer, P, Q, n_inner):
    """out[o, p, i] = sum_q op(table[p, q]) * src[o, q, i]; table element (p, q) at table.flat[p * s_p + q * s_q]."""
    lib = _lib.load()
    out = torch.empty(n_outer * P * n_inner, dtype=torch.complex64, device=src.device)
    _lib.check(lib.sc_table_contract(_ptr(table), s_p, s_q, int(conj), _ptr(src), _ptr(out), n_outer, P, Q, n_inner,
                                     _stream_ptr(src.device)), "sc_table_contract")
    return out


def _pair_reduce(a, b, out, s_p, s_q, n_outer, P, Q, n_inner):
    """out.flat[p * s_p + q * s_q] = sum_{o,i} conj(a[o,p,i]) * b[o,q,i]."""
    lib = _lib.load()
    _lib.check(lib.sc_pair_reduce(_ptr(a), _ptr(b), _ptr(out), s_p, s_q, n_outer, P, Q, n_inner, _stream_ptr(a.device)),
               "sc_pair_reduce")
    return out


class _SpectralConvTucker(torch.autograd.Function):
    """y = SpectralConv.forward(x) with a Tucker weight, contracted factor by factor (einsum `abcd,fghi,bf,eg,ch,di->aecd`,
    reference :86-98):  xm -> U_in -> (core expanded along the mode axes with the kept rows of the mode factors) -> U_out.
    Inputs: x, core (r_in, r_out, r_1..r_d), U_in (Ci, r_in), U_out (Co, r_out), mode factors ALREADY sliced to the kept rows
    (k_j, r_j) -- autograd handles the slicing --, bias.  `plan_kept` is a plan whose weight extents equal the kept modes.
    One C call per direction (`sc_forward_tucker` / `sc_backward_tucker`): the chain of ~20 launches is issued by the library
    from one workspace, the only Python-side allocations are the outputs and the opaque saved-activation buffer."""

    @staticmethod
    def _args(plan, B, Ci, Co, core):
        lib = _lib.load()
        ranks = _rank_array(core)
        ws_bytes = int(lib.sc_tucker_workspace_bytes(plan.handle, B, Ci, Co, ranks))
        saved_elems = int(lib.sc_tucker_saved_elems(plan.handle, B, Ci, Co, ranks))
        return ranks, ws_bytes, saved_elems

    @staticmethod
    def forward(ctx, x, bias, plan, plan_kept, core, u_in, u_out, *u_modes):
        lib = _lib.load()
        dev = x.device
        B, Ci = x.shape[:2]
        Co = u_out.shape[0]
        d = plan.ndim
        core = core.contiguous()
        ranks, ws_bytes, saved_elems = _SpectralConvTucker._args(plan, B, Ci, Co, core)
        y = torch.empty((B, Co, *plan.out_grid), dtype=torch.float32, device=dev)
        saved = torch.empty(saved_elems, dtype=torch.complex64, device=dev)
        ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
        modes_ptrs = _ptr_array(u_modes)
        b = bias.reshape(-1) if bias is not None else None
        with torch.cuda.device(dev):
            _lib.check(lib.sc_forward_tucker(plan.handle, plan_kept.handle, _ptr(x), _ptr(core), _ptr(u_in), _ptr(u_out), modes_ptrs, _ptr(b),
                                             _ptr(y), _ptr(saved), B, Ci, Co, ranks, _ptr(ws), ws.numel(), _stream_ptr(dev)),
                       "sc_forward_tucker")
        ctx.x_dtype = x.dtype            # dx is stored like x (16-bit image storage)
        ctx.plan, ctx.plan_kept, ctx.d = plan, plan_kept, d
        ctx.bias_shape = bias.shape if bias is not None else None
        ctx.dims = (B, Ci, Co)
        ctx.save_for_backward(saved, core, u_in, u_out, *u_modes)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        lib = _lib.load()
        plan, plan_kept, d = ctx.plan, ctx.plan_kept, ctx.d
        B, Ci, Co = ctx.dims
        saved, core, u_in, u_out = ctx.saved_tensors[:4]
        u_modes = ctx.saved_tensors[4:4 + d]
        dev = gy.device
        gy = gy.contiguous()
        if gy.dtype != torch.float32:
            gy = gy.float()
        ranks, ws_bytes, _ = _SpectralConvTucker._args(plan, B, Ci, Co, core)
        dx = torch.empty((B, Ci, *plan.grid), dtype=ctx.x_dtype, device=dev)
        d_core = torch.empty_like(core)
        d_u_in = torch.empty_like(u_in)
        d_u_out = torch.empty_like(u_out)
        d_modes = [torch.empty_like(u) for u in u_modes]
        db = torch.empty(Co, dtype=torch.float32, device=dev) if ctx.bias_shape is not None else None
        ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
        modes_ptrs = _ptr_array(u_modes)
        dmodes_ptrs = _ptr_array(d_modes)
        with torch.cuda.device(dev):
            _lib.check(lib.sc_backward_tucker(plan.handle, plan_kept.handle, _ptr(gy), _ptr(core), _ptr(u_in), _ptr(u_out), modes_ptrs,
                                              _ptr(saved), _ptr(dx), _ptr(d_core), _ptr(d_u_in), _ptr(d_u_out), dmodes_ptrs, _ptr(db),
                                              B, Ci, Co, ranks, _ptr(ws), ws.numel(), _stream_ptr(dev)), "sc_backward_tucker")
        if db is not None:
            db = db.reshape(ctx.bias_shape)
        return (dx, db, None, None, d_core, d_u_in, d_u_out, *d_modes)


# --------------------------------------------------------------------------------------------------
# CP-factorized contraction without reconstructing the weight (reference `_contract_cp`, :55-73)
# --------------------------------------------------------------------------------------------------
def _cp_factor_args(u_modes, kept):
    d = len(u_modes)
    ptrs = (ctypes.c_void_p * d)(*[u.data_ptr() for u in u_modes])      # host array of device pointers
    ks = (ctypes.c_int32 * d)(*[int(k) for k in kept])
    return ptrs, ks, d


class _SpectralConvCP(torch.autograd.Function):
    """y = SpectralConv.forward(x) with a CP weight (einsum `abcd,e,be,fe,ce,de->afcd`, reference :58-71):
    xm -> U_in -> pointwise scale[e, m] = lambda_e prod_j U_j[m_j, e] -> U_out.  Mode factors arrive already sliced to the
    kept rows (k_j, R)."""

    @staticmethod
    def forward(ctx, x, bias, plan, lam, u_in, u_out, *u_modes):
        lib = _lib.load()
        dev = x.device
        B, Ci = x.shape[:2]
        Co, R = u_out.shape
        kept = plan.kept
        M = plan.n_modes_total
        st = _stream_ptr(dev)
        with torch.cuda.device(dev):
            xm = analyze(plan, x)
            ptrs, ks, d = _cp_factor_args(u_modes, kept)
            scale = torch.empty(R * M, dtype=torch.complex64, device=dev)
            _lib.check(lib.sc_cp_scale(ptrs, ks, d, _ptr(lam), _ptr(scale), R, st), "sc_cp_scale")
            t1 = _table_contract(u_in, 1, R, False, xm, B, R, Ci, M)                # T[p=e, q=i] = U_in[i, e]
            t2 = torch.empty_like(t1)
            _lib.check(lib.sc_cp_apply(_ptr(t1), _ptr(scale), _ptr(t2), 0, B, R * M, st), "sc_cp_apply")
            ym = _table_contract(u_out, R, 1, False, t2, B, Co, R, M)               # T[p=o, q=e] = U_out[o, e]
            y = synthesize(plan, ym.view(B, Co, *kept), bias)
        ctx.plan = plan
        ctx.bias_shape = bias.shape if bias is not None else None
        ctx.dims = (B, Ci, Co, R, M)
        ctx.save_for_backward(xm, t1, t2, scale, lam, u_in, u_out, *u_modes)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        lib = _lib.load()
        plan = ctx.plan
        B, Ci, Co, R, M = ctx.dims
        kept = plan.kept
        xm, t1, t2, scale, lam, u_in, u_out = ctx.saved_tensors[:7]
        u_modes = ctx.saved_tensors[7:]
        dev = gy.device
        gy = gy.contiguous()
        cplx = dict(dtype=torch.complex64, device=dev)
        st = _stream_ptr(dev)
        with torch.cuda.device(dev):
            gm = analyze(plan, gy, adjoint=True)
            db = None
            if ctx.bias_shape is not None:
                db = torch.empty(Co, dtype=torch.float32, device=dev)
                _lib.check(lib.sc_bias_grad(plan.handle, _ptr(gm), _ptr(db), B, Co, st), "sc_bias_grad")
                db = db.reshape(ctx.bias_shape)
            g2 = _table_contract(u_out, 1, R, True, gm, B, R, Co, M)                # T[p=e, q=o] = conj(U_out[o, e])
            d_u_out = _pair_reduce(t2, gm, torch.empty(Co, R, **cplx), 1, R, B, R, Co, M)
            dscale = torch.empty(R * M, **cplx)
            _lib.check(lib.sc_cp_dscale(_ptr(t1), _ptr(g2), _ptr(dscale), B, R * M, st), "sc_cp_dscale")
            g1 = torch.empty_like(g2)
            _lib.check(lib.sc_cp_apply(_ptr(g2), _ptr(scale), _ptr(g1), 1, B, R * M, st), "sc_cp_apply")
            d_u_in = _pair_reduce(xm, g1, torch.empty(Ci, R, **cplx), R, 1, B, Ci, R, M)
            dxm = _table_contract(u_in, R, 1, True, g1, B, Ci, R, M)                # T[p=i, q=e] = conj(U_in[i, e])
            dx = synthesize(plan, dxm.view(B, Ci, *kept), adjoint=True)
            ptrs, ks, d = _cp_factor_args(u_modes, kept)
            d_lam = torch.empty(R, **cplx)
            _lib.check(lib.sc_cp_factor_grad(ptrs, ks, d, _ptr(lam), _ptr(dscale), _ptr(d_lam), -1, R, st), "sc_cp_factor_grad")
            d_modes = []
            for j in range(d):
                g = torch.empty(kept[j], R, **cplx)
                _lib.check(lib.sc_cp_factor_grad(ptrs, ks, d, _ptr(lam), _ptr(dscale), _ptr(g), j, R, st), "sc_cp_factor_grad")
                d_modes.append(g)
        return (dx, db, None, d_lam, d_u_in, d_u_out, *d_modes)


# --------------------------------------------------------------------------------------------------
# TT-factorized contraction without reconstructing the weight (reference `_contract_tt`, :106-127)
# --------------------------------------------------------------------------------------------------
class _SpectralConvTT(torch.autograd.Function):
    """y = SpectralConv.forward(x) with a tensor-train weight  W[i,o,m] = G0[0,i,:] G1[:,o,:] G2[:,m_1,:] .. G_{d+1}[:,m_d,0].
    The mode cores (already sliced to the kept rows) are multiplied right to left into V[r2, m]; G1 V gives a rank-r1
    weight block (r1, Co, modes) that the dense mode GEMM applies to xm G0."""

    @staticmethod
    def forward(ctx, x, bias, plan, plan_kept, g0, g1c, *cores):
        dev = x.device
        B, Ci = x.shape[:2]
        r1, Co, r2 = g1c.shape
        kept = plan.kept
        M = plan.n_modes_total
        d = plan.ndim
        with torch.cuda.device(dev):
            xm = analyze(plan, x)
            chain = [cores[d - 1].contiguous()]                                      # A_{d-1}: (ra, k_{d-1}) since rb = 1
            inner = kept[d - 1]
            for j in range(d - 2, -1, -1):
                ra, kj, rb = cores[j].shape
                chain.append(_table_contract(cores[j], rb, 1, False, chain[-1], 1, ra * kj, rb, inner))
                inner *= kj
            v = chain[-1]                                                            # (r2, M)
            wc = _table_contract(g1c, r2, 1, False, v, 1, r1 * Co, r2, M)            # (r1, Co, M)
            t1 = _table_contract(g0, 1, r1, False, xm, B, r1, Ci, M)                 # T[p=r, q=i] = G0[0, i, r]
            ym = contract_dense(plan_kept, t1.view(B, r1, *kept), wc.view(r1, Co, *kept))
            y = synthesize(plan, ym, bias)
        ctx.plan, ctx.plan_kept, ctx.d = plan, plan_kept, d
        ctx.bias_shape = bias.shape if bias is not None else None
        ctx.dims = (B, Ci, Co, r1, r2, M)
        ctx.save_for_backward(xm, t1, wc, g0, g1c, *cores, *chain)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        lib = _lib.load()
        plan, plan_kept, d = ctx.plan, ctx.plan_kept, ctx.d
        B, Ci, Co, r1, r2, M = ctx.dims
        kept = plan.kept
        saved = ctx.saved_tensors
        xm, t1, wc, g0, g1c = saved[:5]
        cores = saved[5:5 + d]
        chain = saved[5 + d:]                     # A_{d-1}, A_{d-2}, ..., A_0 (= V)
        dev = gy.device
        gy = gy.contiguous()
        cplx = dict(dtype=torch.complex64, device=dev)
        with torch.cuda.device(dev):
            gm = analyze(plan, gy, adjoint=True)
            db = None
            if ctx.bias_shape is not None:
                db = torch.empty(Co, dtype=torch.float32, device=dev)
                _lib.check(lib.sc_bias_grad(plan.handle, _ptr(gm), _ptr(db), B, Co, _stream_ptr(dev)), "sc_bias_grad")
                db = db.reshape(ctx.bias_shape)
            g1, d_wc, _ = contract_dense_backward(plan_kept, t1.view(B, r1, *kept), gm, wc.view(r1, Co, *kept),
                                                  need_dbias=False)
            d_g0 = _pair_reduce(xm, g1, torch.empty(1, Ci, r1, **cplx), r1, 1, B, Ci, r1, M)
            dxm = _table_contract(g0, r1, 1, True, g1, B, Ci, r1, M)                 # T[p=i, q=r] = conj(G0[0, i, r])
            dx = synthesize(plan, dxm.view(B, Ci, *kept), adjoint=True)
            v = chain[-1]
            d_g1 = _pair_reduce(v, d_wc, torch.empty(r1, Co, r2, **cplx), 1, r2, 1, r2, r1 * Co, M)
            d_a = _table_contract(g1c, 1, r2, True, d_wc, 1, r2, r1 * Co, M)         # dV (r2, M)
            d_cores = [None] * d
            inner = M
            for j in range(d - 1):
                ra, kj, rb = cores[j].shape
                inner //= kj
                a_next = chain[d - 2 - j]                                            # A_{j+1}: (rb, inner)
                d_cores[j] = _pair_reduce(a_next, d_a, torch.empty(ra, kj, rb, **cplx), 1, rb, 1, rb, ra * kj, inner)
                d_a = _table_contract(cores[j], 1, rb, True, d_a, 1, rb, ra * kj, inner)
            d_cores[d - 1] = d_a.view(cores[d - 1].shape)
        return (dx, db, None, None, d_g0, d_g1, *d_cores)


# --------------------------------------------------------------------------------------------------
# CP / TT chains as ONE C call per direction (sc_forward_cp / sc_backward_cp, sc_forward_tt / sc_backward_tt): the same launches as
# `_SpectralConvCP` / `_SpectralConvTT` above, issued by the library from one saved buffer and one workspace.  They were written
# after the round's GPU minutes were spent, so the Python-orchestrated chains (validated on hardware) stay the default; set
# `FACTORIZED_CHAINS_IN_C = True` (or SC_FACTORIZED_C=1 in the environment) to route CP / TT through the C entry points.
# --------------------------------------------------------------------------------------------------
import os as _os

FACTORIZED_CHAINS_IN_C = _os.environ.get("SC_FACTORIZED_C", "0") == "1"


class _SpectralConvCPCall(torch.autograd.Function):
    """`_SpectralConvCP` behind one C call per direction."""

    @staticmethod
    def forward(ctx, x, bias, plan, lam, u_in, u_out, *u_modes):
        lib = _lib.load()
        dev = x.device
        B, Ci = x.shape[:2]
        Co, R = u_out.shape
        saved = torch.empty(int(lib.sc_cp_saved_elems(plan.handle, B, Ci, Co, R)), dtype=torch.complex64, device=dev)
        ws = torch.empty(max(int(lib.sc_cp_workspace_bytes(plan.handle, B, Ci, Co, R)), 16), dtype=torch.uint8, device=dev)
        y = torch.empty((B, Co, *plan.out_grid), dtype=torch.float32, device=dev)
        b = bias.reshape(-1) if bias is not None else None
        with torch.cuda.device(dev):
            _lib.check(lib.sc_forward_cp(plan.handle, _ptr(x), _ptr(lam), _ptr(u_in), _ptr(u_out), _ptr_array(u_modes), _ptr(b), _ptr(y),
                                         _ptr(saved), B, Ci, Co, R, _ptr(ws), ws.numel(), _stream_ptr(dev)), "sc_forward_cp")
        ctx.x_dtype = x.dtype            # dx is stored like x (16-bit image storage)
        ctx.plan = plan
        ctx.bias_shape = bias.shape if bias is not None else None
        ctx.dims = (B, Ci, Co, R)
        ctx.save_for_backward(saved, lam, u_in, u_out, *u_modes)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        lib = _lib.load()
        plan = ctx.plan
        B, Ci, Co, R = ctx.dims
        saved, lam, u_in, u_out = ctx.saved_tensors[:4]
        u_modes = ctx.saved_tensors[4:]
        dev = gy.device
        gy = gy.contiguous()
        if gy.dtype != torch.float32:
            gy = gy.float()
        dx = torch.empty((B, Ci, *plan.grid), dtype=ctx.x_dtype, device=dev)
        d_lam, d_u_in, d_u_out = torch.empty_like(lam), torch.empty_like(u_in), torch.empty_like(u_out)
        d_modes = [torch.empty_like(u) for u in u_modes]
        db = torch.empty(Co, dtype=torch.float32, device=dev) if ctx.bias_shape is not None else None
        ws = torch.empty(max(int(lib.sc_cp_workspace_bytes(plan.handle, B, Ci, Co, R)), 16), dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.sc_backward_cp(plan.handle, _ptr(gy), _ptr(lam), _ptr(u_in), _ptr(u_out), _ptr_array(u_modes), _ptr(saved),
                                          _ptr(dx), _ptr(d_lam), _ptr(d_u_in), _ptr(d_u_out), _ptr_array(d_modes), _ptr(db),
                                          B, Ci, Co, R, _ptr(ws), ws.numel(), _stream_ptr(dev)), "sc_backward_cp")
        if db is not None:
            db = db.reshape(ctx.bias_shape)
        return (dx, db, None, d_lam, d_u_in, d_u_out, *d_modes)


class _SpectralConvTTCall(torch.autograd.Function):
    """`_SpectralConvTT` behind one C call per direction."""

    @staticmethod
    def _ranks(g1c, cores):
        return (ctypes.c_int32 * (1 + len(cores)))(int(g1c.shape[0]), *[int(c.shape[0]) for c in cores])

    @staticmethod
    def forward(ctx, x, bias, plan, plan_kept, g0, g1c, *cores):
        lib = _lib.load()
        dev = x.device
        B, Ci = x.shape[:2]
        Co = g1c.shape[1]
        cores = tuple(c.contiguous() for c in cores)
        ranks = _SpectralConvTTCall._ranks(g1c, cores)
        saved = torch.empty(int(lib.sc_tt_saved_elems(plan.handle, B, Ci, Co, ranks)), dtype=torch.complex64, device=dev)
        ws = torch.empty(max(int(lib.sc_tt_workspace_bytes(plan.handle, B, Ci, Co, ranks)), 16), dtype=torch.uint8, device=dev)
        y = torch.empty((B, Co, *plan.out_grid), dtype=torch.float32, device=dev)
        b = bias.reshape(-1) if bias is not None else None
        with torch.cuda.device(dev):
            _lib.check(lib.sc_forward_tt(plan.handle, plan_kept.handle, _ptr(x), _ptr(g0), _ptr(g1c), _ptr_array(cores), _ptr(b), _ptr(y),
                                         _ptr(saved), B, Ci, Co, ranks, _ptr(ws), ws.numel(), _stream_ptr(dev)), "sc_forward_tt")
        ctx.x_dtype = x.dtype            # dx is stored like x (16-bit image storage)
        ctx.plan, ctx.plan_kept = plan, plan_kept
        ctx.bias_shape = bias.shape if bias is not None else None
        ctx.dims = (B, Ci, Co)
        ctx.save_for_backward(saved, g0, g1c, *cores)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        lib = _lib.load()
        plan, plan_kept = ctx.plan, ctx.plan_kept
        B, Ci, Co = ctx.dims
        saved, g0, g1c = ctx.saved_tensors[:3]
        cores = ctx.saved_tensors[3:]
        dev = gy.device
        gy = gy.contiguous()
        if gy.dtype != torch.float32:
            gy = gy.float()
        ranks = _SpectralConvTTCall._ranks(g1c, cores)
        dx = torch.empty((B, Ci, *plan.grid), dtype=ctx.x_dtype, device=dev)
        d_g0, d_g1 = torch.empty_like(g0), torch.empty_like(g1c)
        d_cores = [torch.empty_like(c) for c in cores]
        db = torch.empty(Co, dtype=torch.float32, device=dev) if ctx.bias_shape is not None else None
        ws = torch.empty(max(int(lib.sc_tt_workspace_bytes(plan.handle, B, Ci, Co, ranks)), 16), dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.sc_backward_tt(plan.handle, plan_kept.handle, _ptr(gy), _ptr(g0), _ptr(g1c), _ptr_array(cores), _ptr(saved),
                                          _ptr(dx), _ptr(d_g0), _ptr(d_g1), _ptr_array(d_cores), _ptr(db), B, Ci, Co, ranks,
                                          _ptr(ws), ws.numel(), _stream_ptr(dev)), "sc_backward_tt")
        if db is not None:
            db = db.reshape(ctx.bias_shape)
        return (dx, db, None, None, d_g0, d_g1, *d_cores)


# --------------------------------------------------------------------------------------------------
# separable (depthwise) contraction, reference `_contract_dense_separable` :49-52
# --------------------------------------------------------------------------------------------------
class _SpectralConvSeparable(torch.autograd.Function):
    """y = SpectralConv.forward(x) with `separable=True`: ym[b,c,m] = xm[b,c,m] * w[c,m]  (w: (C, *kept), the kept block of the
    weight).  Backward: dxm = gm * conj(w), dw = sum_b conj(xm) * gm, db from the DC slot."""

    @staticmethod
    def forward(ctx, x, w, bias, plan):
        lib = _lib.load()
        dev = x.device
        B, C = x.shape[:2]
        M = plan.n_modes_total
        with torch.cuda.device(dev):
            xm = analyze(plan, x)
            ym = torch.empty_like(xm)
            _lib.check(lib.sc_cp_apply(_ptr(xm), _ptr(w), _ptr(ym), 0, B, C * M, _stream_ptr(dev)), "sc_cp_apply")
            y = synthesize(plan, ym, bias)
        ctx.plan = plan
        ctx.bias_shape = bias.shape if bias is not None else None
        ctx.save_for_backward(xm, w)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        lib = _lib.load()
        plan = ctx.plan
        xm, w = ctx.saved_tensors
        B, C = xm.shape[:2]
        M = plan.n_modes_total
        dev = gy.device
        gy = gy.contiguous()
        st = _stream_ptr(dev)
        with torch.cuda.device(dev):
            gm = analyze(plan, gy, adjoint=True)
            db = None
            if ctx.bias_shape is not None:
                db = torch.empty(C, dtype=torch.float32, device=dev)
                _lib.check(lib.sc_bias_grad(plan.handle, _ptr(gm), _ptr(db), B, C, st), "sc_bias_grad")
                db = db.reshape(ctx.bias_shape)
            dw = torch.empty_like(w)
            _lib.check(lib.sc_cp_dscale(_ptr(xm), _ptr(gm), _ptr(dw), B, C * M, st), "sc_cp_dscale")
            dxm = torch.empty_like(gm)
            _lib.check(lib.sc_cp_apply(_ptr(gm), _ptr(w), _ptr(dxm), 1, B, C * M, st), "sc_cp_apply")
            dx = synthesize(plan, dxm, adjoint=True)
        return dx, dw, db, None


# --------------------------------------------------------------------------------------------------
# the module
# --------------------------------------------------------------------------------------------------
class _SpectralResample(torch.autograd.Function):
    """`resample` for 3-D and higher inputs (reference resample.py:52-69): rfftn(norm="forward"), copy the low-frequency block
    both grids have (leading dims: bins [0, m//2) and [-m//2, 0) with m = min(old, new); last dim: the first
    min(old//2+1, new//2+1) bins), irfftn on the new grid -- i.e. this library's truncated analysis followed by its zero-padded
    synthesis with no contraction in between.  Even m on the leading dims (for odd m the reference's block [-m//2-1, m//2) is not
    the centred block the kernels index)."""

    @staticmethod
    def _plan(x, out_shape):
        grid = list(x.shape[2:])
        stored = []
        for j, (n, m) in enumerate(zip(grid, out_shape)):
            if j == len(grid) - 1:
                stored.append(min(n // 2 + 1, m // 2 + 1))
            else:
                k = min(n, m)
                if k % 2 != 0:
                    raise NotImplementedError("spectral resampling with an odd common size along a leading dim is not covered")
                stored.append(k)
        return get_plan(x.device, grid, list(out_shape), stored, stored, "forward", flags=_lib.FLAG_RESAMPLE)

    @staticmethod
    def forward(ctx, x, out_shape):
        if not x.is_cuda:
            raise RuntimeError("neuraloperator_b200 has no CPU path")
        plan = _SpectralResample._plan(x, out_shape)
        ctx.plan = plan
        return synthesize(plan, analyze(plan, x))

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        plan = ctx.plan
        gm = analyze(plan, gy.contiguous().float(), adjoint=True)
        return synthesize(plan, gm, adjoint=True), None


# --------------------------------------------------------------------------------------------------
# complex_data=True (reference :439-441, :470-479, :500-519, :531-538): C2C transforms along every dim
# --------------------------------------------------------------------------------------------------
class ComplexPlan:
    """Kept-mode index set and twiddle tables of the complex-data path.  Every dim is a complex table product (there is no
    half spectrum), so the whole chain runs on the library's complex table kernel (`sc_table_contract`) and the dense
    mode-wise contraction; nothing here is specific to a grid size.  Index rules (restated from the reference, pinned by the
    oracle's `kept_mode_plan_complex` against the live module): every dim is FFT-shifted unless the conv is 1-D; the weight is
    cut centrally along every dim; the last dim nevertheless takes the FIRST k entries of its (shifted) spectrum; on the way
    back only the leading dims are un-shifted, so the last dim's slots are synthesised at their own index."""

    def __init__(self, device, grid, out_grid, n_modes, max_n_modes, fft_norm, table_device=None):
        import math
        d = len(grid)
        table_device = device if table_device is None else table_device      # (tests build the tables without a GPU)
        self.ndim, self.grid, self.out_grid = d, tuple(grid), tuple(out_grid)
        self.kept, self.w_start, self.analysis, self.synthesis = [], [], [], []
        if fft_norm == "forward":
            s_fwd, s_inv = 1.0 / math.prod(grid), 1.0
        elif fft_norm == "backward":
            s_fwd, s_inv = 1.0, 1.0 / math.prod(out_grid)
        else:
            s_fwd, s_inv = 1.0 / math.sqrt(math.prod(grid)), 1.0 / math.sqrt(math.prod(out_grid))
        for j in range(d):
            last = j == d - 1
            N, M = int(grid[j]), int(out_grid[j])
            k = min(N, int(n_modes[j]))
            start = int(max_n_modes[j]) - k
            if start < 0:
                raise ValueError("n_modes exceeds max_n_modes (weight too small for the requested modes)")
            shift = N // 2 if d > 1 else 0
            pos = list(range(k)) if last else list(range(N // 2 - k // 2, N // 2 + k // 2 + k % 2))
            in_bins = torch.tensor([(q - shift) % N for q in pos], dtype=torch.float64)
            out_pos = torch.tensor(pos if last else [(q - shift) % N for q in pos], dtype=torch.float64)
            n_in = torch.arange(N, dtype=torch.float64)
            n_out = torch.arange(M, dtype=torch.float64)
            ang_a = -2.0 * math.pi * torch.remainder(in_bins[:, None] * n_in[None, :], N) / N               # [k x N]
            ang_s = 2.0 * math.pi * torch.remainder(n_out[:, None] * out_pos[None, :], M) / M              # [M x k]
            a = torch.polar(torch.full_like(ang_a, s_fwd if last else 1.0), ang_a)
            sy = torch.polar(torch.full_like(ang_s, s_inv if last else 1.0), ang_s) * (out_pos[None, :] < M)   # ifftn(s=M) crops the end
            self.kept.append(k)
            self.w_start.append(start // 2 if start else 0)
            self.analysis.append(a.to(torch.complex64).contiguous().to(table_device))
            self.synthesis.append(sy.to(torch.complex64).contiguous().to(table_device))
        self.kept = tuple(self.kept)
        # the dense mode GEMM only needs a plan whose kept block is (k_1..k_d) with weight extents == kept
        self.contract_plan = get_plan(device, [*self.kept[:-1], 2 * self.kept[-1]], [*self.kept[:-1], 2 * self.kept[-1]],
                                      list(self.kept), list(self.kept), "forward")


_COMPLEX_PLANS: "OrderedDict[tuple, ComplexPlan]" = OrderedDict()


def get_complex_plan(device, grid, out_grid, n_modes, max_n_modes, fft_norm) -> ComplexPlan:
    idx = device.index if device.index is not None else torch.cuda.current_device()
    key = (idx, tuple(grid), tuple(out_grid), tuple(n_modes), tuple(max_n_modes), fft_norm)
    with _PLAN_LOCK:
        plan = _COMPLEX_PLANS.get(key)
        if plan is None:
            plan = _COMPLEX_PLANS[key] = ComplexPlan(torch.device("cuda", idx), grid, out_grid, n_modes, max_n_modes, fft_norm)
            while len(_COMPLEX_PLANS) > _PLAN_CACHE_MAX:
                _COMPLEX_PLANS.popitem(last=False)
        return plan


def _apply_tables(tables, src, lead, sizes_in, sizes_out, order, adjoint):
    """Applies one table per dim to `src` (lead, *sizes_in) -> (lead, *sizes_out): `order` lists the dims in the order they are
    transformed.  adjoint: the conjugate transpose of every table."""
    cur = src.reshape(-1)
    sizes = list(sizes_in)
    for j in order:
        P, Q = sizes_out[j], sizes_in[j]
        outer = lead
        for l in range(j):
            outer *= sizes[l]
        inner = 1
        for l in range(j + 1, len(sizes)):
            inner *= sizes[l]
        t = tables[j]
        if adjoint:      # T'[p, q] = conj(T[q, p]),  T is (Q x P) row-major
            cur = _table_contract(t, 1, P, True, cur, outer, P, Q, inner)
        else:            # T is (P x Q) row-major
            cur = _table_contract(t, Q, 1, False, cur, outer, P, Q, inner)
        sizes[j] = P
    return cur.view(lead, *sizes) if isinstance(lead, int) else cur


class _SpectralConvComplex(torch.autograd.Function):
    """y = SpectralConv.forward(x) for complex data and a dense kept-block weight (B,Ci,*grid) -> (B,Co,*out_grid), without the
    bias: C2C analysis (one complex table product per dim, last dim first), mode-wise contraction, C2C synthesis.  The
    contraction is the dense mode GEMM (w_kept: (Ci, Co, *kept)) or, for `separable` (w_kept: (C, *kept),
    `_contract_dense_separable` :49-52), the mode-wise product."""

    @staticmethod
    def forward(ctx, x, w_kept, plan: ComplexPlan, separable=False):
        lib = _lib.load()
        B, Ci = x.shape[:2]
        Co = Ci if separable else w_kept.shape[1]
        d = plan.ndim
        with torch.cuda.device(x.device):
            xm = _apply_tables(plan.analysis, x, B * Ci, plan.grid, plan.kept, range(d - 1, -1, -1), False).view(B, Ci, *plan.kept)
            if separable:
                ym = torch.empty_like(xm)
                _lib.check(lib.sc_cp_apply(_ptr(xm), _ptr(w_kept), _ptr(ym), 0, B, xm[0].numel(), _stream_ptr(x.device)), "sc_cp_apply")
            else:
                ym = contract_dense(plan.contract_plan, xm, w_kept)
            y = _apply_tables(plan.synthesis, ym, B * Co, plan.kept, plan.out_grid, range(d), False).view(B, Co, *plan.out_grid)
        ctx.plan = plan
        ctx.separable = separable
        ctx.save_for_backward(xm, w_kept)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        lib = _lib.load()
        plan = ctx.plan
        xm, w_kept = ctx.saved_tensors
        B, Ci = xm.shape[:2]
        Co = Ci if ctx.separable else w_kept.shape[1]
        d = plan.ndim
        gy = gy.contiguous()
        if gy.dtype != torch.complex64:
            gy = gy.to(torch.complex64)
        st = _stream_ptr(gy.device)
        with torch.cuda.device(gy.device):
            gm = _apply_tables(plan.synthesis, gy, B * Co, plan.out_grid, plan.kept, range(d - 1, -1, -1), True).view(B, Co, *plan.kept)
            if ctx.separable:
                per = xm[0].numel()
                dw = torch.empty_like(w_kept)
                _lib.check(lib.sc_cp_dscale(_ptr(xm), _ptr(gm), _ptr(dw), B, per, st), "sc_cp_dscale")
                dxm = torch.empty_like(gm)
                _lib.check(lib.sc_cp_apply(_ptr(gm), _ptr(w_kept), _ptr(dxm), 1, B, per, st), "sc_cp_apply")
            else:
                dxm, dw, _ = contract_dense_backward(plan.contract_plan, xm, gm, w_kept, need_dbias=False)
            dx = _apply_tables(plan.analysis, dxm, B * Ci, plan.kept, plan.grid, range(d), True).view(B, Ci, *plan.grid)
        return dx, dw, None, None


# --------------------------------------------------------------------------------------------------
# reduced spectral precision, fno_block_precision = "half" / "mixed" (reference :436-437, :451-462; einsum_utils.py:10-36)
# --------------------------------------------------------------------------------------------------
def _round_half_(t: torch.Tensor) -> torch.Tensor:
    """Rounds a float32 / complex64 device tensor to the nearest fp16 values IN PLACE (what `.half()` / `.chalf()` keep)."""
    lib = _lib.load()
    flat = torch.view_as_real(t) if t.is_complex() else t
    if flat.numel():
        with torch.cuda.device(t.device):
            _lib.check(lib.sc_pointwise(_lib.POINTWISE_ROUND_HALF, _ptr(flat), None, _ptr(flat), flat.numel(), _stream_ptr(t.device)),
                       "sc_pointwise")
    return t


class _SpectralConvDenseReduced(torch.autograd.Function):
    """SpectralConv.forward with fno_block_precision "mixed" (full-precision transform, fp16 modes and contraction, :451-462) or
    "half" (the input is cast to fp16 first, :436-437), dense weight.  The kernels keep computing in fp32; the tensors are rounded
    to fp16 at the points where the reference casts -- x (half only), the kept input modes (`x.chalf()`), the weight
    (`einsum_complexhalf` casts it, einsum_utils.py:20-23) and the contracted modes (the chalf output spectrum) -- so the result
    differs from the reference's by fp16 rounding noise only (its half FFTs and fp16 products round more often, not less).  The
    casts are straight-through for gradients, as autograd treats `.half()`; backward is the full-precision backward on the
    rounded tensors.  There is no bandwidth gain yet: the mode tensors are still stored as complex64."""

    @staticmethod
    def forward(ctx, x, weight, bias, plan: Plan, round_input: bool):
        if round_input:
            x = _round_half_(x.clone())
        xm = _round_half_(analyze(plan, x))
        w_r = _round_half_(weight.detach().clone())
        ym = _round_half_(contract_dense(plan, xm, w_r))
        y = synthesize(plan, ym, bias)
        ctx.plan = plan
        ctx.bias_shape = bias.shape if bias is not None else None
        ctx.save_for_backward(xm, w_r)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, gy):
        plan = ctx.plan
        xm, w_r = ctx.saved_tensors
        gy = gy.contiguous()
        if gy.dtype != torch.float32:
            gy = gy.float()
        need_dx, need_dw, need_db = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.bias_shape is not None and ctx.needs_input_grad[2]
        gm = analyze(plan, gy, adjoint=True)
        dxm, dw, db = contract_dense_backward(plan, xm, gm, w_r, need_dxm=need_dx, need_dweight=need_dw, need_dbias=need_db)
        dx = synthesize(plan, dxm, adjoint=True) if need_dx else None
        if db is not None:
            db = db.reshape(ctx.bias_shape)
        return dx, dw, db, None, None


def _validate_scaling_factor(factor, n_dim) -> Optional[List[float]]:
    """Single-layer case of neuralop/utils.py:151-197 (`validate_scaling_factor(..., n_layers=None)`)."""
    if factor is None:
        return None
    if isinstance(factor, (int, float)):
        return [float(factor)] * n_dim
    if isinstance(factor, (list, tuple)) and len(factor) > 0 and all(isinstance(s, (int, float)) for s in factor):
        if len(factor) == n_dim:
            return [float(s) for s in factor]
        return [[float(s)] * n_dim for s in factor]
    return None


class BaseSpectralConv(nn.Module):
    """Plugin contract of the reference (`neuralop/layers/base_spectral_conv.py:4-27`)."""

    def __init__(self, device=None, dtype=None):
        super().__init__()
        self.dtype = dtype
        self.device = device

    def transform(self, x):
        return x


class SpectralConv(BaseSpectralConv):
    """Fourier-layer spectral convolution (real data, full precision) on hand-written sm_100a kernels.

    Parameters: identical to the reference class (spectral_convolution.py:183-305). `complex_data=True` runs C2C transforms on the
    complex table kernels (any grid; dense or reconstructed weights). `fno_block_precision` "half" / "mixed" round the tensors to
    fp16 where the reference casts (dense or reconstructed weights, real data); combinations the kernels do not cover raise
    `NotImplementedError` at construction.
    """

    def __init__(
        self,
        in_channels,
        out_channels,
        n_modes,
        complex_data=False,
        max_n_modes=None,
        bias=True,
        separable=False,
        resolution_scaling_factor: Optional[Union[Number, List[Number]]] = None,
        fno_block_precision="full",
        rank=1.0,
        factorization=None,
        implementation="reconstructed",
        enforce_hermitian_symmetry=True,
        fixed_rank_modes=False,
        decomposition_kwargs: Optional[dict] = None,
        init_std="auto",
        fft_norm="forward",
        device=None,
    ):
        super().__init__(device=device)
        if separable and in_channels != out_channels:
            raise ValueError("To use separable Fourier Conv, in_channels must be equal "
                             f"to out_channels, but got in_channels={in_channels} and out_channels={out_channels}")
        if fno_block_precision not in ("full", "half", "mixed"):
            raise ValueError(f"Got fno_block_precision={fno_block_precision}, expected 'full', 'half' or 'mixed'")
        if fno_block_precision != "full" and (complex_data or separable):
            raise NotImplementedError("fno_block_precision 'half' / 'mixed' is built for real data and a non-separable weight")
        # (reduced precision with implementation="factorized": the weight is reconstructed in fp32 and rounded to fp16 ONCE, where the
        #  reference's einsum_complexhalf rounds after every pairwise contraction of the factors -- fewer roundings, same fp16 noise level)
        if implementation not in ("reconstructed", "factorized"):
            raise ValueError(f'Got implementation={implementation}, expected "reconstructed" or "factorized"')
        if fft_norm not in _lib.NORMS:
            raise ValueError(f"Got fft_norm={fft_norm}, expected one of {sorted(_lib.NORMS)}")

        self.in_channels = in_channels
        self.out_channels = out_channels
        self.complex_data = complex_data
        self.n_modes = n_modes
        self.order = len(self.n_modes)
        if max_n_modes is None:
            max_n_modes = self.n_modes
        elif isinstance(max_n_modes, int):
            max_n_modes = [max_n_modes]
        self.max_n_modes = max_n_modes
        self.fno_block_precision = fno_block_precision
        self.rank = rank
        self.factorization = factorization
        self.implementation = implementation
        # the kernels always apply the Hermitian rules of the reference's default path (:547-559); with the flag
        # off the reference calls irfftn, whose C2R step ignores the same imaginary parts (identical on CPU)
        self.enforce_hermitian_symmetry = enforce_hermitian_symmetry
        self.resolution_scaling_factor = _validate_scaling_factor(resolution_scaling_factor, self.order)
        if init_std == "auto":
            init_std = (2 / (in_channels + out_channels)) ** 0.5
        if isinstance(fixed_rank_modes, bool):
            fixed_rank_modes = [0] if fixed_rank_modes else None
        self.fft_norm = fft_norm
        self.separable = separable
        # optional neuraloperator_b200.GradientAllReducer: backward then overlaps the dweight/dbias all-reduce with dx
        self.gradient_reducer = None

        # separable: one channel axis only (:346-356)
        weight_shape = (in_channels, *self.max_n_modes) if separable else (in_channels, out_channels, *self.max_n_modes)
        tensor_kwargs = decomposition_kwargs if decomposition_kwargs is not None else {}
        self.weight = FactorizedWeight.new(weight_shape, rank=self.rank, factorization=factorization or "Dense",
                                           fixed_rank_modes=fixed_rank_modes, dtype=torch.cfloat, device=device,
                                           **tensor_kwargs)
        self.weight.normal_(0, init_std)
        if bias:
            self.bias = nn.Parameter(init_std * torch.randn(*((self.out_channels,) + (1,) * self.order), device=device))
        else:
            self.bias = None

    # -- n_modes: stored with the last dim already halved, mutable at run time (:400-415) -------------
    @property
    def n_modes(self):
        return self._n_modes

    @n_modes.setter
    def n_modes(self, n_modes):
        n_modes = [n_modes] if isinstance(n_modes, int) else list(n_modes)
        if not self.complex_data:
            n_modes[-1] = n_modes[-1] // 2 + 1
        self._n_modes = n_modes

    def _output_grid(self, in_grid, output_shape):
        if output_shape is not None:
            return [int(s) for s in output_shape]
        if self.resolution_scaling_factor is not None:
            return [round(s * r) for s, r in zip(in_grid, self.resolution_scaling_factor)]
        return list(in_grid)

    def transform(self, x, output_shape=None):
        """Skip-connection transform (:383-398): identity unless the conv changes resolution, else the reference's `resample`
        (neuralop/layers/resample.py:7-71).  1-D / 2-D: spatial interpolation (linear / bicubic, align_corners=True) -- the very
        `F.interpolate` call the reference makes; it is the skip path of the FNO block, not the spectral-conv hot path.
        3-D and up: spectral resampling -- all modes both grids share are kept and synthesised on the new grid -- on this
        library's own transform kernels (identity contraction)."""
        in_shape = list(x.shape[2:])
        out_shape = [int(s) for s in self._output_grid(in_shape, output_shape)]
        if in_shape == out_shape:
            return x
        d = len(in_shape)
        if x.is_complex():
            raise NotImplementedError("SpectralConv.transform with a resolution change is not available for complex data "
                                      "(the reference's `resample` interpolates real tensors)")
        if d == 1:
            return torch.nn.functional.interpolate(x, size=out_shape[0], mode="linear", align_corners=True)
        if d == 2:
            return torch.nn.functional.interpolate(x, size=tuple(out_shape), mode="bicubic", align_corners=True)
        return _SpectralResample.apply(x.contiguous().float(), tuple(out_shape))

    @staticmethod
    def _kept_rows(factor, plan: Plan, j: int, axis: int = 0):
        """Rows of mode factor j the kept block uses (`weight[slices_w]`, :489); the factor itself when that is all of them."""
        lo, hi = plan.weight_row_range(j)
        if lo == 0 and hi == factor.shape[axis]:
            return factor if factor.is_contiguous() else factor.contiguous()
        return factor.narrow(axis, lo, hi - lo).contiguous()

    def _plan_kept(self, plan: Plan) -> Plan:
        if plan.plan_kept is None:
            plan.plan_kept = plan if plan.max_n_modes == plan.kept else \
                get_plan(plan.device, plan.grid, plan.out_grid, list(plan.kept), list(plan.kept), self.fft_norm)
        return plan.plan_kept

    def _forward_complex(self, x, output_shape):
        """complex_data=True (:439-441, :470-479, :531-538): C2C transforms, every weight form contracted as a reconstructed
        dense kept block (`weight[slices_w]`, differentiable: autograd scatters dweight back and reconstructs factor gradients)."""
        if x.dtype != torch.complex64:
            raise TypeError(f"SpectralConv(complex_data=True, full precision) expects complex64 input, got {x.dtype}")
        for name, prm in self.named_parameters():
            if prm.device != x.device:
                raise RuntimeError(f"SpectralConv parameter {name} lives on {prm.device} but the input on {x.device}")
        grid = list(x.shape[2:])
        out_grid = self._output_grid(grid, output_shape)
        plan = get_complex_plan(x.device, grid, out_grid, self.n_modes, self.max_n_modes, self.fft_norm)
        if x.shape[0] == 0:
            z = (x.sum() * 0).real
            for prm in self.parameters():
                z = z + (prm.real.sum() if prm.is_complex() else prm.sum()) * 0
            return x.new_zeros((0, self.out_channels, *out_grid)) + z
        w = self.weight.to_tensor()
        lead = 1 if self.separable else 2                                     # separable: one channel axis (:346-356)
        for j in range(self.order):
            if plan.w_start[j] != 0 or plan.kept[j] != w.shape[lead + j]:
                w = w.narrow(lead + j, plan.w_start[j], plan.kept[j])
        y = _SpectralConvComplex.apply(x.contiguous(), w.contiguous(), plan, self.separable)
        return y + self.bias if self.bias is not None else y                  # (:567-568; real bias on complex data)

    def _forward_separable(self, x, plan: Plan):
        """Depthwise spectral conv (`separable=True`, `_contract_dense_separable` :49-52): the weight (C, *max_n_modes) --
        reconstructed first if it is stored factorized -- is cut to the kept block (`weight[slices_w]`, :471-489) and
        multiplied mode by mode on the device."""
        w = self.weight.to_tensor()
        for j in range(self.order):
            lo, hi = plan.weight_row_range(j)
            if lo != 0 or hi != w.shape[1 + j]:
                w = w.narrow(1 + j, lo, hi - lo)
        return _SpectralConvSeparable.apply(x, w.contiguous(), self.bias, plan)

    def _forward_tucker(self, x, plan: Plan):
        """Factor-by-factor contraction (reference implementation="factorized", `_contract_tucker` :76-103)."""
        w = self.weight
        factors = list(w.factors)
        u_modes = [self._kept_rows(factors[2 + j], plan, j) for j in range(self.order)]
        return _SpectralConvTucker.apply(x, self.bias, plan, self._plan_kept(plan), w.core, factors[0].contiguous(),
                                         factors[1].contiguous(), *u_modes)

    def _forward_cp(self, x, plan: Plan):
        """Factor-by-factor contraction (reference implementation="factorized", `_contract_cp` :55-73)."""
        w = self.weight
        factors = list(w.factors)
        u_modes = [self._kept_rows(factors[2 + j], plan, j) for j in range(self.order)]
        fn = _SpectralConvCPCall if FACTORIZED_CHAINS_IN_C else _SpectralConvCP
        return fn.apply(x, self.bias, plan, w.weights.contiguous(), factors[0].contiguous(), factors[1].contiguous(), *u_modes)

    def _forward_tt(self, x, plan: Plan):
        """Core-by-core contraction (reference implementation="factorized", `_contract_tt` :106-127)."""
        factors = list(self.weight.factors)
        cores = [self._kept_rows(factors[2 + j], plan, j, axis=1) for j in range(self.order)]
        fn = _SpectralConvTTCall if FACTORIZED_CHAINS_IN_C else _SpectralConvTT
        return fn.apply(x, self.bias, plan, self._plan_kept(plan), factors[0].contiguous(), factors[1].contiguous(), *cores)

    def forward(self, x: torch.Tensor, output_shape: Optional[Tuple[int]] = None):
        if x.ndim != self.order + 2:
            raise ValueError(f"expected input of shape (batch, channels, {self.order} spatial dims), got {tuple(x.shape)}")
        if x.shape[1] != self.in_channels:
            raise ValueError(f"expected {self.in_channels} input channels, got {x.shape[1]}")
        if not x.is_cuda:
            raise RuntimeError("neuraloperator_b200.SpectralConv has no CPU path: move the module and input to a B200")
        if self.complex_data:
            return self._forward_complex(x, output_shape)
        if x.dtype not in _GRID_FLAGS:
            raise TypeError(f"SpectralConv (real data) expects float32, float16 or bfloat16 input, got {x.dtype}")
        if torch.is_autocast_enabled("cuda"):
            # the result must not depend on autocast: a 16-bit x runs the 16-bit storage path, and nothing in between (a factorized
            # weight's reconstruction, say) may be recast
            with torch.autocast("cuda", enabled=False):
                return self._forward_real(x, output_shape)
        return self._forward_real(x, output_shape)

    def _forward_real(self, x: torch.Tensor, output_shape):
        """Real data in float32, float16 or bfloat16 (the lifting layer's output under torch.autocast): y is float32 whatever the
        input dtype, as the reference's complex64 output spectrum makes it (:456-462); dx comes back in x's dtype."""
        # the kernels read the parameters through raw pointers: complex64 / float32 on x's device, nothing else
        for name, prm in self.named_parameters():
            want = torch.float32 if name == "bias" else torch.complex64
            if prm.dtype != want:
                raise TypeError(f"SpectralConv parameter {name} is {prm.dtype}; the kernels need {want} "
                                "(module.double() / .half() are not supported: full precision, spectral_convolution.py:459-462)")
            if prm.device != x.device:
                raise RuntimeError(f"SpectralConv parameter {name} lives on {prm.device} but the input on {x.device}")
        grid = list(x.shape[2:])
        out_grid = self._output_grid(grid, output_shape)
        reduced = self.fno_block_precision != "full"
        if reduced and x.dtype != torch.float32:
            x = x.float()       # the reduced path rounds where the reference casts; autograd rounds dx back to x's dtype
        plan = get_plan(x.device, grid, out_grid, self.n_modes, self.max_n_modes, self.fft_norm, flags=_GRID_FLAGS[x.dtype])
        if x.shape[0] == 0:
            # empty batch (torch.fft accepts it in the reference): nothing to launch; stay connected to the autograd graph
            z = x.sum() * 0
            for prm in self.parameters():
                z = z + (prm.real.sum() if prm.is_complex() else prm.sum()) * 0
            return x.new_zeros((0, self.out_channels, *out_grid), dtype=torch.float32) + z
        x = x.contiguous()
        if reduced:
            w = self.weight.to_tensor()
            return _SpectralConvDenseReduced.apply(x, w if w.is_contiguous() else w.contiguous(), self.bias, plan,
                                                   self.fno_block_precision == "half")
        if self.separable:
            return self._forward_separable(x, plan)
        if self.implementation == "factorized" and getattr(self.weight, "kind", "") == "tucker":
            return self._forward_tucker(x, plan)
        if self.implementation == "factorized" and getattr(self.weight, "kind", "") == "cp":
            return self._forward_cp(x, plan)
        if self.implementation == "factorized" and getattr(self.weight, "kind", "") == "tt":
            return self._forward_tt(x, plan)
        # dense weight goes straight to the kernels; other factorized forms are reconstructed first (differentiably)
        w = self.weight.to_tensor()
        if not w.is_contiguous():
            w = w.contiguous()
        return spectral_conv_dense(x, w, self.bias, plan, self.gradient_reducer if self.factorization is None else None)
