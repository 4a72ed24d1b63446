"""GPU tier of the 16-bit image storage (-m gpu): float16 / bfloat16 x, float32 y, dx in x's dtype.

The contract is stated against the float32 path on the widened input, which the 16-bit path must reproduce BIT FOR BIT: every
16-bit value is exact in fp32, and the 16-bit plan runs the very same kernels on an fp32 copy of x.  So y, dweight and dbias are
compared with torch.equal, and dx with torch.equal against the fp32 dx cast to x's dtype.  The shapes reach every kernel family:
fused 2-D and 3-D tensor-core transforms, the last-dim ("rows") tensor-core kernels, the generic SIMT chain."""
import math

import pytest
import torch

import neuraloperator_b200 as nb
from neuraloperator_b200 import spectral_conv as sc
from oracle import spectral_conv_oracle as O

pytestmark = pytest.mark.gpu
DTYPES = [torch.float16, torch.bfloat16]


def rel_err(a, ref):
    a, ref = a.detach().float().cpu(), ref.detach().float().cpu()
    return (a - ref).abs().max().item() / max(ref.abs().max().item(), 1e-20)


def _params(conv):
    return [p for _, p in sorted(conv.named_parameters())]


def _run(conv, x, gy, **kw):
    conv.zero_grad(set_to_none=True)
    x = x.detach().clone().requires_grad_(True)
    y = conv(x, **kw)
    y.backward(gy)
    torch.cuda.synchronize()
    return y.detach(), x.grad, [p.grad.clone() for p in _params(conv)]


def _assert_half_equals_float(conv, x16, gy, **kw):
    y16, dx16, g16 = _run(conv, x16, gy, **kw)
    y32, dx32, g32 = _run(conv, x16.float(), gy, **kw)
    assert y16.dtype == torch.float32 and torch.equal(y16, y32), "y"
    assert dx16.dtype == x16.dtype and torch.equal(dx16, dx32.to(x16.dtype)), "dx"
    for i, (a, b) in enumerate(zip(g16, g32)):
        assert torch.equal(a, b), f"parameter gradient {i}"
    return y16, dx16, dx32


def _inputs(dev, B, Ci, Co, grid, dtype, seed=0, out_grid=None):
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn(B, Ci, *grid, device=dev, generator=g).to(dtype)
    gy = torch.randn(B, Co, *(out_grid or grid), device=dev, generator=g)
    return x, gy


SHAPES = [
    (32, 64, (128, 128), (32, 32)),     # fused 2-D (the headline shape)
    (4, 8, (64, 64), (32, 32)),
    (2, 8, (64, 64, 64), (16, 16, 16)),  # fused slices + leading-dim table kernel
    (16, 32, (1024,), (16,)),            # rows kernels
    (2, 16, (256, 256), (64, 64)),
    (2, 6, (30, 20), (12, 9)),           # generic
    (2, 3, (6, 6, 6, 6), (4, 4, 4, 4)),
]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B,C,grid,modes", SHAPES)
def test_dense_half_io_is_the_float_path(cuda_device, dtype, B, C, grid, modes):
    torch.manual_seed(1)
    conv = nb.SpectralConv(C, C, modes).to(cuda_device)
    x, gy = _inputs(cuda_device, B, C, C, grid, dtype)
    _assert_half_equals_float(conv, x, gy)


@pytest.mark.parametrize("dtype", DTYPES)
def test_generic_chain_and_misaligned_view(cuda_device, dtype):
    torch.manual_seed(2)
    B, C, grid, modes = 4, 8, (64, 64), (32, 32)
    conv = nb.SpectralConv(C, C, modes).to(cuda_device)
    x, gy = _inputs(cuda_device, B, C, C, grid, dtype)
    # a 16-byte misaligned (2-byte offset) contiguous view
    buf = torch.empty(x.numel() + 1, dtype=dtype, device=cuda_device)
    xv = buf[1:].view_as(x)
    xv.copy_(x)
    assert xv.data_ptr() % 16 != 0
    _assert_half_equals_float(conv, xv, gy)
    # the same shape with the tensor-core path switched off
    for dt in (dtype, torch.float32):
        sc.get_plan(cuda_device, grid, grid, conv.n_modes, conv.max_n_modes, "forward", flags=sc._GRID_FLAGS[dt]).set_fast_path(False)
    try:
        _assert_half_equals_float(conv, x, gy)
    finally:
        for dt in (dtype, torch.float32):
            sc.get_plan(cuda_device, grid, grid, conv.n_modes, conv.max_n_modes, "forward", flags=sc._GRID_FLAGS[dt]).set_fast_path(True)


@pytest.mark.parametrize("dtype", DTYPES)
def test_headline_shape_against_oracle(cuda_device, dtype):
    B, C, grid, modes = 32, 64, (128, 128), (32, 32)
    x, w, bias, gy = O.make_inputs(B, C, C, grid, modes, seed=3)
    x16 = x.to(dtype)
    y_ref, dx_ref, dws_ref, db_ref = O.spectral_conv_fwd_bwd(x16.float(), w, bias, gy, modes)
    conv = nb.SpectralConv(C, C, modes).to(cuda_device)
    with torch.no_grad():
        conv.weight.tensor.copy_(w.tensor.to(cuda_device))
        conv.bias.copy_(bias.to(cuda_device))
    xd = x16.to(cuda_device).requires_grad_(True)
    y = conv(xd)
    y.backward(gy.to(cuda_device))
    assert rel_err(y, y_ref) < 1e-4
    assert rel_err(xd.grad, dx_ref.to(dtype)) < 1e-2       # dx itself is rounded to 16 bits
    assert rel_err(conv.weight.tensor.grad, dws_ref[0]) < 1e-4
    assert rel_err(conv.bias.grad, db_ref) < 1e-4


CHAINS = [
    ("tucker factorized", dict(factorization="tucker", rank=0.5, implementation="factorized"), {}),
    ("tucker reconstructed", dict(factorization="tucker", rank=0.5, implementation="reconstructed"), {}),
    ("cp python", dict(factorization="cp", rank=0.5, implementation="factorized"), {"c": False}),
    ("cp c", dict(factorization="cp", rank=0.5, implementation="factorized"), {"c": True}),
    ("tt python", dict(factorization="tt", rank=0.5, implementation="factorized"), {"c": False}),
    ("tt c", dict(factorization="tt", rank=0.5, implementation="factorized"), {"c": True}),
    ("separable", dict(separable=True), {}),
    ("max_n_modes", dict(max_n_modes=(24, 20)), {}),
    ("resolution scaling", dict(resolution_scaling_factor=2), {}),
    ("output_shape", {}, {"output_shape": (40, 24)}),
]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name,ctor,extra", CHAINS, ids=[c[0] for c in CHAINS])
def test_every_chain_is_the_float_path(cuda_device, monkeypatch, dtype, name, ctor, extra):
    torch.manual_seed(4)
    if "c" in extra:
        monkeypatch.setattr(sc, "FACTORIZED_CHAINS_IN_C", extra["c"])
    B, C, grid, modes = 4, 8, (64, 48), (16, 12)
    conv = nb.SpectralConv(C, C, modes, **ctor).to(cuda_device)
    kw = {"output_shape": extra["output_shape"]} if "output_shape" in extra else {}
    out = list(extra.get("output_shape", [2 * g for g in grid] if "resolution_scaling_factor" in ctor else grid))
    x, gy = _inputs(cuda_device, B, C, C, grid, dtype, seed=5, out_grid=out)
    _assert_half_equals_float(conv, x, gy, **kw)


@pytest.mark.parametrize("dtype", DTYPES)
def test_n_modes_changed_at_run_time(cuda_device, dtype):
    torch.manual_seed(6)
    conv = nb.SpectralConv(8, 8, (24, 24)).to(cuda_device)
    x, gy = _inputs(cuda_device, 2, 8, 8, (64, 64), dtype)
    _assert_half_equals_float(conv, x, gy)
    conv.n_modes = (12, 16)
    _assert_half_equals_float(conv, x, gy)


@pytest.mark.parametrize("precision", ["mixed", "half"])
@pytest.mark.parametrize("dtype", DTYPES)
def test_reduced_precision_accepts_16_bit_x(cuda_device, dtype, precision):
    B, C, grid, modes = 2, 8, (128, 128), (32, 32)
    x, w, bias, gy = O.make_inputs(B, C, C, grid, modes, seed=4)
    x16 = x.to(dtype)
    xr = x16.float().requires_grad_(True)
    wt = w.tensor.clone().requires_grad_(True)
    y_ref = O.spectral_conv_forward_reduced(xr, O.Weight("dense", tensor=wt), bias.clone(), modes, precision)
    y_ref.backward(gy)
    conv = nb.SpectralConv(C, C, modes, fno_block_precision=precision).to(cuda_device)
    with torch.no_grad():
        conv.weight.tensor.copy_(w.tensor.to(cuda_device))
        conv.bias.copy_(bias.to(cuda_device))
    xd = x16.to(cuda_device).requires_grad_(True)
    y = conv(xd)
    y.backward(gy.to(cuda_device))
    assert y.dtype == torch.float32 and xd.grad.dtype == dtype
    assert rel_err(y, y_ref) < 4e-3
    assert rel_err(xd.grad, xr.grad) < 2e-3 + (1e-2 if dtype == torch.bfloat16 else 1e-3)
    assert rel_err(conv.weight.tensor.grad, wt.grad) < 2e-3


@pytest.mark.parametrize("dtype", [torch.float32, *DTYPES])
@pytest.mark.parametrize("autocast_dtype", DTYPES)
def test_autocast_does_not_reach_inside(cuda_device, dtype, autocast_dtype):
    torch.manual_seed(7)
    for ctor in ({}, dict(factorization="tucker", rank=0.5, implementation="reconstructed")):
        conv = nb.SpectralConv(8, 8, (16, 16), **ctor).to(cuda_device)
        x, gy = _inputs(cuda_device, 4, 8, 8, (64, 64), dtype)
        y0, dx0, g0 = _run(conv, x, gy)
        with torch.autocast("cuda", dtype=autocast_dtype):
            conv.zero_grad(set_to_none=True)
            xa = x.detach().clone().requires_grad_(True)
            ya = conv(xa)
        ya.backward(gy)
        assert ya.dtype == torch.float32 and torch.equal(ya.detach(), y0)
        assert xa.grad.dtype == dtype and torch.equal(xa.grad, dx0)
        for a, b in zip([p.grad for p in _params(conv)], g0):
            assert torch.equal(a, b)


def test_against_the_reference_fp16_autocast_op_sequence(cuda_device):
    """The reference under float16 autocast: cuFFT half rfftn, the complex-half contraction (einsum_complexhalf: real and imaginary
    parts as fp16 real products), a complex64 output spectrum and a float32 inverse.  Agreement: fp16 noise."""
    torch.manual_seed(8)
    B, C, grid, modes = 4, 16, (64, 64), (16, 16)
    conv = nb.SpectralConv(C, C, modes).to(cuda_device)
    x, gy = _inputs(cuda_device, B, C, C, grid, torch.float16)
    W = conv.weight.tensor.detach().clone().requires_grad_(True)
    bias = conv.bias.detach().clone()

    def reference(xin, w):
        kx, ky = modes[0], modes[1] // 2 + 1
        xf = torch.fft.rfftn(xin, dim=(-2, -1), norm="forward")            # complex32
        xf = torch.fft.fftshift(xf, dim=-2)
        c = grid[0] // 2
        xk = xf[..., c - kx // 2:c + kx // 2, :ky]
        xr, xi = xk.real, xk.imag                                            # fp16
        wr, wi = w.real.half(), w.imag.half()
        yr = torch.einsum("bixy,ioxy->boxy", xr, wr) - torch.einsum("bixy,ioxy->boxy", xi, wi)
        yi = torch.einsum("bixy,ioxy->boxy", xr, wi) + torch.einsum("bixy,ioxy->boxy", xi, wr)
        out = torch.zeros(B, C, grid[0], grid[1] // 2 + 1, dtype=torch.complex64, device=xin.device)
        out[..., c - kx // 2:c + kx // 2, :ky] = torch.complex(yr.float(), yi.float())
        out = torch.fft.ifftshift(out, dim=-2)
        return torch.fft.irfftn(out, s=grid, dim=(-2, -1), norm="forward") + bias

    xr = x.detach().clone().requires_grad_(True)
    y_ref = reference(xr, W)
    y_ref.backward(gy)
    xo = x.detach().clone().requires_grad_(True)
    y = conv(xo)
    y.backward(gy)
    assert y.dtype == torch.float32 and xo.grad.dtype == torch.float16
    assert rel_err(y, y_ref) < 1e-2
    assert rel_err(xo.grad, xr.grad) < 2e-2


def test_dx_overflow_matches_the_cast(cuda_device):
    """float16 only: a float32 dx beyond bfloat16's range would be (nearly) beyond float32's own."""
    torch.manual_seed(9)
    conv = nb.SpectralConv(8, 8, (16, 16)).to(cuda_device)
    x, gy = _inputs(cuda_device, 2, 8, 8, (64, 64), torch.float16)
    _, _, dx32 = _assert_half_equals_float(conv, x, gy)
    scale = 4 * torch.finfo(torch.float16).max / dx32.abs().max().item()      # the largest |dx| lands near 4x the fp16 maximum
    _, dx16, dx32 = _assert_half_equals_float(conv, x, gy * scale)
    assert torch.isinf(dx16).any() and torch.isfinite(dx16).any() and torch.isfinite(dx32).all()


def test_dtypes_rejected_and_empty_batch(cuda_device):
    conv = nb.SpectralConv(4, 6, (8, 8)).to(cuda_device)
    for dt in (torch.float64, torch.int32):
        with pytest.raises(TypeError, match="float32, float16 or bfloat16"):
            conv(torch.zeros(2, 4, 16, 16, device=cuda_device, dtype=dt))
    cplx = nb.SpectralConv(4, 6, (8, 8), complex_data=True).to(cuda_device)
    for dt in DTYPES:
        with pytest.raises(TypeError, match="complex64"):
            cplx(torch.zeros(2, 4, 16, 16, device=cuda_device, dtype=dt))
        x = torch.zeros(0, 4, 16, 16, device=cuda_device, dtype=dt, requires_grad=True)
        y = conv(x)
        assert y.dtype == torch.float32 and y.shape == (0, 6, 16, 16) and y.requires_grad
        y.sum().backward()
        assert x.grad is not None and x.grad.dtype == dt


def test_amp_training_loop(cuda_device):
    """Conv1d lifting, the spectral conv with a Conv1d skip, GELU, Conv1d projection; torch.autocast(float16), loss scaling, Adam.
    torch.amp.GradScaler's unscale kernel has no complex implementation (the spectral weight is complex64), so the loop applies the
    scaler's rule by hand: scaled backward, unscale, skip the step and halve the scale on a non-finite gradient."""
    torch.manual_seed(10)
    dev = cuda_device
    C, N, modes = 16, 128, 16

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.lift = torch.nn.Conv1d(1, C, 1)
            self.conv = nb.SpectralConv(C, C, (modes,))
            self.skip = torch.nn.Conv1d(C, C, 1)
            self.proj = torch.nn.Conv1d(C, 1, 1)

        def forward(self, a):
            h = self.lift(a)
            h = torch.nn.functional.gelu(self.conv(h) + self.skip(h))
            return self.proj(h)

    net = Net().to(dev)
    opt = torch.optim.Adam(net.parameters(), lr=3e-3)
    scale = 2.0 ** 12
    t = torch.linspace(0, 2 * math.pi, N, device=dev)
    a = torch.sin(t[None, None] * torch.randint(1, 5, (32, 1, 1), device=dev).float())
    target = torch.roll(a, 7, dims=-1) * 0.5
    losses = []
    seen_half = []
    net.conv.register_forward_pre_hook(lambda m, args: seen_half.append(args[0].dtype))
    for _ in range(100):
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.float16):
            loss = torch.nn.functional.mse_loss(net(a).float(), target)
        (loss * scale).backward()
        grads = [p.grad for p in net.parameters()]
        for g in grads:
            g.div_(scale)
        if all(bool(torch.isfinite(torch.view_as_real(g) if g.is_complex() else g).all()) for g in grads):
            opt.step()
        else:
            scale /= 2
        losses.append(loss.item())
    assert seen_half[0] == torch.float16
    assert all(math.isfinite(v) for v in losses)
    assert losses[-1] < 0.5 * losses[0], losses[::10]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B,C,grid,modes", [SHAPES[0]])
def test_fused_kernels_read_and_write_16_bit_directly(cuda_device, dtype, B, C, grid, modes):
    """On the fused tensor-core shapes the 16-bit step launches exactly the kernels of the float32 step: no conversion pass and no
    fall-back chain (either would add launches)."""
    from neuraloperator_b200 import _lib
    torch.manual_seed(11)
    conv = nb.SpectralConv(C, C, modes).to(cuda_device)
    x, gy = _inputs(cuda_device, B, C, C, grid, dtype)
    counts = {}
    for dt in (torch.float32, dtype):
        _run(conv, x.to(dt), gy)                       # plans and tensor maps built
        before = _lib.launch_count()
        _run(conv, x.to(dt), gy)
        counts[dt] = _lib.launch_count() - before
    assert counts[dtype] == counts[torch.float32], counts
    assert sc.get_plan(cuda_device, grid, grid, conv.n_modes, conv.max_n_modes, "forward", flags=sc._GRID_FLAGS[dtype]).uses_fast_path() & 9 == 9
