"""The oracle against what the UNMODIFIED reference module returned for the same inputs on CPU, stored by
oracle/make_golden_reference_checks.py (inputs and weights are redrawn here from the same seeds).  Run live, the two agree bit for
bit; against stored results they are held to a few float32 ulps of the largest magnitude, the rounding by which CPU FFT / BLAS
kernels may differ between machines."""
import pytest
import torch

from conftest import reference_checks, stored_rel_err
from oracle import spectral_conv_oracle as O
from oracle.make_golden_reference_checks import conv_case_inputs

ULPS = 4e-7

BIT_EXACT_CASES = [
    ((64,), (16,), {}),
    ((32, 32), (16, 16), {}),
    ((16, 16, 16), (8, 8, 8), {}),
    ((9, 11), (5, 4), {}),
    ((16, 12), (5, 4), {"max_n_modes": (8, 6)}),
    ((12, 12), (10, 8), {"resolution_scaling_factor": 2}),
]
RESAMPLE_CASES = [((2, 3, 16), (24,)), ((2, 3, 12, 10), (18, 20)), ((1, 2, 8, 8, 8), (12, 12, 12)),
                  ((1, 2, 12, 8, 10), (8, 8, 6)), ((1, 2, 8, 6, 10), (8, 12, 16))]
COMPLEX_CASES = [
    ((16,), (6,), {}), ((16, 12), (8, 6), {}), ((9, 11), (4, 5), {}), ((8, 6, 10), (4, 4, 6), {}), ((12, 12), (16, 16), {}),
    ((16, 12), (6, 4), {"max_n_modes": (8, 6)}), ((16, 12), (5, 3), {"max_n_modes": (8, 6)}),
    ((12, 12), (10, 8), {"resolution_scaling_factor": 2}), ((12, 12), (10, 8), {"resolution_scaling_factor": 0.5}),
    ((12, 12), (10, 8), {"fft_norm": "ortho"}),
    ((16, 12), (8, 6), {"separable": True}), ((16,), (6,), {"separable": True}), ((8, 6, 10), (4, 4, 6), {"separable": True}),
    ((16, 12), (5, 3), {"separable": True, "max_n_modes": (8, 6)}),
]


def _assert_stored(store, key, results):
    for name, got in results:
        assert stored_rel_err(store, f"{key}__{name}", got) <= ULPS, name


@pytest.mark.parametrize("grid,modes,kw", BIT_EXACT_CASES)
def test_live_reference_bit_exact(grid, modes, kw):
    store, meta = reference_checks()
    i = BIT_EXACT_CASES.index((grid, modes, kw))
    case = meta[f"conv{i}"]
    x, w, bias, gen = conv_case_inputs((2, 4, *grid), torch.float32, case["w_shape"], case["b_shape"], torch.float32, 7 + i)
    g = torch.randn(*store[f"conv{i}__y"][0], generator=gen)
    okw = {}
    if "max_n_modes" in kw:
        okw["max_n_modes"] = case["max_n_modes"]
    if "resolution_scaling_factor" in kw:
        okw["resolution_scaling_factor"] = [float(kw["resolution_scaling_factor"])] * len(grid)
    y2, dx2, dws, db = O.spectral_conv_fwd_bwd(x, O.Weight("dense", tensor=w), bias, g, modes, **okw)
    _assert_stored(store, f"conv{i}", [("y", y2), ("dx", dx2), ("dw", dws[0]), ("dw_modes", dws[0].sum(dim=(0, 1))), ("db", db)])


def test_reference_fno_blocks_accept_the_plugin_class():
    """The constructor calls the reference `FNOBlocks(conv_module=neuraloperator_b200.SpectralConv)` makes (fno_block.py:210-240,
    stored) construct this package's class, and the host-side attribute traffic of its n_modes setter (:460-464) works. No forward
    here: that needs the GPU."""
    import neuraloperator_b200 as nb
    _, meta = reference_checks()
    calls = meta["conv_module_calls"]
    convs = [nb.SpectralConv(*c["args"], **c["kwargs"]) for c in calls["default"]]      # FNOBlocks(8, 8, (12, 12), n_layers=2)
    assert len(convs) == 2
    assert convs[0].n_modes == [12, 7]
    for conv in convs:
        conv.n_modes = (8, 8)
    assert convs[1].n_modes == [8, 5]
    tf = [nb.SpectralConv(*c["args"], **c["kwargs"]) for c in calls["tucker"]]   # ... n_layers=1, factorization="tucker", rank=0.5
    assert len(tf) == 1 and tf[0].weight.name.lower().endswith("tucker")


@pytest.mark.parametrize("shape,out", RESAMPLE_CASES)
def test_resample_restatement_equals_the_reference(shape, out):
    """`SpectralConv.transform` is tested on the GPU against oracle.resample_restated; here that restatement is pinned to what the
    unmodified reference function (neuralop/layers/resample.py) returned."""
    store, _ = reference_checks()
    torch.manual_seed(0)
    x = torch.randn(*shape)
    assert stored_rel_err(store, f"resample{RESAMPLE_CASES.index((shape, out))}", O.resample_restated(x, out)) <= ULPS


@pytest.mark.parametrize("grid,modes,kw", COMPLEX_CASES)
def test_live_reference_bit_exact_complex_data(grid, modes, kw):
    """complex_data=True: forward and every gradient of the oracle restatement equal the reference's."""
    store, meta = reference_checks()
    i = COMPLEX_CASES.index((grid, modes, kw))
    case = meta[f"cconv{i}"]
    x, w, b, gen = conv_case_inputs((2, 3, *grid), torch.cfloat, case["w_shape"], case["b_shape"],
                                    torch.cfloat if case["b_complex"] else torch.float32, 11 + i)
    g = torch.randn(*store[f"cconv{i}__y"][0], generator=gen, dtype=torch.cfloat)
    okw = {"max_n_modes": case["max_n_modes"], "fft_norm": kw.get("fft_norm", "forward"), "separable": bool(kw.get("separable"))}
    if "resolution_scaling_factor" in kw:
        okw["resolution_scaling_factor"] = [float(kw["resolution_scaling_factor"])] * len(grid)
    x2, w2, b2 = (t.requires_grad_(True) for t in (x, w, b))
    y2 = O.spectral_conv_forward_complex(x2, w2, b2, modes, **okw)
    y2.backward(g)
    _assert_stored(store, f"cconv{i}", [("y", y2), ("dx", x2.grad), ("dw", w2.grad), ("dw_modes", w2.grad.sum(dim=(0, 1))),
                                        ("db", b2.grad)])
