"""`neuraloperator_b200.FNOBlocks` end to end WITHOUT a GPU, against golden vectors minted from the unmodified reference FNOBlocks.

Two things are replaced: (1) the four layer-epilogue kernels run through their host checks (`sc_hostcheck_*`: the kernels' own tile
functions executed thread by thread on CPU buffers), (2) the spectral convolution inside the block is the CPU oracle (the CUDA conv
has its own GPU tiers).  Everything else is the product code: which skip becomes which operand of the fused op, the activation per
layer index, pre / post-activation order, the resampling of the skips, the autograd wiring of every gradient, state-dict names."""
import contextlib

import pytest
import torch

import neuraloperator_b200 as nb
from neuraloperator_b200 import _lib, fno_block as fb
from conftest import block_ctor_kwargs, block_golden_index, load_block_golden, reference_checks, stored_rel_err
from oracle import spectral_conv_oracle as O
from oracle.make_golden_reference_checks import parameter_specs, seeded_tensors

CASES = sorted(block_golden_index().keys())


class _HostLib:
    """The layer entry points of the C ABI, served by the library's own host checks (same arguments minus the stream)."""

    def __init__(self, lib):
        self._lib = lib
        self.calls = []

    def sc_channel_mix(self, *a):
        self.calls.append("sc_channel_mix")
        return self._lib.sc_hostcheck_channel_mix(*a[:-1])

    def sc_channel_mix_act_backward(self, *a):
        self.calls.append("sc_channel_mix_act_backward")
        return self._lib.sc_hostcheck_channel_mix_act_backward(*a[:-1])

    def sc_channel_mix_weight_grad(self, *a):
        self.calls.append("sc_channel_mix_weight_grad")
        return self._lib.sc_hostcheck_channel_mix_weight_grad(*a[:-1])

    def sc_pointwise(self, *a):
        self.calls.append("sc_pointwise")
        return self._lib.sc_hostcheck_pointwise(*a[:-1])

    def sc_last_error(self):
        return self._lib.sc_last_error()


def _oracle_conv_forward(self, x, output_shape=None):
    """SpectralConv.forward served by the CPU oracle (differentiable through torch.fft), from the module's own parameters."""
    kind = getattr(self.weight, "kind", "dense")
    if self.complex_data:
        return O.spectral_conv_forward_complex(x, self.weight.to_tensor(), self.bias, list(self.n_modes), max_n_modes=list(self.max_n_modes),
                                               output_shape=output_shape, fft_norm=self.fft_norm)
    if kind == "dense":
        w = O.Weight("dense", tensor=self.weight.tensor)
    elif kind == "tucker":
        w = O.Weight("tucker", core=self.weight.core, factors=list(self.weight.factors))
    elif kind == "cp":
        w = O.Weight("cp", weights=self.weight.weights, factors=list(self.weight.factors))
    else:
        w = O.Weight("tt", factors=list(self.weight.factors))
    user_modes = list(self.n_modes)
    user_modes[-1] = (user_modes[-1] - 1) * 2            # the oracle takes USER modes and halves the last one itself
    return O.spectral_conv_forward(x, w, self.bias, user_modes, max_n_modes=list(self.max_n_modes), output_shape=output_shape,
                                   resolution_scaling_factor=self.resolution_scaling_factor, fft_norm=self.fft_norm)


def _oracle_transform(self, x, output_shape=None):
    in_shape = list(x.shape[2:])
    out_shape = [int(s) for s in self._output_grid(in_shape, output_shape)]
    return x if in_shape == out_shape else O.resample_restated(x, out_shape)


@pytest.fixture
def host(monkeypatch):
    real = _lib.load()
    h = _HostLib(real)
    monkeypatch.setattr(fb._lib, "load", lambda: h)
    monkeypatch.setattr(fb._lib, "check", lambda rc, what: (_ for _ in ()).throw(RuntimeError(f"{what}: {real.sc_last_error()}")) if rc else None)
    monkeypatch.setattr(fb, "_require_device_tensor", lambda t, what: None)
    monkeypatch.setattr(fb, "_require_complex_input", lambda x: None)
    monkeypatch.setattr(fb, "_stream_ptr", lambda dev: None)
    monkeypatch.setattr(torch.cuda, "device", lambda dev: contextlib.nullcontext())
    monkeypatch.setattr(nb.SpectralConv, "forward", _oracle_conv_forward)
    monkeypatch.setattr(nb.SpectralConv, "transform", _oracle_transform)
    return h


def rel_err(a, ref):
    assert a.shape == ref.shape, (a.shape, ref.shape)
    return (a.detach() - ref).abs().max().item() / max(ref.abs().max().item(), 1e-20)


def grad_err(got, ref, all_refs):
    """rel_err of one parameter gradient -- unless the reference gradient vanishes identically in exact arithmetic (the conv bias in
    front of an instance / group norm: the normalisation removes per-channel constants): then both sides are rounding noise, and what
    is checked is that ours is as negligible as the reference's, on the scale of the case's largest gradient."""
    scale = max(float(g.abs().max()) for g in all_refs.values())
    if float(ref.abs().max()) < 1e-5 * scale:
        assert got.shape == ref.shape
        return float(got.detach().abs().max()) / scale
    return rel_err(got, ref)


def _our_name(pname):
    return pname.replace("weight.factors.", "weight.factors.factor_")


def _build(meta):
    ctor = block_ctor_kwargs(meta)
    return nb.FNOBlocks(meta["in_channels"], meta["out_channels"], tuple(meta["n_modes"]), n_layers=meta["n_layers"], **ctor)


@pytest.mark.parametrize("name", CASES)
def test_block_module_matches_reference_golden(host, name):
    meta, io, params, grads = load_block_golden(name)
    blk = _build(meta)
    ours = dict(blk.named_parameters())
    assert sorted(_our_name(p) for p in meta["params"]) == sorted(ours.keys())          # same parameter set and names as the reference block
    with torch.no_grad():
        for pname, val in params.items():
            assert ours[_our_name(pname)].shape == val.shape, pname
            ours[_our_name(pname)].copy_(val)
    if "ada_in_embedding" in io:
        blk.set_ada_in_embeddings(io["ada_in_embedding"])
    x = io["x"].clone().requires_grad_(True)
    kw = {k: tuple(v) for k, v in meta["forward"].items()}
    y = blk(x, meta["index"], **kw)
    assert y.dtype == (torch.complex64 if meta["ctor"].get("complex_data") else torch.float32) and list(y.shape[2:]) == meta["out_grid"]
    y.backward(io["gy"])
    for bname, buf in blk.named_buffers():                       # batch norm: running statistics after this (training-mode) forward
        want = io["b__" + bname.replace(".", "__")]
        assert rel_err(buf.float(), want.float()) < 2e-5, bname
    assert rel_err(y, io["y"]) < 2e-5, "y"
    assert rel_err(x.grad, io["dx"]) < 2e-5, "dx"
    for pname in meta["params"]:
        p = ours[_our_name(pname)]
        if pname in meta["touched"]:
            assert p.grad is not None, pname
            assert grad_err(p.grad, grads[pname], grads) < 3e-5, pname
        else:
            assert p.grad is None, pname
    assert "sc_channel_mix" in host.calls                                                    # the fused kernels' code did the work


def test_launch_counts_of_the_default_layer(host):
    """Default layer (linear skip, ChannelMLP + soft gating), no resolution change: f1 is ONE mixing launch, f2 two; backward is
    3 activation-backward + 3 input-gradient + 3 weight-gradient launches."""
    meta, io, params, _ = load_block_golden("block_d2_default_mid")
    blk = _build(meta)
    x = io["x"].clone().requires_grad_(True)
    y = blk(x, 0)
    assert host.calls == ["sc_channel_mix"] * 3
    host.calls.clear()
    y.backward(io["gy"])
    assert sorted(host.calls) == sorted(["sc_channel_mix_act_backward"] * 3 + ["sc_channel_mix"] * 3 + ["sc_channel_mix_weight_grad"] * 3)
    host.calls.clear()
    with torch.no_grad():
        blk(io["x"], 1)                                 # last layer: identity activation, still three launches
    assert host.calls == ["sc_channel_mix"] * 3


def test_state_dict_round_trip_with_the_reference(host):
    """A reference FNOBlocks state dict loads into ours (and back) by name: same keys, shapes and dtypes, and with the same parameters the
    same outputs as the reference returned (stored by oracle/make_golden_reference_checks.py)."""
    store, checks = reference_checks()
    ours = nb.FNOBlocks(6, 6, (8, 8), n_layers=3, implementation="reconstructed")
    assert {k: [list(v.shape), str(v.dtype)] for k, v in ours.state_dict().items()} == checks["state_dict"]
    ours.load_state_dict(seeded_tensors(parameter_specs(ours), 4), strict=False)
    x = torch.randn(2, 6, 16, 16, generator=torch.Generator().manual_seed(5))
    for i in range(3):
        assert stored_rel_err(store, f"sd_layer{i}", ours(x, i)) < 2e-5
    # the whole stack, layer after layer, as FNO.forward applies it (fno.py:376-379)
    a = x
    for i in range(3):
        a = ours(a, i)
    assert stored_rel_err(store, "sd_stack", a) < 5e-5


def test_unsupported_configurations_raise():
    for kw in (dict(complex_data=True, norm="group_norm"), dict(complex_data=True, resolution_scaling_factor=2),
               dict(conv_bias_kernel=3, complex_data=True), dict(non_linearity=torch.nn.functional.elu)):
        with pytest.raises(NotImplementedError):
            nb.FNOBlocks(4, 4, (4, 4), **kw)
    with pytest.raises(ValueError):
        nb.FNOBlocks(4, 4, (4, 4), fno_skip="bogus")
    with pytest.raises(ValueError):
        nb.FNOBlocks(4, 4, (4, 4), norm="bogus")
    with pytest.raises(ValueError):
        nb.FNOBlocks(4, 4, (4, 4), conv_bias_kernel=3, fno_skip="soft-gating")
    with pytest.raises(ValueError):
        nb.FNOBlocks(4, 6, (4, 4))                       # soft gating needs in == out channels (skip_connections.py:74-79)


def test_dropout_eval_identity_and_training_masks_like_the_reference(host):
    meta, io, params, _ = load_block_golden("block_d2_default_mid")
    plain, dropped = _build(meta), nb.FNOBlocks(meta["in_channels"], meta["out_channels"], tuple(meta["n_modes"]), n_layers=2,
                                                 implementation="reconstructed", channel_mlp_dropout=0.3)
    dropped.load_state_dict(plain.state_dict())
    dropped.eval()
    with torch.no_grad():
        assert rel_err(dropped(io["x"], 0), plain(io["x"], 0)) == 0.0            # eval mode: the identity
    dropped.train()
    torch.manual_seed(1)
    a = dropped(io["x"], 0)
    torch.manual_seed(2)
    b = dropped(io["x"], 0)
    assert rel_err(a, b.detach()) > 1e-2                                          # training mode: a different mask per draw
    # same generator state, same masks: F.dropout(ones) draws what the reference's F.dropout(x) draws (channel_mlp.py:110-111); the
    # reference's results for these parameters are stored by oracle/make_golden_reference_checks.py
    store, _ = reference_checks()
    dropped.load_state_dict(seeded_tensors(parameter_specs(dropped), 6), strict=False)
    for index in (0, 1):
        x2 = io["x"].clone().requires_grad_(True)
        torch.manual_seed(7)
        y = dropped(x2, index)
        y.backward(io["gy"])
        key = f"dropout{index}"
        assert stored_rel_err(store, f"{key}__y", y) < 2e-5 and stored_rel_err(store, f"{key}__dx", x2.grad) < 2e-5
        for n, p in dropped.named_parameters():
            if f"{key}__g__{n}" in store:                    # the reference's gradient is not None
                assert stored_rel_err(store, f"{key}__g__{n}", p.grad) < 5e-5, n
        dropped.zero_grad(set_to_none=True)


def test_no_cpu_path():
    blk = nb.FNOBlocks(4, 4, (4, 4))
    with pytest.raises(RuntimeError, match="no CPU path"):
        blk(torch.randn(1, 4, 8, 8))
    with pytest.raises(RuntimeError, match="no CPU path"):
        nb.ChannelMLP(4)(torch.randn(1, 4, 8))


def test_layer_views_share_the_parameters(host):
    """`blocks[i]` (fno_block.py:466-500): one layer as a module of its own, same parameters, same result."""
    meta, io, params, _ = load_block_golden("block_d2_default_mid")
    blk = _build(meta)
    with torch.no_grad():
        assert rel_err(blk[1](io["x"]), blk(io["x"], 1)) == 0.0
    assert [id(p) for p in blk[0].parameters()] == [id(p) for p in blk.parameters()]
    with pytest.raises(ValueError):
        nb.FNOBlocks(4, 4, (4, 4), n_layers=1).get_block(0)


def test_n_modes_setter_reaches_every_conv():
    blk = nb.FNOBlocks(4, 4, (8, 8), n_layers=2)
    blk.n_modes = (4, 6)
    assert blk.n_modes == (4, 6) and all(c.n_modes == [4, 4] for c in blk.convs)
