"""Model-level integration without a GPU (kernels through their host checks, conv through the CPU oracle, as in
tests/test_block_host_logic.py):
(1) the drop-ins stacked as the reference `FNO` stacks them (lifting -> n_layers x FNOBlocks -> projection) against goldens minted from
    the unmodified reference model (oracle/make_golden_fno.py): y, dx, every parameter gradient;
(2) `neuraloperator_b200.use_b200_layers(model)` on reference FNO / TFNO / UNO models -- stand-ins with the class names, attributes,
    parameter names and buffers recorded from the reference (the swap recognises modules by those), seeded parameters -- every
    installed module against what the reference module computed (oracle/make_golden_reference_checks.py);
(3) batch-norm running statistics against stored results of the reference block."""
import re

import pytest
import torch

import neuraloperator_b200 as nb
from conftest import build_fno_stack, fno_golden_index, load_fno_golden, reference_checks, stored_rel_err
from oracle.make_golden_reference_checks import CONVERTIBLE, parameter_specs, seeded_tensors, swap_calls, swap_input
from test_block_host_logic import grad_err, host, rel_err  # noqa: F401  (fixture)


@pytest.mark.parametrize("name", sorted(fno_golden_index().keys()))
def test_stacked_drop_ins_match_reference_fno_golden(host, name):  # noqa: F811
    meta, io, params, grads = load_fno_golden(name)
    mods, forward = build_fno_stack(meta, params)
    x = io["x"].clone().requires_grad_(True)
    y = forward(x)
    y.backward(io["gy"])
    assert rel_err(y, io["y"]) < 3e-5 and rel_err(x.grad, io["dx"]) < 3e-5
    ours = dict(mods.named_parameters())
    for k, g in grads.items():
        assert rel_err(ours[k.replace("weight.factors.", "weight.factors.factor_")].grad, g) < 5e-5, k


SWAP_FNO_CASES = [dict(n_modes=(8, 8), in_channels=2, out_channels=3, hidden_channels=8, n_layers=2),
                  dict(n_modes=(8, 6), in_channels=1, out_channels=1, hidden_channels=6, n_layers=2, factorization="tucker",
                       implementation="factorized", rank=[3, 3, 4, 3]),
                  dict(n_modes=(10,), in_channels=1, out_channels=1, hidden_channels=4, n_layers=3, stabilizer="tanh",
                       fno_skip="soft-gating", channel_mlp_skip="linear"),
                  dict(n_modes=(8, 8), in_channels=1, out_channels=1, hidden_channels=6, n_layers=2, norm="group_norm"),
                  dict(n_modes=(8, 8), in_channels=1, out_channels=1, hidden_channels=6, n_layers=2, norm="instance_norm"),
                  dict(n_modes=(8, 8), in_channels=1, out_channels=1, hidden_channels=6, n_layers=2, norm="batch_norm"),
                  dict(n_modes=(8, 8), in_channels=1, out_channels=1, hidden_channels=6, n_layers=2, complex_data=True,
                       positional_embedding=None),
                  dict(n_modes=(8, 8), in_channels=1, out_channels=1, hidden_channels=6, n_layers=2, conv_bias_kernel=3,
                       channel_mlp_dropout=0.2, non_linearity="silu")]
SWAP_ELU_CASE = dict(n_modes=(8, 6), in_channels=1, out_channels=1, hidden_channels=8, n_layers=2, max_n_modes=(10, 8))
SWAP_UNO_CASE = dict(in_channels=1, out_channels=1, hidden_channels=8, n_layers=3, uno_out_channels=[8, 8, 8],
                     uno_n_modes=[[6, 6], [4, 4], [6, 6]], uno_scalings=[[0.5, 0.5], [1, 1], [2, 2]], channel_mlp_skip="linear")
_STAND_IN_CLASSES = {}


def _attribute(v):
    if isinstance(v, dict):
        return getattr(torch.nn.functional, v["function"]) if set(v) == {"function"} else {k: _attribute(e) for k, e in v.items()}
    return [_attribute(e) for e in v] if isinstance(v, list) else v


def _dtype(name):
    return getattr(torch, name.split(".")[-1])


def stand_in(tree):
    """A module with the class name, class module, attributes, parameters (zeros), buffers and children recorded from a reference
    module (oracle/make_golden_reference_checks.py: module_tree) -- what use_b200_layers reads of it -- without the reference's code.
    torch containers are rebuilt as themselves (the swap indexes and assigns into them)."""
    if tree["module"].startswith("torch.nn") and tree["class"] in ("ModuleList", "Sequential"):
        m = getattr(torch.nn, tree["class"])()
    else:
        key = (tree["module"], tree["class"])
        if key not in _STAND_IN_CLASSES:
            _STAND_IN_CLASSES[key] = type(tree["class"], (torch.nn.Module,), {"__module__": tree["module"]})
        m = _STAND_IN_CLASSES[key]()
        for name, v in tree["attrs"].items():
            setattr(m, name, _attribute(v))
    for name, spec in tree["params"].items():
        m.register_parameter(name, None if spec is None else torch.nn.Parameter(torch.zeros(*spec[0], dtype=_dtype(spec[1]))))
    for name, (values, dtype) in tree["buffers"].items():
        m.register_buffer(name, torch.tensor(values, dtype=_dtype(dtype)))
    for name, child in tree["children"].items():
        m.add_module(name, stand_in(child))
    return m


def _our_param_name(ref_name):
    return re.sub(r"factors\.(\d+)", r"factors.factor_\1", ref_name)


def swap_stand_in_model(case):
    """The stand-in of reference model `case` holding the seeded parameters, and the seeded inputs of its convertible modules
    [(path, layer index, input, generator of the output gradient)], drawn as the generator drew them."""
    _, checks = reference_checks()
    rec = checks["swap_models"][case]
    model = stand_in(rec["tree"])
    model.load_state_dict(seeded_tensors(parameter_specs(model), 30 + case), strict=False)
    calls = []
    for j, (path, m) in enumerate(model.named_modules()):
        if type(m).__name__ in CONVERTIBLE:
            for i in swap_calls(m):
                x, gen = swap_input(m, rec["n_dim"], 1000 * case + 10 * j + i)
                calls.append((path, i, x, gen))
    return model, calls


def check_swapped_modules(model, case, calls):
    """Every module use_b200_layers installed (a drop-in whose parent is not one) against what the reference module at that path
    returned for the same input and parameters: forward, input gradient, every parameter gradient.  Returns the paths checked."""
    store, _ = reference_checks()
    done = set()
    modules = dict(model.named_modules())
    for path, i, x, gen in calls:
        m, parent = modules.get(path), modules[path.rpartition(".")[0]]
        if m is None or not type(m).__module__.startswith("neuraloperator_b200") or type(parent).__module__.startswith("neuraloperator_b200"):
            continue
        key = f"swap{case}__{path}__{i}"
        x = x.clone().requires_grad_(True)
        y = m(x, i) if type(m).__name__ == "FNOBlocks" else m(x)
        y.backward(torch.randn(*y.shape, generator=gen, dtype=y.dtype))
        assert stored_rel_err(store, f"{key}__y", y) < 3e-5 and stored_rel_err(store, f"{key}__dx", x.grad) < 3e-5, key
        grads = {k[len(key) + 5:]: v for k, v in store.items() if k.startswith(f"{key}__g__")}
        scale = max([g[1] for g in grads.values()] + [1e-20])
        ours = dict(m.named_parameters())
        for pname, (_, absmax, _) in grads.items():
            p = ours[_our_param_name(pname)]
            if absmax < 1e-5 * scale:     # vanishes in exact arithmetic (a conv bias in front of a norm): ours as negligible
                assert float(p.grad.abs().max()) / scale < 5e-5, (key, pname)
            else:
                assert stored_rel_err(store, f"{key}__g__{pname}", p.grad) < 5e-5, (key, pname)
        for pname, p in ours.items():
            if p.grad is not None and pname not in {_our_param_name(k) for k in grads}:
                assert float(p.grad.abs().max()) == 0.0, (key, pname)
        m.zero_grad(set_to_none=True)
        done.add(path)
    return done


@pytest.mark.parametrize("kw", SWAP_FNO_CASES)
def test_use_b200_layers_on_a_live_reference_model(host, kw):  # noqa: F811
    """A reference FNO / TFNO (stand-in with the recorded structure, attributes and seeded parameters): the block and the lifting /
    projection MLPs move over, parameter names are kept, and each installed module computes what the reference's did."""
    case = SWAP_FNO_CASES.index(kw)
    model, calls = swap_stand_in_model(case)
    names = sorted(k for k, _ in model.named_parameters())
    out = nb.use_b200_layers(model)
    assert out is model
    mlp_type = nb.ComplexValued if kw.get("complex_data") else nb.ChannelMLP
    assert type(model.fno_blocks) is nb.FNOBlocks and type(model.lifting) is mlp_type and type(model.projection) is mlp_type
    assert sorted(k.replace("factors.factor_", "factors.") for k, _ in model.named_parameters()) == names
    assert {"fno_blocks", "lifting", "projection"} <= check_swapped_modules(model, case, calls)
    nb.use_b200_layers(model)                              # idempotent: nothing left to convert
    assert type(model.fno_blocks) is nb.FNOBlocks


def test_blocks_without_a_drop_in_keep_the_reference_block_and_swap_its_convs(host):  # noqa: F811
    """non_linearity=F.elu (an activation the kernels do not have): the reference FNOBlocks and the lifting / projection MLPs stay, with a
    warning each; the SpectralConvs and the (GELU) ChannelMLPs inside the block move over and compute what the reference's did."""
    case = len(SWAP_FNO_CASES)
    model, calls = swap_stand_in_model(case)
    with pytest.warns(UserWarning, match="stays the reference module"):
        nb.use_b200_layers(model)
    assert type(model.fno_blocks).__module__.startswith("neuralop.")                    # the block is still the reference's
    assert all(type(c) is nb.SpectralConv for c in model.fno_blocks.convs)              # ... its convs are ours
    assert all(type(m) is nb.ChannelMLP for m in model.fno_blocks.channel_mlp)          # ... and its (GELU) channel MLPs
    assert type(model.lifting).__module__.startswith("neuralop.")                       # an elu MLP has no drop-in
    assert model.fno_blocks.convs[0].n_modes == [8, 4] and list(model.fno_blocks.convs[0].max_n_modes) == [10, 8]
    want = {f"fno_blocks.{part}.{i}" for part in ("convs", "channel_mlp") for i in range(2)}
    assert want <= check_swapped_modules(model, case, calls)


def test_use_b200_layers_on_another_model_family_uno(host):  # noqa: F811
    """The swap is by module class, not by model: a reference U-shaped neural operator (neuralop/models/uno.py: FNOBlocks with
    different channel counts / modes / scalings per layer, stand-alone linear skips) ends up without a single reference layer class
    from this package's list, and every installed module computes what the reference's did."""
    case = len(SWAP_FNO_CASES) + 1
    model, calls = swap_stand_in_model(case)
    nb.use_b200_layers(model)
    left = {type(m).__name__ for m in model.modules() if type(m).__module__.startswith("neuralop.")}
    assert not left & {"FNOBlocks", "SpectralConv", "ChannelMLP", "Flattened1dConv", "SoftGating"}, left
    top = {path for path, *_ in calls if "." not in path or path.rpartition(".")[0] in ("fno_blocks", "horizontal_skips")}
    assert top and top <= check_swapped_modules(model, case, calls)


def test_batch_norm_eval_mode_uses_the_running_statistics(host):  # noqa: F811
    """Two training steps move the running statistics as the reference's did, and eval mode then uses them as the reference did (its
    results for the same parameters and inputs stored by oracle/make_golden_reference_checks.py)."""
    store, checks = reference_checks()
    ours = nb.FNOBlocks(4, 4, (6, 6), n_layers=2, norm="batch_norm", implementation="reconstructed")
    ours.load_state_dict(seeded_tensors(parameter_specs(ours), 8), strict=False)
    gen = torch.Generator().manual_seed(9)
    x, x2 = torch.randn(3, 4, 12, 12, generator=gen), torch.randn(2, 4, 12, 12, generator=gen)
    for i in range(2):                                       # two training steps: the running statistics move the same way
        assert stored_rel_err(store, f"bn_train{i}", ours(x, i)) < 3e-5
    assert [n for n, _ in ours.named_buffers()] == checks["bn_buffers"]
    for na, a in ours.named_buffers():
        assert stored_rel_err(store, f"bn_buffer__{na}", a.float()) < 1e-5, na
    ours.eval()
    with torch.no_grad():
        assert stored_rel_err(store, "bn_eval", ours(x2, 0)) < 3e-5     # eval: running statistics instead of the batch's
        assert rel_err(ours(x2, 0), ours.train()(x2, 0)) > 1e-3
    ours.eval()


def test_unsupported_reference_modules_are_reported():
    class ChannelMLP(torch.nn.Module):                     # a reference-like ChannelMLP with an activation the kernels do not have
        in_channels = out_channels = hidden_channels = 4
        n_layers = 2
        non_linearity = staticmethod(torch.nn.functional.elu)
        dropout = None
    holder = torch.nn.Module()
    holder.mlp = ChannelMLP()
    with pytest.warns(UserWarning, match="stays the reference module"):
        nb.use_b200_layers(holder)
    assert type(holder.mlp) is ChannelMLP                  # left in place, and said so
