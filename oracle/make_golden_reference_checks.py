"""Stored results of the UNMODIFIED reference for the tests that compare with it directly (live-class comparisons), so that those
tests run anywhere: tests/golden/reference_checks.npz, reference_suite.npz, reference_checks.json and reference_swap_models.json.gz
(the module trees of the use_b200_layers cases).

Inputs and parameters are not stored: both sides draw them from `seeded_tensors` with fixed seeds, so only what the reference
returned is kept: of a tensor its shape, its largest magnitude and the values at `sample_index` positions; the bias gradients of the
conv cases, and their weight gradients summed over the channel axes (one value per mode), whole (the files stay small; `stored_rel_err` in tests/conftest.py compares against them).
TEST INFRASTRUCTURE; run in the build container:  python oracle/make_golden_reference_checks.py"""
import gzip
import importlib
import json
import os
import sys
import zlib

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, "tests", "golden")
SAMPLE = 64          # stored entries of a tensor in reference_checks.npz; up to WHOLE entries are stored whole where asked
WHOLE = 4096
SWAP_SAMPLE = 16     # ... of a tensor of the use_b200_layers cases (about 500 tensors)
SUITE_SAMPLE = 24    # ... in reference_suite.npz (about 600 tensors)


def sample_index(shape, key, k):
    """Flat positions of the stored entries of the tensor stored under `key`: all of them for a small tensor, else k of them drawn
    with a seed derived from the key."""
    n = int(np.prod(shape, dtype=np.int64))
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(zlib.crc32(key.encode())).choice(n, size=k, replace=False))


class Store:
    """Stored tensors, packed into a few flat arrays (one small array per tensor would make the file mostly zip headers)."""

    def __init__(self):
        self.keys, self.shapes, self.absmax, self.is_complex, self.values = [], [], [], [], []

    def add(self, key, t, k=SAMPLE, whole=False):
        t = t.detach().cpu()
        k = max(k, t.numel()) if whole and t.numel() <= WHOLE else k
        flat = t.reshape(-1)[torch.from_numpy(sample_index(tuple(t.shape), key, k))]
        self.keys.append(key)
        self.shapes.append(list(t.shape))
        self.absmax.append(t.abs().max().item() if t.numel() else 0.0)
        self.is_complex.append(flat.is_complex())
        self.values.append((torch.view_as_real(flat) if flat.is_complex() else flat).reshape(-1).float().numpy())

    def save(self, path):
        ndim = max(len(s) for s in self.shapes)
        np.savez_compressed(path, keys=np.array(self.keys), shapes=np.array([s + [-1] * (ndim - len(s)) for s in self.shapes], dtype=np.int64),
                            absmax=np.array(self.absmax, dtype=np.float64), is_complex=np.array(self.is_complex),
                            counts=np.array([v.size for v in self.values], dtype=np.int64), values=np.concatenate(self.values))


def load_store(path):
    """{key: (shape, largest magnitude, stored values)} of a file written by Store.save."""
    d = np.load(path)
    ends = np.cumsum(d["counts"])
    out = {}
    for i, key in enumerate(d["keys"]):
        vals = torch.from_numpy(d["values"][ends[i] - d["counts"][i]:ends[i]].copy())
        if d["is_complex"][i]:
            vals = torch.view_as_complex(vals.reshape(-1, 2))
        out[str(key)] = (tuple(int(n) for n in d["shapes"][i] if n >= 0), float(d["absmax"][i]), vals)
    return out


def seeded_tensors(specs, seed, scale=0.5):
    """[(name, shape, dtype)] -> {name: tensor}, drawn in sorted name order from a generator seeded with `seed`."""
    gen = torch.Generator().manual_seed(seed)
    return {name: scale * torch.randn(*shape, generator=gen, dtype=dtype) for name, shape, dtype in sorted(specs, key=lambda s: s[0])}


def parameter_specs(module):
    return [(n, tuple(p.shape), p.dtype) for n, p in module.named_parameters()]


def conv_case_inputs(x_shape, x_dtype, w_shape, b_shape, b_dtype, seed):
    """x, weight, bias of a SpectralConv comparison (the output gradient is drawn next from the returned generator)."""
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(*x_shape, generator=gen, dtype=x_dtype)
    w = 0.5 * torch.randn(*w_shape, generator=gen, dtype=torch.cfloat)
    b = torch.randn(*b_shape, generator=gen, dtype=b_dtype)
    return x, w, b, gen


def _tests_module(name):
    tests = os.path.join(ROOT, "tests")
    if tests not in sys.path:
        sys.path.insert(0, tests)
    return importlib.import_module(name)


def _conv_cases(ref, store, meta):
    T = _tests_module("test_oracle_vs_reference")
    for i, (grid, modes, kw) in enumerate(T.BIT_EXACT_CASES):
        key = f"conv{i}"
        conv = ref.SpectralConv(4, 6, modes, **kw)
        w_shape, b_shape = tuple(conv.weight.tensor.shape), tuple(conv.bias.shape)
        x, w, b, gen = conv_case_inputs((2, 4, *grid), torch.float32, w_shape, b_shape, torch.float32, 7 + i)
        with torch.no_grad():
            conv.weight.tensor.copy_(w)
            conv.bias.copy_(b)
        x.requires_grad_(True)
        y = conv(x)
        g = torch.randn(*y.shape, generator=gen)
        y.backward(g)
        meta[key] = {"w_shape": list(w_shape), "b_shape": list(b_shape), "max_n_modes": list(conv.max_n_modes)}
        dw = conv.weight.tensor.grad
        for name, t in (("y", y), ("dx", x.grad), ("dw", dw), ("dw_modes", dw.sum(dim=(0, 1))), ("db", conv.bias.grad)):
            store.add(f"{key}__{name}", t, whole=name in ("dw_modes", "db"))

    resample = importlib.import_module("neuralop.layers.resample").resample
    for i, (shape, out) in enumerate(T.RESAMPLE_CASES):
        torch.manual_seed(0)
        x = torch.randn(*shape)
        store.add(f"resample{i}", resample(x, 1.0, list(range(2, x.ndim)), output_shape=out))

    for i, (grid, modes, kw) in enumerate(T.COMPLEX_CASES):
        key = f"cconv{i}"
        conv = ref.SpectralConv(3, 3 if kw.get("separable") else 4, modes, complex_data=True, **kw)
        w_shape, b_shape = tuple(conv.weight.tensor.shape), tuple(conv.bias.shape)
        x, w, b, gen = conv_case_inputs((2, 3, *grid), torch.cfloat, w_shape, b_shape, conv.bias.dtype, 11 + i)
        with torch.no_grad():
            conv.weight.tensor.copy_(w)
            conv.bias.copy_(b)
        x.requires_grad_(True)
        y = conv(x)
        g = torch.randn(*y.shape, generator=gen, dtype=y.dtype)
        y.backward(g)
        meta[key] = {"w_shape": list(w_shape), "b_shape": list(b_shape), "b_complex": conv.bias.is_complex(),
                     "max_n_modes": list(conv.max_n_modes)}
        dw = conv.weight.tensor.grad
        for name, t in (("y", y), ("dx", x.grad), ("dw", dw), ("dw_modes", dw.sum(dim=(0, 1))), ("db", conv.bias.grad)):
            store.add(f"{key}__{name}", t, whole=name in ("dw_modes", "db"))


def _conv_module_calls(meta):
    """The constructor calls the reference FNOBlocks makes to a `conv_module` that is this package's SpectralConv."""
    import neuraloperator_b200 as nb
    fno_block = importlib.import_module("neuralop.layers.fno_block")
    out = {}
    for name, args, kw in [("default", (8, 8, (12, 12)), dict(n_layers=2)),
                           ("tucker", (8, 8, (12, 12)), dict(n_layers=1, factorization="tucker", rank=0.5, implementation="factorized"))]:
        calls = []

        class Recording(nb.SpectralConv):
            def __init__(self, *a, **k):
                calls.append({"args": [list(v) if isinstance(v, tuple) else v for v in a],
                              "kwargs": {kk: (list(v) if isinstance(v, tuple) else v) for kk, v in k.items()}})
                super().__init__(*a, **k)

        fno_block.FNOBlocks(*args, conv_module=Recording, **kw)
        out[name] = calls
    meta["conv_module_calls"] = out


def _block_cases(store, meta):
    fb = importlib.import_module("neuralop.layers.fno_block")
    C = _tests_module("conftest")
    T = _tests_module("test_block_oracle")
    for name in T.LIVE_CASES:
        bmeta, io, params, _ = C.load_block_golden(name)
        blk = fb.FNOBlocks(bmeta["in_channels"], bmeta["out_channels"], tuple(bmeta["n_modes"]), n_layers=bmeta["n_layers"], **bmeta["ctor"])
        specs = parameter_specs(blk)
        assert sorted(specs, key=lambda s: s[0]) == sorted([(k, tuple(v.shape), v.dtype) for k, v in params.items()], key=lambda s: s[0])
        blk.load_state_dict(seeded_tensors(specs, 99), strict=False)
        gen = torch.Generator().manual_seed(100)
        x = torch.randn(*io["x"].shape, generator=gen, dtype=io["x"].dtype).requires_grad_(True)
        y = blk(x, bmeta["index"], **{k: tuple(v) for k, v in bmeta["forward"].items()})
        gy = torch.randn(*y.shape, generator=gen, dtype=y.dtype)
        y.backward(gy)
        key = f"block_{name}"
        store.add(f"{key}__y", y)
        store.add(f"{key}__dx", x.grad)
        touched = sorted(n for n, p in blk.named_parameters() if p.grad is not None)
        for pname, p in blk.named_parameters():
            if p.grad is not None:
                store.add(f"{key}__g__{pname}", p.grad)
        meta[key] = {"touched": touched}


def _half_contraction(store):
    eu = importlib.import_module("neuralop.layers.einsum_utils")
    T = _tests_module("test_reduced_precision")
    for i, shape in enumerate(T.HALF_CASES):
        xm, w = T.half_case_inputs(shape)
        sym = "cdef"[: len(shape[3])]
        ref = eu.einsum_complexhalf(f"ab{sym},bz{sym}->az{sym}", xm.chalf(), w)
        store.add(f"half{i}", torch.view_as_complex(torch.view_as_real(ref).float()))


def _block_state(store, meta):
    fb = importlib.import_module("neuralop.layers.fno_block")
    # state dict round trip: FNOBlocks(6, 6, (8, 8), n_layers=3)
    ref = fb.FNOBlocks(6, 6, (8, 8), n_layers=3, implementation="reconstructed")
    ref.load_state_dict(seeded_tensors(parameter_specs(ref), 4), strict=False)
    meta["state_dict"] = {k: [list(v.shape), str(v.dtype)] for k, v in ref.state_dict().items()}
    x = torch.randn(2, 6, 16, 16, generator=torch.Generator().manual_seed(5))
    with torch.no_grad():
        for i in range(3):
            store.add(f"sd_layer{i}", ref(x, i))
        a = x
        for i in range(3):
            a = ref(a, i)
        store.add("sd_stack", a)

    # batch norm: two training steps, then eval mode
    ref = fb.FNOBlocks(4, 4, (6, 6), n_layers=2, norm="batch_norm", implementation="reconstructed")
    ref.load_state_dict(seeded_tensors(parameter_specs(ref), 8), strict=False)
    gen = torch.Generator().manual_seed(9)
    x, x2 = torch.randn(3, 4, 12, 12, generator=gen), torch.randn(2, 4, 12, 12, generator=gen)
    with torch.no_grad():
        for i in range(2):
            store.add(f"bn_train{i}", ref(x, i))
        meta["bn_buffers"] = [n for n, _ in ref.named_buffers()]
        for n, b in ref.named_buffers():
            store.add(f"bn_buffer__{n}", b.float())
        ref.eval()
        store.add("bn_eval", ref(x2, 0))

    # training-mode dropout under equal seeds: block_d2_default_mid's layer, channel_mlp_dropout=0.3
    C = _tests_module("conftest")
    bmeta, io, _, _ = C.load_block_golden("block_d2_default_mid")
    ref = fb.FNOBlocks(bmeta["in_channels"], bmeta["out_channels"], tuple(bmeta["n_modes"]), n_layers=2, implementation="reconstructed",
                       channel_mlp_dropout=0.3)
    ref.load_state_dict(seeded_tensors(parameter_specs(ref), 6), strict=False)
    for index in (0, 1):
        x1 = io["x"].clone().requires_grad_(True)
        torch.manual_seed(7)
        y = ref(x1, index)
        y.backward(io["gy"])
        store.add(f"dropout{index}__y", y)
        store.add(f"dropout{index}__dx", x1.grad)
        for n, p in ref.named_parameters():
            if p.grad is not None:
                store.add(f"dropout{index}__g__{n}", p.grad)
        ref.zero_grad(set_to_none=True)


CONVERTIBLE = ("FNOBlocks", "ChannelMLP", "SpectralConv", "Flattened1dConv", "SoftGating", "ComplexValued")


def _attribute_value(v):
    """A JSON form of a module attribute, or raises TypeError: plain values, lists / dicts of them, torch.nn.functional functions."""
    if v is None or isinstance(v, (bool, int, float, str)):
        return v
    if isinstance(v, (list, tuple)):
        return [_attribute_value(e) for e in v]
    if isinstance(v, dict):
        return {str(k): _attribute_value(e) for k, e in v.items()}
    if callable(v) and getattr(torch.nn.functional, getattr(v, "__name__", ""), None) is v:
        return {"function": v.__name__}
    raise TypeError(type(v))


def module_tree(m):
    """Class, attributes, parameter specs, buffers and children of a module, recursively (what a converter can read of it)."""
    attrs = {}
    for name in dir(m):
        if (name.startswith("_") or name in m._parameters or name in m._buffers or name in m._modules
                or (name != "training" and hasattr(torch.nn.Module, name))):
            continue
        try:
            attrs[name] = _attribute_value(getattr(m, name))
        except Exception:                     # methods, tensors, other objects: not read by the converters
            pass
    return {"class": type(m).__name__, "module": type(m).__module__, "attrs": attrs,
            "params": {n: (None if p is None else [list(p.shape), str(p.dtype)]) for n, p in m._parameters.items()},
            "buffers": {n: [b.tolist(), str(b.dtype)] for n, b in m._buffers.items() if b is not None},
            "children": {n: module_tree(c) for n, c in m._modules.items()}}


def swap_input(m, n_dim, seed):
    """Seeded input of a convertible module (2 samples, 16 points per dimension) and whether it is complex."""
    cplx = type(m).__name__ == "ComplexValued" or (type(m).__name__ in ("FNOBlocks", "SpectralConv") and m.complex_data)
    inner = m.fr if type(m).__name__ == "ComplexValued" else m
    if type(inner).__name__ == "Flattened1dConv":
        ch = inner.conv.in_channels
    else:
        ch = inner.in_features if type(inner).__name__ == "SoftGating" else inner.in_channels
    gen = torch.Generator().manual_seed(seed)
    return torch.randn(2, ch, *[16] * n_dim, generator=gen, dtype=torch.cfloat if cplx else torch.float32), gen


def swap_calls(m):
    """The forward calls recorded of a convertible module: every layer index of an FNOBlocks, else one call."""
    return range(m.n_layers) if type(m).__name__ == "FNOBlocks" else range(1)


def _swap_models():
    load_fno = importlib.import_module("make_golden_fno").load_reference_fno
    fno = load_fno()
    uno = importlib.import_module("neuralop.models.uno")
    T = _tests_module("test_integration_cpu")
    models = []
    for kw in T.SWAP_FNO_CASES:
        kw = {k: (getattr(torch.nn.functional, v) if k == "non_linearity" else v) for k, v in kw.items()}
        models.append((fno.FNO(**kw), len(kw["n_modes"])))
    models.append((fno.FNO(**T.SWAP_ELU_CASE, non_linearity=torch.nn.functional.elu), 2))
    models.append((uno.UNO(**T.SWAP_UNO_CASE), 2))
    return models


def _swap_cases(store, meta):
    """use_b200_layers: the module trees of reference models, and what each convertible module in them returns for seeded inputs
    and parameters (forward, input gradient, parameter gradients)."""
    import copy
    import warnings
    import neuraloperator_b200 as nb
    sys.path.insert(0, HERE)
    out = []
    for c, (model, n_dim) in enumerate(_swap_models()):
        if getattr(model.fno_blocks, "channel_mlp_dropout", 0):
            model.eval()                                          # (training-mode dropout is compared under equal seeds elsewhere)
        model.load_state_dict(seeded_tensors(parameter_specs(model), 30 + c), strict=False)
        out.append({"n_dim": n_dim, "tree": module_tree(model)})
        with warnings.catch_warnings():                           # which paths the swap installs a module at: only those are stored
            warnings.simplefilter("ignore")
            swapped = dict(nb.use_b200_layers(copy.deepcopy(model)).named_modules())
        for j, (path, m) in enumerate(model.named_modules()):
            parent = swapped.get(path.rpartition(".")[0])
            if (type(m).__name__ not in CONVERTIBLE or not type(swapped.get(path)).__module__.startswith("neuraloperator_b200")
                    or type(parent).__module__.startswith("neuraloperator_b200")):
                continue
            for i in swap_calls(m):
                x, gen = swap_input(m, n_dim, 1000 * c + 10 * j + i)
                x.requires_grad_(True)
                y = m(x, i) if type(m).__name__ == "FNOBlocks" else m(x)
                y.backward(torch.randn(*y.shape, generator=gen, dtype=y.dtype))
                key = f"swap{c}__{path}__{i}"
                store.add(f"{key}__y", y, SWAP_SAMPLE)
                store.add(f"{key}__dx", x.grad, SWAP_SAMPLE)
                for pname, p in m.named_parameters():
                    if p.grad is not None:
                        store.add(f"{key}__g__{pname}", p.grad, SWAP_SAMPLE)
                m.zero_grad(set_to_none=True)
    return out


class _LiveTwin:
    """The reference class holding the weights of a conv of the suite; `check` stores what it returns instead of comparing."""

    def __init__(self, module, case, store):
        self.module, self.case, self.store, self.n = module, case, store, 0

    @property
    def n_modes(self):
        return self.module.n_modes

    @n_modes.setter
    def n_modes(self, value):
        self.module.n_modes = value

    def check(self, out, x, tol):
        with torch.no_grad():
            self.store.add(f"{self.case}__{self.n}", self.module(x.cpu()), SUITE_SAMPLE)
        self.n += 1


def _suite(ref, store):
    T = _tests_module("test_reference_suite_cpu")
    with __import__("pytest").MonkeyPatch.context() as mp:
        T.emulate_device(mp)
        for case in T.GRID_1:
            twins = []

            def twin_of(conv, **ctor):
                with torch.random.fork_rng(devices=[]):            # the suite's own draws go on as in the test
                    module = ref.SpectralConv(conv.in_channels, conv.out_channels if not conv.separable else conv.in_channels,
                                              tuple(ctor.pop("user_modes")), bias=conv.bias is not None, factorization=None,
                                              implementation="reconstructed", separable=conv.separable, complex_data=conv.complex_data,
                                              **ctor)
                with torch.no_grad():
                    module.weight.tensor.copy_(conv.weight.to_tensor())
                    if conv.bias is not None:
                        module.bias.copy_(conv.bias)
                twins.append(_LiveTwin(module, T.case_key("g1", case, len(twins)), store))
                return twins[-1]
            T.suite_factorized_vs_dense(torch.device("cpu"), *case, 2e-5, twin_of=twin_of)
        for case in T.GRID_2:
            hermitian, dim, side, scaling, modes = case

            def twin_of(conv):
                with torch.random.fork_rng(devices=[]):
                    module = ref.SpectralConv(3, 4, modes[:dim], enforce_hermitian_symmetry=hermitian, complex_data=False,
                                              resolution_scaling_factor=scaling)
                with torch.no_grad():
                    module.weight.tensor.copy_(conv.weight.to_tensor())
                    module.bias.copy_(conv.bias)
                return _LiveTwin(module, T.case_key("g2", case, 0), store)
            T.suite_real_output_shapes(torch.device("cpu"), hermitian, dim, side, scaling, modes, 2e-5, twin_of=twin_of)


def main():
    sys.path.insert(0, ROOT)
    from oracle.load_reference import load_reference_spectral_conv
    ref = load_reference_spectral_conv()
    store, suite, meta = Store(), Store(), {}
    _conv_cases(ref, store, meta)
    _conv_module_calls(meta)
    _block_cases(store, meta)
    _half_contraction(store)
    _block_state(store, meta)
    swap_models = _swap_cases(store, meta)
    _suite(ref, suite)
    store.save(os.path.join(OUT, "reference_checks.npz"))
    suite.save(os.path.join(OUT, "reference_suite.npz"))
    with gzip.open(os.path.join(OUT, "reference_swap_models.json.gz"), "wt") as f:
        json.dump(swap_models, f, separators=(",", ":"))
    with open(os.path.join(OUT, "reference_checks.json"), "w") as f:
        json.dump({"reference": "neuraloperator@93d3f06", "generator": "oracle/make_golden_reference_checks.py", **meta}, f, indent=1)
    print(len(store.keys), "tensors in reference_checks.npz,", len(suite.keys), "in reference_suite.npz")


if __name__ == "__main__":
    main()
