import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def golden_index():
    with open(os.path.join(GOLDEN_DIR, "index.json")) as f:
        return json.load(f)["cases"]


def load_golden(name):
    meta = golden_index()[name]
    data = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    return meta, {k: torch.from_numpy(data[k]) for k in data.files}


def golden_weight(meta, arrays):
    """Builds the oracle's Weight from a golden file's parameter tensors."""
    from oracle.spectral_conv_oracle import Weight
    kind = meta["weight_kind"]
    p = {k[3:].replace("__", "."): v for k, v in arrays.items() if k.startswith("p__")}
    nf = len([k for k in p if k.startswith("weight.factors.")])
    factors = [p[f"weight.factors.{i}"] for i in range(nf)]
    sep = bool(meta["ctor"].get("separable", False))
    if kind == "dense":
        return Weight("dense", tensor=p["weight.tensor"], separable=sep)
    if kind == "tucker":
        return Weight("tucker", core=p["weight.core"], factors=factors, separable=sep)
    if kind == "cp":
        return Weight("cp", weights=p["weight.weights"], factors=factors, separable=sep)
    if kind == "tt":
        return Weight("tt", factors=factors, separable=sep)
    raise ValueError(kind)


def golden_grads(meta, arrays):
    g = {k[3:].replace("__", "."): v for k, v in arrays.items() if k.startswith("g__")}
    kind = meta["weight_kind"]
    nf = len([k for k in g if k.startswith("weight.factors.")])
    factors = [g[f"weight.factors.{i}"] for i in range(nf)]
    if kind == "dense":
        w = [g["weight.tensor"]]
    elif kind == "tucker":
        w = [g["weight.core"], *factors]
    elif kind == "cp":
        w = [g["weight.weights"], *factors]
    else:
        w = factors
    return w, g.get("bias")


def forward_kwargs(meta):
    kw = {}
    ctor = meta["ctor"]
    if "max_n_modes" in ctor:
        kw["max_n_modes"] = ctor["max_n_modes"]
    if "resolution_scaling_factor" in ctor:
        kw["resolution_scaling_factor"] = [float(ctor["resolution_scaling_factor"])] * len(meta["grid"])
    if "fft_norm" in ctor:
        kw["fft_norm"] = ctor["fft_norm"]
    if "output_shape" in meta["forward"]:
        kw["output_shape"] = meta["forward"]["output_shape"]
    return kw


@pytest.fixture(scope="session")
def cuda_device():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def complex_golden_index():
    with open(os.path.join(GOLDEN_DIR, "complex_index.json")) as f:
        return json.load(f)["cases"]


def load_complex_golden(name):
    """complex_data=True cases (oracle/make_golden_complex.py): complex tensors are stored as (..., 2) arrays under `<key>__c`."""
    meta = complex_golden_index()[name]
    data = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    out = {}
    for k in data.files:
        t = torch.from_numpy(data[k])
        if k.endswith("__c"):
            out[k[:-3]] = torch.view_as_complex(t.contiguous())
        else:
            out[k] = t
    return meta, out


BLOCK_ACTIVATIONS = {"relu": torch.nn.functional.relu, "silu": torch.nn.functional.silu, "tanh": torch.tanh}


def block_ctor_kwargs(meta):
    """Constructor keywords of a block golden with the activation name resolved to the callable."""
    ctor = dict(meta["ctor"])
    if "max_n_modes" in ctor:
        ctor["max_n_modes"] = tuple(ctor["max_n_modes"])
    if "non_linearity" in ctor:
        ctor["non_linearity"] = BLOCK_ACTIVATIONS[ctor["non_linearity"]]
    return ctor


def block_golden_index():
    with open(os.path.join(GOLDEN_DIR, "block_index.json")) as f:
        return json.load(f)["cases"]


def load_block_golden(name):
    """Fourier-layer cases (oracle/make_golden_block.py): returns meta, {x, gy, y, dx}, params {ref name: tensor}, grads {ref name: tensor}."""
    meta = block_golden_index()[name]
    data = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    io, params, grads = {}, {}, {}
    for k in data.files:
        t = torch.from_numpy(data[k])
        key = k
        if k.endswith("__c"):
            t, key = torch.view_as_complex(t.contiguous()), k[:-3]
        if key.startswith("p__"):
            params[key[3:].replace("__", ".")] = t
        elif key.startswith("g__"):
            grads[key[3:].replace("__", ".")] = t
        else:
            io[key] = t                    # x, gy, y, dx; ada_in_embedding; b__<buffer name>: buffers after the forward pass
    return meta, io, params, grads


def block_oracle_kwargs(meta):
    """Keyword arguments of oracle.fno_block_oracle.fno_block_forward for a golden case."""
    ctor = meta["ctor"]
    kw = dict(n_modes=meta["n_modes"], n_layers=meta["n_layers"], weight_kind=meta["weight_kind"],
              fno_skip=ctor.get("fno_skip", "linear"), channel_mlp_skip=ctor.get("channel_mlp_skip", "soft-gating"),
              use_channel_mlp=ctor.get("use_channel_mlp", True), stabilizer=ctor.get("stabilizer"),
              preactivation=ctor.get("preactivation", False), resolution_scaling_factor=ctor.get("resolution_scaling_factor"),
              norm=ctor.get("norm"), norm_groups=ctor.get("norm_groups", 1))
    if "non_linearity" in ctor:
        kw["non_linearity"] = BLOCK_ACTIVATIONS[ctor["non_linearity"]]
    if "max_n_modes" in ctor:
        from oracle.spectral_conv_oracle import stored_n_modes
        kw["max_n_modes"] = stored_n_modes(ctor["max_n_modes"])
    if "output_shape" in meta["forward"]:
        kw["output_shape"] = meta["forward"]["output_shape"]
    if ctor.get("complex_data"):           # oracle.fno_block_oracle.fno_block_forward_complex: dense weight, no norm, no resampling
        kw = {k: kw[k] for k in ("n_modes", "n_layers", "fno_skip", "channel_mlp_skip", "use_channel_mlp", "stabilizer", "preactivation")}
    return kw


def fno_golden_index():
    with open(os.path.join(GOLDEN_DIR, "fno_index.json")) as f:
        return json.load(f)["cases"]


def load_fno_golden(name):
    """Model-level cases (oracle/make_golden_fno.py): meta, {x, gy, y, dx}, params, grads keyed by the reference's parameter names."""
    meta = fno_golden_index()[name]
    data = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    io, params, grads = {}, {}, {}
    for k in data.files:
        t = torch.from_numpy(data[k])
        key = k
        if k.endswith("__c"):
            t, key = torch.view_as_complex(t.contiguous()), k[:-3]
        if key.startswith("p__"):
            params[key[3:].replace("__", ".")] = t
        elif key.startswith("g__"):
            grads[key[3:].replace("__", ".")] = t
        else:
            io[key] = t
    return meta, io, params, grads


_REFERENCE_CHECKS = {}


def reference_checks(name="reference_checks"):
    """(store, meta) of the stored reference results (oracle/make_golden_reference_checks.py): store = {key: (shape, largest
    magnitude, values at the sampled positions)} of `name`.npz, meta = reference_checks.json with the module trees of
    reference_swap_models.json.gz as meta["swap_models"]."""
    if name not in _REFERENCE_CHECKS:
        import gzip
        from oracle.make_golden_reference_checks import load_store
        with open(os.path.join(GOLDEN_DIR, "reference_checks.json")) as f:
            meta = json.load(f)
        with gzip.open(os.path.join(GOLDEN_DIR, "reference_swap_models.json.gz"), "rt") as f:
            meta["swap_models"] = json.load(f)
        _REFERENCE_CHECKS[name] = (load_store(os.path.join(GOLDEN_DIR, name + ".npz")), meta)
    return _REFERENCE_CHECKS[name]


def stored_rel_err(store, key, got):
    """Largest difference between `got` and the reference tensor stored under `key`, at the stored positions, over the reference's
    largest magnitude; also the difference of the two largest magnitudes, so that no entry of `got` can outgrow the reference's."""
    from oracle.make_golden_reference_checks import sample_index
    shape, absmax, values = store[key]
    assert tuple(got.shape) == shape, (key, tuple(got.shape), shape)
    got = got.detach().cpu()
    flat = got.reshape(-1)[torch.from_numpy(sample_index(shape, key, values.shape[0]))].to(values.dtype)
    peak = abs(float(got.abs().max()) - absmax) if got.numel() else 0.0
    return max(float((flat - values).abs().max()) if values.numel() else 0.0, peak) / max(absmax, 1e-20)


def build_fno_stack(meta, params, device=None):
    """lifting -> FNOBlocks -> projection from this package's drop-ins, as `FNO.__init__` builds them (fno.py:289-345, defaults:
    lifting / projection channel ratio 2), holding the golden's parameters.  Returns (modules dict, forward function)."""
    import neuraloperator_b200 as nb
    kw = dict(meta["ctor"])
    hidden, n_layers = kw.pop("hidden_channels"), kw.pop("n_layers")
    cin, cout, modes = kw.pop("in_channels"), kw.pop("out_channels"), tuple(kw.pop("n_modes"))
    mods = torch.nn.ModuleDict({
        "lifting": nb.ChannelMLP(cin, out_channels=hidden, hidden_channels=2 * hidden, n_layers=2),
        "fno_blocks": nb.FNOBlocks(hidden, hidden, modes, n_layers=n_layers, **kw),
        "projection": nb.ChannelMLP(hidden, out_channels=cout, hidden_channels=2 * hidden, n_layers=2),
    })
    ours = dict(mods.named_parameters())
    assert sorted(ours) == sorted(k.replace("weight.factors.", "weight.factors.factor_") for k in params), "parameter names differ"
    with torch.no_grad():
        for k, v in params.items():
            ours[k.replace("weight.factors.", "weight.factors.factor_")].copy_(v)
    if device is not None:
        mods = mods.to(device)

    def forward(x):
        x = mods["lifting"](x)
        for i in range(n_layers):
            x = mods["fno_blocks"](x, i)
        return mods["projection"](x)
    return mods, forward
