"""The Fourier-layer oracle (oracle/fno_block_oracle.py) against golden vectors minted from the UNMODIFIED reference `FNOBlocks`
(oracle/make_golden_block.py) and against stored results of the live class for fresh parameters: forward, dx and the gradient of
every parameter the layer touches.  CPU only."""
import pytest
import torch

from conftest import block_golden_index, block_oracle_kwargs, load_block_golden, reference_checks, stored_rel_err
from oracle import fno_block_oracle as BO
from oracle.make_golden_reference_checks import seeded_tensors

CASES = sorted(block_golden_index().keys())


def rel_err(a, ref):
    assert a.shape == ref.shape, (a.shape, ref.shape)
    return (a - ref).abs().max().item() / max(ref.abs().max().item(), 1e-20)


@pytest.mark.parametrize("name", CASES)
def test_block_oracle_matches_golden(name):
    meta, io, params, grads = load_block_golden(name)
    if "ada_in_embedding" in io:
        params = dict(params, ada_in_embedding=io["ada_in_embedding"])
    y, dx, g = BO.fno_block_fwd_bwd(io["x"], params, meta["index"], io["gy"], **block_oracle_kwargs(meta))
    g.pop("ada_in_embedding", None)
    assert list(y.shape[2:]) == meta["out_grid"]
    assert rel_err(y, io["y"]) < 2e-5, "y"
    assert rel_err(dx, io["dx"]) < 2e-5, "dx"
    assert sorted(g.keys()) == sorted(meta["touched"])         # the layer touches exactly the parameters the reference's does
    for pname in meta["touched"]:
        assert rel_err(g[pname], grads[pname]) < 2e-5, pname


LIVE_CASES = ["block_d2_default_mid", "block_d2_default_last", "block_d3_mid", "block_d2_tanh", "block_d2_preactivation_mid",
              "block_d2_upsample", "block_d2_no_mlp_mid", "block_d2_tucker"]


@pytest.mark.parametrize("name", LIVE_CASES)
def test_block_oracle_matches_live_reference(name):
    """Fresh random parameters and inputs (not the ones of the golden file), drawn from seeds, through the restatement, against what
    the reference class returned for them (oracle/make_golden_reference_checks.py)."""
    meta, io, params, _ = load_block_golden(name)
    store, checks = reference_checks()
    key = f"block_{name}"
    params = seeded_tensors([(k, tuple(v.shape), v.dtype) for k, v in params.items()], 99)
    gen = torch.Generator().manual_seed(100)
    x = torch.randn(*io["x"].shape, generator=gen, dtype=io["x"].dtype)
    gy = torch.randn(*store[f"{key}__y"][0], generator=gen, dtype=io["y"].dtype)
    y2, dx2, g2 = BO.fno_block_fwd_bwd(x, params, meta["index"], gy, **block_oracle_kwargs(meta))
    assert stored_rel_err(store, f"{key}__y", y2) < 1e-6
    assert stored_rel_err(store, f"{key}__dx", dx2) < 1e-6
    assert sorted(g2.keys()) == checks[key]["touched"]
    for pname in checks[key]["touched"]:
        assert stored_rel_err(store, f"{key}__g__{pname}", g2[pname]) < 1e-6, pname
