"""The reference's OWN test file for this path (`neuralop/layers/tests/test_spectral_convolution.py`: `test_SpectralConv` :7-90,
`test_SpectralConv2` :93-125) against `neuraloperator_b200.SpectralConv` on the GPU: its whole parameter grid (4 factorizations x 2
implementations x separable x 1-4 dims x real / complex data; Hermitian flag x dims x even / odd sizes x resolution scaling x modes)
and its assertions, as stated by `suite_factorized_vs_dense` / `suite_real_output_shapes` in tests/test_reference_suite_cpu.py (where
the same suite runs on CPU with the device primitives emulated and every result is also compared with stored results of the
reference class).
Closeness uses this repo's parity tolerance (1e-4 of max|ref|; contract 1e-3) instead of torch's fp32 defaults: the transforms run as
bf16x3 / fp32 table products.  (Named zzz_a: added after the round's GPU minutes were spent, so it runs after the tiers that were
validated on hardware.)"""
import pytest
import torch

from test_reference_suite_cpu import GRID_1, GRID_2, suite_factorized_vs_dense, suite_real_output_shapes

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(180, method="thread")]


@pytest.mark.parametrize("factorization,implementation,separable,dim,complex_data", GRID_1)
def test_SpectralConv(cuda_device, factorization, implementation, separable, dim, complex_data):
    suite_factorized_vs_dense(cuda_device, factorization, implementation, separable, dim, complex_data, 1e-4)
    torch.cuda.synchronize()


@pytest.mark.parametrize("enforce_hermitian_symmetry,dim,spatial_size,resolution_scaling_factor,modes", GRID_2)
def test_SpectralConv2(cuda_device, enforce_hermitian_symmetry, dim, spatial_size, modes, resolution_scaling_factor):
    suite_real_output_shapes(cuda_device, enforce_hermitian_symmetry, dim, spatial_size, resolution_scaling_factor, modes, 1e-4)
    torch.cuda.synchronize()
