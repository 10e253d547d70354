"""The 10 m step's entry points without a GPU: host tensors are refused before anything reaches the device, and the
C ABI declares the new symbols with the shapes the bindings use."""
import pytest
import torch

from hsr_b200 import _lib, kernels


def test_fine_entry_points_refuse_host_tensors():
    src = torch.zeros((3, 4, 5))
    coeffs = torch.zeros((3, 3), dtype=torch.float64)
    with pytest.raises(TypeError):
        kernels.bilinear_fine_mask(src, 6)
    with pytest.raises(TypeError):
        kernels.bilinear_apply(src, 6, coeffs)
    with pytest.raises(TypeError):
        kernels.masked_percentiles_union([(src, None)], (2, 98), factor=6)


def test_fine_symbols_are_bound():
    for name in ("hsr_bilinear_fine_mask_u8", "hsr_bilinear_apply_f32", "hsr_union_select_count_bilinear"):
        assert name in _lib.SIGNATURES
    assert len(_lib.SIGNATURES["hsr_bilinear_apply_f32"][1]) == 15
    assert len(_lib.SIGNATURES["hsr_union_select_count_bilinear"][1]) == 12
