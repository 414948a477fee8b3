"""Host-side checks of the head widths the DGL-API attention layers run at (no GPU needed)."""
import pytest

from re_gnn_b200.layer.conv import _kernel_head_dim


@pytest.mark.parametrize('width,kernel', [(3, 4), (128, 128), (129, 256), (200, 256), (256, 256), (300, 512),
                                          (349, 512), (512, 512)])
def test_kernel_head_dim_pads_to_a_power_of_two_up_to_512(width, kernel):
    assert _kernel_head_dim(width) == kernel


@pytest.mark.parametrize('width', [513, 1024])
def test_kernel_head_dim_refuses_heads_wider_than_512(width):
    with pytest.raises(ValueError, match='at most 512'):
        _kernel_head_dim(width)
