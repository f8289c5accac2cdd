"""Host-side planning of the block-1 input-gradient entry point (no GPU needed): which implementation TMF_CONV_AUTO picks,
read through the workspace it asks for (the tcgen05 kernel needs none, the CUDA-core path stages dy)."""
from transmf_ad_b200 import _lib as L


def _ws(ng, impl, B, D, H, W, cout=32):
    return int(L.load().tmf_conv1_dgrad_fused_workspace_bytes(ng, impl, B, D, H, W, cout))


def _dy_bytes(B, D, H, W, cout=32):
    return (B * D * H * W * cout * 2 + 255) // 256 * 256


def test_auto_takes_tcgen05_up_to_128_columns(built_lib):
    assert _ws(2, L.CONV_AUTO, 8, 91, 109, 91) == 0
    assert _ws(1, L.CONV_AUTO, 1, 3, 5, 128) == 0
    assert _ws(1, L.CONV_UMMA, 2, 11, 13, 12) == 0


def test_auto_routes_wide_rows_and_other_widths_to_cuda_cores(built_lib):
    assert _ws(1, L.CONV_AUTO, 1, 6, 7, 133) == _dy_bytes(1, 6, 7, 133)
    assert _ws(2, L.CONV_AUTO, 2, 9, 9, 9, cout=16) == 2 * _dy_bytes(2, 9, 9, 9, cout=16)
    assert _ws(2, L.CONV_DIRECT, 8, 91, 109, 91) == 2 * _dy_bytes(8, 91, 109, 91)
