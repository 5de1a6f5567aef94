"""CPU suite: the nearest-2x upsample fold of the packed weights (program.up2_parity_weights) -- no device work."""
import pytest
import torch
import torch.nn.functional as F

from stable_diffusion_pytorch_b200.program import up2_parity_weights


@pytest.mark.parametrize("n, c, h, w", [(5, 3, 4, 6), (8, 16, 7, 5), (1, 1, 1, 1)])
def test_up2_parity_weights_equal_upsample_then_conv(n, c, h, w):
    """Output pixel (2i+py, 2j+px) of conv3x3(upsample2x(x)) is the 2x2 conv of parity (py, px) over the input window whose
    top-left pixel is (i-1+py, j-1+px)."""
    g = torch.Generator().manual_seed(n * 1000 + c * 100 + h * 10 + w)
    wt = torch.randn((n, c, 3, 3), generator=g, dtype=torch.float64)
    x = torch.randn((2, c, h, w), generator=g, dtype=torch.float64)
    ref = F.conv2d(F.interpolate(x, scale_factor=2, mode="nearest"), wt, padding=1)
    wp = up2_parity_weights(wt)
    assert wp.shape == (2, 2, n, c, 2, 2) and wp.dtype == torch.float64
    xp = F.pad(x, (1, 1, 1, 1))
    for py in (0, 1):
        for px in (0, 1):
            got = F.conv2d(xp, wp[py, px])[:, :, py:py + h, px:px + w]
            torch.testing.assert_close(got, ref[:, :, py::2, px::2], rtol=1e-12, atol=1e-12)
