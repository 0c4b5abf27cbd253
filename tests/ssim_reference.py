"""Float64 SSIM on the CPU: the yardstick of the ``pnp_ssim`` kernel (tests only; the package never imports it).

Standard SSIM of Wang et al. (2004) in the form of pytorch-msssim / BasicSR: ``clamp(output, 0, 1)`` against ``gt`` (not
clamped), normalised 11-tap Gaussian window with sigma 1.5 applied separably with valid filtering, population moments,
C1 = 0.01^2, C2 = 0.03^2, mean over the (H-10) x (W-10) map.  It is not a restatement of the reference's
``calculate_ssim`` (evaluation/utils/transformations.py:61-95), which is not in this repository; parity with it is not
claimed.  It lives here rather than in ``oracle/``, whose functions restate reference code and are pinned to vectors the
reference produced.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F


def gaussian_window() -> torch.Tensor:
    k = torch.arange(11, dtype=torch.float64)
    g = torch.exp(-(k - 5) ** 2 / (2 * 1.5 ** 2))
    return g / g.sum()


def ssim(output: torch.Tensor, gt: torch.Tensor) -> torch.Tensor:
    """``[N,...,H,W]`` vs ``[N,...,H,W]`` or one shared ``[H,W]`` -> float64 ``[N,1]``."""
    N = output.shape[0]
    H, W = output.shape[-2:]
    X = torch.clamp(output.real if output.is_complex() else output, 0, 1).to(torch.float64).reshape(N, 1, H, W)
    Y = gt.to(torch.float64).reshape(-1, 1, H, W).expand(N, 1, H, W)
    g = gaussian_window()
    gh, gv = g.reshape(1, 1, 1, 11), g.reshape(1, 1, 11, 1)

    def filt(a):
        return F.conv2d(F.conv2d(a, gh), gv)

    mx, my = filt(X), filt(Y)
    sxx = filt(X * X) - mx * mx
    syy = filt(Y * Y) - my * my
    sxy = filt(X * Y) - mx * my
    c1, c2 = 0.01 ** 2, 0.03 ** 2
    m = ((2 * mx * my + c1) * (2 * sxy + c2)) / ((mx * mx + my * my + c1) * (sxx + syy + c2))
    return m.reshape(N, -1).mean(dim=1, keepdim=True)
