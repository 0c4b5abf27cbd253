"""Float64 restatement of each launch of the denoiser plan, with a per-element error bound (tests only; the package never
imports it).

Every function takes the launch's actual inputs (the NHWC bf16 tensors an earlier launch wrote, or the fp32 denoiser
input), computes the operation in float64 with plain torch (``conv2d``, ``max_pool2d``, ``interpolate``, ``pad``) on the
device of its inputs, and returns ``(ref, bound)`` in the layout of the launch's output.  A kernel is right when
``|got - ref| <= bound`` everywhere.  The bounds follow from what the kernels compute and how they round:

* ``S`` is the same convolution applied to ``|x|`` and ``|w|``, plus ``|b|``: the fp32 accumulation of the
  tensor-core convs errs by at most ``2^-12 S``, the 19-term CUDA-core first conv by at most ``2^-20 S``;
* a bf16 output is the fp32 value rounded once (relative ``2^-9``; the bound allows ``2^-8``);
* LeakyReLU is 1-Lipschitz, so a pre-activation bound carries through it;
* the upsample's fp32 interpolation weights ``s u - floor(s u)`` with ``s = (h-1)/(2h-1)`` rounded to fp32 err by up
  to ``2^-23 h`` (the product ``s u`` is below ``h``), which moves the result by that much times the corner spread;
* the max pool and the clamp of the FINAL epilogue are exact.

What the launches restate (reference evaluation/noise.py): the noise-level-map concat and the first conv
(noise.py:161-162, fp32 weights), ``ConvLayer`` (noise.py:75-89, bf16 weights, fp32 bias), ``MaxPool2d(2)`` (floor
mode, noise.py:23), ``up``'s x2 bilinear upsample with ``align_corners=True`` and its zero pad (noise.py:39,46-53), the
skip-first concat (noise.py:59), and the 1x1 output conv plus the global residual (noise.py:64-71, 132-133).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

SLOPE = 0.2
REL_BF16 = 2.0 ** -8          # bf16 output rounding (2^-9) with a factor 2 to spare
ACC_UMMA = 2.0 ** -12         # fp32 accumulation of the tensor-core convs, relative to S
ACC_FIRST = 2.0 ** -20        # fp32 accumulation of the 19-term first conv, relative to S
ARITH_FINAL = 2.0 ** -18      # fp32 arithmetic of the 33-term 1x1 conv and the residual add


def nchw(t: torch.Tensor) -> torch.Tensor:
    """NHWC (any dtype) -> NCHW float64."""
    return t.to(torch.float64).permute(0, 3, 1, 2)


def nhwc(t: torch.Tensor) -> torch.Tensor:
    return t.permute(0, 2, 3, 1).contiguous()


def bf16r(t: torch.Tensor) -> torch.Tensor:
    """Round to bf16 (round to nearest even) and return float64."""
    return t.to(torch.bfloat16).to(torch.float64)


def _conv_with_s(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor):
    """(conv2d(x, w) + b, conv2d(|x|, |w|) + |b|), 3x3, zero pad 1, float64 NCHW."""
    w = w.to(x.device, torch.float64)
    b = b.to(x.device, torch.float64)
    pre = F.conv2d(x, w, b, padding=1)
    s = F.conv2d(x.abs(), w.abs(), b.abs(), padding=1)
    return pre, s


def first_conv(v: torch.Tensor, sigma: torch.Tensor, w: torch.Tensor, b: torch.Tensor):
    """``v`` [B,H,W] fp32, ``sigma`` [B]; ``w`` fp32 [32,2,3,3], ``b`` [32] -> NHWC [B,H,W,32]."""
    B, H, W = v.shape
    x = torch.stack([v.to(torch.float64), sigma.to(v.device, torch.float64).view(B, 1, 1).expand(B, H, W)], dim=1)
    pre, s = _conv_with_s(x, w, b)
    ref = F.leaky_relu(pre, SLOPE)
    return nhwc(ref), nhwc(REL_BF16 * ref.abs() + ACC_FIRST * s)


def conv3x3(in0: torch.Tensor, in1: torch.Tensor | None, w: torch.Tensor, b: torch.Tensor):
    """bf16 epilogue conv: ``cat(in0, in1)`` (skip segment first) NHWC, ``w`` [Cout,Cin,3,3] as the kernel holds it
    (bf16-rounded for the tensor-core convs), fp32 ``b`` -> NHWC [B,H,W,Cout]."""
    x = nchw(in0 if in1 is None else torch.cat([in0, in1], dim=-1))
    pre, s = _conv_with_s(x, w, b)
    ref = F.leaky_relu(pre, SLOPE)
    return nhwc(ref), nhwc(REL_BF16 * ref.abs() + ACC_UMMA * s)


def maxpool(out: torch.Tensor) -> torch.Tensor:
    """MaxPool2d(2), floor mode, of the launch's own NHWC output: exact, so compared bit for bit."""
    return nhwc(F.max_pool2d(nchw(out), 2))


def upsample(x: torch.Tensor, Ho: int, Wo: int):
    """x2 bilinear upsample (align_corners=True) of NHWC ``x`` [B,h,w,C], zero-padded to [B,Ho,Wo,C] with the pad split
    (dx // 2, dx - dx // 2) as noise.py:49-53.  Returns (ref, bound, inside): ``inside`` is the [Ho,Wo] bool map of the
    upsampled region; outside it the output must be exactly 0 (and the bound is 0)."""
    B, h, w, C = x.shape
    xd = nchw(x)
    up = F.interpolate(xd, scale_factor=2, mode="bilinear", align_corners=True)
    # largest |corner| of each output pixel: the source rows / columns it interpolates between
    def src(n_in):
        u = torch.arange(2 * n_in, dtype=torch.float64, device=x.device)
        pos = u * (n_in - 1) / max(2 * n_in - 1, 1)
        i0 = pos.floor().long().clamp(0, n_in - 1)
        return i0, (i0 + 1).clamp(max=n_in - 1)
    y0, y1 = src(h)
    x0, x1 = src(w)
    a = xd.abs()
    rows = torch.maximum(a[:, :, y0, :], a[:, :, y1, :])
    corner = torch.maximum(rows[:, :, :, x0], rows[:, :, :, x1])
    bound = REL_BF16 * up.abs() + (2.0 ** -22 * (h + w) + 2.0 ** -20) * corner
    dy, dx = Ho - 2 * h, Wo - 2 * w
    pad = (dx // 2, dx - dx // 2, dy // 2, dy - dy // 2)
    inside = torch.zeros(1, 1, 2 * h, 2 * w, dtype=torch.float64, device=x.device)
    inside = F.pad(inside + 1, pad)[0, 0] > 0
    return nhwc(F.pad(up, pad)), nhwc(F.pad(bound, pad)), inside


def final(in0: torch.Tensor, w: torch.Tensor, b: torch.Tensor, wout: torch.Tensor, bout: torch.Tensor, v: torch.Tensor):
    """FINAL epilogue: 3x3 conv (bf16 weights) + bias + LeakyReLU, un-rounded, then the 1x1 output conv with fp32
    ``wout`` [32] / ``bout`` [1], plus the denoiser input ``v`` [B,H,W].  Returns the preclamp (ref, bound) [B,H,W]."""
    x = nchw(in0)
    pre, s = _conv_with_s(x, w, b)
    a = F.leaky_relu(pre, SLOPE)
    wo = wout.to(x.device, torch.float64).reshape(1, -1, 1, 1)
    bo = bout.to(x.device, torch.float64).reshape(())
    vv = v.to(x.device, torch.float64).reshape(a.shape[0], a.shape[2], a.shape[3])
    ref = vv + (a * wo).sum(dim=1) + bo
    bound = (ACC_UMMA * (s * wo.abs()).sum(dim=1)
             + ARITH_FINAL * ((a * wo).abs().sum(dim=1) + bo.abs() + vv.abs()))
    return ref, bound


def compare(got: torch.Tensor, ref: torch.Tensor, bound: torch.Tensor):
    """(max err / bound, index of that element, number of elements over their bound).  A zero bound demands equality."""
    err = (got.to(torch.float64) - ref.to(got.device, torch.float64)).abs()
    bound = bound.to(err.device)
    ratio = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, torch.inf, 0.0))
    ratio = torch.nan_to_num(ratio, nan=torch.inf)
    flat = int(ratio.argmax())
    idx = []
    for n in reversed(ratio.shape):
        idx.append(flat % n)
        flat //= n
    return float(ratio.max()), tuple(reversed(idx)), int((ratio > 1).sum())
