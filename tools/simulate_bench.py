#!/usr/bin/env python
"""Measurement simulator alone (pnp_simulate_measurements through the C-ABI, CUDA events over many launches after warm-up).

Per size: us per call with and without ATy0, and the share of the HBM floor at the algorithmic bytes - read gt 4 and
mask 1, write y0, x0 and ATy0 8 each: 29 B per pixel (21 B without ATy0) - over the data sheet's 7.7 TB/s.  The three
passes move about 61 B per pixel (T is written and read twice in x0), so about 0.5 of the floor is the most this path can
reach.  Sizes whose 29 B/pixel working set fits the 126 MB L2 stay there between launches (no cache flush); the script
says which.  For context it times the same computation written in PyTorch on the GPU (shifts, torch.fft.fft2 with
norm='ortho', torch.randn noise, mask, inverse, clamp) and prints the max |diff| of y0 and x0 against it with sigma_n = 0.
"""
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dt4image_restoration_b200 import _lib, ops  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
L2_BYTES = 126e6
SIZES = [(1, 256, 256), (64, 256, 256), (256, 256, 256), (64, 512, 512), (64, 130, 130)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, mhz = [s.strip() for s in q[torch.cuda.current_device()].split(",")]
    return name, power, float(mhz)


def torch_simulate(gt, mask, sigma_n):
    """The PyTorch composition a user would write: [B,H,W] fp32 gt, bool mask, scalar sigma_n -> (y0, x0, ATy0)."""
    dims = (-2, -1)
    k = torch.fft.fftshift(torch.fft.fft2(torch.fft.ifftshift(gt, dim=dims), norm="ortho"), dim=dims)
    if sigma_n > 0:
        k = k + (sigma_n / 255.0) * torch.randn_like(k)        # complex randn: variance 1 split over re / im
    y0 = k * mask
    aty0 = torch.fft.fftshift(torch.fft.ifft2(torch.fft.ifftshift(y0, dim=dims), norm="ortho"), dim=dims)
    x0 = torch.view_as_complex(torch.view_as_real(aty0).clamp(min=0))
    return y0, x0, aty0


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(10):
        fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e-3


def main():
    l = _lib.lib()
    name, power, mhz = card()
    print(f"card: {name}, power limit {power} W, max SM clock {mhz:.0f} MHz")
    print(f"floor: HBM {HBM_BYTES_PER_S / 1e12:.1f} TB/s (data sheet); 29 B/pixel with ATy0, 21 B/pixel without")
    warm = torch.rand(64, 1, 512, 512, device="cuda")
    wm = torch.ones(1, 512, 512, dtype=torch.uint8, device="cuda")
    wout = tuple(torch.empty(64, 1, 512, 512, dtype=torch.complex64, device="cuda") for _ in range(3))
    for _ in range(200):                                   # the clocks leave their idle state first
        ops.simulate_measurements(warm, wm, 10.0, 0, out=wout)
    torch.cuda.synchronize()
    del warm, wm, wout
    for B, H, W in SIZES:
        g = torch.Generator(device="cuda").manual_seed(B * 1000 + H)
        gt = torch.rand(B, 1, H, W, device="cuda", generator=g)
        mask = ops.cartesian_masks(B, H, W, 4, 0)
        sig = torch.full((1,), 10.0, device="cuda")
        seeds = torch.arange(B, dtype=torch.int64, device="cuda")
        y0, x0, at = (torch.empty(B, 1, H, W, dtype=torch.complex64, device="cuda") for _ in range(3))
        st = _lib.stream_ptr()

        def fn(aty0=True):
            rc = l.pnp_simulate_measurements(gt.data_ptr(), H * W, mask.data_ptr(), H * W, sig.data_ptr(), 0,
                                             seeds.data_ptr(), y0.data_ptr(), x0.data_ptr(),
                                             at.data_ptr() if aty0 else None, B, H, W, st)
            assert rc == 0, l.pnp_last_error()

        px = B * H * W
        t = timed(fn, 200)
        t21 = timed(lambda: fn(False), 200)
        f29, f21 = 29 * px / HBM_BYTES_PER_S, 21 * px / HBM_BYTES_PER_S
        mb = mask.reshape(B, 1, H, W).bool()
        t_ref = timed(lambda: torch_simulate(gt, mb, 10.0), 50)
        ry0, rx0, _ = torch_simulate(gt, mb, 0.0)
        gy0, gx0, _ = ops.simulate_measurements(gt, mask, 0.0, seeds)
        dy = float((gy0 - ry0).abs().max() / ry0.abs().max())
        dx = float((gx0 - rx0).abs().max())
        path = "radix" if (H & (H - 1)) == 0 and (W & (W - 1)) == 0 else "dense DFT"
        print(f"simulate {H:4d}x{W:<4d} B={B:4d} ({path:9s}): {t * 1e6:8.1f} us (HBM floor {f29 * 1e6:6.1f} us, "
              f"{f29 / t:4.2f})  no ATy0 {t21 * 1e6:8.1f} us ({f21 / t21:4.2f})  29 B/px set {29 * px / 1e6:6.1f} MB "
              f"{'fits' if 29 * px <= L2_BYTES else 'exceeds'} L2  |  torch {t_ref * 1e6:8.1f} us ({t_ref / t:5.1f}x)  "
              f"sigma 0: max|dy0|/max|y0| {dy:.1e}, max|dx0| {dx:.1e}")
    passes(64, 256, 256)
    passes(64, 512, 512)


def passes(B, H, W, iters=50):
    """Per-kernel device time of the three passes from torch.profiler (a separate run after the timed ones)."""
    from torch.profiler import ProfilerActivity, profile
    gt = torch.rand(B, 1, H, W, device="cuda")
    mask = ops.cartesian_masks(B, H, W, 4, 0)
    out = tuple(torch.empty(B, 1, H, W, dtype=torch.complex64, device="cuda") for _ in range(3))
    ops.simulate_measurements(gt, mask, 10.0, 0, out=out)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            ops.simulate_measurements(gt, mask, 10.0, 0, out=out)
        torch.cuda.synchronize()
    px = B * H * W
    # B/pixel each pass moves (ATy0 written); the op type names the pass: radix_rows_kernel<N, SimRowsFwd> etc.
    pass_bytes = {"SimRowsFwd": 12, "SimCols": 25, "SimRowsInv": 24}
    for ev in prof.key_averages():
        for k, nb in pass_bytes.items():
            if k in ev.key:
                us = ev.device_time                          # average over the calls, us
                print(f"  pass {k:13s} {H}x{W} B={B}: {us:7.1f} us  {nb * px / (us * 1e-6) / 1e12:5.2f} TB/s at {nb} B/pixel")


if __name__ == "__main__":
    main()
