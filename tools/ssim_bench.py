#!/usr/bin/env python
"""SSIM kernel alone (pnp_ssim through the C-ABI, CUDA events over many launches after warm-up).

Per size: us per call, GB/s at 8 B per input pixel (x and gt read once), and the share of the two floors:
  HBM floor  = 8 B H W per image over the HBM bandwidth (7.7 TB/s, data sheet);
  FP32 floor = OPS_PER_PIXEL FMA-pipe operations per output pixel over (SMs x 128 lanes x max SM clock).
Sizes whose inputs fit the 126 MB L2 are read from L2 after the first launch (no cache flush between launches); the
script says which.  For context it also times the same metric written in PyTorch on the GPU (separable grouped conv2d
over a stacked [B, 5, H, W] tensor) and prints the max |diff| against it.
"""
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dt4image_restoration_b200 import _lib, ops  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
L2_BYTES = 126e6
FMA_LANES_PER_SM = 128
# FMA-pipe operations per output pixel: X.X, Y.Y, X.Y (3), the horizontal and the vertical 11-tap pass over five
# quantities (2 x 55), the SSIM formula (about 12; the division is not counted)
OPS_PER_PIXEL = 3 + 2 * 55 + 12
SIZES = [(1, 128), (64, 128), (1024, 128), (1, 256), (64, 256), (1024, 256), (1, 512), (64, 512), (1, 1024), (64, 1024)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, mhz = [s.strip() for s in q[torch.cuda.current_device()].split(",")]
    return name, power, float(mhz)


def torch_ssim(x, gt):
    X = x.clamp(0, 1)
    k = torch.arange(11, dtype=torch.float32, device=x.device)
    g = torch.exp(-(k - 5) ** 2 / (2 * 1.5 ** 2))
    g = g / g.sum()
    st = torch.cat([X, gt, X * X, gt * gt, X * gt], dim=1)                        # [B, 5, H, W]
    f = F.conv2d(F.conv2d(st, g.reshape(1, 1, 1, 11).expand(5, 1, 1, 11), groups=5),
                 g.reshape(1, 1, 11, 1).expand(5, 1, 11, 1), groups=5)
    mx, my, exx, eyy, exy = f.unbind(1)
    sxx, syy, sxy = exx - mx * mx, eyy - my * my, exy - mx * my
    c1, c2 = 0.01 ** 2, 0.03 ** 2
    m = ((2 * mx * my + c1) * (2 * sxy + c2)) / ((mx * mx + my * my + c1) * (sxx + syy + c2))
    return m.reshape(x.shape[0], -1).mean(1)


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(5):
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
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    fma_per_s = sms * FMA_LANES_PER_SM * mhz * 1e6
    print(f"card: {name}, power limit {power} W, max SM clock {mhz:.0f} MHz, {sms} SMs")
    warm = torch.rand(64, 1, 1024, 1024, device="cuda")
    warm_work = ops.aligned_empty(l.pnp_ssim_workspace_bytes(64, 1024, 1024), "cuda", align=16)
    warm_out = torch.empty(64, device="cuda")
    for _ in range(300):                                   # ~0.2 s of work: the clocks leave their idle state first
        l.pnp_ssim(warm.data_ptr(), warm.data_ptr(), 1024 * 1024, warm_out.data_ptr(), warm_work.data_ptr(), 64, 1024,
                   1024, _lib.stream_ptr())
    torch.cuda.synchronize()
    del warm, warm_work, warm_out
    print(f"floors: HBM {HBM_BYTES_PER_S / 1e12:.1f} TB/s (data sheet); FP32 {fma_per_s / 1e12:.1f} T FMA-pipe ops/s "
          f"at the max SM clock; {OPS_PER_PIXEL} ops per output pixel")
    for B, S in SIZES:
        H = W = S
        g = torch.Generator(device="cuda").manual_seed(B * 1000 + S)
        x = torch.rand(B, 1, H, W, device="cuda", generator=g) * 1.4 - 0.2
        gt = torch.rand(B, 1, H, W, device="cuda", generator=g)
        out = torch.empty(B, device="cuda")
        work = ops.aligned_empty(l.pnp_ssim_workspace_bytes(B, H, W), "cuda", align=16)

        def fn():
            rc = l.pnp_ssim(x.data_ptr(), gt.data_ptr(), H * W, out.data_ptr(), work.data_ptr(), B, H, W,
                            _lib.stream_ptr())
            assert rc == 0, l.pnp_last_error()

        in_bytes = 8 * B * H * W
        t = timed(fn, 200 if in_bytes < 1e9 else 50)
        t_hbm = in_bytes / HBM_BYTES_PER_S
        t_fma = B * (H - 10) * (W - 10) * OPS_PER_PIXEL / fma_per_s
        bound = "FP32" if t_fma >= t_hbm else "HBM"
        t_ref = timed(lambda: torch_ssim(x, gt), 20 if in_bytes < 1e9 else 5)
        diff = float((out - torch_ssim(x, gt)).abs().max())
        print(f"ssim {S:4d}x{S:<4d} B={B:4d}: {t * 1e6:8.1f} us  {in_bytes / t / 1e9:6.0f} GB/s  "
              f"FP32 floor {t_fma * 1e6:7.1f} us ({t_fma / t:4.2f})  HBM floor {t_hbm * 1e6:7.1f} us ({t_hbm / t:4.2f})  "
              f"bound: {bound}  inputs {in_bytes / 1e6:7.1f} MB {'fit' if in_bytes <= L2_BYTES else 'exceed'} L2  |  "
              f"torch conv2d {t_ref * 1e6:8.1f} us ({t_ref / t:5.1f}x)  max|d| {diff:.1e}")


if __name__ == "__main__":
    main()
