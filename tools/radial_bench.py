#!/usr/bin/env python
"""Radial masks alone (pnp_radial_masks through the C-ABI, CUDA events over many launches after warm-up).

Per (B, size, frac): us per call, the number of lines (the mean and the largest of the batch: one CTA per image draws its
lines in order, so the image with the most lines is the critical path) and us per line on that path.  Masks are small
(B*H*W bytes written, nothing read but frac and seeds), so the time is the sequential per-line loop, not HBM; nothing is
flushed between launches.  For context: synth.radial_mask's host time for one mask times B (the host loop makes every
distinct mask separately, which is what a per-episode seeded mask asks of it), and ops.simulate_measurements at the same
batch and size (sigma_n = 10, with ATy0), so the mask's share of making an episode on the device is visible.
"""
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dt4image_restoration_b200 import _lib, ops, synth  # noqa: E402

BATCHES = [1, 64, 256]
SIZES = [128, 256, 512, 1024]
FRACS = [0.2, 0.3]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, mhz = [s.strip() for s in q[torch.cuda.current_device()].split(",")]
    return name, power, float(mhz)


def timed(fn, iters, warm=10):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e-3


def host_time(H, W, frac):
    reps = 5 if H * W <= 256 * 256 else 2
    t0 = time.perf_counter()
    for _ in range(reps):
        synth.radial_mask(H, W, frac)
    return (time.perf_counter() - t0) / reps


def main():
    l = _lib.lib()
    name, power, mhz = card()
    print(f"card: {name}, power limit {power} W, max SM clock {mhz:.0f} MHz")
    print("radial masks: one CTA of 512 threads per image, seeds = arange(B) (rotated patterns), CUDA events over 200 "
          "launches after 10 warm-up launches; simulate = ops.simulate_measurements on the same masks")
    st = _lib.stream_ptr()
    warm = ops.radial_masks(256, 256, 256, 1.0, 0)          # the clocks leave their idle state first
    for _ in range(50):
        ops.radial_masks(256, 256, 256, 1.0, 0, out=warm)
    torch.cuda.synchronize()
    for N in SIZES:
        H = W = N
        host = {f: host_time(H, W, f) for f in FRACS}
        for B in BATCHES:
            seeds = torch.arange(B, dtype=torch.int64, device="cuda")
            mask = torch.empty(B, H, W, dtype=torch.uint8, device="cuda")
            lines = torch.empty(B, dtype=torch.int32, device="cuda")
            for f in FRACS:
                fr = torch.full((1,), f, dtype=torch.float64, device="cuda")

                def fn():
                    rc = l.pnp_radial_masks(fr.data_ptr(), 0, seeds.data_ptr(), mask.data_ptr(), lines.data_ptr(), B, H, W,
                                            st)
                    assert rc == 0, l.pnp_last_error()

                t = timed(fn, 200)
                n_mean, n_max = float(lines.double().mean()), int(lines.max())
                print(f"radial {H:4d}x{W:<4d} B={B:4d} frac {f:.1f}: {t * 1e6:8.1f} us per call  lines mean {n_mean:6.1f} "
                      f"max {n_max:4d}  {t * 1e6 / n_max:6.3f} us per line  |  synth.radial_mask x B on the host "
                      f"{host[f] * B * 1e3:10.1f} ms ({host[f] * B / t:9.0f}x)", flush=True)
            gt = torch.rand(B, 1, H, W, device="cuda")
            sig = torch.full((1,), 10.0, device="cuda")
            outs = tuple(torch.empty(B, 1, H, W, dtype=torch.complex64, device="cuda") for _ in range(3))

            def sim():
                rc = l.pnp_simulate_measurements(gt.data_ptr(), H * W, mask.data_ptr(), H * W, sig.data_ptr(), 0,
                                                 seeds.data_ptr(), outs[0].data_ptr(), outs[1].data_ptr(),
                                                 outs[2].data_ptr(), B, H, W, st)
                assert rc == 0, l.pnp_last_error()

            t1 = timed(sim, 1, warm=2)                       # one launch sizes the timed window to about a second
            iters = max(5, min(200, int(1.0 / t1)))
            ts = timed(sim, iters, warm=2)
            t3 = timed(fn, 200)                              # the mask at frac 0.3 again, next to the simulator
            path = "radix" if N <= 512 else "dense DFT"
            print(f"  simulate {H}x{W} B={B} ({path}, {iters} launches): {ts * 1e6:10.1f} us; radial mask (frac 0.3) "
                  f"{t3 * 1e6:8.1f} us = {t3 / (t3 + ts):.2f} of mask + simulate", flush=True)
            del gt, outs
    for B, N in ((1, 256), (148, 256), (1, 1024), (148, 1024)):   # long loops: the per-line cost without fixed costs
        seeds = torch.arange(B, dtype=torch.int64, device="cuda")
        mask = torch.empty(B, N, N, dtype=torch.uint8, device="cuda")
        lines = torch.empty(B, dtype=torch.int32, device="cuda")
        t = timed(lambda: ops.radial_masks(B, N, N, 1.0, seeds, out=mask, lines_out=lines), 20, warm=3)
        n_max = int(lines.max())
        print(f"radial {N}x{N} B={B} frac 1.0: {t * 1e6:9.1f} us per call, max lines {n_max}, "
              f"{t * 1e6 / n_max:6.3f} us per line", flush=True)


if __name__ == "__main__":
    main()
