#!/usr/bin/env python
"""Variable-density masks alone (pnp_variable_density_masks through the C-ABI), CUDA events over 200 launches after warm-up.

Per (size, B, accel) at power 3, plus power 0 at 256^2: us per call and the HBM floor of the mask write (B*H*W bytes at
7.7 TB/s, the data-sheet rate; nothing is read but accel and seeds).  Alongside each point, in the same run:
  - radial_masks at frac 0.3 on the same batch and size (the other seeded mask on the device);
  - simulate_measurements on the same batch with these masks (sigma_n = 10, with ATy0), i.e. the rest of making an episode;
    above 512^2 it is the dense-DFT path, timed over a ~1 s window instead of 200 launches;
  - torch.topk(largest=False, sorted=False) over the same float32 keys uploaded, ACS keys set to +inf, k = the number of
    non-ACS samples: the selection alone, without computing a key.  Keys come from tests/vd_reference.py for up to 16
    distinct seeds and are tiled over the batch.
Masks are checked against the reference for the first images of every point.

    python tools/vd_bench.py [--out profiles/r03_vd_bench.txt]
"""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from dt4image_restoration_b200 import _lib, ops  # noqa: E402
from vd_reference import acs_block, acs_size, keys, n_keep, vd_mask  # noqa: E402

SIZES = [128, 256, 512, 1024]
BATCHES = [1, 64, 256]
ACCELS = [2, 4, 8]
HBM = 7.7e12


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


def timed_window(fn, seconds=1.0, most=200):
    t1 = timed(fn, 1, warm=2)
    n = max(5, min(most, int(seconds / t1)))
    return timed(fn, n, warm=1), n


def main():
    lines = []

    def out(s):
        print(s, flush=True)
        lines.append(s)

    l = _lib.lib()
    st = _lib.stream_ptr()
    name, power, mhz = card()
    out(f"card: {name}, power limit {power} W, max SM clock {mhz:.0f} MHz")
    out("variable-density masks: one cluster per image, seeds = arange(B), ACS = max(1, round(0.08 N)) square; CUDA events "
        "over 200 launches after 10 warm-up launches; HBM floor = B*H*W bytes at 7.7 TB/s")
    warm = ops.variable_density_masks(256, 256, 256, 4, 0)        # the clocks leave their idle state first
    for _ in range(50):
        ops.variable_density_masks(256, 256, 256, 4, 0, out=warm)
    torch.cuda.synchronize()
    del warm
    points = [(N, B, a, 3) for N in SIZES for B in BATCHES for a in ACCELS] + [(256, B, a, 0) for B in BATCHES for a in ACCELS]
    ctx, host_keys = {}, {}
    for (N, B, accel, pw) in points:
        H = W = N
        a = acs_size(N)
        seeds = torch.arange(B, dtype=torch.int64, device="cuda")
        acc = torch.full((1,), accel, dtype=torch.int32, device="cuda")
        mask = torch.empty(B, H, W, dtype=torch.uint8, device="cuda")

        def fn():
            rc = l.pnp_variable_density_masks(acc.data_ptr(), 0, seeds.data_ptr(), a, a, pw, mask.data_ptr(), B, H, W, st)
            assert rc == 0, l.pnp_last_error()

        t = timed(fn, 200)
        got = mask[:2].cpu().numpy()
        for b in range(min(B, 2)):
            assert np.array_equal(got[b], vd_mask(H, W, accel, b, pw, a, a)), (N, B, accel, pw, b)
        if (N, B) not in ctx:                                  # radial and the simulator do not depend on accel
            fr = torch.full((1,), 0.3, dtype=torch.float64, device="cuda")
            rmask = torch.empty(B, H, W, dtype=torch.uint8, device="cuda")
            tr = timed(lambda: l.pnp_radial_masks(fr.data_ptr(), 0, seeds.data_ptr(), rmask.data_ptr(), None, B, H, W, st),
                       200)
            del rmask
            gt = torch.rand(B, 1, H, W, device="cuda")
            sig = torch.full((1,), 10.0, device="cuda")
            sim_out = tuple(torch.empty(B, 1, H, W, dtype=torch.complex64, device="cuda") for _ in range(3))

            def sim():
                rc = l.pnp_simulate_measurements(gt.data_ptr(), H * W, mask.data_ptr(), H * W, sig.data_ptr(), 0,
                                                 seeds.data_ptr(), sim_out[0].data_ptr(), sim_out[1].data_ptr(),
                                                 sim_out[2].data_ptr(), B, H, W, st)
                assert rc == 0, l.pnp_last_error()

            ts, ns = timed_window(sim) if N > 512 else (timed(sim, 200), 200)
            del gt, sim_out
            ctx[(N, B)] = (tr, ts, ns)
        tr, ts, ns = ctx[(N, B)]
        if (N, pw) not in host_keys:
            host = np.stack([keys(H, W, s, pw).reshape(-1) for s in range(16)])
            host[:, acs_block(H, W, a, a).reshape(-1)] = np.inf
            host_keys[(N, pw)] = host
        nd = min(B, 16)
        kt = torch.from_numpy(host_keys[(N, pw)][:nd]).cuda().repeat((B + nd - 1) // nd, 1)[:B].contiguous()
        extra = max(0, n_keep(H, W, accel) - a * a)
        ttk, ntk = timed_window(lambda: torch.topk(kt, extra, dim=1, largest=False, sorted=False), 2.0)
        del kt
        floor = B * H * W / HBM
        out(f"vd {N:4d}^2 B={B:3d} accel {accel} power {pw}: {t * 1e6:8.1f} us  (write floor {floor * 1e6:6.2f} us, "
            f"{floor / t:5.3f})  |  radial 0.3 {tr * 1e6:8.1f} us  |  simulate {ts * 1e6:10.1f} us ({ns} launches), "
            f"mask {t / (t + ts):.2f} of mask + simulate  |  torch.topk {ttk * 1e6:9.1f} us ({ntk} launches, "
            f"{ttk / t:5.2f}x the vd time)")
    if "--out" in sys.argv:
        path = sys.argv[sys.argv.index("--out") + 1]
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
