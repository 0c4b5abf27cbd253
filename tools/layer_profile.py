#!/usr/bin/env python
"""Per-launch timing table of the denoiser (CUDA events around every launch, pnp_unet_profile)."""
import argparse, ctypes as C, json, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dt4image_restoration_b200 import _lib
from dt4image_restoration_b200.noise import UNetDenoiser2D, random_init_state_dict

ap = argparse.ArgumentParser(); ap.add_argument("--batch", type=int, default=64); ap.add_argument("--size", type=int, default=256)
ap.add_argument("--reps", type=int, default=5); ap.add_argument("--out", default="")
a = ap.parse_args()
B, S = a.batch, a.size
den = UNetDenoiser2D(state_dict=random_init_state_dict(0, "default")).to("cuda")
plan = den.plan(B, S, S)
v = torch.rand(B, 1, S, S, device="cuda"); sg = torch.full((B,), 0.1, device="cuda"); x = torch.empty_like(v)
l = _lib.lib()
blocks = [("inc", [(2, 32), (32, 32), (32, 32)], 0), ("down1", [(32, 64), (64, 64), (64, 64)], 1), ("down2", [(64, 128), (128, 128), (128, 128)], 2),
          ("down3", [(128, 256), (256, 256), (256, 256)], 3), ("down4", [(256, 512), (512, 512), (512, 512)], 4),
          ("up1", [(768, 256), (256, 256), (256, 256)], 3), ("up2", [(384, 128), (128, 128), (128, 128)], 2),
          ("up3", [(192, 64), (64, 64), (64, 64)], 1), ("up4", [(96, 32), (32, 32), (32, 32)], 0)]
info = {}
order = []
for bi, (bn, convs, lvl) in enumerate(blocks):
    if bn.startswith("up"): info[200 + lvl] = (f"{bn}.upsample", None); order.append(200 + lvl)
    for i, (ci, co) in enumerate(convs):
        info[bi * 3 + i] = (f"{bn}.conv{i} {ci}->{co} @{S >> lvl}", (ci, co, lvl)); order.append(bi * 3 + i)
CAP = 4096
n = C.c_int(CAP); ms = (C.c_float * CAP)(); kinds = (C.c_int * CAP)(); ids = (C.c_int * CAP)()
acc = {}
for r in range(a.reps + 1):
    n.value = CAP
    _lib.check(l.pnp_unet_profile(plan.handle, v.data_ptr(), sg.data_ptr(), x.data_ptr(), _lib.stream_ptr(), ms, kinds, ids, C.byref(n)))
    if r:
        for i in range(n.value): acc[ids[i]] = acc.get(ids[i], 0.0) + ms[i] / a.reps
rows = []
tot_f = tot_t = 0.0
T = sum(acc.values())
for k in order:
    name, sh = info[k]
    t = acc.get(k, 0.0)
    fl = 2.0 * 9 * sh[0] * sh[1] * (S >> sh[2]) ** 2 * B if sh else 0.0
    rows.append({"launch": name, "id": k, "ms": t, "gflop": fl / 1e9, "tflops": fl / (t * 1e-3) / 1e12 if sh and t else 0.0})
    if sh and k > 0: tot_f += fl; tot_t += t
print(f"launches per forward: {n.value}")
print(f"{'layer (all chunks summed)':34s} {'ms':>8s} {'GFLOP':>9s} {'TFLOP/s':>8s} {'share':>6s}")
for r in rows: print(f"{r['launch']:34s} {r['ms']:8.4f} {r['gflop']:9.1f} {r['tflops']:8.1f} {100 * r['ms'] / T:5.1f}%")
print(f"total {T:.3f} ms; tcgen05 convs {tot_t:.3f} ms = {tot_f / tot_t / 1e9:.1f} TFLOP/s; image-iters/s (denoiser only) {B / T * 1e3:.0f}")
if a.out: json.dump({"batch": B, "size": S, "rows": rows, "total_ms": float(T), "umma_tflops": tot_f / tot_t / 1e9}, open(a.out, "w"), indent=1)
