#!/usr/bin/env python
"""Bitwise A/B of the line-pass paths against libpnp_b200.so built from another commit, with timing.

    python tools/line_pass_ab.py --old-lib PATH

Build the other library from a git worktree of that commit with the same build module
(``python -m dt4image_restoration_b200.build``) and pass its ``csrc/libpnp_b200.so``.  This tree's library is loaded
through ``_lib``, the other one with ``ctypes.CDLL`` and ``_lib.SIGNATURES``.  Both run the same seeded inputs through
pnp_fft2c (forward, inverse, in place), pnp_prox_dual (per-image and shared masks, mu of 1 and of B entries, v on and off),
pnp_prox_prepare + pnp_prox_dual_prepared_kind (kinds -1 / 0 / 1), pnp_step_prepared_active (the per-image active
predicate) and pnp_simulate_measurements (with and without ATy0, shared gt / mask, unaligned gt), at radix and dense-DFT
sizes, and every output buffer must be torch.equal.  Then old and new are timed alternately (CUDA events, warm-up, several
rounds, median per call) at user sizes, and old against old in the same way, which is the noise floor of the ratio.
"""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dt4image_restoration_b200 import _lib, ops  # noqa: E402

DEV = "cuda"
RADIX = [(32, 32), (64, 128), (128, 64), (512, 512)]
DENSE = [(2, 3), (130, 130), (136, 120), (1000, 1024)]


def load_old(path):
    lib = C.CDLL(os.path.abspath(path))
    for name, (res, args) in _lib.SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    rc = lib.pnp_init()
    assert rc == 0, lib.pnp_last_error()
    return lib


def call(lib, name, *args):
    rc = getattr(lib, name)(*args)
    assert rc == 0, f"{name}: {rc} {lib.pnp_last_error()}"


def ptr(t):
    return None if t is None else t.data_ptr()


class Checker:
    def __init__(self):
        self.n, self.bad = 0, []

    def eq(self, what, a, b):
        self.n += 1
        if not torch.equal(a, b):
            d = (a.view(torch.float32) - b.view(torch.float32)).abs().max().item() if a.is_floating_point() or \
                a.is_complex() else float("nan")
            self.bad.append(what)
            print(f"  DIFFERS: {what} (max |diff| {d:.3e})")


def cplx(g, *shape):
    return torch.complex(torch.randn(*shape, generator=g), torch.randn(*shape, generator=g)).to(DEV)


def ab_fft2c(libs, ck, B, H, W):
    g = torch.Generator().manual_seed(H * 131 + W)
    src = cplx(g, B, 1, H, W)
    st = _lib.stream_ptr()
    for inv in (0, 1):
        outs = []
        for L in libs:
            dst = torch.full_like(src, float("nan"))
            call(L, "pnp_fft2c", ptr(src), ptr(dst), B, H, W, inv, st)
            inplace = src.clone()
            call(L, "pnp_fft2c", ptr(inplace), ptr(inplace), B, H, W, inv, st)
            outs.append((dst, inplace))
        for k, nm in enumerate(("dst", "in place")):
            ck.eq(f"fft2c {H}x{W} B={B} inverse={inv} {nm}", outs[0][k], outs[1][k])


def prox_inputs(B, H, W, per_image_mask, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 1, H, W, generator=g).to(DEV)
    u = cplx(g, B, 1, H, W) * 0.1
    y0 = cplx(g, B, 1, H, W)
    nb = B if per_image_mask else 1
    mask = (torch.rand(nb, 1, H, W, generator=g) < 0.3).to(torch.uint8).to(DEV)
    return x, u, y0, mask


def ab_prox(libs, ck, B, H, W):
    st = _lib.stream_ptr()
    for per_image in (True, False):
        x, u, y0, mask = prox_inputs(B, H, W, per_image, H * 7 + W + per_image)
        for mu_n, want_v in ((1, True), (B, False)):
            mu = torch.linspace(0.2, 0.9, mu_n).to(DEV)
            outs = []
            for L in libs:
                z, un = torch.full_like(u, float("nan")), torch.full_like(u, float("nan"))
                v = torch.full_like(x, float("nan")) if want_v else None
                work = ops.aligned_empty(L.pnp_prox_workspace_bytes(B, H, W), DEV)
                call(L, "pnp_prox_dual", ptr(x), ptr(u), ptr(y0), ptr(mask), H * W if per_image else 0, ptr(mu),
                     0 if mu_n == 1 else 1, ptr(z), ptr(un), ptr(v), ptr(work), B, H, W, st)
                outs.append((z, un, v))
            tag = f"prox {H}x{W} B={B} mask {'per image' if per_image else 'shared'} mu[{mu_n}] v {'on' if want_v else 'off'}"
            for k, nm in enumerate(("z", "u", "v")):
                if outs[0][k] is not None:
                    ck.eq(f"{tag}: {nm}", outs[0][k], outs[1][k])


def prepared_buffers(L, B, H, W):
    yb, mb = C.c_size_t(), C.c_size_t()
    call(L, "pnp_prox_prepared_bytes", B, H, W, C.byref(yb), C.byref(mb))
    return ops.aligned_empty(yb.value, DEV).zero_(), ops.aligned_empty(mb.value, DEV).zero_()


def ab_prepared(libs, ck, B, H, W):
    st = _lib.stream_ptr()
    g = torch.Generator().manual_seed(H + 5)
    cols = (torch.rand(B, 1, 1, W, generator=g) < 0.3).expand(B, 1, H, W).to(torch.uint8).contiguous().to(DEV)
    for mask_kind, mask, kinds in (("column-only per image", cols, (-1, 1)), ("general shared", None, (-1, 0))):
        x, u, y0, gmask = prox_inputs(B, H, W, False, H * 3 + 1)
        if mask is None:
            mask = gmask
        mstride = H * W if mask.shape[0] == B else 0
        mu = torch.linspace(0.3, 0.7, B).to(DEV)
        for kind in kinds:
            outs = []
            for L in libs:
                y0p, maskp = prepared_buffers(L, B, H, W)
                call(L, "pnp_prox_prepare", ptr(y0), ptr(mask), mstride, ptr(y0p), ptr(maskp), B, H, W, st)
                z, un, v = torch.zeros_like(u), torch.zeros_like(u), torch.zeros_like(x)
                call(L, "pnp_prox_dual_prepared_kind", ptr(x), ptr(u), ptr(y0p), ptr(maskp), mstride, ptr(mu), 1, ptr(z),
                     ptr(un), ptr(v), B, H, W, kind, st)
                outs.append((y0p, maskp, z, un, v))
            for k, nm in enumerate(("y0p (copies, Yt, scratch)", "maskp", "z", "u", "v")):
                ck.eq(f"prepared {H}x{W} B={B} {mask_kind} kind {kind}: {nm}", outs[0][k], outs[1][k])


def ab_active(libs, ck, B, H, W):
    """pnp_step_prepared_active: inactive images keep x, z, u, v (the prox epilogue's per-image predicate)."""
    st = _lib.stream_ptr()
    g = torch.Generator().manual_seed(11)
    flat = (torch.randn(_lib.load().pnp_unet_num_params(), generator=g) * 0.05).to(DEV)
    x, u, y0, mask = prox_inputs(B, H, W, True, H + 17)
    vin = torch.rand(B, 1, H, W, generator=g).to(DEV)
    sigma = torch.full((B,), 0.1, device=DEV)
    mu = torch.full((1,), 0.5, device=DEV)
    active = torch.tensor([1, 0] * (B // 2) + [1] * (B % 2), dtype=torch.uint8, device=DEV)
    for kind in (-1, 0):
        outs = []
        for L in libs:
            packed = ops.aligned_empty(L.pnp_unet_packed_bytes(), DEV).zero_()
            call(L, "pnp_unet_pack_weights", ptr(flat), ptr(packed), st)
            nbytes = L.pnp_unet_workspace_bytes(B, H, W)
            ws = ops.aligned_empty(nbytes, DEV)
            h = C.c_void_p()
            call(L, "pnp_unet_plan_create", C.byref(h), ptr(packed), ptr(ws), nbytes, B, H, W)
            y0p, maskp = prepared_buffers(L, B, H, W)
            call(L, "pnp_prox_prepare", ptr(y0), ptr(mask), H * W, ptr(y0p), ptr(maskp), B, H, W, st)
            xs, zs, us, vs = x.clone(), torch.zeros_like(u), u.clone(), vin.clone()
            call(L, "pnp_step_prepared_active", h, ptr(vs), ptr(sigma), ptr(us), ptr(y0p), ptr(maskp), H * W, ptr(mu), 0,
                 ptr(xs), ptr(zs), ptr(us), ptr(vs), kind, ptr(active), st)
            torch.cuda.synchronize()
            L.pnp_unet_plan_destroy(h)
            outs.append((xs, zs, us, vs))
        for k, nm in enumerate(("x", "z", "u", "v")):
            ck.eq(f"step active {H}x{W} B={B} kind {kind}: {nm}", outs[0][k], outs[1][k])


def ab_simulate(libs, ck, B, H, W):
    st = _lib.stream_ptr()
    g = torch.Generator().manual_seed(H * 3 + W)
    base = torch.rand(B * H * W + 1, generator=g).to(DEV)
    masks = (torch.rand(B, H, W, generator=g) < 0.4).to(torch.uint8).to(DEV)
    sigma = torch.linspace(0.0, 20.0, B).to(DEV)
    seeds = torch.arange(100, 100 + B, dtype=torch.int64, device=DEV)
    cases = [("per-image gt/mask, ATy0", base[:B * H * W], H * W, masks, H * W, True),
             ("per-image, no ATy0", base[:B * H * W], H * W, masks, H * W, False),
             ("shared gt and mask", base[:H * W], 0, masks[:1], 0, True),
             ("unaligned gt", base[1:], H * W, masks, H * W, True)]
    for name, gt, gstride, mask, mstride, want_aty0 in cases:
        outs = []
        for L in libs:
            y0, x0 = (torch.full((B, H, W), float("nan"), dtype=torch.complex64, device=DEV) for _ in range(2))
            aty0 = torch.full_like(y0, float("nan")) if want_aty0 else None
            call(L, "pnp_simulate_measurements", ptr(gt), gstride, ptr(mask), mstride, ptr(sigma), 1, ptr(seeds), ptr(y0),
                 ptr(x0), ptr(aty0), B, H, W, st)
            outs.append((y0, x0, aty0))
        for k, nm in enumerate(("y0", "x0", "ATy0")):
            if outs[0][k] is not None:
                ck.eq(f"simulate {H}x{W} B={B} {name}: {nm}", outs[0][k], outs[1][k])


# ---------------------------------------------------------------- timing
def time_pair(fa, fb, iters, rounds=7):
    """Median us per call of fa and fb, timed alternately with CUDA events after a warm-up."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for f in (fa, fb):
        for _ in range(max(3, iters // 4)):
            f()
    torch.cuda.synchronize()
    ta, tb = [], []
    for _ in range(rounds):
        for f, acc in ((fa, ta), (fb, tb)):
            ev[0].record()
            for _ in range(iters):
                f()
            ev[1].record()
            torch.cuda.synchronize()
            acc.append(ev[0].elapsed_time(ev[1]) * 1e3 / iters)
    return statistics.median(ta), statistics.median(tb)


def timed_cases(old, new):
    st = _lib.stream_ptr()
    cases = []

    def prox(B, H, W):
        x, u, y0, mask = prox_inputs(B, H, W, True, 3)
        mu = torch.full((1,), 0.5, device=DEV)
        bufs = {}
        for L in (old, new):
            bufs[id(L)] = (torch.empty_like(u), torch.empty_like(u), torch.empty_like(x),
                           ops.aligned_empty(L.pnp_prox_workspace_bytes(B, H, W), DEV))

        def run(L):
            z, un, v, work = bufs[id(L)]
            call(L, "pnp_prox_dual", ptr(x), ptr(u), ptr(y0), ptr(mask), H * W, ptr(mu), 0, ptr(z), ptr(un), ptr(v),
                 ptr(work), B, H, W, st)
        return run

    def simulate(B, H, W):
        g = torch.Generator().manual_seed(B + H)
        gt = torch.rand(B, H, W, generator=g).to(DEV)
        mask = ops.cartesian_masks(B, H, W, 4, 0)
        sig = torch.full((1,), 10.0, device=DEV)
        seeds = torch.arange(B, dtype=torch.int64, device=DEV)
        y0, x0, aty0 = (torch.empty(B, H, W, dtype=torch.complex64, device=DEV) for _ in range(3))

        def run(L):
            call(L, "pnp_simulate_measurements", ptr(gt), H * W, ptr(mask), H * W, ptr(sig), 0, ptr(seeds), ptr(y0),
                 ptr(x0), ptr(aty0), B, H, W, st)
        return run

    def fft2c(B, H, W):
        g = torch.Generator().manual_seed(B)
        src = cplx(g, B, H, W)
        dst = torch.empty_like(src)

        def run(L):
            call(L, "pnp_fft2c", ptr(src), ptr(dst), B, H, W, 0, st)
        return run

    cases = [("prox general path 512x512 B=128", prox(128, 512, 512), 20),
             ("prox dense 130x130 B=64", prox(64, 130, 130), 20),
             ("simulate 256x256 B=64", simulate(64, 256, 256), 50),
             ("simulate 512x512 B=64", simulate(64, 512, 512), 20),
             ("simulate 130x130 B=64 (dense)", simulate(64, 130, 130), 20),
             ("fft2c 512x512 B=64", fft2c(64, 512, 512), 50)]
    print("timing: median us per call over 7 alternating rounds after warm-up (CUDA events)")
    for name, run, iters in cases:
        t_old, t_new = time_pair(lambda: run(old), lambda: run(new), iters)
        t_o1, t_o2 = time_pair(lambda: run(old), lambda: run(old), iters)
        print(f"  {name:34s} old {t_old:9.1f}  new {t_new:9.1f}  new/old {t_new / t_old:6.3f}   "
              f"old/old (noise floor) {t_o2 / t_o1:6.3f}")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--old-lib", required=True, help="libpnp_b200.so built from the commit to compare against")
    ap.add_argument("--no-timing", action="store_true")
    a = ap.parse_args()
    new = _lib.lib()
    old = load_old(a.old_lib)
    print(f"card: {card()}")
    print(f"new: {_lib.LIB_PATH}\nold: {os.path.abspath(a.old_lib)}")
    libs = (old, new)
    ck = Checker()
    for H, W in RADIX + DENSE:
        B = 2 if H * W >= 1 << 20 else 3
        ab_fft2c(libs, ck, B, H, W)
        ab_prox(libs, ck, B, H, W)
        ab_simulate(libs, ck, B, H, W)
    for H, W in ((64, 64), (512, 512)):
        ab_prepared(libs, ck, 4, H, W)
        ab_active(libs, ck, 4, H, W)
    torch.cuda.synchronize()
    print(f"bitwise: {ck.n - len(ck.bad)} of {ck.n} outputs equal")
    if not a.no_timing:
        timed_cases(old, new)
    if ck.bad:
        sys.exit(1)


if __name__ == "__main__":
    main()
