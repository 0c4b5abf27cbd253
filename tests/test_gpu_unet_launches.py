"""Every launch of the denoiser plan checked alone against a float64 restatement of that one operation
(tests/unet_launch_reference.py), fed the launch's own inputs as the GPU produced them.  Needs a B200.

The plan runs one launch at a time (``UNetPlan.forward_ops(i, i + 1)``); each launch's outputs are cloned right after it
runs, before a later launch recycles the slot, and its inputs are the clones of what earlier launches wrote.  The bound
is then a few bf16 ulps per element instead of an error compounded along the chain, so a wrong tile, a dropped edge row
of the fused pool or an off-by-one pad is found and located: the failure names the launch, its kernel and the worst
element (image, y, x, channel, tile).
"""
import functools
import json
import os
import subprocess
import sys

import pytest
import torch

from dt4image_restoration_b200 import _lib, ops
from oracle import pnp_oracle as O
import unet_launch_reference as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
BLOCKS = ("inc", "down1", "down2", "down3", "down4", "up1", "up2", "up3", "up4")

# (B, H, W): what each shape exercises
SHAPES = [
    (2, 64, 64),        # fast upsample at every level
    (1, 16, 16),        # level 4 is 1x1: the upsample into level 3 takes the general path with h = 1
    (2, 31, 17),        # odd at every level: pads, odd-H / odd-W pools, first-conv edges, ragged tiles
    (1, 45, 51), (3, 36, 52), (2, 130, 130),      # non-power-of-two sizes, mixed exact / padded levels
    (2, 256, 256),      # the benchmark size: many tiles per CTA, both sweep directions
    (1, 512, 512),      # BASELINE config 4
    (96, 32, 32),       # many images, small tiles
]
SMALL = [(2, 64, 64), (1, 16, 16), (2, 31, 17), (1, 45, 51), (3, 36, 52), (96, 32, 32)]
CASES = ([(s, "kaiming", -1) for s in SHAPES] + [(s, "default", -1) for s in SMALL]
         + [(s, "kaiming", m) for s in [(1, 16, 16), (2, 31, 17), (3, 36, 52), (2, 64, 64)] for m in (0, 1)])


def case_id(c):
    (B, H, W), kind, mode = c
    return f"{B}x{H}x{W}-{kind}-splitk{mode}"


@functools.lru_cache(maxsize=None)
def weights(kind):
    params = O.init_unet_params(1, kind)
    return params, ops.pack_unet_weights(ops.flatten_state_dict(params).to(DEV))


def layer_weights(params, li):
    p = f"{O._block_prefix(BLOCKS[li // 3])}.conv-{li % 3}.conv2d"
    return params[p + ".weight"], params[p + ".bias"]


class splitk:
    """Kernel choice of plans created inside the block (-1 auto, 0 never split-K, 1 every eligible conv), restored after."""

    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        self.old = _lib.lib().pnp_unet_set_splitk(self.mode)

    def __exit__(self, *exc):
        _lib.lib().pnp_unet_set_splitk(self.old)


def make_plan(kind, B, H, W, mode):
    _, packed = weights(kind)
    with splitk(mode):
        plan = ops.UNetPlan(packed, B, H, W)
    assert _lib.lib().pnp_unet_micro_batch(plan.handle) == B
    return plan


def inputs(B, H, W, seed=0):
    g = torch.Generator().manual_seed(seed * 7919 + H * 131 + W)
    v = torch.rand(B, H, W, generator=g)
    sigma = torch.rand(B, generator=g) * 0.2 + 0.02
    return v.to(DEV), sigma.to(DEV)


def run_launches(plan, v, sigma):
    """Run the plan one launch at a time.  Returns (descriptors, inputs, outputs): per launch a dict of the clones of the
    workspace tensors it read ("in0", "in1") and one of what it wrote ("out", "pool"; FINAL: "x", "pre")."""
    desc = plan.describe()
    x = torch.empty_like(v)
    pre = torch.empty_like(v)
    latest, ins, outs = {}, [], []
    for i, d in enumerate(desc):
        ins.append({k: latest[d[k + "_off"]] for k in ("in0", "in1") if d[k + "_off"] >= 0})
        plan.forward_ops(i, i + 1, v, sigma, x, pre)
        o = {}
        if d["out_off"] >= 0:
            o["out"] = latest[d["out_off"]] = plan.tensor_at(d["out_off"], d["out_C"], d["H"], d["W"]).clone()
        if d["pool_off"] >= 0:
            o["pool"] = latest[d["pool_off"]] = plan.tensor_at(d["pool_off"], d["pool_C"], d["H"] // 2, d["W"] // 2).clone()
        if d["kernel"] == "final":
            o["x"], o["pre"] = x.clone(), pre.clone()
        outs.append(o)
    torch.cuda.synchronize()
    return desc, ins, outs


def where(d, idx):
    """Human-readable position of an NHWC (or [B,H,W]) index, with its output tile."""
    b, y, xx = idx[:3]
    c = idx[3] if len(idx) > 3 else 0
    tw, th = d["tile_w"] or 16, d["tile_h"] or 16
    return f"image {b}, y {y}, x {xx}, channel {c}, tile (ty {y // th}, tx {xx // tw})"


def check_launch(i, d, ins, outs, params, v, sigma):
    """Compare launch i with its float64 reference; raise AssertionError naming the launch and the worst element."""
    def expect(name, got, ref, bound):
        ratio, idx, n = R.compare(got, ref, bound)
        assert n == 0, (f"launch {i} ({d['kernel']}, layer {d['id']}, {name}): max |err| / bound = {ratio:.3g} at "
                        f"{where(d, idx)}; {n} elements over the bound; descriptor {d}")

    kern = d["kernel"]
    if kern == "first":
        ref, bound = R.first_conv(v, sigma, *layer_weights(params, 0))
        expect("out", outs["out"], ref, bound)
    elif kern in ("ups_fast", "ups_general"):
        ref, bound, _ = R.upsample(ins["in0"], d["H"], d["W"])
        expect("out", outs["out"], ref, bound)         # the pad region has bound 0: exactly 0 there
    elif kern == "final":
        w, b = layer_weights(params, d["id"])
        ref, bound = R.final(ins["in0"], R.bf16r(w), b, params["outc.conv.weight"].reshape(-1),
                             params["outc.conv.bias"], v)
        expect("preclamp", outs["pre"], ref, bound)
        assert torch.equal(outs["x"], outs["pre"].clamp(0, 1)), f"launch {i}: x_out != clamp(preclamp, 0, 1)"
    else:
        w, b = layer_weights(params, d["id"])
        ref, bound = R.conv3x3(ins["in0"], ins.get("in1"), R.bf16r(w), b)
        expect("out", outs["out"], ref, bound)
        if "pool" in outs:
            pref = R.maxpool(outs["out"])
            expect("pool", outs["pool"], pref, torch.zeros_like(pref))


def variant(d):
    """The dispatch facts a launch exercises (the coverage key).  The split-K kernel has no sweep direction."""
    if d["kind"] != 1:
        return (d["kernel"],)
    sweep = "-" if d["kernel"] == "splitk" else "rev" if d["rev"] else "fwd"
    return (d["kernel"], d["kc"], d["bn"], sweep, "pool" if d["pool_off"] >= 0 else "-",
            "wres" if d["wres"] else "stream", "ragged_x" if d["W"] % d["tile_w"] else "-",
            "ragged_y" if d["H"] % d["tile_h"] else "-")


def tiles_per_cta(d):
    """Output tiles one CTA (one CTA pair) walks through, at most."""
    units = d["grid"] // 2 if d["kernel"] == "pair" else d["grid"]
    return -(-d["tiles"] // units)


def check_case(shape, kind, mode):
    """Per-launch check of one plan, plus: a second forward gives the same bits at every launch.  Returns the variants."""
    B, H, W = shape
    params, _ = weights(kind)
    plan = make_plan(kind, B, H, W, mode)
    v, sigma = inputs(B, H, W)
    desc, ins, outs = run_launches(plan, v, sigma)
    assert [d["id"] for d in desc][:3] == [0, 1, 2] and desc[-1]["kernel"] == "final" and len(desc) == 31
    for i, d in enumerate(desc):
        check_launch(i, d, ins[i], outs[i], params, v.view(B, H, W), sigma)
    # determinism (covers the split-K cluster reduction): the same plan again, bit for bit at every launch
    _, _, outs2 = run_launches(plan, v, sigma)
    for i, (a, b) in enumerate(zip(outs, outs2)):
        for k in a:
            assert torch.equal(a[k], b[k]), f"launch {i} ({desc[i]['kernel']}, layer {desc[i]['id']}) {k}: second run differs"
    # the launches one at a time are the forward pass
    x = plan.forward(v, sigma)
    assert torch.equal(x, outs[-1]["x"])
    return {variant(d) for d in desc}


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_launches_match_float64_reference(case):
    check_case(*case)


@pytest.mark.parametrize("shape", [(3, 36, 52), (2, 31, 17), (4, 64, 64)])
def test_image_output_independent_of_batch(shape):
    """With split-K off every conv's kernel, tile shape and summation order depend on the layer only, so an image's
    denoised output is bitwise the same at any batch size and any position in the batch."""
    B, H, W = shape
    v, sigma = inputs(B, H, W, seed=3)
    whole = make_plan("kaiming", B, H, W, 0).forward(v, sigma)
    rev = make_plan("kaiming", B, H, W, 0).forward(v.flip(0).contiguous(), sigma.flip(0).contiguous())
    assert torch.equal(rev.flip(0), whole)
    one = make_plan("kaiming", 1, H, W, 0)
    for b in range(B):
        assert torch.equal(one.forward(v[b:b + 1].contiguous(), sigma[b:b + 1].contiguous()), whole[b:b + 1]), b


def test_forward_ops_rejects_bad_ranges_and_micro_batched_plans():
    plan = make_plan("kaiming", 1, 16, 16, -1)
    v, sigma = inputs(1, 16, 16)
    x = torch.empty_like(v)
    n = len(plan.describe())
    for first, end in ((-1, 1), (0, n + 1), (3, 2)):
        with pytest.raises(_lib.PnpError):
            plan.forward_ops(first, end, v, sigma, x)
    plan.forward_ops(5, 5, v, sigma, x)              # empty range: nothing runs
    l = _lib.lib()
    old = l.pnp_unet_set_workspace_cap(l.pnp_unet_workspace_bytes(2, 32, 32))
    try:
        _, packed = weights("kaiming")
        small = ops.UNetPlan(packed, 5, 32, 32)
        assert l.pnp_unet_micro_batch(small.handle) < 5
        with pytest.raises(_lib.PnpError):
            small.describe()
        v5, s5 = inputs(5, 32, 32)
        with pytest.raises(_lib.PnpError):
            small.forward_ops(0, 1, v5, s5, torch.empty_like(v5))
    finally:
        l.pnp_unet_set_workspace_cap(old)


PAIR_SCRIPT = r"""
import json, sys
sys.path.insert(0, "tests")
import test_gpu_unet_launches as T
seen = set()
for shape, mode in [((2, 31, 17), 0), ((2, 130, 130), -1)]:
    seen |= T.check_case(shape, "kaiming", mode)
print("VARIANTS " + json.dumps(sorted(seen)))
"""


def pair_env_variants(pair):
    env = dict(os.environ, PNP_CONV_PAIR=pair)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", PAIR_SCRIPT], cwd=root, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    line = [s for s in r.stdout.splitlines() if s.startswith("VARIANTS ")][-1]
    return {tuple(v) for v in json.loads(line[len("VARIANTS "):])}


@pytest.mark.parametrize("pair", ["0", "1"])
def test_launches_with_conv_pair_forced(pair):
    """PNP_CONV_PAIR=0 / 1 forces the single-CTA / CTA-pair kernel on every eligible conv; it is read once per process,
    hence the subprocess.  Both plans pass the per-launch check (split-K off at 2x31x17, so that every 64-channel-slice
    conv takes the kernel the switch forces; the product's choice at 2x130x130)."""
    seen = pair_env_variants(pair)
    kernels = {v[:3] for v in seen if len(v) > 1}
    if pair == "0":
        assert not any(k[0] == "pair" for k in kernels) and ("umma", 64, 128) in kernels, sorted(kernels)
    else:
        assert ("pair", 32, 64) in kernels and ("umma", 32, 64) not in kernels, sorted(kernels)


# ------------------------------------------------------------------------------------------------
# coverage of the dispatch
# ------------------------------------------------------------------------------------------------
# Variants the cases above must exercise: (kernel, KC or split-K S, BN, sweep, fused pool, weights resident or streamed,
# ragged tile in x, in y).  A change to the dispatch (use_kws, weights_fit, the split-K or the pair rule) that drops one
# of them fails here instead of leaving it untested.
#
# Variants the plan cannot produce (not tested, by construction):
# * kws with a fused pool or a reversed sweep: kws only serves up4.conv-0, which pools nothing and is launch 28 (even).
# * the first conv's reversed sweep (it is launch 0) and a reversed fast upsample (the upsamples are launches 15, 19,
#   23 and 27); the general upsample has no sweep direction.
# * umma(32, 64) with a pool, streamed weights or a forward sweep: only down1.conv-0 (36 KB of weights, launch 3)
#   takes it.
# * pair(64, 64) in a reversed sweep or with resident weights: only up3.conv-0 (launch 24, 216 KB of weights) takes it;
#   pair(64, 128) with resident weights only in a forward sweep: only down2.conv-0 (launch 6) keeps them.
# * the FINAL epilogue in a reversed sweep or with a pool (launch 30, the last conv).
# * pair(32, 64): only with PNP_CONV_PAIR=1 (test_launches_with_conv_pair_forced); umma(64, 128): only with
#   PNP_CONV_PAIR=0.
# * the split-K kernel ignores the sweep direction and never keeps weights resident.
# * the kws kernel's pool path and the first conv's and the fast upsample's reversed walks are dead code of the plan.
REQUIRED = {
    ("first",), ("ups_fast",), ("ups_general",),
    # inc.conv-1/2 and up4.conv-1 (32 -> 32), down1.conv-0 (32 -> 64), down1.conv-1/2 and up3.conv-1/2 (64 -> 64)
    ("umma", 32, 32, "rev", "-", "wres", "-", "-"), ("umma", 32, 32, "rev", "-", "wres", "ragged_x", "ragged_y"),
    ("umma", 32, 32, "fwd", "pool", "wres", "-", "-"), ("umma", 32, 32, "fwd", "pool", "wres", "ragged_x", "ragged_y"),
    ("umma", 32, 64, "rev", "-", "wres", "-", "-"), ("umma", 32, 64, "rev", "-", "wres", "ragged_x", "ragged_y"),
    ("umma", 64, 64, "fwd", "-", "wres", "-", "-"), ("umma", 64, 64, "fwd", "-", "wres", "ragged_x", "ragged_y"),
    ("umma", 64, 64, "rev", "-", "wres", "-", "-"), ("umma", 64, 64, "rev", "-", "wres", "ragged_x", "ragged_y"),
    ("umma", 64, 64, "rev", "pool", "wres", "-", "-"), ("umma", 64, 64, "rev", "pool", "wres", "ragged_x", "ragged_y"),
    # up4.conv-2 (FINAL) and up4.conv-0 (kw-stacked, 12-pixel-wide tiles)
    ("final", 32, 32, "fwd", "-", "wres", "-", "-"), ("final", 32, 32, "fwd", "-", "wres", "ragged_x", "ragged_y"),
    ("kws", 32, 32, "fwd", "-", "wres", "ragged_x", "-"), ("kws", 32, 32, "fwd", "-", "wres", "ragged_x", "ragged_y"),
    # CTA pairs: resident weights (down2.conv-0) and streamed ones, both sweeps, the fused pool in both sweeps
    ("pair", 64, 64, "fwd", "-", "stream", "-", "-"), ("pair", 64, 64, "fwd", "-", "stream", "ragged_x", "ragged_y"),
    ("pair", 64, 128, "fwd", "-", "wres", "-", "-"), ("pair", 64, 128, "fwd", "-", "wres", "ragged_x", "ragged_y"),
    ("pair", 64, 128, "fwd", "-", "stream", "-", "-"), ("pair", 64, 128, "fwd", "-", "stream", "ragged_x", "ragged_y"),
    ("pair", 64, 128, "rev", "-", "stream", "-", "-"), ("pair", 64, 128, "rev", "-", "stream", "ragged_x", "ragged_y"),
    ("pair", 64, 128, "fwd", "pool", "stream", "-", "-"), ("pair", 64, 128, "fwd", "pool", "stream", "ragged_x", "ragged_y"),
    ("pair", 64, 128, "rev", "pool", "stream", "ragged_x", "ragged_y"),
    # split-K clusters of 1, 2, 4 and 8 CTAs, with and without the fused pool
    ("splitk", 1, 32, "-", "-", "stream", "-", "-"), ("splitk", 1, 32, "-", "-", "stream", "ragged_x", "ragged_y"),
    ("splitk", 1, 32, "-", "pool", "stream", "-", "-"), ("splitk", 1, 32, "-", "pool", "stream", "ragged_x", "ragged_y"),
    ("splitk", 2, 32, "-", "-", "stream", "-", "-"), ("splitk", 2, 32, "-", "-", "stream", "ragged_x", "ragged_y"),
    ("splitk", 2, 32, "-", "pool", "stream", "-", "-"), ("splitk", 2, 32, "-", "pool", "stream", "ragged_x", "ragged_y"),
    ("splitk", 4, 32, "-", "-", "stream", "-", "-"), ("splitk", 4, 32, "-", "-", "stream", "ragged_x", "ragged_y"),
    ("splitk", 4, 32, "-", "pool", "stream", "-", "-"), ("splitk", 4, 32, "-", "pool", "stream", "ragged_x", "ragged_y"),
    ("splitk", 8, 32, "-", "-", "stream", "ragged_x", "ragged_y"),
}
# Kernels whose CTAs must, in some case, walk more output tiles than they have accumulator stages (4 at BN = 32, 2
# otherwise), so that the stages are reused.
REQUIRED_REUSE = {"umma": 4, "final": 4, "kws": 2, "pair": 2}


def test_dispatch_coverage():
    """The descriptors of every plan the cases above build (plan creation only, no launch) cover REQUIRED."""
    seen, walk = set(), {}
    for (B, H, W), kind, mode in CASES:
        for d in make_plan(kind, B, H, W, mode).describe():
            seen.add(variant(d))
            if d["kind"] == 1:
                walk[d["kernel"]] = max(walk.get(d["kernel"], 0), tiles_per_cta(d))
    out = os.environ.get("PNP_COVERAGE_OUT")
    if out:
        with open(out, "w") as f:
            json.dump(sorted(map(list, seen)), f, indent=0)
    missing = REQUIRED - seen
    assert not missing, f"variants no longer covered: {sorted(missing)}; covered: {sorted(seen)}"
    for kern, nacc in REQUIRED_REUSE.items():
        assert walk.get(kern, 0) > nacc, f"no {kern} CTA walks more than {nacc} tiles: {walk}"
