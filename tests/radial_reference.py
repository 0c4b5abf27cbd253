"""Float64 NumPy restatement of the seeded golden-angle radial masks (``pnp_radial_masks``; the definition is in
include/pnp_b200.h).  The count after each line is kept incrementally (the distinct in-image pixels of the line that were
not yet set), not by re-summing the mask as ``synth.radial_mask`` does, so the two agree only if both follow the definition."""
import math

import numpy as np

from measure_reference import philox4x32_10, seed_key

GOLDEN = np.pi * (np.sqrt(5.0) - 1.0) / 2.0       # 0x1.f10d6bc8e0e35p+0
PI_2M32 = np.pi * 2.0 ** -32                       # 0x1.921fb54442d18p-31


def half_length(H: int, W: int) -> int:
    """R = 1 + the smallest integer r with 4 r^2 >= H^2 + W^2."""
    s = H * H + W * W
    r = math.isqrt(s) // 2
    while 4 * r * r < s:
        r += 1
    return r + 1


def phi(seed) -> float:
    """Rotation of the seeded pattern: 0 without a seed, else Philox word 0 at counter (0, 2, 0, 0) times pi 2^-32."""
    if seed is None:
        return 0.0
    w0 = int(philox4x32_10((0, 2, 0, 0), seed_key(seed))[0])
    return float(np.float64(w0) * PI_2M32)


def radial_mask(H: int, W: int, frac: float, seed=None, sincos=None, max_lines=None):
    """(uint8 ``[H, W]`` mask, number of lines).  ``sincos(ang) -> (sin, cos)`` replaces NumPy's sin / cos when given;
    ``max_lines`` stops after that many lines (to look at the count before the last line)."""
    cy, cx = H // 2, W // 2
    R = half_length(H, W)
    t = np.arange(-R, R + 1, dtype=np.float64)
    ph = phi(seed)
    target = frac * H * W
    cap = 8 * max(H, W) if max_lines is None else min(8 * max(H, W), max_lines)
    flat = np.zeros(H * W, dtype=np.uint8)
    count, n = 0, 0
    while count < target and n < cap:
        ang = np.float64(n) * GOLDEN + ph
        s, c = (np.sin(ang), np.cos(ang)) if sincos is None else sincos(ang)
        yy = np.rint(cy + t * s).astype(np.int64)
        xx = np.rint(cx + t * c).astype(np.int64)
        ok = (yy >= 0) & (yy < H) & (xx >= 0) & (xx < W)
        p = np.unique(yy[ok] * W + xx[ok])
        new = p[flat[p] == 0]
        flat[new] = 1
        count += new.size
        n += 1
    return flat.reshape(H, W), n
