"""Float64 NumPy restatement of the seeded variable-density random masks (``pnp_variable_density_masks``; the definition is
in include/pnp_b200.h).  Every step is one IEEE operation on float64 arrays (``+ - * /``, ``sqrt``, the cast to float32), so
the keys, and with them the masks, are bit for bit those of the device."""
import numpy as np

from measure_reference import philox4x32_10, seed_key


def n_keep(H: int, W: int, accel: int) -> int:
    return max(1, (H * W) // accel) if accel >= 1 else H * W


def acs_block(H: int, W: int, acs_h: int, acs_w: int):
    """bool ``[H, W]``: rows [cy - acs_h/2, +acs_h) x columns [cx - acs_w/2, +acs_w)."""
    r0, c0 = H // 2 - acs_h // 2, W // 2 - acs_w // 2
    acs = np.zeros((H, W), dtype=bool)
    acs[r0:r0 + acs_h, c0:c0 + acs_w] = True
    return acs


def density(H: int, W: int, power: int):
    """(w, r), float64 ``[H, W]``: w = (1 - r)^power, rounded after every multiplication."""
    cy, cx = H // 2, W // 2
    ky = (np.arange(H, dtype=np.int64) - cy).astype(np.float64) / np.float64(cy)
    kx = (np.arange(W, dtype=np.int64) - cx).astype(np.float64) / np.float64(cx)
    r = np.sqrt(0.5 * ((ky * ky)[:, None] + (kx * kx)[None, :]))
    w = np.ones((H, W), dtype=np.float64)
    for _ in range(power):
        w = w * (1.0 - r)
    return w, r


def uniforms(H: int, W: int, seed: int):
    """u = (Philox word 0 at counter (p, 3, 0, 0) + 0.5) * 2^-32, float64 ``[H, W]``."""
    p = np.arange(H * W, dtype=np.uint64)
    w0 = philox4x32_10((p, 3, 0, 0), seed_key(seed))[0]
    return ((w0.astype(np.float64) + 0.5) * 2.0 ** -32).reshape(H, W)


def keys(H: int, W: int, seed: int, power: int):
    """float32 ``[H, W]``: key = float32(u / w) (w = 0, or a quotient beyond the float32 range, gives +inf)."""
    w, _ = density(H, W, power)
    with np.errstate(divide="ignore", over="ignore"):
        return (uniforms(H, W, seed) / w).astype(np.float32)


def vd_mask(H: int, W: int, accel: int, seed: int, power: int, acs_h: int, acs_w: int):
    """uint8 ``[H, W]``: the ACS block plus the max(0, n_keep - |ACS|) other pixels with the smallest (key, p)."""
    acs = acs_block(H, W, acs_h, acs_w).reshape(-1)
    extra = max(0, n_keep(H, W, accel) - int(acs.sum()))
    key = keys(H, W, seed, power).reshape(-1)
    cand = np.flatnonzero(~acs)
    order = cand[np.lexsort((cand, key[cand]))]          # primary key, then p
    m = acs.copy()
    m[order[:extra]] = True
    return m.astype(np.uint8).reshape(H, W)


def acs_size(N: int, acs_frac: float = 0.08) -> int:
    """``ops.variable_density_masks``' ACS edge: max(1, round(acs_frac N))."""
    return max(1, int(round(acs_frac * N)))
