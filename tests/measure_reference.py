"""Float64 NumPy restatement of the measurement simulator and the Cartesian masks (``pnp_simulate_measurements``,
``pnp_cartesian_masks``; the definition is in include/pnp_b200.h).  Philox4x32-10 is computed on uint64 arrays (products of
uint32 words never overflow 64 bits), the transforms are ``synth.centered_fft2 / centered_ifft2``."""
import numpy as np

from dt4image_restoration_b200 import synth

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
KEY_INC0, KEY_INC1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
LO32 = np.uint64(0xFFFFFFFF)
SH32 = np.uint64(32)


def philox4x32_10(counter, key):
    """``counter``: 4 uint32-valued arrays (broadcast together), ``key``: 2 ints -> 4 uint64 arrays of uint32 words."""
    c = [np.asarray(x, dtype=np.uint64) & LO32 for x in counter]
    k0, k1 = np.uint64(key[0] & 0xFFFFFFFF), np.uint64(key[1] & 0xFFFFFFFF)
    for r in range(10):
        if r:
            k0, k1 = (k0 + KEY_INC0) & LO32, (k1 + KEY_INC1) & LO32
        p0, p1 = c[0] * M0, c[2] * M1
        c = [(p1 >> SH32) ^ c[1] ^ k0, p1 & LO32, (p0 >> SH32) ^ c[3] ^ k1, p0 & LO32]
    return c


def seed_key(seed: int):
    s = int(seed) & 0xFFFFFFFFFFFFFFFF          # an int64 seed is read as its uint64 bit pattern
    return s & 0xFFFFFFFF, s >> 32


def noise(seed: int, H: int, W: int):
    """(n_r, n_i), float64 ``[H, W]`` each: Box-Muller on the first two words of Philox at counter (i*W + j, 0, 0, 0)."""
    p = np.arange(H * W, dtype=np.uint64)
    w = philox4x32_10((p, 0, 0, 0), seed_key(seed))
    u1 = (w[0].astype(np.float64) + 0.5) * 2.0 ** -32
    u2 = (w[1].astype(np.float64) + 0.5) * 2.0 ** -32
    r = np.sqrt(-2.0 * np.log(u1))
    return (r * np.cos(2 * np.pi * u2)).reshape(H, W), (r * np.sin(2 * np.pi * u2)).reshape(H, W)


def simulate(gt, mask, sigma_n: float, seed: int):
    """One image: complex128 ``y0``, ``ATy0`` and ``x0`` (real and imaginary parts clipped at 0), each ``[H, W]``."""
    H, W = gt.shape
    k = synth.centered_fft2(np.asarray(gt, dtype=np.float64))
    n_r, n_i = noise(seed, H, W)
    y0 = np.where(np.asarray(mask) != 0, k + (sigma_n / 255.0) * (n_r + 1j * n_i), 0)
    aty0 = synth.centered_ifft2(y0)
    x0 = np.maximum(aty0.real, 0) + 1j * np.maximum(aty0.imag, 0)
    return y0, aty0, x0


def cartesian_mask(H: int, W: int, accel: int, seed: int, acs_cols: int):
    """uint8 ``[H, W]``: the ACS band plus the non-ACS columns with the smallest (Philox key, column index)."""
    n_keep = max(1, W // accel) if accel >= 1 else W
    n_acs = min(n_keep, acs_cols)
    c0 = W // 2 - n_acs // 2
    cols = np.zeros(W, dtype=bool)
    cols[c0:c0 + n_acs] = True
    j = np.arange(W, dtype=np.uint64)
    keys = philox4x32_10((j, 1, 0, 0), seed_key(seed))[0]
    cand = np.flatnonzero(~cols)
    order = cand[np.lexsort((cand, keys[cand]))]         # primary key_j, then j
    cols[order[:n_keep - n_acs]] = True
    return np.repeat(cols[None, :], H, axis=0).astype(np.uint8)


def acs_cols(W: int, acs_frac: float = 0.08) -> int:
    return max(1, int(round(acs_frac * W)))


def make_item(gt, mask, sigma_n: float, seed: int) -> dict:
    """``synth.make_item``'s dict for one image, with this generator's noise."""
    H, W = gt.shape
    y0, aty0, x0 = simulate(gt, mask, sigma_n, seed)
    ri = lambda z: np.stack([z.real, z.imag], axis=-1).astype(np.float32).reshape(1, 1, H, W, 2)
    return {"x0": ri(x0), "y0": ri(y0), "ATy0": ri(aty0), "mask": np.asarray(mask, dtype=np.uint8).reshape(1, H, W).copy(),
            "gt": np.asarray(gt, dtype=np.float32).reshape(1, 1, H, W)}
