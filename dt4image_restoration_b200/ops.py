"""Tensor-level wrappers over the C-ABI (``include/pnp_b200.h``).

Every function takes CUDA tensors, launches on ``torch.cuda.current_stream()`` and returns CUDA tensors;
nothing here computes on the CPU.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import check


def _req(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise _lib.PnpError(f"{name}: expected a CUDA tensor (no CPU path exists)")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    _lib.check_device(t.device)
    return t.contiguous()


def aligned_empty(nbytes: int, device, align: int = 1024) -> torch.Tensor:
    """uint8 CUDA buffer whose data_ptr is ``align``-byte aligned."""
    raw = torch.empty(nbytes + align, dtype=torch.uint8, device=device)
    off = (-raw.data_ptr()) % align
    return raw[off:off + nbytes]


# ------------------------------------------------------------------------------------------------
def psnr(x: torch.Tensor, gt: torch.Tensor) -> torch.Tensor:
    """``[N,...]`` vs ``[N,...]`` (or one shared gt) -> fp32 ``[N]`` on the device (env.py:120-125)."""
    if x.is_complex():
        x = x.real
    N = x.shape[0]
    x = _req(x.reshape(N, -1).float(), torch.float32, "x")
    gt = _req(gt.float(), torch.float32, "gt")
    HW = x.shape[1]
    if gt.numel() == N * HW:
        stride = HW
    elif gt.numel() == HW:
        stride = 0
    else:
        raise RuntimeError(f"psnr: gt has {gt.numel()} elements, expected {N * HW} or {HW}")
    out = torch.empty(N, dtype=torch.float32, device=x.device)
    check(_lib.lib().pnp_psnr(x.data_ptr(), gt.data_ptr(), stride, out.data_ptr(), N, HW, _lib.stream_ptr()), "pnp_psnr")
    return out


def ssim(x: torch.Tensor, gt: torch.Tensor) -> torch.Tensor:
    """SSIM per image (Gaussian 11x11 window, sigma 1.5, valid filtering; see ``pnp_ssim`` in include/pnp_b200.h):
    ``[N,...,H,W]`` vs ``[N,...,H,W]`` (or one shared ``[H,W]`` gt) -> fp32 ``[N]`` on the device.  ``x`` is clamped to
    [0, 1], ``gt`` is not."""
    if x.is_complex():
        x = x.real
    N, (H, W) = x.shape[0], x.shape[-2:]
    x = _req(x.reshape(N, H * W).float(), torch.float32, "x")
    gt = _req(gt.float(), torch.float32, "gt")
    if gt.numel() == N * H * W:
        stride = H * W
    elif gt.numel() == H * W:
        stride = 0
    else:
        raise RuntimeError(f"ssim: gt has {gt.numel()} elements, expected {N * H * W} or {H * W}")
    l = _lib.lib()
    out = torch.empty(N, dtype=torch.float32, device=x.device)
    work = aligned_empty(max(int(l.pnp_ssim_workspace_bytes(N, H, W)), 16), x.device, align=16)
    check(l.pnp_ssim(x.data_ptr(), gt.data_ptr(), stride, out.data_ptr(), work.data_ptr(), N, H, W, _lib.stream_ptr()),
          "pnp_ssim")
    return out


def fft2c(x: torch.Tensor, inverse: bool = False) -> torch.Tensor:
    """Centred orthonormal 2-D (i)FFT over the last two dims (transformations.py:6-19)."""
    if not x.is_complex():
        x = torch.complex(x.float(), torch.zeros_like(x, dtype=torch.float32))
    x = _req(x, torch.complex64, "x")
    H, W = x.shape[-2:]
    B = x.numel() // (H * W)
    out = torch.empty_like(x)
    check(_lib.lib().pnp_fft2c(x.data_ptr(), out.data_ptr(), B, H, W, int(inverse), _lib.stream_ptr()), "pnp_fft2c")
    return out


def _mask_arg(mask: torch.Tensor, B: int, H: int, W: int):
    """bool/uint8 mask(s) of B images or one shared image -> (uint8 CUDA tensor, batch stride ``H*W`` or 0)."""
    if mask.dtype == torch.bool:
        mask = mask.contiguous().view(torch.uint8)
    mask = _req(mask, torch.uint8, "mask")
    if mask.numel() not in (B * H * W, H * W):
        raise IndexError(f"mask with {mask.numel()} elements does not match {B} images of {H}x{W}")
    return mask, H * W if mask.numel() == B * H * W else 0


def _check_out(t: torch.Tensor, dtype, numel: int, name: str = "out"):
    """A caller-provided output buffer: contiguous, on the device, of ``dtype`` and ``numel`` elements."""
    if not t.is_cuda or t.dtype != dtype or not t.is_contiguous() or t.numel() != numel:
        raise _lib.PnpError(f"{name} must be a contiguous {dtype} CUDA tensor with {numel} elements")


def _seed_tensor(seeds, B: int, device) -> torch.Tensor:
    """int64 ``[B]`` seeds on the device; an int ``s0`` stands for ``s0 + arange(B)`` (synth.make_batch's image numbering)."""
    if isinstance(seeds, int):
        return torch.arange(seeds, seeds + B, dtype=torch.int64, device=device)
    seeds = _req(seeds.reshape(-1), torch.int64, "seeds")
    if seeds.numel() != B:
        raise RuntimeError(f"seeds must have {B} elements, got {seeds.numel()}")
    return seeds


def _per_image(val, B: int, dtype, name: str, device):
    """A host scalar (one value for the batch, stride 0) or a CUDA ``[B]`` tensor (stride 1)."""
    if torch.is_tensor(val):
        val = _req(val.reshape(-1), dtype, name)
        if val.numel() not in (1, B):
            raise RuntimeError(f"{name} must have 1 or {B} elements, got {val.numel()}")
        return val, 0 if val.numel() == 1 else 1
    return torch.full((1,), val, dtype=dtype, device=device), 0


def _batch_size(gt, mask, sigma_n, seeds) -> int:
    """Images in a simulator call: gt's batch, else the length of seeds / sigma_n / mask, else 1."""
    H, W = gt.shape[-2:]
    if gt.dim() > 2:
        return gt.numel() // (H * W)
    if torch.is_tensor(seeds):
        return seeds.numel()
    if torch.is_tensor(sigma_n) and sigma_n.numel() > 1:
        return sigma_n.numel()
    return max(1, mask.numel() // (H * W)) if mask is not None else 1


def simulate_measurements(gt, mask, sigma_n, seeds, aty0: bool = True, out=None):
    """Undersampled, noisy k-space measurements of fully-sampled images (``pnp_simulate_measurements``, definition in
    include/pnp_b200.h): ``y0 = mask . (fft_c(gt) + sigma_n/255 (n_r + i n_i))``, ``ATy0 = ifft_c(y0)``, ``x0 = max(ATy0, 0)``
    componentwise.

    ``gt`` fp32 ``[B,1,H,W]`` / ``[B,H,W]`` or one shared ``[H,W]``; ``mask`` bool/uint8 ``[B or 1, ..., H, W]``;
    ``sigma_n`` a float or fp32 ``[B]``; ``seeds`` int64 ``[B]`` or an int ``s0`` meaning ``s0 + arange(B)``.  CUDA tensors
    only.  Returns complex64 ``[B,1,H,W]`` tensors ``(y0, x0, ATy0)`` (``ATy0`` is None with ``aty0=False``), written into
    ``out=(y0, x0, aty0)`` when given."""
    gt = _req(gt, torch.float32, "gt")
    H, W = gt.shape[-2:]
    B = _batch_size(gt, mask, sigma_n, seeds)
    gt_stride = H * W if gt.numel() == B * H * W else 0
    if gt.numel() not in (B * H * W, H * W):
        raise RuntimeError(f"gt has {gt.numel()} elements, expected {B * H * W} or {H * W}")
    mask, mstride = _mask_arg(mask, B, H, W)
    sig, sstride = _per_image(sigma_n, B, torch.float32, "sigma_n", gt.device)
    seeds = _seed_tensor(seeds, B, gt.device)
    if out is None:
        y0 = torch.empty(B, 1, H, W, dtype=torch.complex64, device=gt.device)
        x0 = torch.empty_like(y0)
        at = torch.empty_like(y0) if aty0 else None
    else:
        y0, x0, at = out
        for t in (y0, x0) + ((at,) if at is not None else ()):
            _check_out(t, torch.complex64, B * H * W)
    check(_lib.lib().pnp_simulate_measurements(gt.data_ptr(), gt_stride, mask.data_ptr(), mstride, sig.data_ptr(), sstride,
                                               seeds.data_ptr(), y0.data_ptr(), x0.data_ptr(),
                                               at.data_ptr() if at is not None else None, B, H, W, _lib.stream_ptr()),
          "pnp_simulate_measurements")
    return y0, x0, at


def cartesian_masks(B: int, H: int, W: int, accel, seeds, acs_frac: float = 0.08, out=None) -> torch.Tensor:
    """Seeded Cartesian masks (``pnp_cartesian_masks``): uint8 ``[B,H,W]`` on the current CUDA device with
    ``synth.cartesian_mask``'s structure - a centred ACS band of ``max(1, round(acs_frac W))`` columns plus random columns
    up to ``max(1, W // accel)``.  ``accel`` an int or int32 ``[B]`` CUDA tensor; ``seeds`` as in ``simulate_measurements``."""
    dev = torch.device("cuda", torch.cuda.current_device())
    if not torch.is_tensor(accel) and int(accel) < 1:
        raise ValueError(f"accel must be >= 1, got {accel}")
    acc, astride = _per_image(accel if torch.is_tensor(accel) else int(accel), B, torch.int32, "accel", dev)
    seeds = _seed_tensor(seeds, B, dev)
    acs_cols = max(1, int(round(acs_frac * W)))
    if out is None:
        out = torch.empty(B, H, W, dtype=torch.uint8, device=dev)
    _check_out(out, torch.uint8, B * H * W)
    check(_lib.lib().pnp_cartesian_masks(acc.data_ptr(), astride, seeds.data_ptr(), acs_cols, out.data_ptr(), B, H, W,
                                         _lib.stream_ptr()), "pnp_cartesian_masks")
    return out


def radial_masks(B: int, H: int, W: int, frac, seeds=None, out=None, lines_out=None) -> torch.Tensor:
    """Golden-angle radial masks (``pnp_radial_masks``): uint8 ``[B,H,W]`` on the current CUDA device.  Lines through the
    k-space centre are added until the sampled fraction reaches ``frac`` (a float or float64 ``[B]`` CUDA tensor).  With
    ``seeds=None`` every mask is ``synth.radial_mask(H, W, frac)``; with ``seeds`` (as in ``simulate_measurements``) image b's
    lines are rotated by a Philox draw of its seed.  The number of lines of each image goes to ``lines_out`` (int32 ``[B]``,
    CUDA) when given."""
    dev = torch.device("cuda", torch.cuda.current_device())
    fr, fstride = _per_image(frac if torch.is_tensor(frac) else float(frac), B, torch.float64, "frac", dev)
    seeds = _seed_tensor(seeds, B, dev) if seeds is not None else None
    if out is None:
        out = torch.empty(B, H, W, dtype=torch.uint8, device=dev)
    _check_out(out, torch.uint8, B * H * W)
    if lines_out is not None:
        _check_out(lines_out, torch.int32, B, "lines_out")
    check(_lib.lib().pnp_radial_masks(fr.data_ptr(), fstride, seeds.data_ptr() if seeds is not None else None,
                                      out.data_ptr(), lines_out.data_ptr() if lines_out is not None else None, B, H, W,
                                      _lib.stream_ptr()), "pnp_radial_masks")
    return out


def variable_density_masks(B: int, H: int, W: int, accel, seeds, power: int = 3, acs_frac: float = 0.08,
                           out=None) -> torch.Tensor:
    """Seeded 2-D variable-density random masks (``pnp_variable_density_masks``): uint8 ``[B,H,W]`` on the current CUDA
    device.  A centred ACS block of ``max(1, round(acs_frac H))`` x ``max(1, round(acs_frac W))`` pixels plus the other
    pixels with the smallest Philox key / ``(1 - r)^power`` (r the normalised k-space radius), up to exactly
    ``max(1, H*W // accel)`` sampled pixels.  ``accel`` an int or int32 ``[B]`` CUDA tensor; ``seeds`` as in
    ``simulate_measurements``; ``power`` in 0..16 (0: uniform)."""
    dev = torch.device("cuda", torch.cuda.current_device())
    if not torch.is_tensor(accel) and int(accel) < 1:
        raise ValueError(f"accel must be >= 1, got {accel}")
    acc, astride = _per_image(accel if torch.is_tensor(accel) else int(accel), B, torch.int32, "accel", dev)
    seeds = _seed_tensor(seeds, B, dev)
    acs_h, acs_w = max(1, int(round(acs_frac * H))), max(1, int(round(acs_frac * W)))
    if out is None:
        out = torch.empty(B, H, W, dtype=torch.uint8, device=dev)
    _check_out(out, torch.uint8, B * H * W)
    check(_lib.lib().pnp_variable_density_masks(acc.data_ptr(), astride, seeds.data_ptr(), acs_h, acs_w, int(power),
                                                out.data_ptr(), B, H, W, _lib.stream_ptr()), "pnp_variable_density_masks")
    return out


def _episode_masks(B: int, H: int, W: int, seeds, mask=None, accel=None, radial=None, vd=None, out=None) -> torch.Tensor:
    """The uint8 ``[B,H,W]`` masks of a batch of episodes (written into ``out`` when given) from exactly one of ``mask``
    (bool/uint8 ``[B or 1, ..., H, W]``, read as ``!= 0``; one mask serves every image), ``accel`` (``cartesian_masks``),
    ``radial`` (``radial_masks``) and ``vd`` (``variable_density_masks``), the last three drawn with ``seeds``."""
    if sum(m is not None for m in (mask, accel, radial, vd)) != 1:
        raise ValueError("pass exactly one of mask / accel / radial / vd")
    if accel is not None:
        return cartesian_masks(B, H, W, accel, seeds, out=out)
    if radial is not None:
        return radial_masks(B, H, W, radial, seeds, out=out)
    if vd is not None:
        return variable_density_masks(B, H, W, vd, seeds, out=out)
    mask = _mask_arg(mask, B, H, W)[0].ne(0).reshape(-1, H, W).expand(B, H, W)
    if out is None:
        return mask.to(torch.uint8).contiguous()
    _check_out(out, torch.uint8, B * H * W)
    out.view(B, H, W).copy_(mask)
    return out


def make_items(gt, sigma_n, seeds, mask=None, accel=None, radial=None, vd=None) -> dict:
    """A batch of episode items on the device with ``synth.make_batch``'s keys, shapes and dtypes (``x0, y0, ATy0`` fp32
    ``[B,1,H,W,2]``, ``mask`` uint8 ``[B,H,W]``, ``gt`` fp32 ``[B,1,H,W]``), ready for ``PnPEnv.reset`` / ``PnPEngine.reset``.
    Pass exactly one of ``mask`` (bool/uint8 ``[B or 1, ..., H, W]``), ``accel`` (Cartesian masks drawn with ``seeds``),
    ``radial`` (the sampled fraction of radial masks rotated by ``seeds``, see ``radial_masks``) and ``vd`` (the
    acceleration of variable-density masks drawn with ``seeds``, default power and ACS of ``variable_density_masks``)."""
    gt = _req(gt, torch.float32, "gt")
    H, W = gt.shape[-2:]
    B = _batch_size(gt, mask, sigma_n, seeds)
    mask = _episode_masks(B, H, W, seeds, mask, accel, radial, vd)
    y0, x0, aty0 = simulate_measurements(gt, mask, sigma_n, seeds)
    return {"x0": torch.view_as_real(x0), "y0": torch.view_as_real(y0), "ATy0": torch.view_as_real(aty0), "mask": mask,
            "gt": gt.reshape(-1, 1, H, W).expand(B, 1, H, W).contiguous()}


def residual_real(z: torch.Tensor, u: torch.Tensor) -> torch.Tensor:
    """``Re(z - u)`` as fp32 (env.py:85-86)."""
    z = _req(z, torch.complex64, "z")
    u = _req(u, torch.complex64, "u")
    v = torch.empty(z.shape, dtype=torch.float32, device=z.device)
    check(_lib.lib().pnp_residual_real(z.data_ptr(), u.data_ptr(), v.data_ptr(), z.numel(), _lib.stream_ptr()),
          "pnp_residual_real")
    return v


class MaskKindProbe:
    """Host-side view of the mask-structure flag that ``pnp_prox_prepare`` leaves on the device, WITHOUT a synchronisation:
    an asynchronous 4-byte copy into pinned memory plus an event.  ``get()`` returns -1 until the copy has landed, then
    1 (every mask depends on the column index only: row kernel) or 0 (general masks: cluster kernel) - the ``kind``
    argument of ``pnp_prox_dual_prepared_kind`` / ``pnp_step_prepared_kind`` (-1 launches both kernels).  Without
    ``maskp`` (nothing prepared yet) ``get()`` stays -1."""

    def __init__(self, maskp: torch.Tensor | None = None, mstride: int = 0, B: int = 0, H: int = 0, W: int = 0):
        self.kind, self.event = -1, None
        if maskp is None:
            return
        self.host = torch.full((1,), -1, dtype=torch.int32).pin_memory()
        check(_lib.lib().pnp_prox_prepared_kind_async(maskp.data_ptr(), mstride, B, H, W, self.host.data_ptr(),
                                                      _lib.stream_ptr()), "pnp_prox_prepared_kind_async")
        self.event = torch.cuda.Event()
        self.event.record()

    def get(self) -> int:
        if (self.kind < 0 and self.event is not None and not torch.cuda.is_current_stream_capturing()
                and self.event.query()):
            self.kind = 1 if int(self.host[0]) != 0 else 0
        return self.kind


class ProxPrepared:
    """Trajectory constants of the prox step (``pnp_prox_prepare``, see include/pnp_b200.h): the buffers ``y0p`` and
    ``maskp``, their mask stride and the host-side mask-kind hint ``probe``.

    ``ProxPrepared(y0, mask)`` then ``prep.prox_dual(x, u, mu)`` per iteration; same results as ``prox_dual``.
    ``ProxPrepared.empty(B, H, W, device)`` allocates the buffers zero-filled and ``prep.prepare(y0, mask)`` (re)fills them
    in place, so CUDA graphs that captured them stay valid for the next trajectory.
    Only for shapes with a prepared path (``supported(H, W)``)."""

    @staticmethod
    def supported(H: int, W: int) -> bool:
        return bool(_lib.lib().pnp_prox_prepared_supported(H, W))

    def __init__(self, y0, mask):
        y0 = _req(y0, torch.complex64, "y0")
        H, W = y0.shape[-2:]
        self._allocate(y0.numel() // (H * W), H, W, y0.device)
        self.prepare(y0, mask)

    @classmethod
    def empty(cls, B: int, H: int, W: int, device) -> "ProxPrepared":
        prep = cls.__new__(cls)
        prep._allocate(B, H, W, device)
        return prep

    def _allocate(self, B: int, H: int, W: int, device):
        n_y, n_m = C.c_size_t(0), C.c_size_t(0)
        check(_lib.lib().pnp_prox_prepared_bytes(B, H, W, C.byref(n_y), C.byref(n_m)), "pnp_prox_prepared_bytes")
        self.B, self.H, self.W = B, H, W
        self.y0p = torch.zeros(n_y.value // 8, dtype=torch.complex64, device=device)
        self.maskp = torch.zeros(n_m.value, dtype=torch.uint8, device=device)
        self.mstride = 0
        self.probe = MaskKindProbe()

    def prepare(self, y0, mask):
        """Prepare ``y0`` (complex64, B images) and ``mask`` (bool/uint8, B masks or one for the batch) into the buffers."""
        B, H, W = self.B, self.H, self.W
        y0 = _req(y0, torch.complex64, "y0")
        if y0.numel() != B * H * W:
            raise IndexError(f"y0 with {y0.numel()} elements does not match {B} images of {H}x{W}")
        mask, self.mstride = _mask_arg(mask, B, H, W)
        check(_lib.lib().pnp_prox_prepare(y0.data_ptr(), mask.data_ptr(), self.mstride, self.y0p.data_ptr(),
                                          self.maskp.data_ptr(), B, H, W, _lib.stream_ptr()), "pnp_prox_prepare")
        self.probe = MaskKindProbe(self.maskp, self.mstride, B, H, W)

    @property
    def column_only(self) -> bool:
        """Did the preparation find every mask of the batch to depend on the column index only? (synchronises)"""
        self.probe.event.synchronize()
        return self.probe.get() == 1

    @property
    def launches(self) -> int:
        """Kernel launches of one ``prox_dual`` with the current host-side hint (the routing of ``pnp_prox_dual_prepared``)."""
        kind = self.probe.get()
        if (self.H, self.W) == (128, 128):
            return 1                          # the 4-CTA cluster kernel serves every mask
        if (self.H, self.W) == (256, 256):
            return 1 if kind >= 0 else 2      # row-only or cluster kernel; both while the kind is unknown
        return {1: 1, 0: 3}.get(kind, 4)      # row-only kernel, the three radix passes, or both

    def prox_dual(self, x, u, mu, want_v: bool = True, out=None, kind: int | None = None):
        """``kind``: None = use the host-side hint once it has landed; -1 forces the both-kernels launch."""
        x = _req(x, torch.float32, "x")
        u = _req(u, torch.complex64, "u")
        mu, mu_stride = _per_image(mu.float(), self.B, torch.float32, "mu", x.device)
        if out is None:
            z, un = torch.empty_like(u), torch.empty_like(u)
            v = torch.empty_like(x) if want_v else None
        else:
            z, un, v = out
        check(_lib.lib().pnp_prox_dual_prepared_kind(x.data_ptr(), u.data_ptr(), self.y0p.data_ptr(), self.maskp.data_ptr(),
                                                     self.mstride, mu.data_ptr(), mu_stride, z.data_ptr(), un.data_ptr(),
                                                     v.data_ptr() if v is not None else None, self.B, self.H, self.W,
                                                     self.probe.get() if kind is None else kind, _lib.stream_ptr()),
              "pnp_prox_dual_prepared_kind")
        return z, un, v


def prox_dual(x, u, y0, mask, mu, want_v: bool = True, out=None, workspace=None):
    """env.py:87-93.  x fp32 ``[B,1,H,W]``; u, y0 c64; mask bool/uint8 ``[B or 1,1,H,W]``; mu fp32 ``[1]`` or ``[B]``.

    Returns ``(z, u_new, v_next)`` as fresh tensors unless ``out=(z, u_new, v)`` is given.
    """
    x = _req(x, torch.float32, "x")
    u = _req(u, torch.complex64, "u")
    y0 = _req(y0, torch.complex64, "y0")
    H, W = x.shape[-2:]
    B = x.numel() // (H * W)
    mask, mstride = _mask_arg(mask, B, H, W)
    mu, mu_stride = _per_image(mu.float(), B, torch.float32, "mu", x.device)
    if out is None:
        z = torch.empty_like(u)
        un = torch.empty_like(u)
        v = torch.empty_like(x) if want_v else None
    else:
        z, un, v = out
    l = _lib.lib()
    if workspace is None:
        workspace = torch.empty(l.pnp_prox_workspace_bytes(B, H, W), dtype=torch.uint8, device=x.device)
    check(l.pnp_prox_dual(x.data_ptr(), u.data_ptr(), y0.data_ptr(), mask.data_ptr(), mstride, mu.data_ptr(), mu_stride,
                          z.data_ptr(), un.data_ptr(), v.data_ptr() if v is not None else None, workspace.data_ptr(),
                          B, H, W, _lib.stream_ptr()), "pnp_prox_dual")
    return z, un, v


def conv3x3_bf16(in0: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, in1: torch.Tensor | None = None):
    """NHWC bf16 3x3 conv + bias + LeakyReLU(0.2) on the tensor cores; ``in1`` = second concat segment."""
    in0 = _req(in0, torch.bfloat16, "in0")
    B, H, W, C0 = in0.shape
    C1 = 0
    if in1 is not None:
        in1 = _req(in1, torch.bfloat16, "in1")
        C1 = in1.shape[-1]
    weight = _req(weight, torch.float32, "weight")
    bias = _req(bias, torch.float32, "bias")
    Cout = weight.shape[0]
    assert weight.shape == (Cout, C0 + C1, 3, 3)
    l = _lib.lib()
    out = torch.empty(B, H, W, Cout, dtype=torch.bfloat16, device=in0.device)
    scratch = aligned_empty(l.pnp_conv3x3_packed_bytes(C0 + C1, Cout), in0.device)
    check(l.pnp_conv3x3_bf16(in0.data_ptr(), C0, in1.data_ptr() if in1 is not None else None, C1, weight.data_ptr(),
                             bias.data_ptr(), out.data_ptr(), scratch.data_ptr(), B, H, W, Cout, _lib.stream_ptr()),
          "pnp_conv3x3_bf16")
    return out


# ------------------------------------------------------------------------------------------------
_UNET_BLOCKS = (("inc.conv", 2, 32), ("down1.mpconv.1", 32, 64), ("down2.mpconv.1", 64, 128), ("down3.mpconv.1", 128, 256),
                ("down4.mpconv.1", 256, 512), ("up1.conv", 768, 256), ("up2.conv", 384, 128), ("up3.conv", 192, 64),
                ("up4.conv", 96, 32))


def unet_state_dict_shapes():
    """(key, shape) of the 56 tensors of the reference ``UNet(2, 1)`` state_dict in registration order."""
    out = []
    for blk, cin, cout in _UNET_BLOCKS:
        for i in range(3):
            out.append((f"{blk}.conv-{i}.conv2d.weight", (cout, cin if i == 0 else cout, 3, 3)))
            out.append((f"{blk}.conv-{i}.conv2d.bias", (cout,)))
    out += [("outc.conv.weight", (1, 32, 1, 1)), ("outc.conv.bias", (1,))]
    return out


def unflatten_state_dict(flat: torch.Tensor):
    """Inverse of ``flatten_state_dict``: flat fp32 vector -> reference-format state_dict."""
    from collections import OrderedDict
    flat = flat.detach().reshape(-1).to(torch.float32).cpu()
    sd, off = OrderedDict(), 0
    for k, shp in unet_state_dict_shapes():
        n = 1
        for d in shp:
            n *= d
        sd[k] = flat[off:off + n].reshape(shp).clone()
        off += n
    if off != flat.numel():
        raise ValueError(f"flat parameter vector has {flat.numel()} entries, the U-Net has {off}")
    return sd


def flatten_state_dict(sd) -> torch.Tensor:
    """Reference ``UNet(2,1)`` state_dict (56 tensors, noise.py:101-113) -> flat fp32 vector in registration order."""
    keys = [k for k, _ in unet_state_dict_shapes()]
    missing = [k for k in keys if k not in sd]
    if missing:
        raise KeyError(f"state_dict is missing U-Net tensors: {missing[:4]}{'...' if len(missing) > 4 else ''}")
    return torch.cat([sd[k].detach().reshape(-1).to(torch.float32).cpu() for k in keys])


class UNetPlan:
    """Launch plan of the denoiser for one ``(B, H, W)`` (tensor maps, activation workspace)."""

    def __init__(self, packed: torch.Tensor, B: int, H: int, W: int):
        l = _lib.lib()
        self.B, self.H, self.W = B, H, W
        self.packed = packed
        nbytes = l.pnp_unet_workspace_bytes(B, H, W)
        self.workspace = aligned_empty(nbytes, packed.device)
        h = C.c_void_p()
        check(l.pnp_unet_plan_create(C.byref(h), packed.data_ptr(), self.workspace.data_ptr(), nbytes, B, H, W),
              "pnp_unet_plan_create")
        self.handle = h

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                _lib.load().pnp_unet_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def forward(self, v: torch.Tensor, sigma: torch.Tensor, out: torch.Tensor | None = None, preclamp: bool = False):
        v = _req(v, torch.float32, "v")
        sigma = _req(sigma.reshape(-1).float(), torch.float32, "sigma")
        assert v.numel() == self.B * self.H * self.W and sigma.numel() == self.B
        if out is None:
            out = torch.empty_like(v)
        pre = torch.empty_like(v) if preclamp else None
        check(_lib.lib().pnp_unet_forward(self.handle, v.data_ptr(), sigma.data_ptr(), out.data_ptr(),
                                          pre.data_ptr() if pre is not None else None, _lib.stream_ptr()),
              "pnp_unet_forward")
        return (out, pre) if preclamp else out

    def activation(self, name: str) -> torch.Tensor:
        """NHWC bf16 view of a named intermediate (valid after ``forward``; later layers may reuse buffers)."""
        off, c, h, w = C.c_size_t(), C.c_int(), C.c_int(), C.c_int()
        rc = _lib.lib().pnp_unet_plan_tensor(self.handle, name.encode(), C.byref(off), C.byref(c), C.byref(h), C.byref(w))
        if rc != 0:
            raise KeyError(name)
        n = self.B * h.value * w.value * c.value
        return self.workspace[off.value:off.value + 2 * n].view(torch.bfloat16).view(self.B, h.value, w.value, c.value)


def pack_unet_weights(flat: torch.Tensor) -> torch.Tensor:
    """fp32 flat parameter vector (CUDA) -> packed bf16 tensor-core blobs (+ fp32 copy)."""
    l = _lib.lib()
    flat = _req(flat, torch.float32, "flat")
    if flat.numel() != l.pnp_unet_num_params():
        raise RuntimeError(f"expected {l.pnp_unet_num_params()} U-Net parameters, got {flat.numel()}")
    packed = aligned_empty(l.pnp_unet_packed_bytes(), flat.device)
    packed.zero_()
    check(l.pnp_unet_pack_weights(flat.data_ptr(), packed.data_ptr(), _lib.stream_ptr()), "pnp_unet_pack_weights")
    return packed
