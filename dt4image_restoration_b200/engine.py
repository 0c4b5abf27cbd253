"""Batched, allocation-free PnP-ADMM engine: the hot loop of ``PnPEnv.step`` (reference
``evaluation/env.py:85-93``) for ``B`` independent trajectories with persistent device buffers.

``PnPEnv`` (env.py in this package) keeps the reference's dict-in/dict-out contract and allocates fresh
``x, z, u`` every step (callers such as the MCTS tree keep references to old ones, reference
``evaluation/mcts.py:15,18``).  This class is the explicit batched API next to it: buffers are reused,
per-image ``mu`` is allowed (the reference only takes a scalar, env.py:88), nothing synchronises with the
host, and the whole step is one C-ABI call (``pnp_step``), so it can be captured in a CUDA graph.
"""
from __future__ import annotations

import torch

from . import _lib, ops
from ._lib import check
from .noise import UNetDenoiser2D


class PnPEngine:
    def __init__(self, denoiser: UNetDenoiser2D, B: int, H: int, W: int, device="cuda"):
        self.B, self.H, self.W = B, H, W
        self.device = torch.device(device)
        _lib.check_device(self.device)            # one process drives one GPU (see _lib.check_device)
        self.denoiser = denoiser.to(self.device)
        self.plan = self.denoiser.plan(B, H, W)
        dev = self.device
        self.x = torch.zeros(B, 1, H, W, dtype=torch.float32, device=dev)
        self.v = torch.zeros(B, 1, H, W, dtype=torch.float32, device=dev)
        self.z = torch.zeros(B, 1, H, W, dtype=torch.complex64, device=dev)
        self.u = torch.zeros(B, 1, H, W, dtype=torch.complex64, device=dev)
        self.y0 = torch.zeros(B, 1, H, W, dtype=torch.complex64, device=dev)
        self.mask = torch.zeros(B, 1, H, W, dtype=torch.uint8, device=dev)
        self.gt = torch.zeros(B, 1, H, W, dtype=torch.float32, device=dev)
        self.actions = torch.zeros(2, B, dtype=torch.float32, device=dev)    # one upload per step: row 0 sigma_d, row 1 mu
        self.sigma = self.actions[0]
        self.mu = self.actions[1]
        self.reward = torch.zeros(B, dtype=torch.float32, device=dev)
        self.ssim_out = torch.zeros(B, dtype=torch.float32, device=dev)
        self.ssim_work = ops.aligned_empty(_lib.lib().pnp_ssim_workspace_bytes(B, H, W), dev, align=16)
        self.work = torch.empty(_lib.lib().pnp_prox_workspace_bytes(B, H, W), dtype=torch.uint8, device=dev)
        # shapes with a prepared prox path keep the trajectory constants derived from y0 / mask (ops.ProxPrepared)
        self.prepared = ops.ProxPrepared.supported(H, W)
        if self.prepared:
            self.prep = ops.ProxPrepared.empty(B, H, W, dev)
        self.iters = 0

    # the prepared buffers and the host-side mask-kind hint, under the names bench.py and tools/ncu_step.py read
    y0T = property(lambda self: self.prep.y0p)
    maskT = property(lambda self: self.prep.maskp)
    probe = property(lambda self: self.prep.probe)

    @property
    def launches_per_step(self) -> int:
        """Kernel launches of one step: the denoiser's op list (depends on L2 chunking) + the FFT-prox launches."""
        return _lib.lib().pnp_unet_num_launches(self.plan.handle) + (self.prep.launches if self.prepared else 3)

    def reset(self, data: dict, non_blocking: bool = False):
        """Same item dict as ``PnPEnv.reset`` (reference env.py:57-71), batch on dim 0."""
        B, H, W = self.B, self.H, self.W
        x0 = torch.view_as_complex(torch.as_tensor(data["x0"]).contiguous()).reshape(B, 1, H, W)
        y0 = torch.view_as_complex(torch.as_tensor(data["y0"]).contiguous()).reshape(B, 1, H, W)
        mask = torch.as_tensor(data["mask"]).reshape(-1, 1, H, W)
        if mask.shape[0] == 1 and B > 1:
            mask = mask.expand(B, -1, -1, -1)
        self.z.copy_(x0, non_blocking=non_blocking)
        self.u.zero_()
        self.y0.copy_(y0, non_blocking=non_blocking)
        if mask.dtype in (torch.uint8, torch.bool) and not mask.is_cuda:
            # raw bytes go up asynchronously (pinned source stays pinned); "!= 0" as in reference env.py:64 on the device
            self.mask.copy_(mask.view(torch.uint8) if mask.dtype == torch.bool else mask, non_blocking=non_blocking)
            self.mask.copy_(self.mask.ne(0))
        else:
            self.mask.copy_(mask.to(self.device, non_blocking=non_blocking).ne(0))
        self.gt.copy_(torch.as_tensor(data["gt"]).reshape(B, 1, H, W), non_blocking=non_blocking)
        self.x.copy_(self.z.real)
        self.v.copy_(self.z.real)           # Re(z - u) with u = 0
        self.prepare()
        self.iters = 0

    def reset_from_gt(self, gt, sigma_n, seeds, mask=None, accel=None, radial=None, vd=None):
        """Start B new trajectories from fully-sampled images, simulating the measurements straight into the engine's
        buffers (``ops.simulate_measurements``; no host<->device copy of image data): ``y0``, ``z`` = x0, ``x`` = ``v`` =
        Re x0, ``u`` = 0, ``mask``, ``gt``.  Same state as
        ``reset(ops.make_items(gt, sigma_n, seeds, mask, accel, radial, vd))``.  ``gt`` fp32 CUDA ``[B,1,H,W]`` / ``[B,H,W]``
        / ``[H,W]``; pass exactly one of ``mask`` (bool/uint8 ``[B or 1, ..., H, W]``, CUDA), ``accel`` (Cartesian masks
        drawn with ``seeds``), ``radial`` (radial masks with this sampled fraction, rotated by ``seeds``) and ``vd`` (the
        acceleration of variable-density masks drawn with ``seeds``)."""
        B, H, W = self.B, self.H, self.W
        seeds = ops._seed_tensor(seeds, B, self.device)
        ops._episode_masks(B, H, W, seeds, mask, accel, radial, vd, out=self.mask)
        self.gt.copy_(ops._req(gt, torch.float32, "gt").reshape(-1, 1, H, W).expand(B, 1, H, W))
        ops.simulate_measurements(self.gt, self.mask, sigma_n, seeds, aty0=False, out=(self.y0, self.z, None))
        self.u.zero_()
        self.x.copy_(self.z.real)
        self.v.copy_(self.z.real)           # Re(z - u) with u = 0
        self.prepare()
        self.iters = 0

    def prepare(self):
        """Refresh the prepared copies after ``y0`` / ``mask`` changed (they are constants of a trajectory)."""
        if self.prepared:
            self.prep.prepare(self.y0, self.mask)

    def set_actions(self, sigma_d, mu):
        """Device-side action buffers: ``sigma_d`` ``[B]``, ``mu`` scalar or ``[B]`` (tensors or floats)."""
        self.sigma.copy_(torch.as_tensor(sigma_d, dtype=torch.float32).reshape(-1).expand(self.B), non_blocking=True)
        self.mu.copy_(torch.as_tensor(mu, dtype=torch.float32).reshape(-1).expand(self.B), non_blocking=True)

    def step(self, active: torch.Tensor | None = None):
        """One PnP-ADMM iteration for all B images (uses the current ``sigma``/``mu`` buffers).

        ``active`` (bool ``[B]``, device): trajectories with ``False`` keep their state untouched, which is what the
        reference's early exit ``if T > 0.5: return states, True`` (env.py:79-81) does for a single image; no host
        synchronisation is involved.
        """
        if self.prepared:
            # per-image early exit: the predicate is applied in the epilogues of the last conv and of the prox kernels
            # (pnp_step_prepared_active), no copies of the state and no select passes
            if active is not None:
                if active.dtype == torch.bool:
                    active = active.view(torch.uint8)
                active = active.reshape(-1)
                if active.numel() != self.B or not active.is_cuda or active.dtype != torch.uint8:
                    raise RuntimeError(f"active must be a bool / uint8 CUDA tensor with {self.B} elements")
            p = self.prep
            check(_lib.lib().pnp_step_prepared_active(self.plan.handle, self.v.data_ptr(), self.sigma.data_ptr(),
                                                      self.u.data_ptr(), p.y0p.data_ptr(), p.maskp.data_ptr(), p.mstride,
                                                      self.mu.data_ptr(), 1, self.x.data_ptr(), self.z.data_ptr(),
                                                      self.u.data_ptr(), self.v.data_ptr(), p.probe.get(),
                                                      active.data_ptr() if active is not None else None,
                                                      _lib.stream_ptr()), "pnp_step_prepared_active")
        else:
            if active is not None:
                prev = [t.clone() for t in (self.x, self.z, self.u, self.v)]
            check(_lib.lib().pnp_step(self.plan.handle, self.v.data_ptr(), self.sigma.data_ptr(), self.u.data_ptr(),
                                      self.y0.data_ptr(), self.mask.data_ptr(), self.H * self.W, self.mu.data_ptr(), 1,
                                      self.x.data_ptr(), self.z.data_ptr(), self.u.data_ptr(), self.v.data_ptr(),
                                      self.work.data_ptr(), _lib.stream_ptr()), "pnp_step")
            if active is not None:
                m = active.reshape(self.B, 1, 1, 1).bool()
                for p, t in zip(prev, (self.x, self.z, self.u, self.v)):
                    t.copy_(torch.where(m, t, p))
        self.iters += 1

    def psnr(self) -> torch.Tensor:
        """Per-image reward of the current ``x`` (reference env.py:112-125), on the device."""
        check(_lib.lib().pnp_psnr(self.x.data_ptr(), self.gt.data_ptr(), self.H * self.W, self.reward.data_ptr(), self.B,
                                  self.H * self.W, _lib.stream_ptr()), "pnp_psnr")
        return self.reward

    def ssim(self) -> torch.Tensor:
        """Per-image SSIM of the current ``x`` against ``gt`` (see ``ops.ssim``), on the device; allocation-free, so it can
        be captured in a CUDA graph.  Returns the same ``[B]`` buffer on every call."""
        check(_lib.lib().pnp_ssim(self.x.data_ptr(), self.gt.data_ptr(), self.H * self.W, self.ssim_out.data_ptr(),
                                  self.ssim_work.data_ptr(), self.B, self.H, self.W, _lib.stream_ptr()), "pnp_ssim")
        return self.ssim_out

    def run(self, sigmas, mus, n_iters: int | None = None):
        """Fixed-schedule trajectory: ``sigmas[k]``, ``mus[k]`` scalars or ``[B]`` per iteration."""
        n = len(sigmas) if n_iters is None else n_iters
        for k in range(n):
            self.set_actions(sigmas[k], mus[k])
            self.step()
        return self.x
