"""Drop-in for the reference environment ``PnPEnv`` (reference ``evaluation/env.py:30-125``).

Call-compatible with the reference's callers (``evaluation/eval.py:75,119,203-212``,
``evaluation/mcts.py:118,126,192,215``): same constructor, ``reset(data, device_type)``,
``step(states, action_dict) -> (states, done)``, ``get_policy_ob``, ``compute_reward``; same state-dict
keys, dtypes, in-place dict mutation and "fresh tensors for x, z, u" ownership (SURVEY.md section 8b).
Differences, all generalisations: any batch ``B`` and any ``H, W`` in 16..1024 (radix FFT kernels for powers of two in
32..512, a dense-DFT path for every other size the reference's ``step`` accepts) instead of the literal
``1 x 128 x 128`` (env.py:64,115), and the compute runs as sm_100a CUDA kernels through the C-ABI
(``include/pnp_b200.h``).  There is no CPU path.
"""
from __future__ import annotations

from collections import OrderedDict

import torch

from . import _lib, ops
from ._lib import check
from .noise import UNetDenoiser2D

# Images per call up to which ``PnPEnv.step`` replays a CUDA graph: below this the step is bound by ~30 kernel launches of
# 5-10 us each (profiles/r01_config1_b1_256_radial30.txt), above it by the kernels themselves.
GRAPH_MAX_PIXELS = 8 * 256 * 256


class _GraphedStep:
    """The body of ``PnPEnv.step`` (reference env.py:85-93) for one ``(B, H, W)`` as ONE CUDA-graph replay.

    Static device buffers: the state ``[x | z | u]`` (one flat allocation), ``sigma_d``, ``mu`` and the prepared prox
    constants (``pnp_prox_prepare`` runs into them once per trajectory, outside the graph, so a new trajectory does not
    re-capture).  The graph reads ``z, u`` from the static state and writes ``x, z, u`` back into it (the prox kernels
    allow ``u_out`` to alias ``u_in``; ``z`` is consumed by the first kernel), so consecutive steps of one trajectory
    need no input copy; the drop-in contract "x, z, u are FRESH tensors every step" (SURVEY section 8b: MCTS nodes keep
    references to old ones, reference mcts.py:15,18) is kept by ONE copy of the flat state into a new allocation."""

    def __init__(self, denoiser: UNetDenoiser2D, B: int, H: int, W: int, device):
        self.B, self.H, self.W, self.dev = B, H, W, device
        n = B * H * W
        self.flat = torch.zeros(n * 5, dtype=torch.float32, device=device)         # x: n floats, z: 2n, u: 2n
        self.x = self.flat[:n].view(B, 1, H, W)
        self.z = torch.view_as_complex(self.flat[n:3 * n].view(B, 1, H, W, 2))
        self.u = torch.view_as_complex(self.flat[3 * n:].view(B, 1, H, W, 2))
        self.v = torch.zeros(B, 1, H, W, dtype=torch.float32, device=device)
        self.sigma = torch.zeros(B, dtype=torch.float32, device=device)
        self.mu = torch.zeros(1, dtype=torch.float32, device=device)
        self.prep = ops.ProxPrepared.empty(B, H, W, device)
        self.plan = denoiser.plan(B, H, W)
        self.prep_key = None
        self.last_out = None                    # (z, u) handed out by the last step and their versions
        self.graph = None

    def prepare(self, y0, mask, traj=None):
        key = (("traj", traj, tuple(mask.shape)) if traj is not None else
               (y0.data_ptr(), y0._version, mask.data_ptr(), mask._version, tuple(mask.shape)))
        if key == self.prep_key:
            return
        mstride = self.prep.mstride
        self.prep.prepare(y0, mask)             # IndexError for a mask that does not match
        if self.prep.mstride != mstride:
            self.graph = None                   # the mask stride is baked into the captured launch
        self.prep_key, self._keep = key, (y0, mask)

    def _body(self):
        l, p = _lib.lib(), self.prep
        n = self.z.numel()
        check(l.pnp_residual_real(self.z.data_ptr(), self.u.data_ptr(), self.v.data_ptr(), n, _lib.stream_ptr()),
              "pnp_residual_real")
        check(l.pnp_step_prepared_kind(self.plan.handle, self.v.data_ptr(), self.sigma.data_ptr(), self.u.data_ptr(),
                                       p.y0p.data_ptr(), p.maskp.data_ptr(), p.mstride, self.mu.data_ptr(), 0,
                                       self.x.data_ptr(), self.z.data_ptr(), self.u.data_ptr(), None, -1,
                                       _lib.stream_ptr()), "pnp_step_prepared_kind")

    @staticmethod
    def _set_action(buf, val):
        """Device tensors are copied on the stream; host scalars travel as a kernel argument (``fill_``), which keeps the
        copy engine - and its switch-over bubbles - out of a 0.2 ms step; host vectors take the pageable copy."""
        if torch.is_tensor(val) and val.is_cuda:
            buf.copy_(val.reshape(-1).expand_as(buf) if val.numel() == 1 else val.reshape(buf.shape), non_blocking=True)
            return
        t = torch.as_tensor(val, dtype=torch.float32).reshape(-1)
        if t.numel() == 1:
            buf.fill_(float(t))
        else:
            buf.copy_(t.reshape(buf.shape), non_blocking=True)

    def run(self, z, u, sigma, mu):
        last = self.last_out
        if not (last is not None and z is last[0] and u is last[1] and z._version == last[2] and u._version == last[3]):
            self.z.copy_(z)
            self.u.copy_(u)
        self._set_action(self.sigma, sigma)
        self._set_action(self.mu, mu)
        if self.graph is None:
            keep = self.flat.clone()
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._body()                     # warm-up outside the capture (lazy kernel attributes)
            torch.cuda.current_stream().wait_stream(s)
            self.flat.copy_(keep)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._body()
            self.graph = g
        self.graph.replay()
        n = self.B * self.H * self.W
        out = self.flat.clone()                  # fresh x, z, u (one copy kernel)
        x = out[:n].view(self.B, 1, self.H, self.W)
        zo = torch.view_as_complex(out[n:3 * n].view(self.B, 1, self.H, self.W, 2))
        uo = torch.view_as_complex(out[3 * n:].view(self.B, 1, self.H, self.W, 2))
        self.last_out = (zo, uo, zo._version, uo._version)
        return x, zo, uo


class PnPEnv:
    _traj_counter = 0

    def __init__(self, max_episode_step, denoiser, device_type, use_graph: bool = True) -> None:
        self.max_episode_step = max_episode_step
        self.denoiser = denoiser.to(device_type)
        self.no_ref_model = None
        self.use_graph = use_graph            # small batches: replay the step as one CUDA graph (see _GraphedStep)
        self._graphed = OrderedDict()         # (B, H, W) -> _GraphedStep
        self._prep_cache = OrderedDict()      # (y0, mask) identity -> ops.ProxPrepared, see _prepared()
        self._load_no_ref()

    def _load_no_ref(self):
        """The reference downloads ARNIQA through torch.hub here (env.py:36-40); that needs the network and third-party
        weights, so nothing is loaded: assign ``env.no_ref_model`` - either the ARNIQA module itself (any ``nn.Module`` with
        its call signature; ``run_no_ref_reward`` then does what the reference does) or a plain ``callable(state) -> float``."""
        self.no_ref_model = None

    @staticmethod
    def no_ref_inputs(state):
        """The two model inputs of the reference's ``run_no_ref_reward`` (env.py:42-50) for one image of any size: ``x`` as a
        3-channel image (grey channel + two zero channels, ``greyscale_to_rgb`` env.py:20-25) at full and at half resolution
        (``torchvision.transforms.Resize`` on a tensor = antialiased bilinear), each with a leading batch dimension."""
        import torch.nn.functional as F
        x = state['x']
        x = x.real if x.is_complex() else x
        H, W = x.shape[-2:]
        img = x.reshape(1, H, W).float()
        img_ds = F.interpolate(img[None], size=(H // 2, W // 2), mode="bilinear", antialias=True, align_corners=False)[0]
        rgb = lambda t: torch.cat((t, torch.zeros(2, *t.shape[-2:], dtype=t.dtype, device=t.device)), dim=0)
        return rgb(img).unsqueeze(0), rgb(img_ds).unsqueeze(0)

    def run_no_ref_reward(self, state):
        """env.py:42-54.  With an ``nn.Module`` installed (ARNIQA or a stand-in with its signature) the call is the
        reference's: ``model(img, img_ds, return_embedding=False, scale_score=True)`` under ``no_grad`` + autocast, mean score
        as a float; a plain callable is called with the state."""
        if self.no_ref_model is None:
            raise NotImplementedError("no-reference reward model not installed (reference env.py:36-54 uses ARNIQA "
                                      "via torch.hub); assign env.no_ref_model = the ARNIQA module, or a callable(state) -> float")
        if isinstance(self.no_ref_model, torch.nn.Module):
            img, img_ds = self.no_ref_inputs(state)
            with torch.no_grad(), torch.autocast(device_type=img.device.type, enabled=img.is_cuda):
                score = self.no_ref_model(img, img_ds, return_embedding=False, scale_score=True)
            return score.mean(0).item()
        return float(self.no_ref_model(state))

    # ------------------------------------------------------------------------------------------
    def reset(self, data, device_type):
        """env.py:57-71 for any ``[B,1,H,W,2]`` item batch."""
        x = torch.as_tensor(data['x0'])
        x = torch.view_as_complex(x.contiguous())
        data['complex_y0'] = data['y0']
        B, _, H, W = x.shape
        z = x.clone().detach()
        u = torch.zeros_like(x)
        mask = torch.as_tensor(data['mask']).reshape(-1, 1, H, W).contiguous().to(torch.bool)
        y0 = torch.view_as_complex(torch.as_tensor(data['y0']).contiguous())
        gt = torch.as_tensor(data['gt'])
        Aty0 = torch.as_tensor(data['ATy0'])[..., 0]
        x, z, u, mask, y0, gt = (t.to(device_type) for t in (x, z, u, mask, y0, gt))
        # '_traj': an id of this trajectory's constants (y0, mask).  It survives copy.deepcopy of the state dict, so callers
        # that copy states per tree node keep hitting the same prepared prox constants instead of re-preparing every step.
        PnPEnv._traj_counter += 1
        return OrderedDict({'x': x, 'y0': y0, 'z': z, 'u': u, 'mask': mask, 'gt': gt, 'ATy0': Aty0, 'T': 0,
                            'complex_y0': data['y0'], '_traj': PnPEnv._traj_counter})

    def _prepared(self, y0, mask, traj=None):
        """``y0`` and ``mask`` are constants of a trajectory (set in ``reset``), so what the prox step derives from them
        (transposed / column-transformed copies, the mask-structure flag) is prepared once and reused by every later
        ``step`` on the same tensors; the key includes the tensors' version counters, so in-place edits re-prepare."""
        H, W = y0.shape[-2:]
        if not ops.ProxPrepared.supported(H, W):
            return None
        key = (("traj", traj, tuple(y0.shape), tuple(mask.shape)) if traj is not None else
               (y0.data_ptr(), y0._version, tuple(y0.shape), mask.data_ptr(), mask._version, tuple(mask.shape)))
        prep = self._prep_cache.get(key)
        if prep is None:
            prep = ops.ProxPrepared(y0, mask)
            prep._keepalive = (y0, mask)          # the key is only valid while these tensors are alive
            self._prep_cache[key] = prep
            while len(self._prep_cache) > 4:
                self._prep_cache.popitem(last=False)
        else:
            self._prep_cache.move_to_end(key)
        return prep

    def step(self, states: OrderedDict, action_dict: OrderedDict):
        """env.py:74-100: denoise -> centred FFT -> masked k-space solve -> inverse FFT -> dual update."""
        T, mu, sigma_d = action_dict['T'], action_dict['mu'], action_dict['sigma_d']
        y0, z, u, mask = states['y0'], states['z'], states['u'], states['mask']

        if T > 0.5:          # tensor -> bool: same early exit (and host sync) as env.py:79-81
            return states, True
        done = False

        dev = z.device
        mu = torch.as_tensor(mu, dtype=torch.float32)
        mu.view(1, 1, 1, 1)                  # scalar mu only, like env.py:88 (RuntimeError otherwise)
        g = self._graphed_step(z, y0, mask, sigma_d, states.get('_traj'))
        if g is not None:
            x, z, u = g.run(z, u, sigma_d, mu)
            states['x'], states['z'], states['u'] = x, z, u
            states['T'] = states['T'] + 1 / 30
            return states, done
        _mu = mu.to(dev).view(1, 1, 1, 1)
        v = ops.residual_real(z, u)          # (z - u).real
        x = self.denoiser(v, torch.as_tensor(sigma_d, dtype=torch.float32, device=dev))
        prep = self._prepared(y0, mask, states.get('_traj')) if (y0.is_cuda and mask.is_cuda) else None
        if prep is not None:
            z, u, _ = prep.prox_dual(x, u, _mu, want_v=False)
        else:
            z, u, _ = ops.prox_dual(x, u, y0, mask, _mu, want_v=False)

        states['x'] = x
        states['z'] = z
        states['u'] = u
        states['T'] = states['T'] + 1 / 30
        return states, done

    def _graphed_step(self, z, y0, mask, sigma_d, traj=None):
        """The CUDA-graph replay of the step body for small calls, or None (large batches, foreign denoisers, CPU tensors,
        a capture already in progress, ``use_graph=False``): the eager path below computes the same thing."""
        if not (self.use_graph and isinstance(self.denoiser, UNetDenoiser2D) and z.is_cuda and y0.is_cuda and mask.is_cuda
                and z.dim() == 4 and z.dtype == torch.complex64):
            return None
        B, _, H, W = z.shape
        if B * H * W > GRAPH_MAX_PIXELS or not ops.ProxPrepared.supported(H, W) or torch.cuda.is_current_stream_capturing():
            return None
        if torch.as_tensor(sigma_d).numel() != B:   # the eager path raises the reference's RuntimeError (noise.py:159)
            return None
        key = (B, H, W, str(z.device))
        g = self._graphed.get(key)
        if g is None:
            g = self._graphed[key] = _GraphedStep(self.denoiser, B, H, W, z.device)
            while len(self._graphed) > 4:
                self._graphed.popitem(last=False)
        try:
            g.prepare(y0, mask, traj)
        except IndexError:
            raise
        return g

    @staticmethod
    def get_policy_ob(state: OrderedDict):
        """env.py:103-109; ``[B, H*W]`` (``[1, H*W]`` for the reference's B=1)."""
        x = state['x']
        policy_ob = x.real if x.is_complex() else x
        return policy_ob.reshape(policy_ob.shape[0], -1)

    @staticmethod
    def compute_reward(x, y0):
        """env.py:112-116: PSNR per image as a CPU ``[N,1]`` tensor (computed on the device)."""
        x = x.detach()
        N = x.shape[0]
        gt = y0.detach().reshape(-1, *x.shape[1:]) if y0.numel() != x[0].numel() else y0.detach()
        dev = x.device if x.is_cuda else (gt.device if gt.is_cuda else torch.device('cuda'))
        return ops.psnr(x.to(dev), gt.to(dev)).reshape(N, 1).cpu()

    @staticmethod
    def compute_ssim(x, gt):
        """SSIM per image (``ops.ssim``) shaped like ``compute_reward``: a CPU ``[N,1]`` tensor computed on the device."""
        x = x.detach()
        N = x.shape[0]
        gt = gt.detach().reshape(-1, *x.shape[1:]) if gt.numel() != x[0].numel() else gt.detach()
        dev = x.device if x.is_cuda else (gt.device if gt.is_cuda else torch.device('cuda'))
        return ops.ssim(x.to(dev), gt.to(dev)).reshape(N, 1).cpu()


def torch_psnr(output, gt):
    """env.py:120-125 on the device; returns ``[N,1]`` on the inputs' device."""
    return ops.psnr(output, gt).unsqueeze(1)
