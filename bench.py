#!/usr/bin/env python
"""Headline benchmark: PnP-ADMM image-iterations/sec at 256x256 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--size S] [--dump-outputs DIR]

One "step" = one PnP-ADMM iteration (U-Net denoise -> centred FFT -> masked k-space solve -> inverse FFT ->
dual update; reference evaluation/env.py:85-93) over one batch of B synthetic 256x256 CS-MRI images
(BASELINE.json configs[1]: batch 64, Cartesian 4x).  Rank 0 prints ONE JSON line.

  value        image-iterations/s, all ranks, inputs resident in HBM, timed with CUDA events (max over ranks)
  e2e          same metric through the public API with host buffers: reset(item) from pinned host memory once per 30-step
               trajectory, per step H2D of the actions and D2H of the rewards, final x to the host
               (e2e_state_roundtrip: every step uploads the whole state and downloads x, z, u)
  roofline     the tcgen05 conv kernel (26 launches/step, >95 % of the step): algorithmic conv FLOPs / summed
               launch durations (CUDA events around every launch, pnp_unet_profile) vs the measured bf16 peak
  cpu_baseline the CPU oracle (restatement of the reference's PyTorch path) on this host's cores, bounded sample
  --impl reference   only the CPU leg, as its own JSON line
  --dump-outputs DIR after the timed steps, rank 0 writes what the timed path computed in its last step as DIR/<name>.npy
                     (float32 or float64; complex arrays get a trailing (re, im) axis; at most 64 MB, a seeded
                     sample of the images when the whole batch is larger): the state x, z, u and, for `ours`, the rewards.
                     Inputs and weights are seeded, so two builds run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "pnp_admm_image_iters_per_sec_256"
UNIT = "image-iters/s"
# conv MACs x2 per image-iteration (SURVEY.md 8a-U / BASELINE.md section 3), 26 tensor-core convs + first conv
GFLOP_PER_IMAGE = {128: 9.684, 256: 38.734, 512: 154.938}


def conv_flops_umma(H, W):
    """2*MACs of the 26 tensor-core convs (everything except the 2->32 first conv and the 1x1 output conv)."""
    chans = [(32, 32), (32, 32),
             (32, 64), (64, 64), (64, 64), (64, 128), (128, 128), (128, 128), (128, 256), (256, 256), (256, 256),
             (256, 512), (512, 512), (512, 512),
             (768, 256), (256, 256), (256, 256), (384, 128), (128, 128), (128, 128), (192, 64), (64, 64), (64, 64),
             (96, 32), (32, 32), (32, 32)]
    lvl = [0, 0, 1, 1, 1, 2, 2, 2, 3, 3, 3, 4, 4, 4, 3, 3, 3, 2, 2, 2, 1, 1, 1, 0, 0, 0]
    return sum(2.0 * 9 * ci * co * (H >> l) * (W >> l) for (ci, co), l in zip(chans, lvl))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def ncu_step_traffic(B, S):
    """Per-kernel DRAM bytes (read + write) of ONE step from the committed ncu capture of the current kernels
    (profiles/r02_ncu_step_b{B}_{S}.csv: `ncu --profile-from-start off --metrics dram__bytes_read.sum,dram__bytes_write.sum,
    gpu__time_duration.sum python tools/ncu_step.py`).  None when no capture of this shape is committed."""
    import csv
    path = os.path.join(ROOT, "profiles", f"r02_ncu_step_b{B}_{S}.csv")
    if not os.path.exists(path):
        return None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    per = {}
    for r in csv.DictReader(l for l in open(path) if l.startswith('"')):
        if r["Metric Name"].startswith("dram__bytes"):
            e = per.setdefault(int(r["ID"]), [r["Kernel Name"].split("(")[0].replace("void ", ""), 0.0])
            e[1] += float(r["Metric Value"].replace(",", "")) * unit.get(r["Metric Unit"], 1.0)
    conv = [b for n, b in per.values() if n.startswith(("conv3x3_umma", "conv3x3_pair", "conv3x3_kws"))]
    unet = [b for n, b in per.values() if n.startswith(("conv", "upsample", "maxpool"))]
    first = lambda pre: next((b for n, b in per.values() if n.startswith(pre)), None)
    return {"source": os.path.relpath(path, ROOT), "conv_launches": len(conv), "conv_bytes_per_launch_mean": sum(conv) / max(len(conv), 1),
            "conv_bytes_per_step": sum(conv), "unet_bytes_per_step": sum(unet), "fftprox_rows256": first("fftprox_rows256"),
            "fftprox_cl": first("fftprox_cl_kernel"), "psnr": first("psnr_kernel")}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,clocks_event_reasons.active,"
         "enforced.power.limit")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, pw, masks = [], [], set(), [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if ts < t0 - 0.05 or ts > t1 + 0.05:
                continue
            f = [x.strip() for x in ln.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except Exception:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
            if len(f) > 7:
                masks.add(f[7])
            if len(f) > 8:
                try:
                    self.power_limit = float(f[8])
                except Exception:
                    pass
        if not sm:   # region shorter than the sampling period: use the nearest samples
            for ts, ln in self.lines[-3:]:
                f = [x.strip() for x in ln.split(",")]
                try:
                    sm.append(float(f[0])); mx.append(float(f[1]))
                except Exception:
                    pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "sm_mhz_min": float(min(sm)) if sm else None, "power_w_max": float(max(pw)) if pw else None,
                "power_limit_w": getattr(self, "power_limit", None), "samples": len(sm), "reasons": sorted(reasons),
                "event_reason_masks": sorted(masks)}


ACCEL, NOISE = 4, 0.0      # Cartesian acceleration and k-space noise sigma of the synthetic batch (--accel / --noise)


def config_dict(B, S, world):
    """``config`` of BOTH arms (ours and ``--impl reference``): identical keys and values for the same command line."""
    return {"workload": workload_name(B, S), "global_batch": world * B,
            "cache": "per-step activations (>1 GB at batch 64) exceed the 126 MB L2; no L2 flush needed"}


def workload_name(B, S):
    """``config.workload`` of both arms (ours and ``--impl reference``): BASELINE.json configs[1] by default."""
    return (f"batch {B} per GPU of {S}x{S} CS-MRI, Cartesian {ACCEL}x, k-space noise sigma {NOISE:g}, fixed (sigma,mu) schedule "
            f"standing in for the DT policy, random-init (PyTorch-default) U-Net")


def make_inputs(B, S, seed0=0):
    from dt4image_restoration_b200 import synth
    # one phantom/mask pair per 8 images is generated and tiled (generation is host-side numpy; values are
    # irrelevant to timing, parity is covered by tests/)
    nuniq = min(B, 8)
    base = synth.make_batch(nuniq, S, S, "cartesian", ACCEL, NOISE, seed0=seed0)
    reps = (B + nuniq - 1) // nuniq
    return {k: np.concatenate([v] * reps, axis=0)[:B] for k, v in base.items()}


DUMP_LIMIT_BYTES = 64_000_000     # --dump-outputs writes at most this much


def dump_index(B, image_bytes, other_bytes):
    """Images whose per-image outputs --dump-outputs writes: all B when they fit under DUMP_LIMIT_BYTES next to
    `other_bytes`, else a fixed seeded sample (sorted), the same on every run with the same arguments.  ValueError when
    not even one image fits."""
    import torch
    n = min(B, (DUMP_LIMIT_BYTES - other_bytes) // image_bytes)
    if n < 1:
        raise ValueError(f"--dump-outputs: x, z and u of one image ({image_bytes} bytes) do not fit in the "
                         f"{DUMP_LIMIT_BYTES}-byte limit; use a smaller --size")
    idx = np.arange(B) if n >= B else np.sort(np.random.default_rng(0).choice(B, n, replace=False))
    return torch.from_numpy(idx)


def write_outputs(out_dir, arrays):
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().cpu()
        if a.is_complex():
            a = torch.view_as_real(a)
        if a.dtype != torch.float64:
            a = a.to(torch.float32)
        np.save(os.path.join(out_dir, f"{name}.npy"), a.numpy())


# ------------------------------------------------------------------------------------------------
def cpu_leg(S, threads, sample_B, steps, warmup):
    """The reference's PyTorch CPU path (oracle restatement) on this host."""
    import torch
    from oracle import pnp_oracle as O
    from dt4image_restoration_b200 import synth
    torch.set_num_threads(threads)
    params = O.init_unet_params(0, "default")
    batch = make_inputs(sample_B, S)
    st = O.reset(batch)
    sig, mus = synth.fixed_schedule(30)
    ts = []
    for k in range(warmup + steps):
        a = {"T": torch.zeros(1), "mu": torch.tensor([mus[k % 30]]), "sigma_d": torch.full((sample_B,), float(sig[k % 30]))}
        t0 = time.perf_counter()
        st, _ = O.step(params, st, a)
        ts.append(time.perf_counter() - t0)
    t = float(np.mean(ts[warmup:]))
    return sample_B / t, t, st


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    S = args.size
    sample_B = 8 if S <= 256 else 2
    v, t, st = cpu_leg(S, threads, sample_B, args.steps, args.warmup)
    if args.dump_outputs:
        idx = dump_index(sample_B, 20 * S * S, 0)      # x fp32 + z, u complex64: 20 bytes per pixel
        write_outputs(args.dump_outputs, {k: st[k].index_select(0, idx) for k in ("x", "z", "u")})
    out = {"metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "impl": "reference",
           "config": config_dict(args.batch, S, args.gpus),
           "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                            "sample": f"{args.steps} steps of {sample_B} images at {S}x{S} on rank 0's host cores, scaled per "
                                      f"image (oracle = PyTorch CPU restatement of reference env.step), {threads} threads"},
           "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(torch, local):
    """Best effort: run this rank on the CPUs of the NUMA node its GPU hangs off, BEFORE any pinned allocation, so that the
    end-to-end legs' pinned host buffers are node-local (8 ranks streaming the state through one socket's memory was the
    limit of ``e2e_state_roundtrip`` in round 1).  Returns a short description for ``run_info``."""
    try:
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return {"gpu_pci": bdf, "numa_node": node, "bound": False}
        cpus = set()
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"gpu_pci": bdf, "numa_node": node, "bound": False}
        os.sched_setaffinity(0, cpus)
        return {"gpu_pci": bdf, "numa_node": node, "bound": True, "cpus": len(cpus)}
    except Exception as ex:  # pragma: no cover - sysfs layout / permissions differ between boxes
        return {"bound": False, "why": repr(ex)[:80]}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from dt4image_restoration_b200 import _lib, synth
    from dt4image_restoration_b200.engine import PnPEngine
    from dt4image_restoration_b200.noise import UNetDenoiser2D, random_init_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line (rank 0).  NCCL prints its banner / INFO lines to stdout when NCCL_DEBUG asks for
    # them; NCCL_DEBUG is left as the caller set it, and file descriptor 1 points at stderr while NCCL initialises and runs
    # its first collective (so the lines land on stderr, where a log reader finds them); the other ranks keep it there.
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(torch, local) if world > 1 else {"bound": False, "why": "single rank"}
    if world > 1:
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)                    # communicator creation happens here
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            if rank == 0:
                os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    B, S, K, Wm = args.batch, args.size, args.steps, args.warmup
    peaks = load_peaks()

    den = UNetDenoiser2D(state_dict=random_init_state_dict(0, "default")).to(dev)
    eng = PnPEngine(den, B, S, S, dev)
    batch = make_inputs(B, S, seed0=rank * B)
    eng.reset({k: torch.from_numpy(v) for k, v in batch.items()})
    sig, mus = synth.fixed_schedule(30)
    sig_d = torch.tensor(sig, device=dev).reshape(30, 1).expand(30, B).contiguous()
    mu_d = torch.tensor(mus, device=dev).reshape(30, 1).expand(30, B).contiguous()

    def one_step(k):
        eng.sigma.copy_(sig_d[k % 30], non_blocking=True)
        eng.mu.copy_(mu_d[k % 30], non_blocking=True)
        eng.step()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the only exchange of the path: all-gather of per-image rewards (MCTS selection).  Fused with the reward kernel over
    # NVLink peer memory (pnp_psnr_allgather) when the symmetric buffer can be set up, else NCCL
    peer = None
    if world > 1 and not os.environ.get("PNP_REWARD_GATHER_NCCL"):
        from dt4image_restoration_b200 import dist as pdist0
        peer = pdist0.make_peer_gather(max(B, (512 + world - 1) // world), dev)
    gather_kind = ("peer-memory fused kernel (pnp_psnr_allgather)" if peer is not None
                   else ("nccl all_gather" if world > 1 else "none (one rank)"))

    IDLE_BEFORE_E2E_S = 1.5

    def settle():
        """The legs before the end-to-end ones (a >= 1 s full-power run, the per-launch profile) leave the GPU at its power
        cap; every leg of this file is meant to start from the same state as the K-step `value` leg, so the end-to-end legs
        begin after a short idle (`run_info.idle_before_e2e_s`); the power-capped rate is `sustained_1s`."""
        torch.cuda.synchronize()
        time.sleep(IDLE_BEFORE_E2E_S)

    # ---------------- device-resident throughput ----------------
    for k in range(max(Wm, 3)):
        one_step(k)
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    for k in range(K):
        one_step(k)
    if peer is not None:
        allr = peer.psnr_allgather(eng.x, eng.gt)
    else:
        rew = eng.psnr()
        if world > 1:
            allr = torch.empty(world * B, dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(allr, rew)
    e1.record()
    barrier()
    t1 = time.time()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop(t0, t1)
    dumped = None
    if args.dump_outputs and rank == 0:
        # copied now: the legs below step the same engine again.  The rewards are those of every rank, in rank order
        reward = rew if world == 1 else (allr[:, :B].reshape(-1) if peer is not None else allr)
        idx = dump_index(B, 20 * S * S, 4 * reward.numel()).to(dev)     # x fp32 + z, u complex64: 20 bytes per pixel
        dumped = {"x": eng.x.index_select(0, idx), "z": eng.z.index_select(0, idx), "u": eng.u.index_select(0, idx),
                  "reward": reward.clone()}
    tmax = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms = float(tmax.item())
    value = world * B * K / (ms * 1e-3)

    # ---------------- per-launch profile of the dominant kernel in the regime of the timed region (rank 0) ----------------
    def profile_convs(reps):
        """CUDA-event pair around every launch of the denoiser (pnp_unet_profile), `reps` passes interleaved with normal steps;
        returns (conv ms, all-launch ms, conv launches) per step."""
        import ctypes as C
        l = _lib.lib()
        CAP = 4096
        n = C.c_int(CAP)
        buf, kinds, ids = (C.c_float * CAP)(), (C.c_int * CAP)(), (C.c_int * CAP)()
        conv_ms = all_ms = 0.0
        n_conv = 0
        for _ in range(reps):
            for k in range(4):            # stay in the power / clock state of the preceding timed region
                one_step(k)
            n.value = CAP
            _lib.check(l.pnp_unet_profile(eng.plan.handle, eng.v.data_ptr(), eng.sigma.data_ptr(), eng.x.data_ptr(),
                                          _lib.stream_ptr(), buf, kinds, ids, C.byref(n)), "pnp_unet_profile")
            t = np.array(buf[:n.value]); kk = np.array(kinds[:n.value])
            conv_ms += float(t[kk == 1].sum()) / reps
            all_ms += float(t.sum()) / reps
            n_conv = int((kk == 1).sum())
        return conv_ms, all_ms, n_conv

    prof_burst = profile_convs(3) if rank == 0 else None     # right after the K-step region: burst clocks, like `value`

    # ---------------- untimed check of the fused reward gather against NCCL (N > 1) ----------------
    gather_check = None
    if world > 1:
        rew = eng.psnr().clone()
        ref_all = torch.empty(world * B, dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(ref_all, rew)
        if peer is not None:
            got = peer.psnr_allgather(eng.x, eng.gt)[:, :B].reshape(-1)
            d = float((got - ref_all).abs().max().item())
            gather_check = {"max_abs_diff_vs_nccl_all_gather": d, "ok": bool(d == 0.0), "ranks": world, "rewards": world * B,
                            "timed_out": bool(peer.timed_out()) if hasattr(peer, "timed_out") else None}
        else:
            gather_check = {"max_abs_diff_vs_nccl_all_gather": 0.0, "ok": True, "ranks": world, "rewards": world * B,
                            "note": "NCCL path in use"}

    # ---------------- a >= 1 s timed run next to the K-step one (sustained clocks / power) ----------------
    sustained = None
    n_sus = max(K, int(1.3 / max(ms / K * 1e-3, 1e-6)))
    barrier()
    e0s, e1s = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0s.record()
    for k in range(n_sus):
        one_step(k)
    e1s.record()
    barrier()
    ts = torch.tensor([e0s.elapsed_time(e1s)], device=dev)
    if world > 1:
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
    sustained = {"value": world * B * n_sus / (float(ts.item()) * 1e-3), "unit": UNIT, "steps": n_sus,
                 "seconds": float(ts.item()) * 1e-3, "ms_per_step": float(ts.item()) / n_sus}

    # ---------------- the same profile right after the >= 1 s run: sustained (power-capped) clocks ----------------
    roof = None
    if rank == 0:
        conv_ms_sus, all_ms_sus, n_conv = profile_convs(3)
        conv_ms, all_ms, _ = prof_burst
        flops = conv_flops_umma(S, S) * B
        ach = flops / (conv_ms * 1e-3) / 1e12               # burst regime (profiled right after the K-step timed region)
        ach_sus = flops / (conv_ms_sus * 1e-3) / 1e12       # sustained regime (profiled right after the >= 1 s run)
        peak = peaks["bf16_tflops"]             # burst peak: the denominator for kernels timed in the burst regime
        tr = ncu_step_traffic(B, S)
        roof = {"bound": "tensor", "kernel": f"conv3x3_umma_kernel / conv3x3_pair_kernel / conv3x3_kws_kernel ({n_conv} launches per step, summed)",
                "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                "frac_burst": ach / peaks["bf16_tflops"], "frac_sustained": ach_sus / peaks["bf16_tflops_sustained"],
                "achieved_sustained": ach_sus, "conv_ms_per_step_sustained": conv_ms_sus,
                "regimes": "frac = frac_burst: launches profiled right after the K-step timed region (burst clocks, as `value`) vs the "
                           "burst bf16 peak; frac_sustained: profiled right after the >= 1 s run (power-capped clocks, as "
                           "`sustained_1s`) vs the sustained bf16 peak",
                "peak_burst": peaks["bf16_tflops"], "peak_sustained": peaks["bf16_tflops_sustained"],
                "traffic": tr["conv_bytes_per_launch_mean"] if tr else None,
                "traffic_note": ("mean dram__bytes_read+write per conv launch over the " + str(tr["conv_launches"]) + " tensor-core conv "
                                 "launches of one step, parsed from " + tr["source"]) if tr else "no ncu capture committed for this shape",
                "traffic_per_step": tr,
                "algorithmic_conv_bytes_per_step": None,
                "peak_source": f"{peaks['source']} bf16_tflops (burst; sustained alongside)", "conv_ms_per_step": conv_ms,
                "conv_ms_note": "sum of per-launch CUDA-event pairs: an UPPER bound (event overhead, no PDL overlap between launches); "
                                "the whole step is ms_per_step",
                "unet_ms_per_step": all_ms, "conv_share_of_unet": conv_ms / all_ms,
                "launches_timed": n_conv}

    # ---------------- end-to-end with host buffers ----------------
    # Every step uploads ITS inputs (v, u, y0, mask, sigma, mu) from pinned host memory and downloads ITS results
    # (x, z, u).  Steps are independent in this protocol, so they are software-pipelined over two device buffer
    # sets and three streams (H2D | compute | D2H); nothing is skipped or cached.
    pin = lambda t: t.cpu().pin_memory()
    h_in = [pin(eng.v), pin(eng.u), pin(eng.y0), pin(eng.mask), pin(eng.sigma), pin(eng.mu)]
    h_out = [[pin(eng.x), pin(eng.z), pin(eng.u)] for _ in range(2)]
    h2d = sum(t.numel() * t.element_size() for t in h_in)
    d2h = sum(t.numel() * t.element_size() for t in h_out[0])
    engs = [eng, PnPEngine(den, B, S, S, dev)]          # second buffer set; the launch plan / workspace is shared
    s_h2d, s_cmp, s_d2h = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()

    def e2e_run(n):
        ev_in = [None, None]; ev_cmp = [None, None]; ev_out = [None, None]
        for k in range(n):
            e = engs[k % 2]
            with torch.cuda.stream(s_h2d):
                if ev_cmp[k % 2] is not None:
                    s_h2d.wait_event(ev_cmp[k % 2])        # inputs of step k-2 have been consumed
                for dst, src in zip((e.v, e.u, e.y0, e.mask, e.sigma, e.mu), h_in):
                    dst.copy_(src, non_blocking=True)
                ev_in[k % 2] = s_h2d.record_event()
            with torch.cuda.stream(s_cmp):
                s_cmp.wait_event(ev_in[k % 2])
                if ev_out[k % 2] is not None:
                    s_cmp.wait_event(ev_out[k % 2])        # results of step k-2 have left the device
                e.prepare()                                # y0 / mask are new every step in this protocol
                e.step()
                ev_cmp[k % 2] = s_cmp.record_event()
            with torch.cuda.stream(s_d2h):
                s_d2h.wait_event(ev_cmp[k % 2])
                for dst, src in zip(h_out[k % 2], (e.x, e.z, e.u)):
                    dst.copy_(src, non_blocking=True)
                ev_out[k % 2] = s_d2h.record_event()
        torch.cuda.current_stream().wait_stream(s_d2h)
        torch.cuda.current_stream().wait_stream(s_cmp)
        torch.cuda.current_stream().wait_stream(s_h2d)

    settle()
    e2e_run(4)
    barrier()
    e0.record()
    e2e_run(K)
    e1.record()
    barrier()
    tm = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    e2e_roundtrip_value = world * B * K / (float(tm.item()) * 1e-3)

    # ---------------- end-to-end through the public API as the reference's loops use it ----------------
    # reset(data) once per 30-step trajectory from pinned HOST arrays (x0, y0, mask, gt: the reference's dataset item,
    # evaluation/eval.py:75), then per step: H2D of that step's actions (sigma_d, mu) from pinned memory, step(), the
    # reward (PSNR per image, env.py:112-116) and its D2H read; after the last step the reconstruction x goes back to
    # the host.  The state lives on the device between steps, exactly as the reference's CUDA path keeps it
    # (env.py:57-71).  Two engines alternate so the next trajectory's upload overlaps the current one's compute.
    TRAJ = 30
    h_item = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in batch.items()}
    h_act = torch.stack([torch.tensor(sig, dtype=torch.float32).reshape(TRAJ, 1).expand(TRAJ, B),
                         torch.tensor(mus, dtype=torch.float32).reshape(TRAJ, 1).expand(TRAJ, B)], dim=1).contiguous().pin_memory()
    h_rew = [torch.empty(TRAJ, B, dtype=torch.float32).pin_memory() for _ in range(2)]
    h_x = [torch.empty(B, 1, S, S, dtype=torch.float32).pin_memory() for _ in range(2)]
    item_bytes = sum(v.numel() * v.element_size() for k, v in h_item.items() if k in ("x0", "y0", "mask", "gt"))
    h2d_traj = (item_bytes + TRAJ * 2 * B * 4) / TRAJ
    d2h_traj = (TRAJ * B * 4 + B * S * S * 4) / TRAJ

    def e2e_traj(n_steps):
        n_traj = (n_steps + TRAJ - 1) // TRAJ
        done = 0
        ev_up = [None, None]; ev_cmp = [None, None]
        def upload(j):
            e = engs[j % 2]
            with torch.cuda.stream(s_h2d):
                if ev_cmp[j % 2] is not None:
                    s_h2d.wait_event(ev_cmp[j % 2])        # the previous trajectory on this engine has finished
                e.reset(h_item, non_blocking=True)
                ev_up[j % 2] = s_h2d.record_event()
        upload(0)
        for j in range(n_traj):
            e = engs[j % 2]
            if j + 1 < n_traj:
                upload(j + 1)
            steps = min(TRAJ, n_steps - done)
            with torch.cuda.stream(s_cmp):
                s_cmp.wait_event(ev_up[j % 2])
                for k in range(steps):
                    e.actions.copy_(h_act[k], non_blocking=True)       # that step's (sigma_d, mu) for every image
                    e.step()
                    h_rew[j % 2][k].copy_(e.psnr(), non_blocking=True)
                h_x[j % 2].copy_(e.x, non_blocking=True)
                ev_cmp[j % 2] = s_cmp.record_event()
            done += steps
        torch.cuda.current_stream().wait_stream(s_cmp)
        torch.cuda.current_stream().wait_stream(s_h2d)

    settle()
    e2e_traj(max(Wm, 3))            # warm-up: the same W steps as the `value` leg (a whole 30-step trajectory here would
    barrier()                       # put the timed one behind 30 full-power steps, i.e. measure the power-capped rate)
    Ke = max(K, TRAJ)
    e0.record()
    e2e_traj(Ke)
    e1.record()
    barrier()
    tm = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    e2e_value = world * B * Ke / (float(tm.item()) * 1e-3)

    # ---------------- named variants of BASELINE.json configs (extra keys of the same JSON line) ----------------
    variants = {}
    if not args.no_variants:
        # config 2 as named: 30 iterations DRIVEN BY a random-init decision transformer (eval mode); T is held at 0
        # so that all 30 iterations execute (a random policy would stop trajectories at random)
        try:
            from dt4image_restoration_b200.policy import DecisionTransformer
            from dt4image_restoration_b200.rollout import BatchedRollout
            torch.manual_seed(0)
            pol_dt = DecisionTransformer()
            ro = BatchedRollout(pol_dt, eng, context_length=6, max_timesteps=30, force_full_length=True)
            data_t = h_item                                 # the item batch in pinned host memory (uploaded by reset)
            task = torch.full((B,), 4, dtype=torch.long)
            rtg0 = (10 + 1.08) / (16.6 + 1.08)          # rtg 10 normalised as reference dataset/datasets.py:204
            # warm-up: W iterations of the same loop (like the `value` leg; a whole 30-iteration rollout right before the
            # timed one would measure the power-capped rate), after the idle that every end-to-end leg starts from
            settle()
            BatchedRollout(pol_dt, eng, context_length=6, max_timesteps=max(Wm, 3), force_full_length=True).run(data_t, task, rtg0)
            barrier()
            t0 = time.perf_counter()
            out_dt = ro.run(data_t, task, rtg0)
            barrier()
            dt_s = torch.tensor([time.perf_counter() - t0], device=dev)
            if world > 1:
                dist.all_reduce(dt_s, op=dist.ReduceOp.MAX)
            variants["dt_driven_rollout"] = {
                "value": world * out_dt["image_iters"] / float(dt_s.item()), "unit": UNIT,
                "note": "reset + 30 iterations on a static context window; per iteration one fused policy kernel (action and "
                        "return heads, pnp_policy_step), the environment step and one fused observation kernel (area mean, "
                        "state encoder, window append, pnp_policy_observe); graph replay: " + str(bool(ro.use_graph)) +
                        ", wall clock",

                "mean_psnr_db": float(out_dt["psnr"].mean().item())}
        except Exception as ex:  # pragma: no cover
            variants["dt_driven_rollout"] = {"error": repr(ex)[:200]}
        # config 3: 512 candidate expansions of one shared state, sharded over the ranks, rewards all-gathered
        try:
            from dt4image_restoration_b200.rollout import CandidateExpander
            from dt4image_restoration_b200 import dist as pdist
            n_cand = 512
            lo, hi = pdist.shard_range(n_cand, rank, world)
            ceng = PnPEngine(den, hi - lo, S, S, dev)
            item = synth.make_item(synth.phantom(S, S, 11), synth.radial_mask(S, S, 0.2), 0.0, 11)
            from dt4image_restoration_b200.env import PnPEnv
            st0 = PnPEnv(30, den, dev).reset({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in item.items()}, dev)
            state = {k: st0[k] for k in ("z", "u", "y0", "mask", "gt")}
            gen = torch.Generator().manual_seed(5)
            sg_all, mu_all = CandidateExpander.sample_actions(0.1, 0.5, n_cand, gen)
            cx = CandidateExpander(ceng)
            for _ in range(2):
                cx.expand_and_gather(state, sg_all[lo:hi], mu_all[lo:hi], n_cand, peer)
            barrier()
            e0.record()
            reps = 5
            for _ in range(reps):
                r_all = cx.expand_and_gather(state, sg_all[lo:hi], mu_all[lo:hi], n_cand, peer)
            e1.record()
            barrier()
            tm3 = torch.tensor([e0.elapsed_time(e1) / reps], device=dev)
            if world > 1:
                dist.all_reduce(tm3, op=dist.ReduceOp.MAX)
            variants["mcts_512_candidates"] = {
                "value": n_cand / (float(tm3.item()) * 1e-3), "unit": "candidate expansions/s (= image-iters/s)",
                "ms_per_expansion_round": float(tm3.item()), "best_candidate": int(torch.argmax(r_all).item()),
                "note": "broadcast of the shared state + one step per candidate + PSNR + all-gather of 512 rewards (" + gather_kind + ")"}
            del ceng, cx
        except Exception as ex:  # pragma: no cover
            variants["mcts_512_candidates"] = {"error": repr(ex)[:200]}

        # config 1: ONE 256x256 image, radial 30 %, 30 iterations through the drop-in PnPEnv.reset/step (rank 0)
        if rank == 0:
            try:
                from collections import OrderedDict as OD
                from dt4image_restoration_b200.env import PnPEnv
                env1 = PnPEnv(30, den, dev)
                it1 = synth.make_item(synth.phantom(S, S, 0), synth.radial_mask(S, S, 0.3), 0.0, 0)
                d1 = {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in it1.items()}

                def traj1():
                    st = env1.reset(dict(d1), dev)
                    for k in range(30):
                        st, _ = env1.step(st, OD(T=0.0, sigma_d=torch.tensor([float(sig[k])]), mu=torch.tensor(float(mus[k]))))
                    return env1.compute_reward(st["x"].reshape(1, S, S), st["gt"].reshape(1, S, S))
                traj1()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(3):
                    r1 = traj1()
                torch.cuda.synchronize()
                t1 = (time.perf_counter() - t0) / 3
                variants["config1_dropin_b1_radial30"] = {
                    "ms_per_iteration": t1 / 30 * 1e3, "value": 30 / t1, "unit": UNIT, "psnr_db": float(r1),
                    "note": "reset (host arrays) + 30 x PnPEnv.step (CUDA-graph replay of the step body + one copy-out that keeps "
                            "the fresh-tensor contract) + compute_reward, wall clock"}
            except Exception as ex:  # pragma: no cover
                variants["config1_dropin_b1_radial30"] = {"error": repr(ex)[:200]}
        # the whole tree search of the reference (30 iterations: selection, batched expansion, greedy rollouts) at its
        # native 128x128, candidates of an expansion sharded over the ranks
        try:
            from dt4image_restoration_b200.mcts import BatchedMCTS
            from dt4image_restoration_b200.policy import DecisionTransformer as DTp
            torch.manual_seed(1234)
            pol = DTp(block_size=18, n_embeds=9, mode="norm")
            with torch.no_grad():
                pol.predict_action[0].bias[0] = -2.0       # stop head biased to "continue" (as tests/test_drivers.py)
            width = 5 if world == 1 else 8 * world - 1
            ms_search = BatchedMCTS(pol, den, 128, 128, width=width, n_iters=30, device=dev, rank=rank, world=world, peer=None)
            itm = synth.make_item(synth.phantom(128, 128, 2), synth.radial_mask(128, 128, 0.3), 0.0, 2)
            dm = {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in itm.items()}
            torch.manual_seed(99)
            ms_search.search(dm, rtg0 if "rtg0" in dir() else (10 + 1.08) / (16.6 + 1.08), torch.tensor([[3]]))
            barrier()
            ms_search.env_steps = 0
            torch.manual_seed(99)
            t0 = time.perf_counter()
            fin, best, progs = ms_search.search(dm, (10 + 1.08) / (16.6 + 1.08), torch.tensor([[3]]))
            barrier()
            tsr = torch.tensor([time.perf_counter() - t0], device=dev)
            if world > 1:
                dist.all_reduce(tsr, op=dist.ReduceOp.MAX)
            variants["mcts_full_search"] = {
                "seconds_per_search": float(tsr.item()), "iterations": 30, "width": width, "programs": len(progs),
                "env_steps_this_rank": int(ms_search.env_steps), "best_program": best, "final_psnr_db": float(fin),
                "note": "reference run_mcts semantics with independent children (mcts.BatchedMCTS) at 128x128: p-UCB selection, "
                        "one batched expansion step per iteration, greedy policy rollout to the horizon, max backprop; "
                        "the reference's CPU loop takes 13.8 s for the same search (SURVEY 6)"}
        except Exception as ex:  # pragma: no cover
            variants["mcts_full_search"] = {"error": repr(ex)[:300]}

        # config 4: batch 128 of 512x512, 8x Cartesian undersampling, complex Gaussian k-space noise sigma 10 (per GPU; the
        # denoiser runs in micro-batches on the capped workspace), and the any-size path at 130x130 (dense-DFT prox)
        for vname, (vB, vS, vkind, vpar, vsn) in (("config4_b128_512_cartesian8", (128, 512, "cartesian", 8, 10.0)),
                                                  ("nonpow2_b64_130_radial30", (64, 130, "radial", 0.3, 0.0))):
            try:
                veng = PnPEngine(den, vB, vS, vS, dev)
                vb = synth.make_batch(8, vS, vS, vkind, vpar, vsn, seed0=40 + rank)
                vb = {k: torch.from_numpy(np.ascontiguousarray(np.concatenate([v] * (vB // 8), 0))) for k, v in vb.items()}
                veng.reset(vb)
                del vb
                for k in range(3):
                    veng.set_actions(float(sig[k]), float(mus[k]))
                    veng.step()
                barrier()
                e0.record()
                nv = 6
                for k in range(nv):
                    veng.set_actions(float(sig[3 + k]), float(mus[3 + k]))
                    veng.step()
                e1.record()
                barrier()
                tv = torch.tensor([e0.elapsed_time(e1) / nv], device=dev)
                if world > 1:
                    dist.all_reduce(tv, op=dist.ReduceOp.MAX)
                variants[vname] = {"value": world * vB / (float(tv.item()) * 1e-3), "unit": "image-iters/s",
                                   "ms_per_step": float(tv.item()), "batch_per_gpu": vB, "size": vS,
                                   "tflops_per_gpu": (GFLOP_PER_IMAGE[vS] * vB / float(tv.item())) if vS in GFLOP_PER_IMAGE else None,
                                   "psnr_db_mean": float(veng.psnr().mean().item()),
                                   "note": f"{vkind} mask ({vpar}), k-space noise sigma {vsn}; 3 warm-up + {nv} timed engine steps, "
                                           "CUDA events, state resident"}
                del veng
                torch.cuda.empty_cache()
            except Exception as ex:  # pragma: no cover
                variants[vname] = {"error": repr(ex)[:300]}

    # ---------------- HBM-bound kernels of the path, timed alone on this batch (rank 0) ----------------
    others = {}
    if rank == 0:
        l = _lib.lib()
        hw = S * S

        def time_fn(fn, n=20):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n * 1e-3

        if eng.prepared:
            prox = lambda: _lib.check(l.pnp_prox_dual_prepared_kind(
                eng.x.data_ptr(), eng.u.data_ptr(), eng.y0T.data_ptr(), eng.maskT.data_ptr(), hw, eng.mu.data_ptr(), 1,
                eng.z.data_ptr(), eng.u.data_ptr(), eng.v.data_ptr(), B, S, S, eng.probe.get(), _lib.stream_ptr()))
        else:
            prox = lambda: _lib.check(l.pnp_prox_dual(
                eng.x.data_ptr(), eng.u.data_ptr(), eng.y0.data_ptr(), eng.mask.data_ptr(), hw, eng.mu.data_ptr(), 1,
                eng.z.data_ptr(), eng.u.data_ptr(), eng.v.data_ptr(), eng.work.data_ptr(), B, S, S, _lib.stream_ptr()))
        t = time_fn(prox)
        gbs = 37.0 * B * hw / t / 1e9
        others["fftprox_dual"] = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                  "frac": gbs / peaks["hbm_gbs"], "us_per_launch": t * 1e6,
                                  "algorithmic_bytes_per_pixel": 37, "images_per_launch": B,
                                  "also_written": "v_next = Re(z - u') fp32 (4 B/pixel, not counted): replaces the next step's residual kernel",
                                  "traffic": (ncu_step_traffic(B, S) or {}).get("fftprox_rows256"),
                                  "kernel": (("fftprox_rows256_kernel" if S == 256 else f"fftprox_rows_generic_kernel<{S}>")
                                             + " (column-only Cartesian mask of this workload: row transforms only)")
                                  if eng.prepared else "general three-launch path"}
        if eng.prepared and S == 256:
            # the same step with a radial 30 % mask (BASELINE configs 1/3): general single-launch cluster kernel
            from dt4image_restoration_b200 import ops
            rm = torch.from_numpy(synth.radial_mask(S, S, 0.3)).to(dev).reshape(1, 1, S, S)
            prep_r = ops.ProxPrepared(eng.y0, rm)
            zr, ur, vr = torch.empty_like(eng.z), torch.empty_like(eng.u), torch.empty_like(eng.v)
            t = time_fn(lambda: prep_r.prox_dual(eng.x, eng.u, eng.mu, out=(zr, ur, vr)))
            gbs = 37.0 * B * hw / t / 1e9
            others["fftprox_dual_radial_mask"] = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                                  "frac": gbs / peaks["hbm_gbs"], "us_per_launch": t * 1e6,
                                                  "algorithmic_bytes_per_pixel": 37, "images_per_launch": B,
                                                  "kernel": "fftprox_cl_kernel<16> (16-CTA cluster, bulk-async loads, st.async "
                                                            "DSMEM exchanges, 2-D transforms)",
                                                  "traffic": (ncu_step_traffic(B, S) or {}).get("fftprox_cl")}
            del prep_r, zr, ur, vr
        if eng.prepared:
            # the reference's native 128x128 with a radial mask: 4-CTA cluster kernel (fftprox_cl128.cuh), B = 1024 images
            from dt4image_restoration_b200 import ops
            Bn, Sn = 1024, 128
            gn = torch.Generator(device=dev).manual_seed(0)
            xn = torch.rand(Bn, 1, Sn, Sn, device=dev, generator=gn)
            un = torch.complex(torch.randn(Bn, 1, Sn, Sn, device=dev, generator=gn), torch.randn(Bn, 1, Sn, Sn, device=dev, generator=gn)) * 0.1
            yn = torch.complex(torch.randn(Bn, 1, Sn, Sn, device=dev, generator=gn), torch.randn(Bn, 1, Sn, Sn, device=dev, generator=gn))
            rmn = torch.from_numpy(synth.radial_mask(Sn, Sn, 0.3)).to(dev).reshape(1, 1, Sn, Sn)
            prep_n = ops.ProxPrepared(yn, rmn)
            mun = torch.full((Bn,), 0.5, device=dev)
            outn = (torch.empty_like(un), torch.empty_like(un), torch.empty_like(xn))
            t = time_fn(lambda: prep_n.prox_dual(xn, un, mun, out=outn))
            gbs = 37.0 * Bn * Sn * Sn / t / 1e9
            others["fftprox_dual_radial_mask_128"] = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                                      "frac": gbs / peaks["hbm_gbs"], "us_per_launch": t * 1e6,
                                                      "algorithmic_bytes_per_pixel": 37, "images_per_launch": Bn,
                                                      "kernel": "fftprox_cl128_kernel (4-CTA cluster)"}
            del prep_n, xn, un, yn, outn
        t = time_fn(lambda: eng.psnr())
        gbs = 8.0 * B * hw / t / 1e9
        others["psnr"] = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                          "frac": gbs / peaks["hbm_gbs"], "us_per_launch": t * 1e6, "algorithmic_bytes_per_pixel": 8,
                          "images_per_launch": B, "note": "latency-bound at this batch (one CTA per image)"}

    # ---------------- CPU baseline (rank 0, N=1 only) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads = os.cpu_count() or 1
        sB = 8 if S <= 256 else 2
        v, t, _ = cpu_leg(S, threads, sB, 3, 1)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"3 steps of {sB} images at {S}x{S} after 1 warm-up (oracle = PyTorch CPU restatement of the "
                         f"reference step), {threads} threads"}
        if S <= 256:            # SURVEY 8d: the one-thread figure next to the all-cores one (2 images, 1 step after 1 warm-up)
            v1, _, _ = cpu_leg(S, 1, 2, 1, 1)
            cpu["value_1_thread"] = v1

    if rank == 0:
        if isinstance(variants.get("dt_driven_rollout"), dict) and "value" in variants["dt_driven_rollout"]:
            variants["dt_driven_rollout"]["fraction_of_value"] = variants["dt_driven_rollout"]["value"] / value
            if sustained:      # a 30-iteration rollout (~0.1 s) runs into the power cap like the >= 1 s leg does
                variants["dt_driven_rollout"]["fraction_of_sustained_1s"] = variants["dt_driven_rollout"]["value"] / sustained["value"]
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(Wm, 3),
               "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
               "data": "synthetic",
               "config": config_dict(B, S, world),
               "run_info": {"parallelism": f"dp{world} (independent trajectories, reward all-gather only)",
                            "reward_gather": gather_kind, "gather_check": gather_check,
                            "idle_before_e2e_s": IDLE_BEFORE_E2E_S, "numa": numa},
               "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_traj, "d2h_bytes_per_step": d2h_traj,
                       "steps": Ke,
                       "protocol": "public API as the reference's loops use it: reset(item) from pinned host arrays once per "
                                   "30-step trajectory, per step H2D of the actions, step(), reward, D2H of the rewards; "
                                   "final x to the host; bytes are per-step averages"},
               "e2e_state_roundtrip": {"value": e2e_roundtrip_value, "unit": UNIT, "h2d_bytes_per_step": h2d,
                                       "d2h_bytes_per_step": d2h,
                                       "protocol": "stricter variant: EVERY step uploads the whole state (v, u, y0, mask, "
                                                   "sigma, mu) and downloads x, z, u; host-bandwidth bound at 8 GPUs"},
               "gpu_launches": K * eng.launches_per_step + 1,
               "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "other_kernels": others, "variants": variants,
               "sustained_1s": sustained,
               "dt_driven": variants.get("dt_driven_rollout"),   # BASELINE config 2 as named (policy in the loop)
               "tflops_whole_step": world * B * K * GFLOP_PER_IMAGE.get(S, 0) / (ms * 1e-3) / 1e3}
        print(json.dumps(out), flush=True)
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--accel", type=int, default=4, help="Cartesian acceleration factor of the synthetic masks")
    ap.add_argument("--noise", type=float, default=0.0, help="complex Gaussian k-space noise sigma (x/255)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs:
        try:            # refused before the run rather than after its timed steps
            dump_index(args.batch, 20 * args.size ** 2, 4 * args.gpus * args.batch)
        except ValueError as ex:
            ap.error(str(ex))
    global ACCEL, NOISE
    ACCEL, NOISE = args.accel, args.noise
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
