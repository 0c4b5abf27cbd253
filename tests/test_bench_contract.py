"""bench.py's reference arm (the CPU leg, `--impl reference`): one JSON line with the contract's keys on rank 0, nothing on the
other ranks.  Runs the oracle on a 64 x 64 sample, so it needs no GPU.  --dump-outputs of both arms against the oracle (the
`ours` arm's test needs the GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env, *extra_args):
    env = dict(os.environ, **extra_env)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--size", "64", "--steps", "1",
                           "--warmup", "1", "--gpus", extra_env.get("WORLD_SIZE", "1"), *extra_args],
                          capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)


def test_reference_arm_prints_one_contract_line_on_rank_0():
    r = _run({})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "pnp_admm_image_iters_per_sec_256" and d["unit"] == "image-iters/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1 and d["dtype"] == "f32"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert "sample" in d["cpu_baseline"] and d["config"]["workload"].startswith("batch 64 per GPU of 64x64")
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_is_silent_on_other_ranks():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def _oracle_after(schedule_steps, B=8, S=64):
    """The oracle stepped as bench.py steps: the seeded batch of make_inputs, the default-init weights of seed 0, and the
    fixed (sigma, mu) schedule at the given indices."""
    import torch
    import bench
    from dt4image_restoration_b200 import synth
    from oracle import pnp_oracle as O
    params = O.init_unet_params(0, "default")
    st = O.reset(bench.make_inputs(B, S))
    sig, mus = synth.fixed_schedule(30)
    for k in schedule_steps:
        st, _ = O.step(params, st, {"T": torch.zeros(1), "mu": torch.tensor([mus[k]]), "sigma_d": torch.full((B,), float(sig[k]))})
    return st


def _check_state(out_dir, st, atol):
    import numpy as np
    import torch
    for name in ("x", "z", "u"):
        got, ref = np.load(out_dir / f"{name}.npy"), st[name]
        ref = (torch.view_as_real(ref) if ref.is_complex() else ref).numpy()
        assert got.dtype == np.float32 and got.shape == ref.shape, name
        np.testing.assert_allclose(got, ref, rtol=0, atol=atol, err_msg=name)


def test_reference_arm_dumps_the_state_of_its_last_step(tmp_path):
    """--dump-outputs: x, z, u after the last timed step, equal to the oracle stepped on the same seeded inputs."""
    r = _run({}, "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["u.npy", "x.npy", "z.npy"]
    _check_state(tmp_path, _oracle_after([0, 1]), 1e-5)          # --warmup 1, then --steps 1


def test_dump_outputs_refuses_a_size_whose_single_image_exceeds_the_limit(tmp_path):
    """One 2048 x 2048 image's x, z, u (80 MiB) cannot be sampled under the 64 MB limit: refused up front, nothing written."""
    r = _run({}, "--size", "2048", "--dump-outputs", str(tmp_path / "out"))
    assert r.returncode == 2 and "do not fit" in r.stderr and r.stdout == ""
    assert not os.path.exists(tmp_path / "out")


@pytest.mark.gpu
def test_gpu_arm_dumps_the_state_and_rewards_of_its_last_step(tmp_path):
    """The timed path (`ours`): after 3 warm-up steps and --steps 1, x, z, u and the rewards of the batch match the oracle
    stepped on the same seeded inputs with the same schedule, within the engine's bf16 tolerances (1e-3, 0.05 dB)."""
    import numpy as np
    from oracle import pnp_oracle as O
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--size", "64", "--batch", "8", "--steps", "1",
                        "--warmup", "3", "--no-cpu", "--no-variants", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["reward.npy", "u.npy", "x.npy", "z.npy"]
    st = _oracle_after([0, 1, 2, 0])             # the warm-up steps, then the timed loop starts the schedule again
    _check_state(tmp_path, st, 1e-3)
    reward = np.load(tmp_path / "reward.npy")
    ref = O.psnr(st["x"].reshape(8, 64, 64), st["gt"].reshape(8, 64, 64)).reshape(-1).numpy()
    assert reward.dtype == np.float32 and reward.shape == (8,)
    np.testing.assert_allclose(reward, ref, rtol=0, atol=0.05)
